// frontend.cu -- K4: range/intensity image projection, LOAM feature extraction and PCL-style VoxelGrid.
//
// Replaces ImageHandler::cloud_handler (image_handler.h_ouster:103-140), laserCloudHandler's numeric body
// (scanRegistration.cpp:152-186, 244-412, 427-589) and pcl::VoxelGrid::filter (scanRegistration.cpp:580-589,
// laserMapping.cpp:608-616, mapOptimization.cpp:368-370).
//
// Everything here is streaming / small-sort work bound by HBM bandwidth and launch latency; no tensor cores.
// Float arithmetic that feeds integer decisions (ring id, curvature order, labels, voxel index) uses explicit
// round-to-nearest intrinsics in the reference's evaluation order (x86-64 SSE2, no FMA).
#include <string.h>

#include "ilsm_host.hpp"
#include "ilsm_voxel.cuh"

namespace ilsm {

// ---------------------------------------------------------------------------------------------------
// projection: 4 consecutive pixels per thread, float4 loads, uchar4 / float4 stores
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void project_one(float x, float y, float z, float inten, unsigned char& r8, unsigned char& i8,
                                            float4& track) {
  const float range = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
  const float ic = (255.0f < inten) ? 255.0f : inten;  // std::min(intensity, 255.0f)
  const float r20m = __fmul_rn(range, 20.f);
  const float r20 = (255.0f < r20m) ? 255.0f : r20m;  // std::min(range * 20, 255.0f)
  r8 = (unsigned char)(__float2int_rz(r20) & 0xFF);
  i8 = (unsigned char)(__float2int_rz(ic) & 0xFF);
  if ((double)range >= 0.1)
    track = make_float4(x, y, z, ic);
  else
    track = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void project_kernel(const float* __restrict__ cloud, int n, int stride_f, int ioff,
                               unsigned char* __restrict__ img_range, unsigned char* __restrict__ img_inten,
                               float4* __restrict__ track) {
  pdl_entry();
  const int i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i0 >= n) return;
  unsigned char r8[4] = {0, 0, 0, 0}, i8[4] = {0, 0, 0, 0};
  float4 tr[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = i0 + k;
    if (i < n) {
      const float* p = cloud + (size_t)i * stride_f;
      float x, y, z, it;
      if ((stride_f & 3) == 0) {  // 16- or 32-byte points: one 128-bit load for xyz(+w)
        const float4 v = __ldg(reinterpret_cast<const float4*>(p));
        x = v.x, y = v.y, z = v.z;
        it = ioff == 3 ? v.w : __ldg(p + ioff);
      } else {
        x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2), it = __ldg(p + ioff);
      }
      project_one(x, y, z, it, r8[k], i8[k], tr[k]);
    }
  }
  if (i0 + 3 < n) {
    *reinterpret_cast<uchar4*>(img_range + i0) = make_uchar4(r8[0], r8[1], r8[2], r8[3]);
    *reinterpret_cast<uchar4*>(img_inten + i0) = make_uchar4(i8[0], i8[1], i8[2], i8[3]);
#pragma unroll
    for (int k = 0; k < 4; ++k) track[i0 + k] = tr[k];
  } else {
    for (int k = 0; k < 4 && i0 + k < n; ++k) {
      img_range[i0 + k] = r8[k];
      img_inten[i0 + k] = i8[k];
      track[i0 + k] = tr[k];
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// sensor_msgs/PointCloud2 blob -> packed xyzi (pcl::fromROSMsg's field map, scanRegistration.cpp:235).  One thread per
// point; the blob is read with the widest aligned loads its layout allows (Ouster: point_step 48, x/y/z at 0/4/8 ->
// one 128-bit load + one 32-bit load per point), the output is one float4 store.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float pc2_f32(const unsigned char* p) {  // unaligned-safe little-endian float
  uint32_t v;
  if ((reinterpret_cast<uintptr_t>(p) & 3) == 0)
    v = __ldg(reinterpret_cast<const uint32_t*>(p));
  else
    v = (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16) | ((uint32_t)__ldg(p + 3) << 24);
  return __uint_as_float(v);
}

__global__ void pc2_unpack_kernel(const unsigned char* __restrict__ data, int n, ilsm_pc2_layout l, float4* __restrict__ out) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char* p = data + (size_t)i * l.point_step;
  float x, y, z;
  if (l.off_y == l.off_x + 4 && l.off_z == l.off_x + 8 && ((reinterpret_cast<uintptr_t>(p) + l.off_x) & 15) == 0) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p + l.off_x));
    x = v.x, y = v.y, z = v.z;
  } else {
    x = pc2_f32(p + l.off_x), y = pc2_f32(p + l.off_y), z = pc2_f32(p + l.off_z);
  }
  float it = 0.f;
  if (l.off_intensity >= 0) {
    const unsigned char* q = p + l.off_intensity;
    switch (l.intensity_datatype) {
      case 7: it = pc2_f32(q); break;
      case 2: it = (float)__ldg(q); break;
      case 4: it = (float)((uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8)); break;
      case 6: it = (float)__float_as_uint(pc2_f32(q)); break;
      case 8: {
        const unsigned long long lo = __float_as_uint(pc2_f32(q)), hi = __float_as_uint(pc2_f32(q + 4));
        it = (float)__longlong_as_double((long long)(lo | (hi << 32)));
        break;
      }
      default: break;
    }
  }
  out[i] = make_float4(x, y, z, it);
}

int Ctx::pc2_unpack_dev(const unsigned char* d_data, int n, const ilsm_pc2_layout& l, float4* d_out) {
  if (n <= 0) return ILSM_OK;
  ILSM_CUDA(launch_pdl(pc2_unpack_kernel, dim3((n + 255) / 256), dim3(256), 0, stream, d_data, n, l, d_out));
  count_launches(1);
  return check_launch("pc2_unpack");
}

// The other direction (pcl::toROSMsg of the clouds the nodes publish): packed xyzi -> point_step-byte records with x / y / z
// / intensity as FLOAT32 at the layout's offsets, every other byte zero (PCL leaves its padding floats as they are in memory;
// subscribers read fields by offset).  One thread per 4 bytes of output: coalesced stores whatever the point step.
__global__ void pc2_pack_kernel(const float4* __restrict__ in, int n, ilsm_pc2_layout l, uint32_t* __restrict__ out) {
  pdl_entry();
  const int wpp = l.point_step >> 2;  // 32-bit words per point (point_step is a multiple of 4)
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= (long long)n * wpp) return;
  const int i = (int)(w / wpp), off = (int)(w - (long long)i * wpp) << 2;
  uint32_t v = 0u;
  if (off == l.off_x || off == l.off_y || off == l.off_z || (l.off_intensity >= 0 && off == l.off_intensity)) {
    const float4 p = __ldg(in + i);
    v = __float_as_uint(off == l.off_x ? p.x : off == l.off_y ? p.y : off == l.off_z ? p.z : p.w);
  }
  out[w] = v;
}

int Ctx::pc2_pack_dev(const float4* d_in, int n, const ilsm_pc2_layout& l, unsigned char* d_out) {
  if (n <= 0) return ILSM_OK;
  const long long words = (long long)n * (l.point_step >> 2);
  ILSM_CUDA(launch_pdl(pc2_pack_kernel, dim3((unsigned)((words + 255) / 256)), dim3(256), 0, stream, d_in, n, l, reinterpret_cast<uint32_t*>(d_out)));
  count_launches(1);
  return check_launch("pc2_pack");
}

// ---------------------------------------------------------------------------------------------------
// feature extraction
// ---------------------------------------------------------------------------------------------------
constexpr int kRings = 64;
constexpr int kMaxSeg = 2048;      // points per (ring, segment) handled by the in-block sort
constexpr int kMaxRingLF = 4096;   // less-flat points of one ring handled by the in-block VoxelGrid

// FeStats layout (ints): [0] first kept index (min), [1] last kept index (max), [2] first index whose unwrapped
// azimuth passes startOri + pi (the halfPassed latch), [3] error flags, [4..67] ring counts, [68..131] per-ring
// sharp / [132..195] less-sharp / [196..259] flat / [260..323] less-flat output counts
constexpr int kStFirst = 0, kStLast = 1, kStStar = 2, kStErr = 3, kStRing = 4, kStSharp = 68, kStLSharp = 132,
              kStFlat = 196, kStLFlat = 260, kStInts = 324;

__global__ void fe_init_kernel(int* st) {
  pdl_entry();
  const int i = threadIdx.x;
  if (i < kStInts) st[i] = (i == kStFirst || i == kStStar) ? INT_MAX : (i == kStLast ? -1 : 0);
}

// pass 1: min-range filter, ring id, raw azimuth; ring histogram, first/last kept point
__global__ void fe_tag_kernel(const float* __restrict__ in, int n, int stride_f, float thr2,
                              unsigned char* __restrict__ scanid, float* __restrict__ ori_raw, int* st,
                              int* __restrict__ chunk_hist) {
  pdl_entry();
  __shared__ int hist[kRings];
  if (threadIdx.x < kRings) hist[threadIdx.x] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int first = INT_MAX, last = -1;
  if (i < n) {
    const float* p = in + (size_t)i * stride_f;
    const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
    unsigned char sid = 254;  // removed by the range filter
    if (!(d2 < thr2)) {
      first = last = i;
      const float ratio = __fdiv_rn(z, __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y))));
      const float at = (float)atan((double)ratio);  // atan evaluated in double, rounded to float
      const float angle = (float)((double)__fmul_rn(at, 180.f) / 3.14159265358979323846);
      const int s = __double2int_rz(((double)angle + 22.5) * 1.41 + 0.5) - 1;
      sid = (s >= 0 && s < kRings) ? (unsigned char)s : 255;
      if (sid < kRings) atomicAdd(&hist[sid], 1);
      ori_raw[i] = -atan2f(y, x);
    }
    scanid[i] = sid;
  }
  first = (int)__reduce_min_sync(0xffffffffu, (unsigned)first);
  last = __reduce_max_sync(0xffffffffu, last);
  if ((threadIdx.x & 31) == 0) {
    if (first != INT_MAX) atomicMin(&st[kStFirst], first);
    if (last >= 0) atomicMax(&st[kStLast], last);
  }
  __syncthreads();
  if (threadIdx.x < kRings) {
    chunk_hist[blockIdx.x * kRings + threadIdx.x] = hist[threadIdx.x];  // ring counts of this 256-point chunk
    if (hist[threadIdx.x]) atomicAdd(&st[kStRing + threadIdx.x], hist[threadIdx.x]);
  }
}

struct OriRef {
  float startOri, endOri;
};
// scanRegistration.cpp:247-262
__device__ __forceinline__ OriRef ori_reference(const float* __restrict__ in, int stride_f, const int* st) {
  OriRef r;
  const float* p0 = in + (size_t)st[kStFirst] * stride_f;
  const float* pN = in + (size_t)st[kStLast] * stride_f;
  r.startOri = -atan2f(__ldg(p0 + 1), __ldg(p0));
  float endOri = (float)((double)(-atan2f(__ldg(pN + 1), __ldg(pN))) + 2 * 3.14159265358979323846);
  const double PI = 3.14159265358979323846;
  if ((double)__fsub_rn(endOri, r.startOri) > 3 * PI)
    endOri = (float)((double)endOri - 2 * PI);
  else if ((double)__fsub_rn(endOri, r.startOri) < PI)
    endOri = (float)((double)endOri + 2 * PI);
  r.endOri = endOri;
  return r;
}

// first-half unwrapping (scanRegistration.cpp:336-349)
__device__ __forceinline__ float ori_first_half(float ori, float startOri) {
  const double PI = 3.14159265358979323846;
  if ((double)ori < (double)startOri - PI / 2)
    ori = (float)((double)ori + 2 * PI);
  else if ((double)ori > (double)startOri + PI * 3 / 2)
    ori = (float)((double)ori - 2 * PI);
  return ori;
}

// pass 2: the halfPassed latch = first valid point (input order) whose first-half azimuth exceeds startOri + pi
__global__ void fe_star_kernel(const float* __restrict__ in, int n, int stride_f, const unsigned char* __restrict__ scanid,
                               const float* __restrict__ ori_raw, int* st) {
  pdl_entry();
  if (st[kStLast] < 0) return;
  const OriRef ref = ori_reference(in, stride_f, st);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int cand = INT_MAX;
  if (i < n && scanid[i] < kRings) {
    const float o1 = ori_first_half(ori_raw[i], ref.startOri);
    if ((double)__fsub_rn(o1, ref.startOri) > 3.14159265358979323846) cand = i;
  }
  cand = (int)__reduce_min_sync(0xffffffffu, (unsigned)cand);
  if ((threadIdx.x & 31) == 0 && cand != INT_MAX) atomicMin(&st[kStStar], cand);
}

// pass 3a: per ring, exclusive prefix of the chunk histograms (one block per ring, chunks scanned 256 at a time)
constexpr int kFeChunk = 256;
__global__ void __launch_bounds__(256) fe_scan_kernel(const int* __restrict__ chunk_hist, int chunks, int* __restrict__ chunk_base) {
  pdl_entry();
  __shared__ int wsum[8];
  __shared__ int carry_s;
  const int ring = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int c0 = 0; c0 < chunks; c0 += 256) {
    const int c = c0 + threadIdx.x;
    const int v = c < chunks ? chunk_hist[c * kRings + ring] : 0;
    int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, inc, off);
      if (lane >= off) inc += o;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < warp) wbase += wsum[w];
      tot += wsum[w];
    }
    const int carry = carry_s;
    if (c < chunks) chunk_base[c * kRings + ring] = carry + wbase + inc - v;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + tot;
    __syncthreads();
  }
}

// pass 3b: stable scatter of every kept point into the ring-concatenated cloud: position = ring offset + points of
// the same ring in earlier chunks + in earlier warps of this chunk + in earlier lanes of this warp (match_any);
// intensity = scanID + 0.1 * relTime (scanRegistration.cpp:334-373)
__global__ void __launch_bounds__(kFeChunk) fe_bucket_kernel(const float* __restrict__ in, int n, int stride_f,
                                                             const unsigned char* __restrict__ scanid,
                                                             const float* __restrict__ ori_raw, const int* __restrict__ st,
                                                             const int* __restrict__ chunk_base, float4* __restrict__ cloud,
                                                             int* __restrict__ src_index) {
  pdl_entry();
  __shared__ int ring_off[kRings];
  __shared__ int wcnt[kFeChunk / 32][kRings];
  if (st[kStLast] < 0) return;
  if (threadIdx.x < kRings) {
    int off = 0;
    for (int r = 0; r < (int)threadIdx.x; ++r) off += st[kStRing + r];
    ring_off[threadIdx.x] = off;
  }
  for (int t = threadIdx.x; t < (kFeChunk / 32) * kRings; t += blockDim.x) (&wcnt[0][0])[t] = 0;
  __syncthreads();
  const OriRef ref = ori_reference(in, stride_f, st);
  const int star = st[kStStar];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * kFeChunk + threadIdx.x;
  const int ring = i < n ? (int)scanid[i] : 255;
  const bool mine = ring < kRings;
  const unsigned peers = __match_any_sync(0xffffffffu, mine ? ring : 255);
  const int rank = __popc(peers & ((1u << lane) - 1u));
  if (mine && rank == 0) wcnt[warp][ring] = __popc(peers);
  __syncthreads();
  if (mine) {
    int wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += wcnt[w][ring];
    const int pos = ring_off[ring] + chunk_base[blockIdx.x * kRings + ring] + wbase + rank;
    const float* p = in + (size_t)i * stride_f;
    float ori = ori_raw[i];
    const double PI = 3.14159265358979323846;
    if (i <= star) {
      ori = ori_first_half(ori, ref.startOri);
    } else {
      ori = (float)((double)ori + 2 * PI);
      if ((double)ori < (double)ref.endOri - PI * 3 / 2)
        ori = (float)((double)ori + 2 * PI);
      else if ((double)ori > (double)ref.endOri + PI / 2)
        ori = (float)((double)ori - 2 * PI);
    }
    const float relTime = __fdiv_rn(__fsub_rn(ori, ref.startOri), __fsub_rn(ref.endOri, ref.startOri));
    const float tag = (float)((double)ring + 0.1 * (double)relTime);
    cloud[pos] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), tag);
    src_index[pos] = i;
  }
}

// pass 4: curvature over the concatenated cloud (scanRegistration.cpp:397-412), exact left-to-right float sums
__global__ void fe_curvature_kernel(const float4* __restrict__ cloud, const int* __restrict__ st, float* __restrict__ curv,
                                    int* __restrict__ label, unsigned char* __restrict__ picked) {
  pdl_entry();
  int N = 0;
  for (int r = 0; r < kRings; ++r) N += st[kStRing + r];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float c = 0.f;
  if (i >= 5 && i < N - 5) {
    float4 p[11];
#pragma unroll
    for (int k = 0; k < 11; ++k) p[k] = __ldg(cloud + i - 5 + k);
    float d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#define C_(k) (a == 0 ? p[k].x : (a == 1 ? p[k].y : p[k].z))
      float s = __fadd_rn(C_(0), C_(1));
      s = __fadd_rn(s, C_(2));
      s = __fadd_rn(s, C_(3));
      s = __fadd_rn(s, C_(4));
      s = __fsub_rn(s, __fmul_rn(10.f, C_(5)));
      s = __fadd_rn(s, C_(6));
      s = __fadd_rn(s, C_(7));
      s = __fadd_rn(s, C_(8));
      s = __fadd_rn(s, C_(9));
      s = __fadd_rn(s, C_(10));
#undef C_
      d[a] = s;
    }
    c = __fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2]));
  }
  curv[i] = c;
  label[i] = 0;
  picked[i] = 0;
}

__device__ __forceinline__ void ring_bounds(const int* st, int ring, int& S, int& E) {
  int off = 0;
  for (int r = 0; r < ring; ++r) off += st[kStRing + r];
  S = off + 5;
  E = off + st[kStRing + ring] - 6;
}

// pass 5: one block per (ring, segment): sort the segment's points by (curvature, index)
// (std::sort(cloudSortInd + sp, cloudSortInd + ep + 1, comp) with the tie order fixed by index)
__global__ void __launch_bounds__(256) fe_sort_kernel(const float* __restrict__ curv, int* __restrict__ st,
                                                      int* __restrict__ sort_ind) {
  pdl_entry();
  __shared__ u64 keys[kMaxSeg];
  const int ring = blockIdx.x / 6, j = blockIdx.x % 6;
  int S, E;
  ring_bounds(st, ring, S, E);
  if (E - S < 6) return;
  const int sp = S + (E - S) * j / 6, ep = S + (E - S) * (j + 1) / 6 - 1;
  const int L = ep - sp + 1;
  if (L <= 0) return;
  if (L > kMaxSeg) {
    if (threadIdx.x == 0) atomicOr(&st[kStErr], 1);
    return;
  }
  int P = 1;
  while (P < L) P <<= 1;
  for (int t = threadIdx.x; t < P; t += blockDim.x)
    keys[t] = t < L ? (((u64)__float_as_uint(curv[sp + t]) << 32) | (uint32_t)(sp + t)) : ~0ull;
  __syncthreads();
  bitonic_sort_smem(keys, P);
  for (int t = threadIdx.x; t < L; t += blockDim.x) sort_ind[sp + t] = (int)(uint32_t)keys[t];
}

// neighbour suppression of scanRegistration.cpp:481-504 by one warp: lanes 1..5 test the forward gaps,
// lanes 6..10 the backward gaps; marking stops at the first gap^2 > 0.05
__device__ __forceinline__ void mark_neighbours(const float4* cloud, unsigned char* picked, int ind, int lane) {
  bool gap = false;
  int a = 0;
  if (lane >= 1 && lane <= 10) {
    const int l = lane <= 5 ? lane : -(lane - 5);
    a = ind + l;
    const int b = l > 0 ? a - 1 : a + 1;
    const float4 pa = cloud[a], pb = cloud[b];  // generic loads: the ring is staged in shared memory when it fits
    const float dx = __fsub_rn(pa.x, pb.x), dy = __fsub_rn(pa.y, pb.y), dz = __fsub_rn(pa.z, pb.z);
    const float g = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    gap = (double)g > 0.05;
  }
  const unsigned gm = __ballot_sync(0xffffffffu, gap);
  const unsigned fwd = (gm >> 1) & 0x1Fu, bwd = (gm >> 6) & 0x1Fu;
  const int nf = fwd ? __ffs(fwd) - 1 : 5, nb = bwd ? __ffs(bwd) - 1 : 5;  // neighbours marked on each side
  if (lane == 0) picked[ind] = 1;
  if (lane >= 1 && lane <= 5 && lane <= nf) picked[a] = 1;
  if (lane >= 6 && lane <= 10 && lane - 5 <= nb) picked[a] = 1;
  __syncwarp();
}

// pass 6: feature picking (scanRegistration.cpp:427-565), one block of six warps per ring.
// Inside a segment the picks are a dependent chain (the first eligible entry in sorted order is taken, its neighbours are
// suppressed, the test is repeated): one warp walks it, 32 sorted entries per window -- the window's indices and curvature
// tests are loaded once, after every pick only the picked flags of the lanes behind it are read again.
// Between segments the reference is sequential too, but the coupling is thin: segment j + 1 depends on segment j only
// through the picked flags segment j's picks leave on the FIRST FIVE points of segment j + 1 (a pick suppresses at most five
// neighbours ahead), and an initially suppressed point changes the outcome only if segment j + 1 would have picked it.
// So the six segments are picked SPECULATIVELY in parallel, each warp on private flags, and then checked in order: a
// segment whose own picks avoid the points its predecessor's final run suppressed is exactly the sequential result;
// otherwise it is re-run with those points suppressed (and its successor is checked against the new run).  Rings with a
// segment shorter than 11 points (a predecessor's suppression could reach past it) and rings that do not fit the staging
// buffers take the sequential order on one warp.
constexpr int kPickCap = 1536;  // ring points staged in shared memory (an OS0-64 ring has 1024)
constexpr int kPickWarps = 6;

struct SegPicks {  // what one segment's run picked, in pick order (labels are written once the run is final)
  int n_sharp, n_lsharp, n_flat;
  int sharp[2], lsharp[20], flat[4];
};

__device__ __forceinline__ void pick_segment(const float4* cloud, const float* curv, const int* sort_ind, unsigned char* picked, int sp,
                                             int ep, int lane, SegPicks* out) {
  int n_sharp = 0, n_lsharp = 0, n_flat = 0;
  // ---- sharp / less sharp: descending curvature
  int largest = 0;
  int k = ep;
  bool stop = false;
  while (k >= sp && !stop) {
    const int kk = k - lane;
    int ind = -1;
    bool low = false;
    if (kk >= sp) {
      ind = sort_ind[kk];
      low = !((double)curv[ind] > 0.1);
    }
    const unsigned lm = __ballot_sync(0xffffffffu, low);
    const int fl = lm ? __ffs(lm) - 1 : 32;  // sorted: from here on the curvature is <= 0.1 and nothing qualifies
    unsigned avail = __ballot_sync(0xffffffffu, kk >= sp && !low) & (fl < 32 ? (1u << fl) - 1u : 0xffffffffu);
    while (avail) {
      const bool elig = ((avail >> lane) & 1u) && picked[ind] == 0;
      const unsigned em = __ballot_sync(0xffffffffu, elig);
      if (!em) break;
      const int fe = __ffs(em) - 1;
      const int pick = __shfl_sync(0xffffffffu, ind, fe);
      ++largest;
      if (largest <= 2) {
        if (lane == 0) out->sharp[n_sharp] = pick, out->lsharp[n_lsharp] = pick;
        ++n_sharp, ++n_lsharp;
      } else if (largest <= 20) {
        if (lane == 0) out->lsharp[n_lsharp] = pick;
        ++n_lsharp;
      } else {
        stop = true;
        break;
      }
      mark_neighbours(cloud, picked, pick, lane);
      avail &= ~((2u << fe) - 1u);  // the lanes up to the pick are behind us (fe = 31: 2u << 31 wraps to 0, mask = all)
    }
    if (fl < 32) break;
    k -= 32;
  }
  // ---- flat: ascending curvature, four picks, the fourth does not suppress its neighbours
  int smallest = 0;
  k = sp;
  stop = false;
  while (k <= ep && !stop) {
    const int kk = k + lane;
    int ind = -1;
    bool high = false;
    if (kk <= ep) {
      ind = sort_ind[kk];
      high = !((double)curv[ind] < 0.1);
    }
    const unsigned hm = __ballot_sync(0xffffffffu, high);
    const int fh = hm ? __ffs(hm) - 1 : 32;
    unsigned avail = __ballot_sync(0xffffffffu, kk <= ep && !high) & (fh < 32 ? (1u << fh) - 1u : 0xffffffffu);
    while (avail) {
      const bool elig = ((avail >> lane) & 1u) && picked[ind] == 0;
      const unsigned em = __ballot_sync(0xffffffffu, elig);
      if (!em) break;
      const int fe = __ffs(em) - 1;
      const int pick = __shfl_sync(0xffffffffu, ind, fe);
      if (lane == 0) out->flat[n_flat] = pick;
      ++n_flat;
      ++smallest;
      if (smallest >= 4) {
        stop = true;
        break;
      }
      mark_neighbours(cloud, picked, pick, lane);
      avail &= ~((2u << fe) - 1u);
    }
    if (fh < 32) break;
    k += 32;
  }
  __syncwarp();
  if (lane == 0) out->n_sharp = n_sharp, out->n_lsharp = n_lsharp, out->n_flat = n_flat;
  __syncwarp();
}

__global__ void __launch_bounds__(32 * kPickWarps) fe_pick_kernel(const float4* __restrict__ g_cloud, const float* __restrict__ g_curv,
                                                                   const int* __restrict__ g_sort_ind, int* __restrict__ st,
                                                                   int* __restrict__ label, unsigned char* __restrict__ g_picked,
                                                                   int* __restrict__ ring_sharp, int* __restrict__ ring_lsharp,
                                                                   int* __restrict__ ring_flat) {
  pdl_entry();
  __shared__ float4 s_cloud[kPickCap];
  __shared__ float s_curv[kPickCap];
  __shared__ int s_sort[kPickCap];
  __shared__ unsigned char s_picked[kPickWarps][kPickCap];
  __shared__ SegPicks s_seg[kPickWarps];
  const int ring = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int S, E;
  ring_bounds(st, ring, S, E);
  if (E - S < 6) return;
  // every access of this ring's picking falls into [S - 5, E + 6): stage it once, the picks then run on shared-memory latency
  const int base = S - 5, cnt = E + 6 - base;
  const bool staged = cnt <= kPickCap;
  const int sp = S + (E - S) * warp / 6, ep = S + (E - S) * (warp + 1) / 6 - 1;  // this warp's segment (:440-441)
  const bool seg_ok = ep - sp + 1 <= kMaxSeg;                                    // larger ones are flagged by the sort kernel and skipped
  const bool parallel = staged && (E - S) / 6 >= 11;                             // every segment at least 11 points long
  if (tid < kPickWarps) s_seg[tid].n_sharp = s_seg[tid].n_lsharp = s_seg[tid].n_flat = 0;
  if (staged) {
    for (int t = tid; t < cnt; t += blockDim.x) {
      s_cloud[t] = g_cloud[base + t];
      s_curv[t] = g_curv[base + t];
      s_sort[t] = g_sort_ind[base + t];
    }
    for (int t = tid; t < kPickWarps * kPickCap / 4; t += blockDim.x) reinterpret_cast<uint32_t*>(&s_picked[0][0])[t] = 0u;
  }
  __syncthreads();
  if (parallel) {
    const float4* cloud = s_cloud - base;
    const float* curv = s_curv - base;
    const int* sort_ind = s_sort - base;
    unsigned char* mine = s_picked[warp] - base;
    if (seg_ok) pick_segment(cloud, curv, sort_ind, mine, sp, ep, lane, &s_seg[warp]);
    __syncthreads();
    // in segment order: the points this segment's predecessor (final run) suppressed among its first five
#pragma unroll 1
    for (int j = 1; j < kPickWarps; ++j) {
      if (warp == j && seg_ok) {
        const unsigned char* prev = s_picked[j - 1] - base;
        const unsigned inc = __ballot_sync(0xffffffffu, lane < 5 && prev[sp + lane] != 0);
        if (inc) {
          const SegPicks& r = s_seg[j];
          bool hit = false;  // did this segment's run pick one of them?  (the lists hold at most 20 + 4 picks)
          if (lane < r.n_lsharp) hit = (unsigned)(r.lsharp[lane] - sp) < 5u && ((inc >> (r.lsharp[lane] - sp)) & 1u);
          if (lane >= 24 && lane - 24 < r.n_flat) hit = (unsigned)(r.flat[lane - 24] - sp) < 5u && ((inc >> (r.flat[lane - 24] - sp)) & 1u);
          if (__any_sync(0xffffffffu, hit)) {  // yes: pick it again, with those points suppressed from the start
            for (int t = sp - 5 + lane; t <= ep + 5; t += 32) mine[t] = 0;
            __syncwarp();
            if (lane < 5 && ((inc >> lane) & 1u)) mine[sp + lane] = 1;
            __syncwarp();
            pick_segment(cloud, curv, sort_ind, mine, sp, ep, lane, &s_seg[j]);
          }
        }
      }
      __syncthreads();
    }
  } else {
    // sequential order on one warp, one set of flags for the whole ring (shared when the ring is staged, else global)
    if (warp == 0) {
      const float4* cloud = staged ? s_cloud - base : g_cloud;
      const float* curv = staged ? s_curv - base : g_curv;
      const int* sort_ind = staged ? s_sort - base : g_sort_ind;
      unsigned char* picked = staged ? s_picked[0] - base : g_picked;
      for (int j = 0; j < 6; ++j) {
        const int spj = S + (E - S) * j / 6, epj = S + (E - S) * (j + 1) / 6 - 1;
        if (epj - spj + 1 > kMaxSeg) continue;
        pick_segment(cloud, curv, sort_ind, picked, spj, epj, lane, &s_seg[j]);
      }
    }
    __syncthreads();
  }
  // ---- labels and the ring's three index lists, segments in order (the reference appends as it goes)
  int o_sharp = 0, o_lsharp = 0, o_flat = 0;
  for (int j = 0; j < warp; ++j) o_sharp += s_seg[j].n_sharp, o_lsharp += s_seg[j].n_lsharp, o_flat += s_seg[j].n_flat;
  const SegPicks& r = s_seg[warp];
  if (lane < r.n_lsharp) {
    const int pick = r.lsharp[lane];
    label[pick] = lane < r.n_sharp ? 2 : 1;  // the first (up to two) picks of a segment are the sharp ones
    ring_lsharp[ring * 120 + o_lsharp + lane] = pick;
    if (lane < r.n_sharp) ring_sharp[ring * 12 + o_sharp + lane] = pick;
  }
  if (lane < r.n_flat) {
    const int pick = r.flat[lane];
    label[pick] = -1;
    ring_flat[ring * 24 + o_flat + lane] = pick;
  }
  if (tid == 0) {
    int ns = 0, nl = 0, nf = 0;
    for (int j = 0; j < kPickWarps; ++j) ns += s_seg[j].n_sharp, nl += s_seg[j].n_lsharp, nf += s_seg[j].n_flat;
    st[kStSharp + ring] = ns;
    st[kStLSharp + ring] = nl;
    st[kStFlat + ring] = nf;
  }
}

// pass 7: one block per ring: collect the ring's less-flat points (label <= 0 inside the six segments, in index
// order) and run VoxelGrid(0.2) on them (scanRegistration.cpp:570-589)
__global__ void __launch_bounds__(256) fe_lessflat_kernel(const float4* __restrict__ cloud, const int* __restrict__ label,
                                                          int* __restrict__ st, float4* __restrict__ ring_pts,
                                                          float4* __restrict__ ring_out, int ring_cap, float leaf) {
  pdl_entry();
  __shared__ u64 keys[kMaxRingLF];
  __shared__ int s_m;
  const int ring = blockIdx.x;
  int S, E;
  ring_bounds(st, ring, S, E);
  if (E - S < 6) return;
  // the six segments tile [S, S + (E-S)*6/6 - 1] = [S, E-1] contiguously
  const int lo = S, hi = S + (E - S) * 6 / 6 - 1;
  if (threadIdx.x == 0) s_m = 0;
  __syncthreads();
  float4* mine = ring_pts + (size_t)ring * ring_cap;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ int wc[8];
  for (int c0 = lo; c0 <= hi; c0 += blockDim.x) {
    const int k = c0 + threadIdx.x;
    const bool take = k <= hi && label[k] <= 0;
    const unsigned b = __ballot_sync(0xffffffffu, take);
    if (lane == 0) wc[warp] = __popc(b);
    __syncthreads();
    int wbase = 0, tot = 0;
    for (int w = 0; w < 8; ++w) {
      if (w < warp) wbase += wc[w];
      tot += wc[w];
    }
    const int base = s_m;
    if (take) {
      const int pos = base + wbase + __popc(b & ((1u << lane) - 1u));
      if (pos < ring_cap) mine[pos] = cloud[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) s_m = base + tot;
    __syncthreads();
  }
  const int m = s_m;
  if (m > kMaxRingLF || m > ring_cap) {
    if (threadIdx.x == 0) atomicOr(&st[kStErr], 4);
    return;
  }
  int P = 1;
  while (P < m) P <<= 1;
  const int nvox = m > 0 ? voxelgrid_block(mine, m, leaf, keys, P, ring_out + (size_t)ring * ring_cap, &st[kStErr]) : 0;
  if (threadIdx.x == 0) st[kStLFlat + ring] = nvox;
}

// pass 8: concatenate the per-ring outputs in ring order (the reference appends ring by ring)
__global__ void fe_compact_kernel(const int* __restrict__ st, const int* __restrict__ ring_sharp,
                                  const int* __restrict__ ring_lsharp, const int* __restrict__ ring_flat,
                                  const float4* __restrict__ ring_out, int ring_cap, int* __restrict__ sharp,
                                  int* __restrict__ lsharp, int* __restrict__ flat, float4* __restrict__ lflat,
                                  int* __restrict__ counts /* n_cloud, n_sharp, n_lsharp, n_flat, n_lflat */) {
  pdl_entry();
  const int ring = blockIdx.x;
  int o_s = 0, o_ls = 0, o_f = 0, o_lf = 0;
  for (int r = 0; r < ring; ++r) {
    o_s += st[kStSharp + r], o_ls += st[kStLSharp + r], o_f += st[kStFlat + r], o_lf += st[kStLFlat + r];
  }
  const int ns = st[kStSharp + ring], nls = st[kStLSharp + ring], nf = st[kStFlat + ring], nlf = st[kStLFlat + ring];
  for (int t = threadIdx.x; t < ns; t += blockDim.x) sharp[o_s + t] = ring_sharp[ring * 12 + t];
  for (int t = threadIdx.x; t < nls; t += blockDim.x) lsharp[o_ls + t] = ring_lsharp[ring * 120 + t];
  for (int t = threadIdx.x; t < nf; t += blockDim.x) flat[o_f + t] = ring_flat[ring * 24 + t];
  for (int t = threadIdx.x; t < nlf; t += blockDim.x) lflat[o_lf + t] = ring_out[(size_t)ring * ring_cap + t];
  if (ring == kRings - 1 && threadIdx.x == 0) {
    int N = 0;
    for (int r = 0; r < kRings; ++r) N += st[kStRing + r];
    counts[0] = N;
    counts[1] = o_s + ns, counts[2] = o_ls + nls, counts[3] = o_f + nf, counts[4] = o_lf + nlf;
    counts[5] = st[kStErr];
  }
}

// gather selected points of a cloud by index (less-sharp / sharp / flat clouds)
__global__ void gather_points_kernel(const float4* __restrict__ cloud, const int* __restrict__ idx, const int* __restrict__ n_ptr,
                                     int slot, float4* __restrict__ out) {
  pdl_entry();
  const int n = n_ptr[slot];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = cloud[idx[i]];
}

// stand-alone VoxelGrid, one block per job (n <= kVoxelMax per job).  The two feature stacks of a frame (corner / surf)
// are two jobs of one launch.
constexpr int kVoxelMax = kVoxelBlockMax;
constexpr int kVgHashMin = 2048;  // clouds above this size take the hash-based VoxelGrid (only the distinct voxels are sorted)
struct VoxJob {
  const float* in;
  float4* packed;
  float4* out;
  int* n_out;
  int n, stride_f, ioff;
  float leaf;
  uint32_t* scratch;  // kVgScratchWords words of global memory for the hash-based path (nullptr: sort-based path only)
};
struct VoxJobs {
  VoxJob j[2];
};
__global__ void __launch_bounds__(1024) voxelgrid_kernel(VoxJobs jobs, int* err) {
  pdl_entry();
  extern __shared__ u64 dyn_keys[];
  const VoxJob jb = blockIdx.x == 0 ? jobs.j[0] : jobs.j[1];  // no dynamic index: the parameters stay in the constant bank
  const int n = jb.n;
  if (n > kVoxelMax) {
    if (threadIdx.x == 0) atomicOr(err, 8), *jb.n_out = 0;
    return;
  }
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    const float* p = jb.in + (size_t)t * jb.stride_f;
    jb.packed[t] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + jb.ioff));
  }
  __syncthreads();
  int P = 1;
  while (P < n) P <<= 1;
  int nvox = 0;
  if (n > kVgHashMin && jb.scratch)
    nvox = voxelgrid_block_hash(jb.packed, n, jb.leaf, reinterpret_cast<unsigned char*>(dyn_keys), jb.scratch, jb.out, err);
  else if (n > 0)
    nvox = voxelgrid_block(jb.packed, n, jb.leaf, dyn_keys, P, jb.out, err);
  if (threadIdx.x == 0) *jb.n_out = nvox;
}

// ---------------------------------------------------------------------------------------------------
// VoxelGrid of clouds that do not fit one block (n > 16384, e.g. mapOptimization's ground + less-flat cloud): the
// same PCL semantics as voxelgrid_block, spread over the GPU.  bbox reduction -> keys (voxel << 24 | order) -> tiled
// bitonic sort (16384-key tiles sorted in registers/shuffles/shared memory, cross-tile stages through global memory)
// -> run heads -> per-chunk head counts + scan -> ordered float centroids.
// ---------------------------------------------------------------------------------------------------
constexpr int kVgTile = 16384;
__device__ __forceinline__ int fenc(float f) {
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float fdec(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF); }

__global__ void vg_init_kernel(VgState* st) {
  pdl_entry();
  if (threadIdx.x < 3) st->mn[threadIdx.x] = fenc(__int_as_float(0x7f800000)), st->mx[threadIdx.x] = fenc(__int_as_float(0xff800000));
  if (threadIdx.x == 3) st->n_out = 0;
}

__global__ void __launch_bounds__(256) vg_pack_bbox_kernel(const float* __restrict__ in, int n, int stride_f, int ioff,
                                                           float4* __restrict__ packed, VgState* st) {
  pdl_entry();
  float mn[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
  float mx[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
    const float* p = in + (size_t)t * stride_f;
    const float4 v = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + ioff));
    packed[t] = v;
    if (isfinite(v.x) && isfinite(v.y) && isfinite(v.z)) {
      mn[0] = fminf(mn[0], v.x), mn[1] = fminf(mn[1], v.y), mn[2] = fminf(mn[2], v.z);
      mx[0] = fmaxf(mx[0], v.x), mx[1] = fmaxf(mx[1], v.y), mx[2] = fmaxf(mx[2], v.z);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], off));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], off));
    }
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) atomicMin(&st->mn[a], fenc(mn[a])), atomicMax(&st->mx[a], fenc(mx[a]));
  }
}

__global__ void __launch_bounds__(256) vg_keys_kernel(const float4* __restrict__ packed, int n, int P, float leaf, const VgState* st,
                                                      u64* __restrict__ keys, int* err) {
  pdl_entry();
  const float inv = __fdiv_rn(1.0f, leaf);
  int min_b[3], div_b[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    min_b[a] = __float2int_rd(__fmul_rn(fdec(st->mn[a]), inv));
    div_b[a] = __float2int_rd(__fmul_rn(fdec(st->mx[a]), inv)) - min_b[a] + 1;
  }
  const long long mul1 = div_b[0], mul2 = (long long)div_b[0] * div_b[1];
  const bool too_small = mul2 * div_b[2] >= (1ll << 31);  // pcl: "Leaf size is too small for the input dataset"
  if (too_small && blockIdx.x == 0 && threadIdx.x == 0) atomicOr(err, 2);
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < P; t += gridDim.x * blockDim.x) {
    u64 key = ~0ull;
    if (t < n && !too_small) {
      const float4 p = packed[t];
      if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
        const int i0 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(p.x, inv)), (float)min_b[0]));
        const int i1 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(p.y, inv)), (float)min_b[1]));
        const int i2 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(p.z, inv)), (float)min_b[2]));
        const long long idx = i0 + i1 * mul1 + i2 * mul2;
        key = ((u64)idx << 24) | (uint32_t)t;
      }
    }
    keys[t] = key;
  }
}

// one 16384-key tile per block (E = 16 keys per thread).  merge_only == 0: full sort of the tile (stages 2 .. tile);
// merge_only == 1: the partner distances tile/2 .. 1 of stage k (after the cross-tile exchanges of that stage).
__global__ void __launch_bounds__(1024) vg_sort_tile_kernel(u64* __restrict__ keys, unsigned k, int merge_only) {
  pdl_entry();
  extern __shared__ u64 tile[];
  const unsigned base = blockIdx.x * (unsigned)kVgTile;
  for (int t = threadIdx.x; t < kVgTile; t += blockDim.x) tile[t] = keys[base + t];
  __syncthreads();
  if (merge_only) bitonic_sort_regs<16>(tile, kVgTile, base, k, k, true);
  else bitonic_sort_regs<16>(tile, kVgTile, base, 2u, (unsigned)kVgTile, false);
  for (int t = threadIdx.x; t < kVgTile; t += blockDim.x) keys[base + t] = tile[t];
}

// cross-tile compare-exchange of stage k at partner distance j >= tile
__global__ void __launch_bounds__(256) vg_sort_global_kernel(u64* __restrict__ keys, unsigned P, unsigned k, unsigned j) {
  pdl_entry();
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < P / 2; t += gridDim.x * blockDim.x) {
    const unsigned i = ((t & ~(j - 1u)) << 1) | (t & (j - 1u));  // index with bit j clear
    const unsigned p = i | j;
    const u64 a = keys[i], b = keys[p];
    const bool up = (i & k) == 0;
    if ((a > b) == up) keys[i] = b, keys[p] = a;
  }
}

__global__ void __launch_bounds__(256) vg_head_count_kernel(const u64* __restrict__ keys, int P, int* __restrict__ chunk_cnt) {
  pdl_entry();
  __shared__ int wc[8];
  const int t = blockIdx.x * 256 + threadIdx.x;
  bool head = false;
  if (t < P && keys[t] != ~0ull) head = t == 0 || (keys[t] >> 24) != (keys[t - 1] >> 24);
  const unsigned b = __ballot_sync(0xffffffffu, head);
  if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(b);
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < 8; ++w) s += wc[w];
    chunk_cnt[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(1024) vg_scan_kernel(const int* __restrict__ chunk_cnt, int chunks, int* __restrict__ chunk_base,
                                                       int* __restrict__ total, int* __restrict__ total2) {
  pdl_entry();
  __shared__ int wsum[32];
  __shared__ int carry_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int c0 = 0; c0 < chunks; c0 += 1024) {
    const int c = c0 + threadIdx.x;
    const int v = c < chunks ? chunk_cnt[c] : 0;
    int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, inc, off);
      if (lane >= off) inc += o;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int wbase = 0, tot = 0;
    for (int w = 0; w < 32; ++w) {
      if (w < warp) wbase += wsum[w];
      tot += wsum[w];
    }
    const int carry = carry_s;
    if (c < chunks) chunk_base[c] = carry + wbase + inc - v;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *total = carry_s;
    if (total2) *total2 = carry_s;
  }
}

__global__ void __launch_bounds__(256) vg_centroid_kernel(const u64* __restrict__ keys, int P, const float4* __restrict__ packed,
                                                          const int* __restrict__ chunk_base, float4* __restrict__ out) {
  pdl_entry();
  __shared__ int wc[8];
  const int t = blockIdx.x * 256 + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool head = false;
  if (t < P && keys[t] != ~0ull) head = t == 0 || (keys[t] >> 24) != (keys[t - 1] >> 24);
  const unsigned b = __ballot_sync(0xffffffffu, head);
  if (lane == 0) wc[warp] = __popc(b);
  __syncthreads();
  if (!head) return;
  int wbase = 0;
  for (int w = 0; w < warp; ++w) wbase += wc[w];
  const int slot = chunk_base[blockIdx.x] + wbase + __popc(b & ((1u << lane) - 1u));
  const u64 vox = keys[t] >> 24;
  int cnt = 1;
  while (t + cnt < P && (keys[t + cnt] >> 24) == vox) ++cnt;
  float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
  for (int e0 = 0; e0 < cnt; e0 += 4) {
    float4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) q[u] = e0 + u < cnt ? packed[(int)(keys[t + e0 + u] & 0xFFFFFF)] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (e0 + u < cnt) sx = __fadd_rn(sx, q[u].x), sy = __fadd_rn(sy, q[u].y), sz = __fadd_rn(sz, q[u].z), si = __fadd_rn(si, q[u].w);
  }
  const float c = (float)cnt;
  out[slot] = make_float4(__fdiv_rn(sx, c), __fdiv_rn(sy, c), __fdiv_rn(sz, c), __fdiv_rn(si, c));
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
int Ctx::project_dev(const float* d_cloud, int n, int stride_bytes, unsigned char* d_range, unsigned char* d_inten,
                     float* d_track) {
  if (n <= 0) return ILSM_OK;
  const int stride_f = stride_bytes / 4, ioff = intensity_word(stride_bytes);
  const int threads = 256, blocks = ((n + 3) / 4 + threads - 1) / threads;
  ILSM_CUDA(launch_pdl(project_kernel, dim3(blocks), dim3(threads), 0, stream, d_cloud, n, stride_f, ioff, d_range, d_inten, reinterpret_cast<float4*>(d_track)));
  count_launches(1);
  return check_launch("project");
}

static inline unsigned __float_as_uint_host(float f) {
  unsigned u;
  memcpy(&u, &f, 4);
  return u;
}

int Ctx::features_dev(const float* d_in, int n, int stride_bytes, float min_range) {
  int rc;
  FeBufs& f = fe;
  const int ring_cap = n < kMaxRingLF ? (n > 0 ? n : 1) : kMaxRingLF;
  if ((rc = f.scanid.reserve(n + 4)) || (rc = f.ori.reserve(n + 4)) || (rc = f.stats.reserve(kStInts + 8)) ||
      (rc = f.cloud.reserve(n + 4)) || (rc = f.src_index.reserve(n + 4)) || (rc = f.curv.reserve(n + 4)) ||
      (rc = f.label.reserve(n + 4)) || (rc = f.picked.reserve(n + 4)) || (rc = f.sort_ind.reserve(n + 4)) ||
      (rc = f.ring_sharp.reserve(kRings * 12)) || (rc = f.ring_lsharp.reserve(kRings * 120)) ||
      (rc = f.ring_flat.reserve(kRings * 24)) || (rc = f.ring_pts.reserve((size_t)kRings * ring_cap)) ||
      (rc = f.ring_out.reserve((size_t)kRings * ring_cap)) || (rc = f.sharp.reserve(kRings * 12)) ||
      (rc = f.lsharp.reserve(kRings * 120)) || (rc = f.flat.reserve(kRings * 24)) || (rc = f.lflat.reserve(n + 4)) ||
      (rc = f.counts.reserve(8)) || (rc = f.chunk_hist.reserve((size_t)(n / 256 + 2) * kRings)) ||
      (rc = f.chunk_base.reserve((size_t)(n / 256 + 2) * kRings)))
    return rc;
  f.n_in = n;
  f.ring_cap = ring_cap;
  // The chain is 10 short kernels whose launch parameters only depend on (input pointer, n, stride, min_range) and on the
  // scratch pointers: it is captured once into a CUDA graph (programmatic-dependent-launch edges included) and replayed
  // with ONE launch call per frame -- 10 launches cost ~32 us of host time, the replay ~8.  Any change of a parameter
  // or a reallocated scratch buffer re-captures.
  unsigned long long key = 1469598103934665603ull;
  auto mix = [&key](unsigned long long v) { key = (key ^ v) * 1099511628211ull; };
  mix((unsigned long long)(uintptr_t)d_in), mix((unsigned long long)n), mix((unsigned long long)stride_bytes), mix((unsigned long long)ring_cap);
  mix((unsigned long long)__float_as_uint_host(min_range));
  const void* ptrs[] = {f.scanid.p, f.ori.p, f.stats.p, f.cloud.p, f.src_index.p, f.curv.p, f.label.p, f.picked.p, f.sort_ind.p,
                        f.ring_sharp.p, f.ring_lsharp.p, f.ring_flat.p, f.ring_pts.p, f.ring_out.p, f.sharp.p, f.lsharp.p, f.flat.p,
                        f.lflat.p, f.counts.p, f.chunk_hist.p, f.chunk_base.p};
  for (const void* q : ptrs) mix((unsigned long long)(uintptr_t)q);
  if (fe_graph_exec && key == fe_graph_key) {
    ILSM_CUDA(cudaGraphLaunch(fe_graph_exec, stream));
    count_launches(n > 0 ? 10 : 2);
    return check_launch("extract_features(graph)");
  }
  bool capturing = false;
  if (fe_graphs_ok) {
    if (fe_graph_exec) cudaGraphExecDestroy(fe_graph_exec), fe_graph_exec = nullptr;
    capturing = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (!capturing) cudaGetLastError(), fe_graphs_ok = false;
  }
  int rcl = features_launch(d_in, n, stride_bytes, min_range, ring_cap);
  if (capturing) {
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(stream, &g);
    if (e == cudaSuccess && rcl == ILSM_OK) e = cudaGraphInstantiate(&fe_graph_exec, g, 0);
    if (g) cudaGraphDestroy(g);
    if (e != cudaSuccess || rcl != ILSM_OK || !fe_graph_exec) {  // capture not possible here: plain launches from now on
      cudaGetLastError();
      fe_graph_exec = nullptr, fe_graphs_ok = false;
      return features_launch(d_in, n, stride_bytes, min_range, ring_cap);
    }
    fe_graph_key = key;
    ILSM_CUDA(cudaGraphLaunch(fe_graph_exec, stream));
    return check_launch("extract_features(graph)");
  }
  return rcl;
}

int Ctx::features_launch(const float* d_in, int n, int stride_bytes, float min_range, int ring_cap) {
  FeBufs& f = fe;
  const int stride_f = stride_bytes / 4;
  const int T = 256, B = (n + T - 1) / T;
  ILSM_CUDA(launch_pdl(fe_init_kernel, dim3(1), dim3(352), 0, stream, f.stats.p));
  if (n > 0) {
    ILSM_CUDA(launch_pdl(fe_tag_kernel, dim3(B), dim3(T), 0, stream, d_in, n, stride_f, min_range * min_range, f.scanid.p, f.ori.p, f.stats.p, f.chunk_hist.p));
    ILSM_CUDA(launch_pdl(fe_star_kernel, dim3(B), dim3(T), 0, stream, d_in, n, stride_f, f.scanid.p, f.ori.p, f.stats.p));
    ILSM_CUDA(launch_pdl(fe_scan_kernel, dim3(kRings), dim3(256), 0, stream, f.chunk_hist.p, B, f.chunk_base.p));
    ILSM_CUDA(launch_pdl(fe_bucket_kernel, dim3(B), dim3(kFeChunk), 0, stream, d_in, n, stride_f, f.scanid.p, f.ori.p, f.stats.p, f.chunk_base.p, f.cloud.p, f.src_index.p));
    ILSM_CUDA(launch_pdl(fe_curvature_kernel, dim3(B), dim3(T), 0, stream, f.cloud.p, f.stats.p, f.curv.p, f.label.p, f.picked.p));
    ILSM_CUDA(launch_pdl(fe_sort_kernel, dim3(kRings * 6), dim3(256), 0, stream, f.curv.p, f.stats.p, f.sort_ind.p));
    ILSM_CUDA(launch_pdl(fe_pick_kernel, dim3(kRings), dim3(32 * kPickWarps), 0, stream, f.cloud.p, f.curv.p, f.sort_ind.p, f.stats.p, f.label.p, f.picked.p, f.ring_sharp.p, f.ring_lsharp.p, f.ring_flat.p));
    ILSM_CUDA(launch_pdl(fe_lessflat_kernel, dim3(kRings), dim3(256), 0, stream, f.cloud.p, f.label.p, f.stats.p, f.ring_pts.p, f.ring_out.p, ring_cap, 0.2f));
    count_launches(8);
  }
  ILSM_CUDA(launch_pdl(fe_compact_kernel, dim3(kRings), dim3(128), 0, stream, f.stats.p, f.ring_sharp.p, f.ring_lsharp.p, f.ring_flat.p, f.ring_out.p, ring_cap, f.sharp.p, f.lsharp.p, f.flat.p, f.lflat.p, f.counts.p));
  count_launches(2);
  return check_launch("extract_features");
}

// one cloud of at most kVoxelMax points as one block of voxelgrid_kernel; returns the dynamic shared memory it needs
static size_t vox_block_job(VoxJob& job, const Ctx::VgCloud& c, float4* packed, uint32_t* scratch, int stride_bytes, int ioff) {
  job = VoxJob{c.in, packed, c.out, c.n_out, c.n, stride_bytes / 4, ioff, c.leaf, scratch};
  int P = 1;
  while (P < c.n) P <<= 1;
  return c.n > kVgHashMin ? kVgHashSmemBytes : (size_t)P * sizeof(u64);
}

// When every cloud fits a block: ONE launch, one block per cloud (the corner and surf stacks of a frame).  Otherwise the
// clouds go one after the other on `s` (they share the scratch buffers), a cloud above kVoxelMax points on the tiled
// multi-block path (a 64-ring sensor that keeps all its beams produces ~25 k less-flat points,
// scanRegistration.cpp:570-589).  The caller's own error word keeps a VoxelGrid running on a side stream from sharing a
// word with the front end that resets its own.
int Ctx::voxelgrid(const VgCloud* clouds, int count, int stride_bytes, int ioff, cudaStream_t s, int* d_err) {
  int rc;
  if ((rc = fe.vox_packed.reserve((size_t)2 * kVoxelMax + 8)) || (rc = fe.stats.reserve(kStInts + 8)) || (rc = fe.vg_hash.reserve(2 * kVgScratchWords)))
    return rc;
  if (!d_err) d_err = fe.stats.p + kStErr;
  ILSM_CUDA(cudaFuncSetAttribute(voxelgrid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVgHashSmemBytes));
  bool fit = true;
  for (int k = 0; k < count; ++k) fit = fit && clouds[k].n <= kVoxelMax;
  if (fit) {
    VoxJobs jobs = {};
    size_t smem = 0;
    for (int k = 0; k < count; ++k)
      smem = std::max(smem, vox_block_job(jobs.j[k], clouds[k], fe.vox_packed.p + (size_t)k * kVoxelMax, fe.vg_hash.p + k * kVgScratchWords,
                                          stride_bytes, ioff));
    ILSM_CUDA(launch_pdl(voxelgrid_kernel, dim3(count), dim3(1024), smem, s, jobs, d_err));
    count_launches(1);
    return check_launch("voxelgrid");
  }
  for (int k = 0; k < count; ++k) {
    const VgCloud& c = clouds[k];
    if (c.n > kVoxelMax) {
      if ((rc = voxelgrid_large_dev(c.in, c.n, stride_bytes, ioff, c.leaf, c.out, c.n_out, s, d_err))) return rc;
    } else {
      VoxJobs jobs = {};
      const size_t smem = vox_block_job(jobs.j[0], c, fe.vox_packed.p, fe.vg_hash.p, stride_bytes, ioff);
      ILSM_CUDA(launch_pdl(voxelgrid_kernel, dim3(1), dim3(1024), smem, s, jobs, d_err));
      count_launches(1);
    }
  }
  return check_launch("voxelgrid(large)");
}

// VoxelGrid of n > 16384 points (up to 2^24): see the vg_* kernels above.  d_n_out receives the voxel count.
int Ctx::voxelgrid_large_dev(const float* d_in, int n, int stride_bytes, int ioff, float leaf, float4* d_out, int* d_n_out,
                             cudaStream_t s, int* d_err) {
  if (n >= (1 << 24)) return fail(ILSM_ERR_INVALID_ARG, "voxelgrid: at most 2^24 points");
  unsigned P = kVgTile;
  while (P < (unsigned)n) P <<= 1;
  const int chunks = (int)(P / 256);
  int rc;
  if ((rc = fe.vox_packed.reserve((size_t)n + 8)) || (rc = fe.vg_keys.reserve(P)) || (rc = fe.vg_state.reserve(1)) ||
      (rc = fe.vg_chunk.reserve(2 * (size_t)chunks + 8)) || (rc = fe.stats.reserve(kStInts + 8)))
    return rc;
  ILSM_CUDA(cudaFuncSetAttribute(vg_sort_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kVgTile * sizeof(u64))));
  const int grid = sm_count * 4;
  int launches = 0;
  ILSM_CUDA(launch_pdl(vg_init_kernel, dim3(1), dim3(32), 0, s, fe.vg_state.p));
  ILSM_CUDA(launch_pdl(vg_pack_bbox_kernel, dim3(grid), dim3(256), 0, s, d_in, n, stride_bytes / 4, ioff, fe.vox_packed.p, fe.vg_state.p));
  ILSM_CUDA(launch_pdl(vg_keys_kernel, dim3(grid), dim3(256), 0, s, (const float4*)fe.vox_packed.p, n, (int)P, leaf,
                       (const VgState*)fe.vg_state.p, fe.vg_keys.p, d_err));
  ILSM_CUDA(launch_pdl(vg_sort_tile_kernel, dim3(P / kVgTile), dim3(1024), kVgTile * sizeof(u64), s, fe.vg_keys.p, 0u, 0));
  launches += 4;
  for (unsigned k = 2u * kVgTile; k <= P; k <<= 1) {
    for (unsigned j = k >> 1; j >= (unsigned)kVgTile; j >>= 1) {
      ILSM_CUDA(launch_pdl(vg_sort_global_kernel, dim3(grid), dim3(256), 0, s, fe.vg_keys.p, P, k, j));
      ++launches;
    }
    ILSM_CUDA(launch_pdl(vg_sort_tile_kernel, dim3(P / kVgTile), dim3(1024), kVgTile * sizeof(u64), s, fe.vg_keys.p, k, 1));
    ++launches;
  }
  ILSM_CUDA(launch_pdl(vg_head_count_kernel, dim3(chunks), dim3(256), 0, s, (const u64*)fe.vg_keys.p, (int)P, fe.vg_chunk.p));
  ILSM_CUDA(launch_pdl(vg_scan_kernel, dim3(1), dim3(1024), 0, s, (const int*)fe.vg_chunk.p, chunks, fe.vg_chunk.p + chunks,
                       &fe.vg_state.p->n_out, d_n_out));
  ILSM_CUDA(launch_pdl(vg_centroid_kernel, dim3(chunks), dim3(256), 0, s, (const u64*)fe.vg_keys.p, (int)P,
                       (const float4*)fe.vox_packed.p, (const int*)(fe.vg_chunk.p + chunks), d_out));
  count_launches(launches + 3);
  return check_launch("voxelgrid_large");
}

int Ctx::gather_dev(const float4* d_cloud, const int* d_idx, const int* d_counts, int slot, int max_n, float4* d_out) {
  if (max_n <= 0) return ILSM_OK;
  ILSM_CUDA(launch_pdl(gather_points_kernel, dim3((max_n + 255) / 256), dim3(256), 0, stream, d_cloud, d_idx, d_counts, slot, d_out));
  count_launches(1);
  return check_launch("gather");
}

}  // namespace ilsm
