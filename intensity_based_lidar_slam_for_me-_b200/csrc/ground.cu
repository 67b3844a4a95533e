// ground.cu -- ground-plane extraction feeding mapOptimization (SURVEY 8f, f2).
//
// Replaces ImageHandler::groundPlaneExtraction (image_handler.h_ouster:41-100): z-band screening, pcl::SACSegmentation
// (SACMODEL_PLANE, SAC_RANSAC, threshold 0.01, optimize coefficients), the 15-degree acceptance test and the selection
// of the points within 0.03 m of the plane.
//
// RANSAC is a sequential loop with an adaptive iteration bound, but its hypotheses do not depend on each other: all
// candidate planes (64 triples from the declared LCG sampler -- PCL's rand() is unpinned) are built and scored against
// the screened cloud in parallel, the host replays PCL's loop (best-so-far, k = log(1-p)/log(1-w^3), skip of
// degenerate samples) over the 64 inlier counts, and the winner is refitted on the device (PCA of its inliers: sums
// in fp64 with a fixed reduction order, 3x3 Jacobi).  Inlier tests use PCL's float expression, left to right, no FMA:
// the counts are integers and match the oracle exactly.
#include <math.h>

#include "ilsm_host.hpp"

namespace ilsm {

constexpr int kGroundHyp = 64;
constexpr int kGroundChunk = 256;

struct GroundModels {
  float co[kGroundHyp][4];
  int valid[kGroundHyp];
};

__device__ __forceinline__ float plane_dist_f(const float* co, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(co[0], x), __fmul_rn(co[1], y)), __fmul_rn(co[2], z)), co[3]);
}

// mode 0: z band (screening);  mode 1: within `band` of the refitted plane and z < 0 (final selection, double math)
__device__ __forceinline__ bool ground_pred(int mode, float x, float y, float z, double z_min, double z_max, const float* coeff,
                                            double band) {
  if (mode == 0) return (double)z >= z_min && (double)z <= z_max;
  if (coeff[4] == 0.f) return false;  // plane rejected by the acceptance test
  const double A = coeff[0], B = coeff[1], C = coeff[2], D = coeff[3];
  const double X = x, Y = y, Z = z;
  const double height = fabs(A * X + B * Y + C * Z + D) / sqrt(A * A + B * B + C * C);
  return height <= band && Z < 0.0;
}

// stable compaction in three steps: per-chunk counts, scan of the chunk counts (one block), scatter
__global__ void __launch_bounds__(kGroundChunk) ground_count_kernel(const float* __restrict__ in, int n, int stride_f, int mode,
                                                                    double z_min, double z_max, const float* __restrict__ coeff,
                                                                    double band, int* __restrict__ chunk_cnt) {
  pdl_entry();
  __shared__ int wc[kGroundChunk / 32];
  const int i = blockIdx.x * kGroundChunk + threadIdx.x;
  bool keep = false;
  if (i < n) {
    const float* p = in + (size_t)i * stride_f;
    keep = ground_pred(mode, __ldg(p), __ldg(p + 1), __ldg(p + 2), z_min, z_max, coeff, band);
  }
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(b);
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < kGroundChunk / 32; ++w) t += wc[w];
    chunk_cnt[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(1024) ground_scan_kernel(const int* __restrict__ chunk_cnt, int chunks, int* __restrict__ chunk_base,
                                                           int* __restrict__ total) {
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
  if (threadIdx.x == 0) *total = carry_s;
}

__global__ void __launch_bounds__(kGroundChunk) ground_scatter_kernel(const float* __restrict__ in, int n, int stride_f, int mode,
                                                                      double z_min, double z_max, const float* __restrict__ coeff,
                                                                      double band, const int* __restrict__ chunk_base,
                                                                      float4* __restrict__ out) {
  pdl_entry();
  __shared__ int wc[kGroundChunk / 32];
  const int i = blockIdx.x * kGroundChunk + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool keep = false;
  float x = 0, y = 0, z = 0;
  if (i < n) {
    const float* p = in + (size_t)i * stride_f;
    x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
    keep = ground_pred(mode, x, y, z, z_min, z_max, coeff, band);
  }
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) wc[warp] = __popc(b);
  __syncthreads();
  if (keep) {
    int wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += wc[w];
    out[chunk_base[blockIdx.x] + wbase + __popc(b & ((1u << lane) - 1u))] = make_float4(x, y, z, 0.f);
  }
}

// SampleConsensusModelPlane::computeModelCoefficients for every sampled triple (float, left to right, no FMA)
__global__ void ground_models_kernel(const float4* __restrict__ scr, const int* __restrict__ triples, GroundModels* __restrict__ gm) {
  pdl_entry();
  const int h = threadIdx.x;
  if (h >= kGroundHyp) return;
  const float4 p0 = scr[triples[3 * h]], p1 = scr[triples[3 * h + 1]], p2 = scr[triples[3 * h + 2]];
  const float a0 = __fsub_rn(p1.x, p0.x), a1 = __fsub_rn(p1.y, p0.y), a2 = __fsub_rn(p1.z, p0.z);
  const float b0 = __fsub_rn(p2.x, p0.x), b1 = __fsub_rn(p2.y, p0.y), b2 = __fsub_rn(p2.z, p0.z);
  const float r0 = __fdiv_rn(a0, b0), r1 = __fdiv_rn(a1, b1), r2 = __fdiv_rn(a2, b2);
  bool ok = !(r0 == r1 && r2 == r1);  // collinear samples
  float n0 = __fsub_rn(__fmul_rn(a1, b2), __fmul_rn(a2, b1));
  float n1 = __fsub_rn(__fmul_rn(a2, b0), __fmul_rn(a0, b2));
  float n2 = __fsub_rn(__fmul_rn(a0, b1), __fmul_rn(a1, b0));
  const float nn = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(n0, n0), __fmul_rn(n1, n1)), __fmul_rn(n2, n2)));
  n0 = __fdiv_rn(n0, nn), n1 = __fdiv_rn(n1, nn), n2 = __fdiv_rn(n2, nn);
  const float d = __fmul_rn(-1.0f, __fadd_rn(__fadd_rn(__fmul_rn(n0, p0.x), __fmul_rn(n1, p0.y)), __fmul_rn(n2, p0.z)));
  ok = ok && isfinite(n0) && isfinite(n1) && isfinite(n2);
  gm->co[h][0] = n0, gm->co[h][1] = n1, gm->co[h][2] = n2, gm->co[h][3] = d;
  gm->valid[h] = ok ? 1 : 0;
}

// countWithinDistance of all hypotheses at once: every block takes a slice of the screened cloud, the planes sit in
// shared memory, counts go through warp ballots and one atomicAdd per (warp, hypothesis)
__global__ void __launch_bounds__(256) ground_score_kernel(const float4* __restrict__ scr, int m, const GroundModels* __restrict__ gm,
                                                           float thr, int* __restrict__ counts) {
  pdl_entry();
  __shared__ float co[kGroundHyp][4];
  __shared__ int cnt[kGroundHyp];
  for (int t = threadIdx.x; t < kGroundHyp * 4; t += blockDim.x) (&co[0][0])[t] = (&gm->co[0][0])[t];
  if (threadIdx.x < kGroundHyp) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  int mine[2] = {0, 0};  // lane L accumulates the warp totals of hypotheses L and L + 32
  for (int i0 = blockIdx.x * blockDim.x; i0 < m; i0 += gridDim.x * blockDim.x) {
    const int i = i0 + threadIdx.x;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool in = i < m;
    if (in) p = scr[i];
#pragma unroll 4
    for (int h = 0; h < kGroundHyp; ++h) {
      const bool hit = in && fabsf(plane_dist_f(co[h], p.x, p.y, p.z)) < thr;
      const int c = __popc(__ballot_sync(0xffffffffu, hit));
      if (lane == (h & 31)) mine[h >> 5] += c;
    }
  }
  atomicAdd(&cnt[lane], mine[0]);
  atomicAdd(&cnt[lane + 32], mine[1]);
  __syncthreads();
  if (threadIdx.x < kGroundHyp && cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], cnt[threadIdx.x]);
}

// optimizeModelCoefficients: PCA of the winner's inliers.  Pass 1: per-block fp64 sums (x, y, z, xx, xy, xz, yy, yz, zz, n)
// in a fixed order;  pass 2 (one block): ordered combine, covariance, 3x3 Jacobi, smallest eigenvector oriented upward,
// float coefficients and the acceptance flag n.z > cos(max_angle).
constexpr int kRefitBlocks = 64;
__global__ void __launch_bounds__(256) ground_refit_sums_kernel(const float4* __restrict__ scr, int m, const GroundModels* __restrict__ gm,
                                                                int best, float thr, double* __restrict__ partial) {
  pdl_entry();
  __shared__ double red[8][10];
  double a[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) a[k] = 0.0;
  float co[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) co[k] = gm->co[best][k];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const float4 p = scr[i];
    if (fabsf(plane_dist_f(co, p.x, p.y, p.z)) < thr) {
      const double x = p.x, y = p.y, z = p.z;
      a[0] += x, a[1] += y, a[2] += z;
      a[3] += x * x, a[4] += x * y, a[5] += x * z, a[6] += y * y, a[7] += y * z, a[8] += z * z;
      a[9] += 1.0;
    }
  }
#pragma unroll
  for (int k = 0; k < 10; ++k) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) a[k] += __shfl_xor_sync(0xffffffffu, a[k], off);
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 10; ++k) red[threadIdx.x >> 5][k] = a[k];
  }
  __syncthreads();
  if (threadIdx.x < 10) {
    double v = 0;
    for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    partial[blockIdx.x * 10 + threadIdx.x] = v;
  }
}

__device__ __forceinline__ void jacobi_rot3(double& app, double& aqq, double& apq, double& arp, double& arq, double (&V)[3][3], int p,
                                            int q) {
  if (apq == 0.0) return;
  const double h = aqq - app;
  const double t = (h >= 0.0 ? 2.0 : -2.0) * apq / (fabs(h) + sqrt(h * h + 4.0 * apq * apq));
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
  app -= t * apq, aqq += t * apq, apq = 0.0;
  const double x = arp, y = arq;
  arp = c * x - s * y, arq = s * x + c * y;
  for (int r = 0; r < 3; ++r) {
    const double vx = V[r][p], vy = V[r][q];
    V[r][p] = c * vx - s * vy, V[r][q] = s * vx + c * vy;
  }
}

__global__ void ground_refit_kernel(const double* __restrict__ partial, const GroundModels* __restrict__ gm, int best, double cos_max,
                                    float* __restrict__ coeff /* a b c d accepted */) {
  pdl_entry();
  if (threadIdx.x != 0) return;
  double s[10];
  for (int k = 0; k < 10; ++k) {
    double v = 0;
    for (int b = 0; b < kRefitBlocks; ++b) v += partial[b * 10 + k];
    s[k] = v;
  }
  float co[4] = {gm->co[best][0], gm->co[best][1], gm->co[best][2], gm->co[best][3]};
  const double n = s[9];
  if (n > 3.0) {
    const double cx = s[0] / n, cy = s[1] / n, cz = s[2] / n;
    double a00 = s[3] / n - cx * cx, a01 = s[4] / n - cx * cy, a02 = s[5] / n - cx * cz;
    double a11 = s[6] / n - cy * cy, a12 = s[7] / n - cy * cz, a22 = s[8] / n - cz * cz;
    double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 40; ++sweep) {
      const double off = a01 * a01 + a02 * a02 + a12 * a12, dg = a00 * a00 + a11 * a11 + a22 * a22;
      if (off <= 1e-34 * dg || off == 0.0) break;
      jacobi_rot3(a00, a11, a01, a02, a12, V, 0, 1);
      jacobi_rot3(a00, a22, a02, a01, a12, V, 0, 2);
      jacobi_rot3(a11, a22, a12, a01, a02, V, 1, 2);
    }
    int k = 0;
    double lmin = a00;
    if (a11 < lmin) lmin = a11, k = 1;
    if (a22 < lmin) lmin = a22, k = 2;
    double nx = V[0][k], ny = V[1][k], nz = V[2][k];
    const double nn = sqrt(nx * nx + ny * ny + nz * nz);
    nx /= nn, ny /= nn, nz /= nn;
    if (nz < 0) nx = -nx, ny = -ny, nz = -nz;
    co[0] = (float)nx, co[1] = (float)ny, co[2] = (float)nz, co[3] = (float)(-(nx * cx + ny * cy + nz * cz));
  }
  coeff[0] = co[0], coeff[1] = co[1], coeff[2] = co[2], coeff[3] = co[3];
  coeff[4] = ((double)co[2] > cos_max) ? 1.f : 0.f;
}

struct GroundBufs {
  DevBuf<float> raw, coeff;
  DevBuf<float4> scr, out;
  DevBuf<int> chunk_cnt, chunk_base, totals, triples, counts;
  DevBuf<GroundModels> models;
  DevBuf<double> partial;
};

}  // namespace ilsm

using namespace ilsm;

struct ilsm_ground {
  Ctx* ctx;
  GroundBufs b;
};

static uint32_t lcg_next(uint32_t& x) {
  x = x * 1664525u + 1013904223u;
  return x >> 8;
}

extern "C" {

ILSM_API void ilsm_ground_opts_default(ilsm_ground_opts* o) {
  if (!o) return;
  o->z_min = -2.0, o->z_max = -0.45, o->distance_threshold = 0.01, o->probability = 0.99;
  o->max_iterations = 50, o->seed = 1;
  o->band = 0.03, o->max_angle_deg = 15.0;
}

ILSM_API int ilsm_ground_create(ilsm_ctx* ctx, ilsm_ground** out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "ground_create: null argument");
  ilsm_ground* g = new (std::nothrow) ilsm_ground();
  if (!g) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  g->ctx = &ctx->c;
  *out = g;
  return ILSM_OK;
}

ILSM_API void ilsm_ground_destroy(ilsm_ground* g) {
  if (!g) return;
  std::lock_guard<std::mutex> lk(g->ctx->mu);
  cudaSetDevice(g->ctx->device);
  cudaStreamSynchronize(g->ctx->stream);
  delete g;
}

}  // extern "C"

namespace ilsm {
// The extraction with the frame taken from the host (from_host) or already on the device; the ground points stay on
// the device in g->b.out (packed xyz0, *n_out of them).  Caller holds the context mutex.
int ground_extract_core(ilsm_ground* g, const float* xyz, bool from_host, int n, int stride_bytes, const ilsm_ground_opts& o,
                        int* n_out, float coeff_abcd[4], ilsm_ground_info* info) {
  *n_out = 0;
  if (info) memset(info, 0, sizeof(*info)), info->best_hypothesis = -1;
  if (coeff_abcd) coeff_abcd[0] = coeff_abcd[1] = coeff_abcd[2] = coeff_abcd[3] = 0.f;
  if (n == 0) return ILSM_OK;
  Ctx& c = *g->ctx;
  GroundBufs& b = g->b;
  const int chunks = (n + kGroundChunk - 1) / kGroundChunk;
  const size_t bytes = (size_t)n * stride_bytes;
  int rc;
  if ((rc = b.raw.reserve(bytes / 4 + 4)) || (rc = b.coeff.reserve(8)) || (rc = b.scr.reserve(n + 4)) || (rc = b.out.reserve(n + 4)) ||
      (rc = b.chunk_cnt.reserve(chunks + 4)) || (rc = b.chunk_base.reserve(chunks + 4)) || (rc = b.totals.reserve(4)) ||
      (rc = b.triples.reserve(3 * kGroundHyp)) || (rc = b.counts.reserve(kGroundHyp)) || (rc = b.models.reserve(1)) ||
      (rc = b.partial.reserve(kRefitBlocks * 10)))
    return rc;
  cudaStream_t s = c.stream;
  const int sf = stride_bytes / 4;
  ILSM_CUDA(cudaMemcpyAsync(b.raw.p, xyz, bytes, from_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  // 1. screening: stable compaction of the z band
  ILSM_CUDA(launch_pdl(ground_count_kernel, dim3(chunks), dim3(kGroundChunk), 0, s, (const float*)b.raw.p, n, sf, 0, o.z_min, o.z_max,
                       (const float*)nullptr, o.band, b.chunk_cnt.p));
  ILSM_CUDA(launch_pdl(ground_scan_kernel, dim3(1), dim3(1024), 0, s, (const int*)b.chunk_cnt.p, chunks, b.chunk_base.p, b.totals.p));
  ILSM_CUDA(launch_pdl(ground_scatter_kernel, dim3(chunks), dim3(kGroundChunk), 0, s, (const float*)b.raw.p, n, sf, 0, o.z_min, o.z_max,
                       (const float*)nullptr, o.band, (const int*)b.chunk_base.p, b.scr.p));
  count_launches(3);
  int* pin = reinterpret_cast<int*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, b.totals.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaStreamSynchronize(s));
  const int m = pin[0];
  if (info) info->n_band = m;
  if (m < 3) return ILSM_OK;
  // 2. hypotheses from the declared sampler, all scored at once
  int* tri = pin + 16;
  uint32_t x = (uint32_t)o.seed;
  for (int h = 0; h < kGroundHyp; ++h) {
    int a = (int)(lcg_next(x) % (uint32_t)m), bb = (int)(lcg_next(x) % (uint32_t)m);
    while (bb == a) bb = (int)(lcg_next(x) % (uint32_t)m);
    int cc = (int)(lcg_next(x) % (uint32_t)m);
    while (cc == a || cc == bb) cc = (int)(lcg_next(x) % (uint32_t)m);
    tri[3 * h] = a, tri[3 * h + 1] = bb, tri[3 * h + 2] = cc;
  }
  ILSM_CUDA(cudaMemcpyAsync(b.triples.p, tri, 3 * kGroundHyp * sizeof(int), cudaMemcpyHostToDevice, s));
  ILSM_CUDA(cudaMemsetAsync(b.counts.p, 0, kGroundHyp * sizeof(int), s));
  ILSM_CUDA(launch_pdl(ground_models_kernel, dim3(1), dim3(kGroundHyp), 0, s, (const float4*)b.scr.p, (const int*)b.triples.p, b.models.p));
  int sblocks = (m + 255) / 256;
  if (sblocks > c.sm_count * 4) sblocks = c.sm_count * 4;
  ILSM_CUDA(launch_pdl(ground_score_kernel, dim3(sblocks), dim3(256), 0, s, (const float4*)b.scr.p, m, (const GroundModels*)b.models.p,
                       (float)o.distance_threshold, b.counts.p));
  count_launches(2);
  int* h_counts = pin + 16 + 3 * kGroundHyp;
  int* h_valid = h_counts + kGroundHyp;
  ILSM_CUDA(cudaMemcpyAsync(h_counts, b.counts.p, kGroundHyp * sizeof(int), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaMemcpyAsync(h_valid, b.models.p->valid, kGroundHyp * sizeof(int), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaStreamSynchronize(s));
  // 3. replay of pcl::RandomSampleConsensus::computeModel over the precomputed counts
  double k = 1.0;
  int it = 0, skipped = 0, h = 0, n_best = 0, best = -1;
  const double log_p = log(1.0 - o.probability), eps = 2.220446049250313e-16;
  while (it < k && skipped < o.max_iterations * 10 && h < kGroundHyp) {
    if (!h_valid[h]) {
      ++skipped, ++h;
      continue;
    }
    if (h_counts[h] > n_best) {
      n_best = h_counts[h], best = h;
      const double w = (double)n_best / (double)m;
      double p_no = 1.0 - w * w * w;
      p_no = p_no < eps ? eps : (p_no > 1.0 - eps ? 1.0 - eps : p_no);
      k = log_p / log(p_no);
    }
    ++it, ++h;
    if (it > o.max_iterations) break;
  }
  if (info) info->best_hypothesis = best, info->n_best_inliers = n_best, info->iterations = it;
  if (best < 0) return ILSM_OK;
  // 4. refit + acceptance on the device, 5. final selection (stable compaction of the whole input)
  ILSM_CUDA(launch_pdl(ground_refit_sums_kernel, dim3(kRefitBlocks), dim3(256), 0, s, (const float4*)b.scr.p, m,
                       (const GroundModels*)b.models.p, best, (float)o.distance_threshold, b.partial.p));
  ILSM_CUDA(launch_pdl(ground_refit_kernel, dim3(1), dim3(32), 0, s, (const double*)b.partial.p, (const GroundModels*)b.models.p, best,
                       cos(o.max_angle_deg * 3.14159265358979323846 / 180.0), b.coeff.p));
  ILSM_CUDA(launch_pdl(ground_count_kernel, dim3(chunks), dim3(kGroundChunk), 0, s, (const float*)b.raw.p, n, sf, 1, o.z_min, o.z_max,
                       (const float*)b.coeff.p, o.band, b.chunk_cnt.p));
  ILSM_CUDA(launch_pdl(ground_scan_kernel, dim3(1), dim3(1024), 0, s, (const int*)b.chunk_cnt.p, chunks, b.chunk_base.p, b.totals.p + 1));
  ILSM_CUDA(launch_pdl(ground_scatter_kernel, dim3(chunks), dim3(kGroundChunk), 0, s, (const float*)b.raw.p, n, sf, 1, o.z_min, o.z_max,
                       (const float*)b.coeff.p, o.band, (const int*)b.chunk_base.p, b.out.p));
  count_launches(5);
  float* pin_f = reinterpret_cast<float*>(pin + 512);
  ILSM_CUDA(cudaMemcpyAsync(pin, b.totals.p + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaMemcpyAsync(pin_f, b.coeff.p, 5 * sizeof(float), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaStreamSynchronize(s));
  const int ng = pin[0];
  *n_out = ng;
  if (coeff_abcd) for (int i = 0; i < 4; ++i) coeff_abcd[i] = pin_f[i];
  if (info) info->accepted = pin_f[4] != 0.f;
  return check_launch("ground_extract");
}

const float4* ground_points_dev(ilsm_ground* g) { return g->b.out.p; }
}  // namespace ilsm

extern "C" {

ILSM_API int ilsm_ground_extract(ilsm_ground* g, const float* xyz, int n, int stride_bytes, const ilsm_ground_opts* opts,
                                 float* out_xyz, int capacity, int* n_out, float coeff_abcd[4], ilsm_ground_info* info) {
  if (!g || !n_out || (n > 0 && !xyz)) return fail(ILSM_ERR_INVALID_ARG, "ground_extract: null argument");
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "ground_extract: bad n/stride");
  ilsm_ground_opts o;
  if (opts) o = *opts; else ilsm_ground_opts_default(&o);
  if (o.max_iterations < 1 || o.max_iterations > 62) return fail(ILSM_ERR_INVALID_ARG, "ground_extract: max_iterations must be in [1, 62]");
  Ctx& c = *g->ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  int rc = ground_extract_core(g, xyz, true, n, stride_bytes, o, n_out, coeff_abcd, info);
  if (rc) return rc;
  const int ng = *n_out;
  if (ng > 0 && out_xyz) {
    const int kcp = ng < capacity ? ng : capacity;
    // pcl::PointXYZ layout: 16-byte points (x, y, z, pad)
    ILSM_CUDA(cudaMemcpyAsync(out_xyz, g->b.out.p, (size_t)kcp * 16, cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
  }
  return ILSM_OK;
}

}  // extern "C"
