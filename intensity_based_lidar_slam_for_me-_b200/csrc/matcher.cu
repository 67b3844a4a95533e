// matcher.cu -- intensity-image feature back end: brute-force Hamming matching of ORB descriptors with cross check,
// selection of the best fraction, and the 3D-3D alignment of the matched points.
//
// Replaces cv::BFMatcher(cv::NORM_HAMMING, true).match(cur, prev) + std::sort + "first 30 %"
// (intensity_feature_tracker.cpp:631-648, 678-686) and feeds p2p_calculateRandT (:880-928), whose Ceres problem
// (front_end_residual blocks, lidarFeaturePointsFunction.hpp:21-58) runs on the same device-side LM solver as the
// LiDAR factors (factor type 3).
//
// The distance matrix is never materialised: one warp per query descriptor streams the train set (32 B per
// descriptor, coalesced) with the query held in registers, 8 x popc(xor) per pair, and keeps the packed minimum
// (distance << 32 | index), i.e. OpenCV's batchDistance semantics: first minimum wins.  Integer work, bit-exact.
#include "ilsm_host.hpp"
#include "ilsm_voxel.cuh"

namespace ilsm {

constexpr int kDescWords = 8;  // 256-bit ORB descriptor

__global__ void __launch_bounds__(128) hamming_argmin_kernel(const uint32_t* __restrict__ q, int nq, const uint32_t* __restrict__ t,
                                                             int nt, int* __restrict__ best_idx, int* __restrict__ best_dist) {
  pdl_entry();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 4 + warp;
  if (i >= nq) return;
  uint32_t qa[kDescWords];
  {
    const uint4* qp = reinterpret_cast<const uint4*>(q + (size_t)i * kDescWords);
    const uint4 a = __ldg(qp), b = __ldg(qp + 1);
    qa[0] = a.x, qa[1] = a.y, qa[2] = a.z, qa[3] = a.w, qa[4] = b.x, qa[5] = b.y, qa[6] = b.z, qa[7] = b.w;
  }
  u64 best = ~0ull;
  for (int j = lane; j < nt; j += 32) {
    const uint4* tp = reinterpret_cast<const uint4*>(t + (size_t)j * kDescWords);
    const uint4 a = __ldg(tp), b = __ldg(tp + 1);
    const int d = __popc(qa[0] ^ a.x) + __popc(qa[1] ^ a.y) + __popc(qa[2] ^ a.z) + __popc(qa[3] ^ a.w) +
                  __popc(qa[4] ^ b.x) + __popc(qa[5] ^ b.y) + __popc(qa[6] ^ b.z) + __popc(qa[7] ^ b.w);
    const u64 key = ((u64)(uint32_t)d << 32) | (uint32_t)j;
    best = key < best ? key : best;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const u64 o = __shfl_xor_sync(0xffffffffu, best, off);
    best = o < best ? o : best;
  }
  if (lane == 0) {
    best_idx[i] = nt > 0 ? (int)(uint32_t)best : -1;
    best_dist[i] = nt > 0 ? (int)(best >> 32) : 0;
  }
}

// cross check, stable compaction in query order (DMatch list of BFMatcher::match), then the good matches: sort by
// (distance, queryIdx) and keep the first ceil(n * fraction).  One block; n_q <= kVoxelBlockMax.
__global__ void __launch_bounds__(1024) match_finalize_kernel(int nq, const int* __restrict__ best_t, const int* __restrict__ dist_q,
                                                              const int* __restrict__ best_q, int cross_check, double fraction,
                                                              ilsm_dmatch* __restrict__ matches, ilsm_dmatch* __restrict__ good,
                                                              int* __restrict__ counts) {
  pdl_entry();
  extern __shared__ u64 keys[];
  __shared__ int wc[32];
  __shared__ int s_base;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i0 = 0; i0 < nq; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    bool keep = false;
    int tj = -1;
    if (i < nq) {
      tj = best_t[i];
      keep = tj >= 0 && (!cross_check || best_q[tj] == i);
    }
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wc[warp] = __popc(b);
    __syncthreads();
    int wbase = 0, tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      if (w < warp) wbase += wc[w];
      tot += wc[w];
    }
    const int base = s_base;
    if (keep) {
      const int pos = base + wbase + __popc(b & ((1u << lane) - 1u));
      ilsm_dmatch m;
      m.queryIdx = i, m.trainIdx = tj, m.imgIdx = 0, m.distance = (float)dist_q[i];
      matches[pos] = m;
      keys[pos] = ((u64)(uint32_t)dist_q[i] << 32) | (uint32_t)i;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base = base + tot;
    __syncthreads();
  }
  const int n = s_base;
  int P = 1;
  while (P < n) P <<= 1;
  for (int t = n + threadIdx.x; t < P; t += blockDim.x) keys[t] = ~0ull;
  __syncthreads();
  if (n > 1) bitonic_sort_smem(keys, P);
  const int n_good = (int)ceil((double)n * fraction);  // for (i = 0; i < matches.size() * fraction; ++i)
  for (int t = threadIdx.x; t < n_good && t < n; t += blockDim.x) {
    const int i = (int)(uint32_t)keys[t];
    ilsm_dmatch m;
    m.queryIdx = i, m.trainIdx = best_t[i], m.imgIdx = 0, m.distance = (float)dist_q[i];
    good[t] = m;
  }
  if (threadIdx.x == 0) counts[0] = n, counts[1] = n_good < n ? n_good : n;
}

// point pairs -> front_end_residual factors (type 3: p = source point, a = destination point)
__global__ void align_factors_kernel(const float* __restrict__ src, const float* __restrict__ dst, int n, int stride_f, int* type,
                                     float4* p, double4* a, double4* b) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* s = src + (size_t)i * stride_f;
  const float* d = dst + (size_t)i * stride_f;
  type[i] = 3;
  p[i] = make_float4(__ldg(s), __ldg(s + 1), __ldg(s + 2), 0.f);
  a[i] = make_double4((double)__ldg(d), (double)__ldg(d + 1), (double)__ldg(d + 2), 0.0);
  b[i] = make_double4(0, 0, 0, 0);
}

}  // namespace ilsm

using namespace ilsm;

extern "C" {

ILSM_API int ilsm_orb_match(ilsm_ctx* ctx, const uint8_t* cur_desc, int n_cur, const uint8_t* prev_desc, int n_prev, int desc_bytes,
                            int cross_check, double keep_fraction, ilsm_dmatch* matches, int* n_matches, ilsm_dmatch* good,
                            int* n_good) {
  if (!ctx || !n_matches || !n_good || (n_cur > 0 && (!cur_desc || !matches || !good)) || (n_prev > 0 && !prev_desc))
    return fail(ILSM_ERR_INVALID_ARG, "orb_match: null argument");
  if (desc_bytes != 32) return fail(ILSM_ERR_INVALID_ARG, "orb_match: 32-byte (256-bit ORB) descriptors only");
  if (n_cur < 0 || n_prev < 0 || n_cur > kVoxelBlockMax || !(keep_fraction >= 0.0 && keep_fraction <= 1.0))
    return fail(ILSM_ERR_INVALID_ARG, "orb_match: bad sizes (at most 16384 query descriptors) or fraction");
  *n_matches = 0, *n_good = 0;
  if (n_cur == 0 || n_prev == 0) return ILSM_OK;
  Ctx& c = ctx->c;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  // scratch layout in out_idx: cur desc | prev desc | best_t[n_cur] dist_q[n_cur] best_q[n_prev] dist_t[n_prev] counts[4]
  //                            | matches | good
  const size_t wq = (size_t)n_cur * 8, wt = (size_t)n_prev * 8;
  const size_t ints = wq + wt + 2 * (size_t)n_cur + 2 * (size_t)n_prev + 4;
  const size_t total = ints + 2 * (size_t)n_cur * 4 + 16;
  int rc;
  if ((rc = c.out_idx.reserve(total))) return rc;
  uint32_t* d_q = reinterpret_cast<uint32_t*>(c.out_idx.p);
  uint32_t* d_t = d_q + wq;
  int* best_t = reinterpret_cast<int*>(d_t + wt);
  int* dist_q = best_t + n_cur;
  int* best_q = dist_q + n_cur;
  int* dist_t = best_q + n_prev;
  int* counts = dist_t + n_prev;
  ilsm_dmatch* d_matches = reinterpret_cast<ilsm_dmatch*>(reinterpret_cast<uintptr_t>(counts + 4 + 3) & ~(uintptr_t)15);
  ilsm_dmatch* d_good = d_matches + n_cur;
  ILSM_CUDA(cudaMemcpyAsync(d_q, cur_desc, wq * 4, cudaMemcpyHostToDevice, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(d_t, prev_desc, wt * 4, cudaMemcpyHostToDevice, c.stream));
  ILSM_CUDA(launch_pdl(hamming_argmin_kernel, dim3((n_cur + 3) / 4), dim3(128), 0, c.stream, d_q, n_cur, d_t, n_prev, best_t, dist_q));
  if (cross_check) ILSM_CUDA(launch_pdl(hamming_argmin_kernel, dim3((n_prev + 3) / 4), dim3(128), 0, c.stream, d_t, n_prev, d_q, n_cur, best_q, dist_t));
  int P = 1;
  while (P < n_cur) P <<= 1;
  const size_t smem = (size_t)P * sizeof(u64);
  ILSM_CUDA(cudaFuncSetAttribute(match_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kVoxelBlockMax * sizeof(u64))));
  ILSM_CUDA(launch_pdl(match_finalize_kernel, dim3(1), dim3(1024), smem, c.stream, n_cur, best_t, dist_q, best_q, cross_check ? 1 : 0, keep_fraction, d_matches, d_good, counts));
  count_launches(cross_check ? 3 : 2);
  if ((rc = check_launch("orb_match"))) return rc;
  int* pin = reinterpret_cast<int*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, counts, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  *n_matches = pin[0], *n_good = pin[1];
  if (pin[0] > 0) ILSM_CUDA(cudaMemcpyAsync(matches, d_matches, (size_t)pin[0] * sizeof(ilsm_dmatch), cudaMemcpyDeviceToHost, c.stream));
  if (pin[1] > 0) ILSM_CUDA(cudaMemcpyAsync(good, d_good, (size_t)pin[1] * sizeof(ilsm_dmatch), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_align_points(ilsm_ctx* ctx, const float* src_xyz, const float* dst_xyz, int n, int stride_bytes, double q[4],
                               double t[3], int max_num_iterations, double huber_a, ilsm_solve_summary* summary) {
  if (!ctx || !q || !t || (n > 0 && (!src_xyz || !dst_xyz))) return fail(ILSM_ERR_INVALID_ARG, "align_points: null argument");
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "align_points: bad n/stride");
  if (max_num_iterations < 0) max_num_iterations = 0;
  if (max_num_iterations > 200) max_num_iterations = 200;
  Ctx& c = ctx->c;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  int rc;
  FactorBufs& f = c.fac;
  const size_t bytes = (size_t)n * stride_bytes;
  if ((rc = f.type.reserve(n + 4)) || (rc = f.p.reserve(n + 1)) || (rc = f.a.reserve(n + 1)) || (rc = f.b.reserve(n + 1)) ||
      (rc = c.stack_raw.reserve(2 * (bytes / 4) + 16)))
    return rc;
  f.n = n, f.nc = n;
  float* d_src = c.stack_raw.p;
  float* d_dst = c.stack_raw.p + bytes / 4;
  if (n > 0) {
    ILSM_CUDA(cudaMemcpyAsync(d_src, src_xyz, bytes, cudaMemcpyHostToDevice, c.stream));
    ILSM_CUDA(cudaMemcpyAsync(d_dst, dst_xyz, bytes, cudaMemcpyHostToDevice, c.stream));
    ILSM_CUDA(launch_pdl(align_factors_kernel, dim3((n + 255) / 256), dim3(256), 0, c.stream, d_src, d_dst, n, stride_bytes / 4, f.type.p, f.p.p, f.a.p, f.b.p));
    count_launches(1);
  }
  ilsm_reg_report rep;
  if ((rc = c.upload_pose(q, t, c.stream)) || (rc = c.solve_launch(max_num_iterations, huber_a, 0)) || (rc = c.lm_finish(q, t, &rep, 1)))
    return rc;
  if (summary) *summary = rep.pass[0];
  return ILSM_OK;
}

}  // extern "C"
