// icp.cu -- K6: loop-closure verification, point-to-point ICP (pcl::IterativeClosestPoint, PCL 1.10, restated in the
// CPU oracle, DESIGN section 2) for a batch of (source, target) pairs in ONE launch.
//
//   icp_cluster_kernel : one thread-block cluster per pair runs the whole do-while loop of IterativeClosestPoint::
//                        computeTransformation and the final getFitnessScore pass.  Per pass every CTA takes 256-point
//                        tiles of the source (tile i -> CTA i % cluster size), each warp 32 points of a tile: pose
//                        transform (double math, float store), exact 1-NN in the target's voxel hash (knn_search<1>), the
//                        correspondence gate, and the tile's fp64 sums about the pair origin o (the guess translation):
//                        count, sum d2, sum (p - o), sum (q - o), sum (p - o)(q - o)^T.  The sums of a tile are a fixed
//                        tree (lane-pair butterfly inside a warp, then warps 0..7 in order); the tiles are summed in tile
//                        order after one cluster barrier by EVERY CTA, which then advances an identical copy of the state
//                        machine (Horn's quaternion solve, DefaultConvergenceCriteria): nothing is broadcast, and the
//                        result depends neither on the cluster size nor on the other pairs of the batch.
// The source has no size limit: no per-point state survives a pass, the tile partials live in HBM (double-buffered by
// pass parity, which the barrier of the pass in between protects).
#include <float.h>
#include <math.h>
#include <stdio.h>

#include "ilsm_host.hpp"

namespace ilsm {
namespace {

constexpr int kIcpThreads = 256, kIcpWarps = kIcpThreads / 32;
constexpr int kIcpTile = kIcpThreads;  // source points per tile: one per thread
constexpr int kIcpSums = 17;           // count, sum d2, sum (p - o) [3], sum (q - o) [3], sum (p - o)(q - o)^T [9]
constexpr int kIcpCluster = 8, kIcpClusterWide = 16;

struct IcpPair {
  GridView g;
  double guess[7];  // qx qy qz qw tx ty tz
  int src_begin, n_src, tile_base, pad;
};

struct IcpParams {
  const float* src;
  int stride_f, max_iter, total_tiles, pad;
  float knn_d2, fit_knn_d2;  // k-NN cut-offs, rounded up to float (0: none)
  double max_corr2, eps_t, rot_thr, eps_fit, fit_range;
};

struct IcpState {
  double q[4], t[3];  // accumulated pose P
  double prev_mse, mse;
  int iter, state, n_corr, done;
};

__device__ __forceinline__ uint32_t icp_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void icp_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Largest-eigenvalue eigenvector of Horn's symmetric 4x4 matrix N by cyclic Jacobi (the rotation of eig3 in the oracle),
// IEEE sqrt / division; returns the unit quaternion (x, y, z, w) with w >= 0.
__device__ void horn_quat(const double S[3][3], double qo[4]) {
  const double sxx = S[0][0], sxy = S[0][1], sxz = S[0][2], syx = S[1][0], syy = S[1][1], syz = S[1][2], szx = S[2][0],
               szy = S[2][1], szz = S[2][2];
  double a[4][4] = {{sxx + syy + szz, syz - szy, szx - sxz, sxy - syx},
                    {syz - szy, sxx - syy - szz, sxy + syx, szx + sxz},
                    {szx - sxz, sxy + syx, -sxx + syy - szz, syz + szy},
                    {sxy - syx, szx + sxz, syz + szy, -sxx - syy + szz}};
  double v[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
  for (int sweep = 0; sweep < 32; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int p = 0; p < 4; ++p) {
      diag = diag + a[p][p] * a[p][p];
      for (int q = p + 1; q < 4; ++q) off = off + a[p][q] * a[p][q];
    }
    if (off == 0.0 || off <= 1e-36 * diag) break;
    for (int p = 0; p < 3; ++p)
      for (int q = p + 1; q < 4; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 4; ++k) {
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 4; ++k) {
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 4; ++k) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq;
          v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int best = 0;
  for (int k = 1; k < 4; ++k)
    if (a[k][k] > a[best][best]) best = k;
  double w = v[0][best], x = v[1][best], y = v[2][best], z = v[3][best];
  const double nrm = sqrt(w * w + x * x + y * y + z * z);
  w = w / nrm, x = x / nrm, y = y / nrm, z = z / nrm;
  if (w < 0) w = -w, x = -x, y = -y, z = -z;
  qo[0] = x, qo[1] = y, qo[2] = z, qo[3] = w;
}

__device__ void quat_mat(const double q[4], double R[3][3]) {
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  R[0][0] = 1.0 - 2.0 * (y * y + z * z), R[0][1] = 2.0 * (x * y - w * z), R[0][2] = 2.0 * (x * z + w * y);
  R[1][0] = 2.0 * (x * y + w * z), R[1][1] = 1.0 - 2.0 * (x * x + z * z), R[1][2] = 2.0 * (y * z - w * x);
  R[2][0] = 2.0 * (x * z - w * y), R[2][1] = 2.0 * (y * z + w * x), R[2][2] = 1.0 - 2.0 * (x * x + y * y);
}

// One iteration's closed-form fit and DefaultConvergenceCriteria::hasConverged (max_iterations_similar_transforms 0,
// failure_after_max_iter false) on the pass's sums S; o = the pair origin.
__device__ void icp_advance(IcpState& s, const double* S, const IcpParams& prm, const double o[3]) {
  const double n = S[0];
  s.n_corr = (int)n;
  s.mse = n > 0 ? S[1] / n : DBL_MAX;
  if (n < 3) {
    s.state = ILSM_ICP_NO_CORRESPONDENCES, s.done = 1;
    return;
  }
  double H[3][3];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) H[a][b] = S[8 + 3 * a + b] - S[2 + a] * S[5 + b] / n;
  double qi[4], R[3][3];
  horn_quat(H, qi);
  quat_mat(qi, R);
  double cp[3], cq[3], ti[3];
  for (int a = 0; a < 3; ++a) cp[a] = S[2 + a] / n + o[a], cq[a] = S[5 + a] / n + o[a];
  for (int a = 0; a < 3; ++a) ti[a] = cq[a] - ((R[a][0] * cp[0] + R[a][1] * cp[1]) + R[a][2] * cp[2]);
  // P <- (R, t) o P
  const double* b = s.q;
  double qn[4] = {qi[3] * b[0] + qi[0] * b[3] + qi[1] * b[2] - qi[2] * b[1],
                  qi[3] * b[1] + qi[1] * b[3] + qi[2] * b[0] - qi[0] * b[2],
                  qi[3] * b[2] + qi[2] * b[3] + qi[0] * b[1] - qi[1] * b[0],
                  qi[3] * b[3] - qi[0] * b[0] - qi[1] * b[1] - qi[2] * b[2]};
  const double qnn = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
  double tn[3];
  for (int a = 0; a < 3; ++a) tn[a] = ((R[a][0] * s.t[0] + R[a][1] * s.t[1]) + R[a][2] * s.t[2]) + ti[a];
  for (int k = 0; k < 4; ++k) s.q[k] = qn[k] / qnn;
  for (int a = 0; a < 3; ++a) s.t[a] = tn[a];
  ++s.iter;
  if (s.iter >= prm.max_iter) {
    s.state = ILSM_ICP_ITERATIONS, s.done = 1;
    return;
  }
  const double cos_angle = 0.5 * (R[0][0] + R[1][1] + R[2][2] - 1.0);
  const double tr2 = ti[0] * ti[0] + ti[1] * ti[1] + ti[2] * ti[2];
  if (cos_angle >= prm.rot_thr && tr2 <= prm.eps_t) {
    s.state = ILSM_ICP_TRANSFORM, s.done = 1;
    return;
  }
  const double dm = fabs(s.mse - s.prev_mse);
  if (dm < 1e-12) {
    s.state = ILSM_ICP_ABS_MSE, s.done = 1;
    return;
  }
  if (dm / s.prev_mse < prm.eps_fit) {
    s.state = ILSM_ICP_REL_MSE, s.done = 1;
    return;
  }
  s.prev_mse = s.mse;
}

// The sums of one 256-point tile under pose (q, t): correspondence pass (fit = false, all 17) or fitness pass (count and
// sum d2).  Thread 0..16 store the tile's partial to dst.
__device__ void icp_tile(const IcpPair& pp, const IcpParams& prm, const int (&bb)[6], const double q[4], const double t[3],
                         const double o[3], bool fit, int tile, WarpScratch& ws, double (*wsum)[kIcpSums], double* dst) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i = tile * kIcpTile + tid;
  const bool have = i < pp.n_src;
  float px = 0.f, py = 0.f, pz = 0.f;
  if (have) {  // pointAssociateToMap: double math, float store
    const float* s = prm.src + (size_t)(pp.src_begin + i) * prm.stride_f;
    const D3 w = quat_rotate(q, d3((double)s[0], (double)s[1], (double)s[2]));
    px = __double2float_rn(dadd(w.x, t[0])), py = __double2float_rn(dadd(w.y, t[1])), pz = __double2float_rn(dadd(w.z, t[2]));
  }
  const unsigned live = __ballot_sync(0xffffffffu, have);  // a prefix of the warp
  const float max_d2 = fit ? prm.fit_knn_d2 : prm.knn_d2;
  float nx = 0.f, ny = 0.f, nz = 0.f, nd2 = 0.f;
  bool found = false;
#pragma unroll 1
  for (int j = 0; j < 32 && ((live >> j) & 1u); ++j) {
    KnnResult<1, true> res;
    knn_search<1, true>(pp.g, bb, __shfl_sync(0xffffffffu, px, j), __shfl_sync(0xffffffffu, py, j),
                        __shfl_sync(0xffffffffu, pz, j), max_d2, (unsigned)lane, ws, res);
    if (lane == j) {
      found = res.key[0] != kSentinel;
      nd2 = cand_d2(res.key[0]), nx = res.x[0], ny = res.y[0], nz = res.z[0];
    }
  }
  const bool ok = found && (double)nd2 <= (fit ? prm.fit_range : prm.max_corr2);
  double c[kIcpSums];
#pragma unroll
  for (int k = 0; k < kIcpSums; ++k) c[k] = 0.0;
  if (ok) {
    c[0] = 1.0, c[1] = (double)nd2;
    if (!fit) {
      const double dp[3] = {(double)px - o[0], (double)py - o[1], (double)pz - o[2]};
      const double dq[3] = {(double)nx - o[0], (double)ny - o[1], (double)nz - o[2]};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        c[2 + a] = dp[a], c[5 + a] = dq[a];
#pragma unroll
        for (int b = 0; b < 3; ++b) c[8 + 3 * a + b] = dp[a] * dq[b];
      }
    }
  }
  const int nsum = fit ? 2 : kIcpSums;
#pragma unroll
  for (int k = 0; k < kIcpSums; ++k) {
    if (k >= nsum) break;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) c[k] = c[k] + __shfl_xor_sync(0xffffffffu, c[k], off);
    if (lane == 0) wsum[warp][k] = c[k];
  }
  __syncthreads();
  if (tid < kIcpSums) {
    double s = 0.0;
    if (tid < nsum) {
      s = wsum[0][tid];
      for (int w = 1; w < kIcpWarps; ++w) s = s + wsum[w][tid];
    }
    __stcg(dst + tid, s);
  }
  __syncthreads();  // wsum is reused by the next tile
}

template <int kCS>
__global__ void __cluster_dims__(kCS, 1, 1) __launch_bounds__(kIcpThreads, 1)
    icp_cluster_kernel(const IcpPair* __restrict__ pairs, IcpParams prm, double* __restrict__ part,
                       ilsm_icp_result* __restrict__ out) {
  pdl_entry();
  __shared__ WarpScratch ws[kIcpWarps];
  __shared__ double wsum[kIcpWarps][kIcpSums];
  __shared__ double tot[kIcpSums];
  __shared__ IcpState st;
  const int tid = threadIdx.x;
  const int pair = blockIdx.x / kCS;
  const int rank = (int)icp_ctarank();
  const IcpPair pp = pairs[pair];
  int bb[6] = {0, 0, 0, 0, 0, 0};
  if (pp.g.n > 0) load_bbox(pp.g, bb);
  const double o[3] = {pp.guess[4], pp.guess[5], pp.guess[6]};
  const int n_tiles = (pp.n_src + kIcpTile - 1) / kIcpTile;
  if (tid == 0) {
    for (int k = 0; k < 4; ++k) st.q[k] = pp.guess[k];
    for (int k = 0; k < 3; ++k) st.t[k] = pp.guess[4 + k];
    st.prev_mse = DBL_MAX, st.mse = DBL_MAX;
    st.iter = 0, st.state = ILSM_ICP_NOT_CONVERGED, st.n_corr = 0, st.done = 0;
  }
  __syncthreads();
#pragma unroll 1
  for (int pass = 0;; ++pass) {
    const bool fit = st.done != 0;  // the loop has ended: this pass is getFitnessScore's
    const double q[4] = {st.q[0], st.q[1], st.q[2], st.q[3]}, t[3] = {st.t[0], st.t[1], st.t[2]};
    double* buf = part + (size_t)(pass & 1) * prm.total_tiles * kIcpSums + (size_t)pp.tile_base * kIcpSums;
#pragma unroll 1
    for (int tile = rank; tile < n_tiles; tile += kCS)
      icp_tile(pp, prm, bb, q, t, o, fit, tile, ws[tid >> 5], wsum, buf + (size_t)tile * kIcpSums);
    icp_cluster_sync();  // every tile partial of this pass is written
    if (tid < kIcpSums) {
      double s = 0.0;
      for (int tile = 0; tile < n_tiles; ++tile) s = s + __ldcg(buf + (size_t)tile * kIcpSums + tid);
      tot[tid] = s;
    }
    __syncthreads();
    if (fit) {
      if (rank == 0 && tid == 0) {
        ilsm_icp_result r;
        for (int k = 0; k < 4; ++k) r.q_xyzw[k] = st.q[k];
        for (int k = 0; k < 3; ++k) r.t[k] = st.t[k];
        r.fitness = tot[0] > 0 ? tot[1] / tot[0] : DBL_MAX;
        r.mse = st.mse;
        r.iterations = st.iter, r.state = st.state, r.n_correspondences = st.n_corr;
        r.converged = st.state != ILSM_ICP_NOT_CONVERGED && st.state != ILSM_ICP_NO_CORRESPONDENCES;
        out[pair] = r;
      }
      return;
    }
    if (tid == 0) icp_advance(st, tot, prm, o);
    __syncthreads();
  }
}

// float cut-off for knn_search that is never below the double gate d2 (0 = no cut-off)
float knn_cutoff(double d2) {
  if (!(d2 < (double)FLT_MAX)) return 0.f;
  float f = (float)d2;
  if ((double)f < d2) f = nextafterf(f, FLT_MAX);
  return f;
}

}  // namespace

// d_src: the first point of pair 0 (offs[0])
int icp_align(Ctx& c, ilsm_map* const* targets, int n_pairs, const float* d_src, const int* offs, int stride_bytes,
              const double* guess7, const ilsm_icp_opts& o, ilsm_icp_result* results) {
  const int base = offs[0];
  long long total_tiles = 0;
  for (int p = 0; p < n_pairs; ++p) total_tiles += (offs[p + 1] - offs[p] + kIcpTile - 1) / kIcpTile;
  const size_t pair_bytes = (size_t)n_pairs * sizeof(IcpPair), res_bytes = (size_t)n_pairs * sizeof(ilsm_icp_result);
  const size_t res_off = (pair_bytes + 255) & ~(size_t)255;
  int rc;
  if ((rc = c.icp_pairs.reserve(pair_bytes)) || (rc = c.icp_res.reserve(n_pairs)) ||
      (rc = c.icp_part.reserve((size_t)2 * total_tiles * kIcpSums + 1)) || (rc = c.icp_pin.reserve(res_off + res_bytes)))
    return rc;
  IcpPair* hp = reinterpret_cast<IcpPair*>(c.icp_pin.p);
  long long tb = 0;
  for (int p = 0; p < n_pairs; ++p) {
    Map* m = &targets[p]->m;
    if ((rc = m->wait_ready(c.stream))) return rc;
    IcpPair& r = hp[p];
    memset(&r, 0, sizeof(r));
    if (m->table_size) r.g = m->view();  // a map that was never built is an empty target
    for (int k = 0; k < 7; ++k) r.guess[k] = guess7 ? guess7[7 * p + k] : (k == 3 ? 1.0 : 0.0);
    r.src_begin = offs[p] - base, r.n_src = offs[p + 1] - offs[p], r.tile_base = (int)tb;
    tb += (r.n_src + kIcpTile - 1) / kIcpTile;
  }
  IcpParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.src = d_src;
  prm.stride_f = stride_bytes / 4;
  prm.max_iter = o.max_iterations;
  prm.total_tiles = (int)total_tiles;
  prm.max_corr2 = o.max_correspondence_distance * o.max_correspondence_distance;
  prm.knn_d2 = knn_cutoff(prm.max_corr2);
  prm.fit_range = o.fitness_max_range;
  prm.fit_knn_d2 = knn_cutoff(o.fitness_max_range);
  prm.eps_t = o.transformation_epsilon;
  prm.rot_thr = o.transformation_rotation_epsilon > 0 ? o.transformation_rotation_epsilon : 1.0 - o.transformation_epsilon;
  prm.eps_fit = o.euclidean_fitness_epsilon;
  ILSM_CUDA(cudaMemcpyAsync(c.icp_pairs.p, hp, pair_bytes, cudaMemcpyHostToDevice, c.stream));
  const IcpPair* dp = reinterpret_cast<const IcpPair*>(c.icp_pairs.p);
  if (wide_cluster(c.icp_wide, icp_cluster_kernel<kIcpClusterWide>, kIcpClusterWide, kIcpThreads))
    ILSM_CUDA(launch_pdl(icp_cluster_kernel<kIcpClusterWide>, dim3((unsigned)n_pairs * kIcpClusterWide), dim3(kIcpThreads), 0,
                         c.stream, dp, prm, c.icp_part.p, c.icp_res.p));
  else
    ILSM_CUDA(launch_pdl(icp_cluster_kernel<kIcpCluster>, dim3((unsigned)n_pairs * kIcpCluster), dim3(kIcpThreads), 0, c.stream,
                         dp, prm, c.icp_part.p, c.icp_res.p));
  count_launches(1);
  if ((rc = check_launch("icp"))) return rc;
  ilsm_icp_result* hr = reinterpret_cast<ilsm_icp_result*>(c.icp_pin.p + res_off);
  ILSM_CUDA(cudaMemcpyAsync(hr, c.icp_res.p, res_bytes, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));  // also: the pinned pair records may be rewritten by the next call
  memcpy(results, hr, res_bytes);
  return ILSM_OK;
}

}  // namespace ilsm

using namespace ilsm;

static int icp_check(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* src, const int* offs, int stride_bytes,
                     const ilsm_icp_opts* opts, ilsm_icp_result* results, const char* who) {
  char msg[160];
  if (!ctx) return snprintf(msg, sizeof(msg), "%s: null ctx", who), fail(ILSM_ERR_INVALID_ARG, msg);
  if (n_pairs < 0) return snprintf(msg, sizeof(msg), "%s: n_pairs < 0", who), fail(ILSM_ERR_INVALID_ARG, msg);
  if (n_pairs == 0) return ILSM_OK;
  if (!targets || !offs || !results)
    return snprintf(msg, sizeof(msg), "%s: null targets / offsets / results", who), fail(ILSM_ERR_INVALID_ARG, msg);
  if (!valid_stride(stride_bytes))
    return snprintf(msg, sizeof(msg), "%s: bad stride", who), fail(ILSM_ERR_INVALID_ARG, msg);
  if (opts && opts->max_iterations < 0)
    return snprintf(msg, sizeof(msg), "%s: max_iterations < 0", who), fail(ILSM_ERR_INVALID_ARG, msg);
  if (offs[0] < 0) return snprintf(msg, sizeof(msg), "%s: negative source offset", who), fail(ILSM_ERR_INVALID_ARG, msg);
  for (int p = 0; p < n_pairs; ++p)
    if (offs[p + 1] < offs[p])
      return snprintf(msg, sizeof(msg), "%s: source offsets decrease at pair %d", who, p), fail(ILSM_ERR_INVALID_ARG, msg);
  if (offs[n_pairs] > offs[0] && !src) return snprintf(msg, sizeof(msg), "%s: null source points", who), fail(ILSM_ERR_INVALID_ARG, msg);
  for (int p = 0; p < n_pairs; ++p) {
    if (!targets[p]) return snprintf(msg, sizeof(msg), "%s: null target %d", who, p), fail(ILSM_ERR_INVALID_ARG, msg);
    if (targets[p]->m.ctx != &ctx->c)
      return snprintf(msg, sizeof(msg), "%s: target %d belongs to another context", who, p), fail(ILSM_ERR_INVALID_ARG, msg);
  }
  return ILSM_OK;
}

static int icp_run(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* src, bool on_device, const int* offs,
                   int stride_bytes, const double* guess7, const ilsm_icp_opts* opts, ilsm_icp_result* results) {
  ilsm_icp_opts o;
  if (opts)
    o = *opts;
  else
    ilsm_icp_opts_default(&o);
  Ctx& c = ctx->c;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  const size_t bytes = (size_t)(offs[n_pairs] - offs[0]) * stride_bytes;
  const float* first = src + (size_t)offs[0] * (stride_bytes / 4);
  if (!on_device) {
    int rc;
    if ((rc = c.icp_src.reserve(bytes / 4 + 4))) return rc;
    if (bytes) ILSM_CUDA(cudaMemcpyAsync(c.icp_src.p, first, bytes, cudaMemcpyHostToDevice, c.stream));
    first = c.icp_src.p;
  }
  return icp_align(c, targets, n_pairs, first, offs, stride_bytes, guess7, o, results);
}

extern "C" {

ILSM_API void ilsm_icp_opts_default(ilsm_icp_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->max_correspondence_distance = sqrt(DBL_MAX);
  o->max_iterations = 10;
  o->transformation_epsilon = 0.0;
  o->transformation_rotation_epsilon = 0.0;
  o->euclidean_fitness_epsilon = -DBL_MAX;
  o->fitness_max_range = DBL_MAX;
}

ILSM_API int ilsm_icp_align_batch(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* src_xyz,
                                  const int* src_offsets, int stride_bytes, const double* guess7, const ilsm_icp_opts* opts,
                                  ilsm_icp_result* results) {
  int rc = icp_check(ctx, targets, n_pairs, src_xyz, src_offsets, stride_bytes, opts, results, "icp_align_batch");
  if (rc || n_pairs == 0) return rc;
  return icp_run(ctx, targets, n_pairs, src_xyz, false, src_offsets, stride_bytes, guess7, opts, results);
}

ILSM_API int ilsm_icp_align_batch_dev(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* d_src_xyz,
                                      const int* src_offsets, int stride_bytes, const double* guess7, const ilsm_icp_opts* opts,
                                      ilsm_icp_result* results) {
  int rc = icp_check(ctx, targets, n_pairs, d_src_xyz, src_offsets, stride_bytes, opts, results, "icp_align_batch_dev");
  if (rc || n_pairs == 0) return rc;
  return icp_run(ctx, targets, n_pairs, d_src_xyz, true, src_offsets, stride_bytes, guess7, opts, results);
}

}  // extern "C"
