// registration.cu -- K2 (per-correspondence line/plane fit, fused behind the k-NN) and K3 (residual + 6-DoF
// Jacobian + J^T J / J^T r reduction with the Levenberg-Marquardt update folded into the last block).
//
// Replaces the association + ceres::Solve block of laserMapping.cpp:640-861 and mapOptimization.cpp:377-450:
//   associate_kernel : pointAssociateToMap (double math, float store) -> exact 5-NN in the voxel hash ->
//                      gate d2[4] < 1 -> 3x3 scatter-matrix eigen (corner) / 5x3 pivoted-QR plane (surf),
//                      one warp per point for the search, one lane per point (of one warp per block) for the fit;
//                      one factor slot per stack point.
//   solve_cluster_kernel (one thread-block cluster per ceres::Solve) / normal_eq_*_kernel (one evaluation over an
//                      ordinary grid): LidarEdgeFactor / LidarPlaneNormFactor residuals with closed-form tangent Jacobians
//                      (hpp:199-293 + EigenQuaternionParameterization), HuberLoss(0.1) corrector, warp-shuffle +
//                      block reduction of cost/JtJ/Jtr, deterministic cross-block sum by the last block, which
//                      then advances the trust-region state machine (Ceres 1.14 TrustRegionMinimizer +
//                      LevenbergMarquardtStrategy restated) and writes the next candidate pose to HBM.
// A registration is therefore a fixed sequence of launches with no host round trip until the final pose.
#include "ilsm_host.hpp"

namespace ilsm {

// ---------------------------------------------------------------------------------------------------
// fits
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void jacobi_rot(double& app, double& aqq, double& apq, double& arp, double& arq, double& v0p,
                                           double& v0q, double& v1p, double& v1q, double& v2p, double& v2q) {
  if (apq == 0.0) return;
  // t = tan(phi) of the annihilating rotation, smaller root: sgn(h) 2 apq / (|h| + sqrt(h^2 + 4 apq^2)), h = aqq - app
  // (one sqrt, one division and one rsqrt per rotation: fp64 div/sqrt are the long-latency ops of this kernel)
  const double h = aqq - app;
  const double t = (h >= 0.0 ? 2.0 : -2.0) * apq * frcp(fabs(h) + fsqrt(h * h + 4.0 * apq * apq));
  const double c = frsqrt(t * t + 1.0), s = t * c;
  app -= t * apq;
  aqq += t * apq;
  apq = 0.0;
  double x = arp, y = arq;
  arp = c * x - s * y;
  arq = s * x + c * y;
  x = v0p, y = v0q, v0p = c * x - s * y, v0q = s * x + c * y;
  x = v1p, y = v1q, v1p = c * x - s * y, v1q = s * x + c * y;
  x = v2p, y = v2q, v2p = c * x - s * y, v2q = s * x + c * y;
}

// laserMapping.cpp:681-722.  nb = the 5 neighbours (float map points widened to double).
__device__ __forceinline__ bool fit_line(const float (&nb)[5][3], double ratio, double (&pa)[3], double (&pb)[3]) {
  double cx = 0, cy = 0, cz = 0;
#pragma unroll
  for (int j = 0; j < 5; ++j) cx = cx + (double)nb[j][0], cy = cy + (double)nb[j][1], cz = cz + (double)nb[j][2];
  cx = cx * 0.2, cy = cy * 0.2, cz = cz * 0.2;
  double a00 = 0, a01 = 0, a02 = 0, a11 = 0, a12 = 0, a22 = 0;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    double zx = (double)nb[j][0] - cx, zy = (double)nb[j][1] - cy, zz = (double)nb[j][2] - cz;
    a00 = a00 + zx * zx, a01 = a01 + zx * zy, a02 = a02 + zx * zz;
    a11 = a11 + zy * zy, a12 = a12 + zy * zz, a22 = a22 + zz * zz;
  }
  double v00 = 1, v01 = 0, v02 = 0, v10 = 0, v11 = 1, v12 = 0, v20 = 0, v21 = 0, v22 = 1;
#pragma unroll 1
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = a01 * a01 + a02 * a02 + a12 * a12;
    double dg = a00 * a00 + a11 * a11 + a22 * a22;
    if (off <= 1e-32 * dg || off == 0.0) break;
    jacobi_rot(a00, a11, a01, a02, a12, v00, v01, v10, v11, v20, v21);  // (p,q)=(0,1), r=2
    jacobi_rot(a00, a22, a02, a01, a12, v00, v02, v10, v12, v20, v22);  // (0,2), r=1
    jacobi_rot(a11, a22, a12, a01, a02, v01, v02, v11, v12, v21, v22);  // (1,2), r=0
  }
  // largest eigenvalue / vector and the middle eigenvalue
  double lmax = a00, lmid, dx = v00, dy = v10, dz = v20;
  double o1 = a11, o2 = a22;
  if (a11 > lmax) lmax = a11, dx = v01, dy = v11, dz = v21, o1 = a00, o2 = a22;
  if (a22 > lmax) lmax = a22, dx = v02, dy = v12, dz = v22, o1 = a00, o2 = a11;
  lmid = o1 > o2 ? o1 : o2;
  if (!(lmax > ratio * lmid)) return false;
  pa[0] = 0.1 * dx + cx, pa[1] = 0.1 * dy + cy, pa[2] = 0.1 * dz + cz;
  pb[0] = -0.1 * dx + cx, pb[1] = -0.1 * dy + cy, pb[2] = -0.1 * dz + cz;
  return true;
}

// laserMapping.cpp:756-796 / mapOptimization.cpp:395-427: A(5x3) n = -1 by Householder QR with column pivoting.
__device__ __forceinline__ bool fit_plane(const float (&nb)[5][3], double tol, double (&nrm)[3], double& d_out) {
  double A[5][3], b[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    b[i] = -1.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) A[i][c] = (double)nb[i][c];
  }
  int perm[3] = {0, 1, 2};
  double rinv[3] = {0, 0, 0};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    double cn[3] = {0, 0, 0};
#pragma unroll
    for (int j = k; j < 3; ++j) {
#pragma unroll
      for (int i = k; i < 5; ++i) cn[j] += A[i][j] * A[i][j];
    }
    int piv = k;
    double best = cn[k];
#pragma unroll
    for (int j = k + 1; j < 3; ++j)
      if (cn[j] > best) best = cn[j], piv = j;
#pragma unroll
    for (int j = k + 1; j < 3; ++j) {
      if (piv == j) {
#pragma unroll
        for (int i = 0; i < 5; ++i) {
          double tmp = A[i][k];
          A[i][k] = A[i][j];
          A[i][j] = tmp;
        }
        int tp = perm[k];
        perm[k] = perm[j];
        perm[j] = tp;
      }
    }
    const double nr = fsqrt(best);
    if (nr == 0.0) {
      rinv[k] = 0.0;
      continue;
    }
    // reflector v = x - alpha e_k with alpha = -sgn(x_k)|x|;  v^T v = 2(|x|^2 - alpha x_k)  =>  2 / v^T v = beta
    const double xk = A[k][k];
    const double alpha = xk > 0.0 ? -nr : nr;
    const double beta = frcp(best - alpha * xk);
    double v[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) v[i] = i >= k ? A[i][k] : 0.0;
    v[k] = xk - alpha;
#pragma unroll
    for (int j = k + 1; j < 3; ++j) {
      double s = 0;
#pragma unroll
      for (int i = k; i < 5; ++i) s += v[i] * A[i][j];
      s *= beta;
#pragma unroll
      for (int i = k; i < 5; ++i) A[i][j] -= s * v[i];
    }
    double s = 0;
#pragma unroll
    for (int i = k; i < 5; ++i) s += v[i] * b[i];
    s *= beta;
#pragma unroll
    for (int i = k; i < 5; ++i) b[i] -= s * v[i];
    A[k][k] = alpha;  // R diagonal
    rinv[k] = frcp(alpha);
  }
  double y[3];
#pragma unroll
  for (int k = 2; k >= 0; --k) {
    double s = b[k];
#pragma unroll
    for (int j = k + 1; j < 3; ++j) s -= A[k][j] * y[j];
    y[k] = s * rinv[k];
  }
  double n[3] = {0, 0, 0};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      if (perm[k] == c) n[c] = y[k];
  }
  const double nn2 = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
  const double d = frsqrt(nn2);  // negative_OA_dot_norm = 1/|n|
  n[0] *= d, n[1] *= d, n[2] *= d;
  bool ok = nn2 > 0.0 && isfinite(d);
#pragma unroll
  for (int j = 0; j < 5; ++j)
    if (fabs(n[0] * (double)nb[j][0] + n[1] * (double)nb[j][1] + n[2] * (double)nb[j][2] + d) > tol) ok = false;
  nrm[0] = n[0], nrm[1] = n[1], nrm[2] = n[2];
  d_out = d;
  return ok;
}

struct FactorView {
  int* type;
  float4* p;
  double4* a;
  double4* b;
  int32_t* knn_idx;  // may be null
  float* knn_d2;     // may be null
};

struct AssocParams {
  float gate_sq;
  double line_ratio, plane_tol;
};

constexpr int kAssocThreads = 128;

constexpr int kAssocWarps = kAssocThreads / 32;
constexpr int kAssocChunk = 32;  // points a block gathers before one warp fits them (8 per warp)
constexpr int kNbStride = 21;    // floats per gathered point (odd: the fitting lanes read conflict-free)

struct AssocShared {
  WarpScratch scratch[kAssocWarps];
  float nb[2][kAssocChunk][kNbStride];  // 5 neighbours (x,y,z), [15] gate flag, [16..18] the point
  int next[2];                          // next unclaimed point of the chunk (chunks of more than one point per warp)
  int bb[12];                           // bounding boxes of the two maps, pose (kept here by the looping variants:
  double pose[7];                       // in registers across the fit they cost spills)
};

#ifdef ILSM_DEBUG_TIMING
#define ASTAMP(k) do { if (lane == 0 && (gid == 5 || gid == nc + 1000)) st->dbg[48 + (gid == 5 ? 0 : 8) + (k)] = clock64(); } while (0)
#else
#define ASTAMP(k) do { } while (0)
#endif

// One warp per stack point for the 5-NN, one LANE per stack point for the fit.  A block works through chunks of
// 4 * per_warp consecutive points: its warps run the searches and leave the five neighbours in shared memory, then the
// lanes of warp 0 fit the chunk together while the other warps start on the next chunk (double-buffered).  A warp
// instruction occupies the fp64 pipe for the same time whether 1 or 32 lanes are active, so fitting on lane 0 of every
// warp -- 20 single-lane instruction streams per SM queueing behind one another -- cost more than the search itself.
//   kLoop = false : the launch has a warp for every point (per-frame stacks): one round, everything in registers
//   kLoop = true  : several rounds; kDynamic: up to 8 points per warp and chunk, claimed through a shared cursor
template <bool kLoop, bool kDynamic>
__device__ __forceinline__ void associate_rounds(AssocShared& sh, const GridView& gc, const GridView& gs,
                                                 const float* __restrict__ corner, int nc, const float* __restrict__ surf, int ns,
                                                 int stride_f, LmState* __restrict__ st, const AssocParams& prm,
                                                 const FactorView& fv, const PoseSrc& src, int per_warp) {
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // pose: the LM state (later passes), or handed in with the launch (first pass; block 0 then seeds the LM state for
  // the solve kernel -- nobody reads the state's pose inside this launch in that case)
  const double* p7 = src.mode == 2 ? src.dptr : (src.mode == 1 ? src.v : st->xq);  // xq[4], xt[3] are contiguous
  int bbr[12];
  double pr[7];
  if (!kLoop) {
    // everything that does not depend on the point is fetched up front so that the latencies overlap
#pragma unroll
    for (int i = 0; i < 6; ++i) bbr[i] = __ldg(gc.bbox + i), bbr[6 + i] = __ldg(gs.bbox + i);
#pragma unroll
    for (int i = 0; i < 7; ++i) pr[i] = p7[i];
    if (src.mode != 0 && blockIdx.x == 0 && threadIdx.x < 7) st->xq[threadIdx.x] = p7[threadIdx.x];
  } else {
    if (threadIdx.x < 7) {
      const double v = p7[threadIdx.x];
      sh.pose[threadIdx.x] = v;
      if (src.mode != 0 && blockIdx.x == 0) st->xq[threadIdx.x] = v;
    }
    if (threadIdx.x >= 32 && threadIdx.x < 38) sh.bb[threadIdx.x - 32] = gc.bbox[threadIdx.x - 32];
    if (threadIdx.x >= 64 && threadIdx.x < 70) sh.bb[6 + threadIdx.x - 64] = gs.bbox[threadIdx.x - 64];
    if (kDynamic && threadIdx.x >= 96 && threadIdx.x < 98) sh.next[threadIdx.x - 96] = 0;
    __syncthreads();
  }
  const int total = nc + ns;
  const int chunk = per_warp * kAssocWarps;
  int it = 0;
#pragma unroll 1
  for (int base = blockIdx.x * chunk; base < total; base += gridDim.x * chunk, ++it) {
    const int buf = kLoop ? (it & 1) : 0;
    const int cn = min(chunk, total - base);
    // the other buffer's cursor was last touched before the barrier that ended the previous chunk
    if (kDynamic && threadIdx.x == 0) sh.next[buf ^ 1] = 0;
#pragma unroll 1
    for (int turn = 0;; ++turn) {
      int j = (int)warp;
      if (kDynamic) {
        if (lane == 0) j = atomicAdd(&sh.next[buf], 1);
        j = __shfl_sync(0xffffffffu, j, 0);
      } else if (turn) {
        break;
      }
      if (j >= cn) break;
      const int gid = base + j;
      ASTAMP(0);
      const bool is_corner = gid < nc;
      const float* pp = is_corner ? corner + (size_t)gid * stride_f : surf + (size_t)(gid - nc) * stride_f;
      const float px = __ldg(pp), py = __ldg(pp + 1), pz = __ldg(pp + 2);
      // pointAssociateToMap: double math, float store
      double q[4], tx, ty, tz;
      if (kLoop) {
        q[0] = sh.pose[0], q[1] = sh.pose[1], q[2] = sh.pose[2], q[3] = sh.pose[3];
        tx = sh.pose[4], ty = sh.pose[5], tz = sh.pose[6];
      } else {
        q[0] = pr[0], q[1] = pr[1], q[2] = pr[2], q[3] = pr[3];
        tx = pr[4], ty = pr[5], tz = pr[6];
      }
      const D3 pw = quat_rotate(q, d3((double)px, (double)py, (double)pz));
      const float qx = __double2float_rn(dadd(pw.x, tx));
      const float qy = __double2float_rn(dadd(pw.y, ty));
      const float qz = __double2float_rn(dadd(pw.z, tz));
      ASTAMP(1);
      KnnResult<5, true> res;  // the neighbours' coordinates travel with the keys: no dependent gather before the fit
      GridView g;  // field-wise select keeps everything in registers (no local-memory copy of the parameter structs)
      g.cells = is_corner ? gc.cells : gs.cells;
      g.sorted = is_corner ? gc.sorted : gs.sorted;
      g.orig = nullptr;
      g.bbox = nullptr;
      g.mask = is_corner ? gc.mask : gs.mask;
      g.log2_size = is_corner ? gc.log2_size : gs.log2_size;
      g.cell = is_corner ? gc.cell : gs.cell;
      g.inv_cell = is_corner ? gc.inv_cell : gs.inv_cell;
      g.n = is_corner ? gc.n : gs.n;
      int bb[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) bb[i] = kLoop ? sh.bb[(is_corner ? 0 : 6) + i] : (is_corner ? bbr[i] : bbr[6 + i]);
      knn_search<5, true>(g, bb, qx, qy, qz, prm.gate_sq, lane, sh.scratch[warp], res);
      ASTAMP(2);
      if (lane == 0) {
        float* r = sh.nb[buf][j];
#pragma unroll
        for (int k = 0; k < 5; ++k) r[3 * k] = res.x[k], r[3 * k + 1] = res.y[k], r[3 * k + 2] = res.z[k];
        r[15] = (res.key[4] != kSentinel && cand_d2(res.key[4]) < prm.gate_sq) ? 1.f : 0.f;
        r[16] = px, r[17] = py, r[18] = pz;
        if (fv.knn_idx) {
#pragma unroll
          for (int k = 0; k < 5; ++k) {
            const bool have = res.key[k] != kSentinel;
            fv.knn_idx[(size_t)gid * 5 + k] = have ? cand_idx(res.key[k]) : -1;
            fv.knn_d2[(size_t)gid * 5 + k] = have ? cand_d2(res.key[k]) : __int_as_float(0x7f800000);
          }
        }
      }
      __syncwarp();
    }
    __syncthreads();
    if (warp == 0 && (int)lane < cn) {
      const float* r = sh.nb[buf][lane];
      const int fid = base + (int)lane;
      int type = 0;
      double a[3] = {0, 0, 0}, b[3] = {0, 0, 0}, w = 0;
      if (r[15] != 0.f) {
        float nb[5][3];
#pragma unroll
        for (int k = 0; k < 5; ++k) nb[k][0] = r[3 * k], nb[k][1] = r[3 * k + 1], nb[k][2] = r[3 * k + 2];
        if (fid < nc) {
          if (fit_line(nb, prm.line_ratio, a, b)) type = 1;
        } else {
          if (fit_plane(nb, prm.plane_tol, a, w)) type = 2;
        }
      }
      fv.type[fid] = type;
      fv.p[fid] = make_float4(r[16], r[17], r[18], 0.f);
      fv.a[fid] = make_double4(a[0], a[1], a[2], w);
      fv.b[fid] = make_double4(b[0], b[1], b[2], 0.0);
    }
    if (!kLoop) break;
  }
}

// kMulti = false: one point per warp and round, statically assigned (per-frame stacks: normally a single round).
template <bool kMulti>
__global__ void __launch_bounds__(kAssocThreads, 5)
    associate_kernel(GridView gc, GridView gs, const float* __restrict__ corner, int nc, const float* __restrict__ surf,
                     int ns, int stride_f, LmState* __restrict__ st, AssocParams prm, FactorView fv,
                     const int* __restrict__ d_counts, PoseSrc src, int per_warp) {
  pdl_entry();
  __shared__ AssocShared sh;
  if (d_counts) nc = d_counts[0], ns = d_counts[1];  // stack sizes produced on the device (VoxelGrid outputs)
  const int total = nc + ns, wave = (int)gridDim.x * kAssocWarps;
  if (kMulti) {
    // with device-side sizes the host only knows an upper bound: the chunk size follows the real total
    if (d_counts) per_warp = min(8, max(1, (total + wave - 1) / wave));
    associate_rounds<true, true>(sh, gc, gs, corner, nc, surf, ns, stride_f, st, prm, fv, src, per_warp);
  } else if (total <= wave) {
    associate_rounds<false, false>(sh, gc, gs, corner, nc, surf, ns, stride_f, st, prm, fv, src, 1);
  } else {
    associate_rounds<true, false>(sh, gc, gs, corner, nc, surf, ns, stride_f, st, prm, fv, src, 1);
  }
}

// ---------------------------------------------------------------------------------------------------
// scan-to-scan odometry association (laserOdometry.cpp:446-565 edges, :568-689 planes)
// The previous frame's less-sharp / less-flat clouds are ring-sorted (scanRegistration appends ring by ring) and
// carry the ring id in int(intensity); after the 1-NN the reference walks the cloud up and down from the closest
// point until the ring id leaves closest +- NEARBY_SCAN.  One warp per feature point: the walk is done 32 points
// per step, candidates are ranked by (float d2, visiting order) so that ties resolve like the sequential strict `<`.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 warp_min_u64(u64 v) {
  const uint32_t hi = (uint32_t)(v >> 32), lo = (uint32_t)v;
  const uint32_t mhi = redux_min_u32(0xffffffffu, hi);
  const uint32_t mlo = redux_min_u32(0xffffffffu, hi == mhi ? lo : 0xFFFFFFFFu);
  return ((u64)mhi << 32) | mlo;
}

// walk one direction; plane == false: edge rule (other rings only -> slot A); plane == true: slot A = same side or
// same ring, slot B = other side (see the reference loops).  order_base keeps upward visits ahead of downward ones.
template <bool kPlane, bool kUp>
__device__ __forceinline__ void ring_walk(const float4* __restrict__ pts, int n, int closest, int cring, float sx, float sy,
                                          float sz, unsigned lane, uint32_t order_base, u64& bestA, u64& bestB) {
  int base = kUp ? closest + 1 : closest - 1;
#pragma unroll 1
  for (;;) {
    const int j = kUp ? base + (int)lane : base - (int)lane;
    const bool in = kUp ? j < n : j >= 0;
    bool stop = false;
    u64 ka = ~0ull, kb = ~0ull;
    if (in) {
      const float4 p = __ldg(pts + j);
      const int rj = (int)p.w;
      stop = kUp ? (double)rj > (double)cring + 2.5 : (double)rj < (double)cring - 2.5;
      const float dx = __fsub_rn(p.x, sx), dy = __fsub_rn(p.y, sy), dz = __fsub_rn(p.z, sz);
      const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
      const uint32_t order = order_base + (uint32_t)(kUp ? j - closest : closest - j);
      const u64 key = ((u64)__float_as_uint(d) << 32) | order;
      const bool near = (double)d < 25.0;  // DISTANCE_SQ_THRESHOLD seeds minPointSqDis2/3
      if (!kPlane) {
        if (near && (kUp ? rj > cring : rj < cring)) ka = key;
      } else {
        if (near && (kUp ? rj <= cring : rj >= cring)) ka = key;
        if (near && (kUp ? rj > cring : rj < cring)) kb = key;
      }
    }
    const unsigned sm = __ballot_sync(0xffffffffu, stop || !in);
    const int first_stop = sm ? __ffs(sm) - 1 : 32;
    if ((int)lane >= first_stop) ka = ~0ull, kb = ~0ull;  // the sequential loop breaks there
    const u64 ma = warp_min_u64(ka);
    bestA = ma < bestA ? ma : bestA;
    if (kPlane) {
      const u64 mb = warp_min_u64(kb);
      bestB = mb < bestB ? mb : bestB;
    }
    if (first_stop < 32) break;
    base = kUp ? base + 32 : base - 32;
  }
}

__global__ void __launch_bounds__(kAssocThreads, 5)
    odom_associate_kernel(GridView gc, GridView gs, const float* __restrict__ sharp, int nsh, const float* __restrict__ flat,
                          int nfl, int stride_f, const LmState* __restrict__ st, FactorView fv) {
  pdl_entry();
  __shared__ WarpScratch scratch[kAssocThreads / 32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = gridDim.x * (kAssocThreads / 32);
  int bbc[6], bbs[6];
  load_bbox(gc, bbc);
  load_bbox(gs, bbs);
  const double q[4] = {st->xq[0], st->xq[1], st->xq[2], st->xq[3]};
  const double tx = st->xt[0], ty = st->xt[1], tz = st->xt[2];
#pragma unroll 1
  for (int gid = blockIdx.x * (kAssocThreads / 32) + warp; gid < nsh + nfl; gid += nwarps) {
    const bool is_corner = gid < nsh;
    const float* pp = is_corner ? sharp + (size_t)gid * stride_f : flat + (size_t)(gid - nsh) * stride_f;
    const float px = __ldg(pp), py = __ldg(pp + 1), pz = __ldg(pp + 2);
    // TransformToStart with s = 1 (DISTORTION 0): q_last_curr * p + t_last_curr, double math, float store
    const D3 pw = quat_rotate(q, d3((double)px, (double)py, (double)pz));
    const float sx = __double2float_rn(dadd(pw.x, tx)), sy = __double2float_rn(dadd(pw.y, ty)),
                sz = __double2float_rn(dadd(pw.z, tz));
    GridView g;
    g.cells = is_corner ? gc.cells : gs.cells;
    g.sorted = is_corner ? gc.sorted : gs.sorted;
    g.orig = is_corner ? gc.orig : gs.orig;
    g.bbox = nullptr;
    g.mask = is_corner ? gc.mask : gs.mask;
    g.log2_size = is_corner ? gc.log2_size : gs.log2_size;
    g.cell = is_corner ? gc.cell : gs.cell;
    g.inv_cell = is_corner ? gc.inv_cell : gs.inv_cell;
    g.n = is_corner ? gc.n : gs.n;
    int bb[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) bb[i] = is_corner ? bbc[i] : bbs[i];
    KnnResult<1, false> res;
    knn_search<1, false>(g, bb, sx, sy, sz, 25.0f, lane, scratch[warp], res);
    int type = 0;
    double a[3] = {0, 0, 0}, b[3] = {0, 0, 0}, w = 0;
    if (res.key[0] != kSentinel && (double)cand_d2(res.key[0]) < 25.0) {  // warp-uniform
      const int closest = cand_idx(res.key[0]);
      const float4 pc = __ldg(g.orig + closest);
      const int cring = (int)pc.w;
      u64 bestA = ~0ull, bestB = ~0ull;
      if (is_corner) {
        ring_walk<false, true>(g.orig, g.n, closest, cring, sx, sy, sz, lane, 0u, bestA, bestB);
        ring_walk<false, false>(g.orig, g.n, closest, cring, sx, sy, sz, lane, 0x40000000u, bestA, bestB);
        if (bestA != ~0ull) {
          const uint32_t ord = (uint32_t)bestA;
          const int j2 = ord < 0x40000000u ? closest + (int)ord : closest - (int)(ord - 0x40000000u);
          const float4 pb = __ldg(g.orig + j2);
          type = 1;
          a[0] = pc.x, a[1] = pc.y, a[2] = pc.z;
          b[0] = pb.x, b[1] = pb.y, b[2] = pb.z;
        }
      } else {
        ring_walk<true, true>(g.orig, g.n, closest, cring, sx, sy, sz, lane, 0u, bestA, bestB);
        ring_walk<true, false>(g.orig, g.n, closest, cring, sx, sy, sz, lane, 0x40000000u, bestA, bestB);
        if (bestA != ~0ull && bestB != ~0ull) {
          const uint32_t oa = (uint32_t)bestA, ob = (uint32_t)bestB;
          const int j2 = oa < 0x40000000u ? closest + (int)oa : closest - (int)(oa - 0x40000000u);
          const int j3 = ob < 0x40000000u ? closest + (int)ob : closest - (int)(ob - 0x40000000u);
          const float4 pl = __ldg(g.orig + j2), pm = __ldg(g.orig + j3);
          // ljm_norm = normalize((j - l) x (j - m));  r = (lp - j) . ljm  ==  ljm . lp + (-j . ljm)
          const double ux = (double)pc.x - (double)pl.x, uy = (double)pc.y - (double)pl.y, uz = (double)pc.z - (double)pl.z;
          const double vx = (double)pc.x - (double)pm.x, vy = (double)pc.y - (double)pm.y, vz = (double)pc.z - (double)pm.z;
          const double nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
          const double inv = 1.0 / sqrt(nx * nx + ny * ny + nz * nz);
          const double n0 = nx * inv, n1 = ny * inv, n2 = nz * inv;
          if (isfinite(n0) && isfinite(n1) && isfinite(n2)) {
            type = 2;
            a[0] = n0, a[1] = n1, a[2] = n2;
            w = -((double)pc.x * n0 + (double)pc.y * n1 + (double)pc.z * n2);
          }
        }
      }
    }
    if (lane == 0) {
      fv.type[gid] = type;
      fv.p[gid] = make_float4(px, py, pz, 0.f);
      fv.a[gid] = make_double4(a[0], a[1], a[2], w);
      fv.b[gid] = make_double4(b[0], b[1], b[2], 0.0);
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------
// residual + Jacobian of one factor, accumulated into the 30 running sums
// ---------------------------------------------------------------------------------------------------
// running sums per evaluation: [0] cost, [1..21] H (upper triangle), [22..27] g, [28] #edge, [29] #plane
constexpr int kSumStride = 32;

__device__ __forceinline__ void acc_row(double (&acc)[kSumStride], const double (&j)[6], double r) {
  int k = 1;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
#pragma unroll
    for (int b = a; b < 6; ++b) acc[k++] += j[a] * j[b];
    acc[22 + a] += j[a] * r;
  }
}

// LidarEdgeFactor (hpp:243-293) / LidarPlaneNormFactor (hpp:199-240) at pose (q,t) with the closed-form tangent
// Jacobians of EigenQuaternionParameterization and the HuberLoss corrector.
// Rp = q * curr_point is passed in: the LM solver rotates with Eigen's _transformVector form (quat_rotate), the bulk
// J^T J kernel with the rotation matrix of the (launch-constant) pose.
__device__ __forceinline__ void eval_factor_rp(int type, const D3 Rp, const double4 fa, const double4 fb,
                                               const double (&t)[3], double huber_a, double (&acc)[kSumStride]) {
  D3 lp = d3(Rp.x + t[0], Rp.y + t[1], Rp.z + t[2]);
  if (type == 1) {
    D3 u = d3(lp.x - fa.x, lp.y - fa.y, lp.z - fa.z), v = d3(lp.x - fb.x, lp.y - fb.y, lp.z - fb.z);
    D3 nu = d3(u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x);
    const double dex = fa.x - fb.x, dey = fa.y - fb.y, dez = fa.z - fb.z;
    const double idn = frsqrt(dex * dex + dey * dey + dez * dez);  // 1/|a-b|
    const double r0 = nu.x * idn, r1 = nu.y * idn, r2 = nu.z * idn;
    const double mx = -dex * idn, my = -dey * idn, mz = -dez * idn;  // (b - a)/|a-b|
    const double sq = r0 * r0 + r1 * r1 + r2 * r2;
    double rho0 = sq, sc = 1.0;
    if (huber_a > 0.0 && sq > huber_a * huber_a) {  // ceres::HuberLoss + Corrector (rho'' <= 0): scale by sqrt(rho')
      const double irr = frsqrt(sq);
      rho0 = 2.0 * huber_a * (sq * irr) - huber_a * huber_a;
      sc = fsqrt(huber_a * irr);
    }
    acc[0] += 0.5 * rho0;
    acc[28] += 1.0;
    // J_t = [m]x ; J_delta = J_t * (-2 [Rp]x)
    const double Jt[3][3] = {{0, -mz, my}, {mz, 0, -mx}, {-my, mx, 0}};
    const double S[3][3] = {{0, 2 * Rp.z, -2 * Rp.y}, {-2 * Rp.z, 0, 2 * Rp.x}, {2 * Rp.y, -2 * Rp.x, 0}};
    const double rr[3] = {r0, r1, r2};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      double jr[6];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        jr[c] = sc * (Jt[a][0] * S[0][c] + Jt[a][1] * S[1][c] + Jt[a][2] * S[2][c]);
        jr[3 + c] = sc * Jt[a][c];
      }
      acc_row(acc, jr, sc * rr[a]);
    }
  } else if (type == 2) {
    const double r0 = fa.x * lp.x + fa.y * lp.y + fa.z * lp.z + fa.w;
    const double sq = r0 * r0;
    double rho0 = sq, sc = 1.0;
    if (huber_a > 0.0 && sq > huber_a * huber_a) {
      const double irr = frsqrt(sq);
      rho0 = 2.0 * huber_a * (sq * irr) - huber_a * huber_a;
      sc = fsqrt(huber_a * irr);
    }
    acc[0] += 0.5 * rho0;
    acc[29] += 1.0;
    double jr[6];
    jr[0] = sc * 2.0 * (Rp.y * fa.z - Rp.z * fa.y);  // n^T (-2[Rp]x) = 2 (Rp x n)^T
    jr[1] = sc * 2.0 * (Rp.z * fa.x - Rp.x * fa.z);
    jr[2] = sc * 2.0 * (Rp.x * fa.y - Rp.y * fa.x);
    jr[3] = sc * fa.x, jr[4] = sc * fa.y, jr[5] = sc * fa.z;
    acc_row(acc, jr, sc * r0);
  } else if (type == 3) {
    // front_end_residual (hpp:21-58): r = q * src + t - dst;  J = [-2 [Rp]x, I]   (fa = destination point)
    const double rr[3] = {lp.x - fa.x, lp.y - fa.y, lp.z - fa.z};
    const double sq = rr[0] * rr[0] + rr[1] * rr[1] + rr[2] * rr[2];
    double rho0 = sq, sc = 1.0;
    if (huber_a > 0.0 && sq > huber_a * huber_a) {
      const double irr = frsqrt(sq);
      rho0 = 2.0 * huber_a * (sq * irr) - huber_a * huber_a;
      sc = fsqrt(huber_a * irr);
    }
    acc[0] += 0.5 * rho0;
    acc[28] += 1.0;  // counted with the 3-row (edge-like) blocks
    const double S[3][3] = {{0, 2 * Rp.z, -2 * Rp.y}, {-2 * Rp.z, 0, 2 * Rp.x}, {2 * Rp.y, -2 * Rp.x, 0}};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      double jr[6];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        jr[c] = sc * S[a][c];
        jr[3 + c] = a == c ? sc : 0.0;
      }
      acc_row(acc, jr, sc * rr[a]);
    }
  }
}

__device__ __forceinline__ void eval_factor(int type, const float4 pf, const double4 fa, const double4 fb,
                                            const double (&q)[4], const double (&t)[3], double huber_a,
                                            double (&acc)[kSumStride]) {
  eval_factor_rp(type, quat_rotate(q, d3((double)pf.x, (double)pf.y, (double)pf.z)), fa, fb, t, huber_a, acc);
}

// Transposing warp reduction: 32 lanes x 32 values -> lane L returns the warp total of value L
// (31 shuffles per lane instead of 32 x 5).  Fixed order => deterministic.
__device__ __forceinline__ double warp_reduce_transpose(double (&v)[kSumStride], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const double send = upper ? v[i] : v[i + off];
      const double keep = upper ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// ---------------------------------------------------------------------------------------------------
// Levenberg-Marquardt state machine (Ceres 1.14 TrustRegionMinimizer + LevenbergMarquardtStrategy restated on
// the 6-dof tangent normal equations; DENSE_QR replaced by an LDL^T solve of the damped normal equations)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void quat_mul_d(const double a[4], const double b[4], double o[4]) {
  o[0] = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
  o[1] = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
  o[2] = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
  o[3] = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
}
// EigenQuaternionParameterization::Plus:  [sin|d|/|d| d, cos|d|] * x.
// sin(u)/u and cos(u) are even in u: for |d| < 0.5 (every LM step of a converging registration) they are evaluated
// as Taylor polynomials in |d|^2 (truncation < 1e-17), which drops sqrt, sincos and a division from the critical
// path of the single-threaded trust-region update; larger steps take the libm path.
__device__ __forceinline__ void quat_plus_d(const double x[4], const double d[3], double o[4]) {
  const double u2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
  if (u2 > 0.0) {
    double sbd, cs;
    if (u2 < 0.25) {
      // sin(u)/u = sum (-1)^k u^2k/(2k+1)!   cos(u) = sum (-1)^k u^2k/(2k)!
      sbd = fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, -7.6471637318198164759e-13, 1.6059043836821614599e-10),
                                                       -2.5052108385441718775e-8), 2.7557319223985890653e-6),
                                    -1.9841269841269841270e-4), 8.3333333333333333333e-3), -1.6666666666666666667e-1), 1.0);
      cs = fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, fma(u2, 4.7794773323873852974e-14, -1.1470745597729724714e-11),
                                                              2.0876756987868098979e-9), -2.7557319223985890653e-7),
                                           2.4801587301587301587e-5), -1.3888888888888888889e-3), 4.1666666666666666667e-2),
                       -0.5), 1.0);
    } else {
      const double nd = sqrt(u2);
      double sn;
      sincos(nd, &sn, &cs);
      sbd = sn / nd;
    }
    double dq[4] = {sbd * d[0], sbd * d[1], sbd * d[2], cs};
    quat_mul_d(dq, x, o);
  } else {
    o[0] = x[0], o[1] = x[1], o[2] = x[2], o[3] = x[3];
  }
}

// Packed lower-triangular index of a symmetric 6x6.
__device__ __forceinline__ constexpr int lt(int i, int j) { return i * (i + 1) / 2 + j; }  // i >= j
// Upper-triangle row-major index used by LmState::H.
__device__ __forceinline__ constexpr int ut(int a, int b) { return a * 6 - a * (a - 1) / 2 + (b - a); }  // a <= b

// A y = b for symmetric positive definite 6x6 (packed lower, destroyed) by in-place LDL^T with reciprocal pivots:
// 6 divisions in all, everything in registers.  Measured alternatives (round 2, clock64 stamps around the update, 3.4-3.6 k
// cycles with this solver): a division-free elimination on the packed triangle with the six reciprocals taken side by
// side -- half the dependency depth on paper -- runs 3.65-4.0 k (its 39 live values spill in this non-inlined function);
// keeping 1/radius and 1/model_cost_change as state, which removes two reciprocals from the chain, changes nothing
// measurable.  The update is not a pure latency chain that shorter algebra would shrink.
__device__ __forceinline__ bool ldlt_solve6(double (&m)[21], const double (&b)[6], double (&x)[6]) {
  // right-looking, in place: once column j is final (w_ij = L_ij d_j), the trailing sub-matrix is updated with
  // m_ic -= L_ij w_cj (one FMA per term) and the column is overwritten with L; no second array, 6 reciprocals
  double dinv[6];
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const double dj = m[lt(j, j)];
    ok = ok && (dj > 0.0);
    dinv[j] = frcp(dj);
    double l[6];
#pragma unroll
    for (int i = j + 1; i < 6; ++i) l[i] = m[lt(i, j)] * dinv[j];
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
#pragma unroll
      for (int c = j + 1; c <= i; ++c) m[lt(i, c)] = fma(-l[i], m[lt(c, j)], m[lt(i, c)]);
    }
#pragma unroll
    for (int i = j + 1; i < 6; ++i) m[lt(i, j)] = l[i];
  }
  if (!ok) return false;
  double z[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s = fma(-m[lt(i, k)], z[k], s);
    z[i] = s;
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = z[i] * dinv[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) s = fma(-m[lt(k, i)], x[k], s);
    x[i] = s;
  }
  return true;
}

__device__ void lm_arm(LmState* s, int max_iter, double huber_a, int pass) {
#pragma unroll
  for (int i = 0; i < 4; ++i) s->cq[i] = s->xq[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) s->ct[i] = s->xt[i];
  s->status = 0, s->phase = 0, s->iteration = 0, s->max_iter = max_iter;
  s->invalid_run = 0, s->reuse_diag = 0;
  s->n_success = s->n_unsuccess = s->n_evals = 0;
  s->n_edge = s->n_plane = 0;
  s->radius = 1e4, s->decrease_factor = 2.0, s->model_cost_change = 0.0;
  s->huber_a = huber_a;
  s->pass = pass;
  s->ticket = 0u;
}

// rep == nullptr: this CTA only mirrors the state machine (another CTA writes the report)
__device__ void lm_terminate(LmState* s, ilsm_reg_report* rep, int code) {
  s->status = 1 + code;
  if (!rep) return;
  ilsm_solve_summary& r = rep->pass[s->pass < ILSM_MAX_OUTER ? s->pass : ILSM_MAX_OUTER - 1];
  r.termination = code;
  r.iterations = s->iteration;
  r.num_successful_steps = s->n_success;
  r.num_unsuccessful_steps = s->n_unsuccess;
  r.num_edge_factors = s->n_edge;
  r.num_plane_factors = s->n_plane;
  r.num_evaluations = s->n_evals;
  r.reserved = 0;
  r.initial_cost = s->initial_cost;
  r.final_cost = s->cost;
  rep->passes = s->pass + 1;
}

// The update runs on ONE thread on purpose.  A warp-cooperative form (one matrix element per lane, LDL^T by shuffles) was
// built and measured in round 2: 4.3-5.0 k cycles per update against 3.4 k for this one in an instrumented build, and 3.6 x
// slower end to end in the release build, where every __shfl_sync inside the warp-0 branch is compiled into a
// WARPSYNC.COLLECTIVE / ENDCOLLECTIVE pair.  Dependent fp64 operations cost ~35 cycles each on this part, so the update is
// bound by its dependency chain (6 sequential pivots), not by issue slots; shuffles only lengthen that chain.
// Consume the sums of the evaluation at the candidate pose and either terminate or emit the next candidate.
// (a template only so that every kernel gets its own copy, compiled to ITS register budget: a shared copy is held to the
// smallest budget of its callers, and the update is faster with the 255 registers a 192-thread block allows)
template <int kCopy>
__device__ __noinline__ void lm_advance(LmState* s, ilsm_reg_report* rep, const double* sums) {
  const double function_tolerance = 1e-6, gradient_tolerance = 1e-10, parameter_tolerance = 1e-8;
  const double min_relative_decrease = 1e-3, min_radius = 1e-32, max_radius = 1e16;
  const double min_diag = 1e-6, max_diag = 1e32;
  s->n_evals += 1;
  const double new_cost = sums[0];
  if (s->phase == 0) {
    s->n_edge = (int)sums[28];
    s->n_plane = (int)sums[29];
    s->cost = new_cost;
    s->initial_cost = new_cost;
#pragma unroll
    for (int i = 0; i < 21; ++i) s->H[i] = sums[1 + i];
#pragma unroll
    for (int i = 0; i < 6; ++i) s->g[i] = sums[22 + i];
    if (s->n_edge + s->n_plane == 0) {  // Ceres: no residual blocks -> parameter blocks dropped -> CONVERGENCE
      lm_terminate(s, rep, ILSM_CONVERGENCE);
      return;
    }
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      s->scale[a] = frcp(1.0 + fsqrt(s->H[k]));
      k += 6 - a;
    }
  } else {
    double step2 = 0, x2 = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double d = s->xq[i] - s->cq[i];
      step2 += d * d;
      x2 += s->xq[i] * s->xq[i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double d = s->xt[i] - s->ct[i];
      step2 += d * d;
      x2 += s->xt[i] * s->xt[i];
    }
    // |step| <= ptol (|x| + ptol); |x| >= ~1 (unit quaternion) so the square-root test is only reached when the
    // cheap squared bound says it can possibly hold
    if (step2 <= 1.001 * parameter_tolerance * parameter_tolerance * (x2 + 1.0) &&
        sqrt(step2) <= parameter_tolerance * (sqrt(x2) + parameter_tolerance)) {
      lm_terminate(s, rep, ILSM_CONVERGENCE);
      return;
    }
    const double cost_change = s->cost - new_cost;
    if (fabs(cost_change) <= function_tolerance * s->cost) {
      lm_terminate(s, rep, ILSM_CONVERGENCE);
      return;
    }
    const double rho = cost_change * frcp(s->model_cost_change);
    if (rho > min_relative_decrease) {
#pragma unroll
      for (int i = 0; i < 4; ++i) s->xq[i] = s->cq[i];
#pragma unroll
      for (int i = 0; i < 3; ++i) s->xt[i] = s->ct[i];
      s->cost = new_cost;
#pragma unroll
      for (int i = 0; i < 21; ++i) s->H[i] = sums[1 + i];
#pragma unroll
      for (int i = 0; i < 6; ++i) s->g[i] = sums[22 + i];
      const double w = 2.0 * rho - 1.0;
      s->radius = s->radius * frcp(fmax(1.0 / 3.0, 1.0 - w * w * w));
      s->radius = fmin(max_radius, s->radius);
      s->decrease_factor = 2.0;
      s->reuse_diag = 0;
      s->n_success += 1;
    } else {
      s->radius = s->radius * frcp(s->decrease_factor);  // decrease_factor is a power of two: exact
      s->decrease_factor *= 2.0;
      s->reuse_diag = 1;
      s->n_unsuccess += 1;
    }
  }
  // FinalizeIterationAndCheckIfMinimizerCanContinue + ComputeTrustRegionStep, repeated over invalid steps
#pragma unroll 1
  for (;;) {
    if (s->iteration >= s->max_iter) {
      lm_terminate(s, rep, ILSM_NO_CONVERGENCE);
      return;
    }
    {  // gradient_max_norm = |x - Plus(x, -g)|_inf in the ambient space; the translation rows are exactly |g_t|,
       // so the quaternion rows (one sincos) only matter when those are already below the tolerance
      double m = fmax(fmax(fabs(s->g[3]), fabs(s->g[4])), fabs(s->g[5]));
      if (m <= gradient_tolerance) {
        double ng[3] = {-s->g[0], -s->g[1], -s->g[2]}, qp[4];
        quat_plus_d(s->xq, ng, qp);
#pragma unroll
        for (int i = 0; i < 4; ++i) m = fmax(m, fabs(s->xq[i] - qp[i]));
        if (m <= gradient_tolerance) {
          lm_terminate(s, rep, ILSM_CONVERGENCE);
          return;
        }
      }
    }
    if (s->radius <= min_radius) {
      lm_terminate(s, rep, ILSM_CONVERGENCE);
      return;
    }
    s->iteration += 1;
    double gs[6], m[21], y[6], step[6];
#pragma unroll
    for (int a = 0; a < 6; ++a) gs[a] = s->g[a] * s->scale[a];
    if (!s->reuse_diag) {
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        const double haa = s->H[ut(a, a)] * s->scale[a] * s->scale[a];
        s->diag[a] = fmin(fmax(haa, min_diag), max_diag);
      }
    }
    const double inv_radius = frcp(s->radius);
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int j = 0; j <= i; ++j)
        m[lt(i, j)] = s->H[ut(j, i)] * s->scale[j] * s->scale[i] + (i == j ? s->diag[i] * inv_radius : 0.0);
    bool ok = ldlt_solve6(m, gs, y);
    s->reuse_diag = 1;
    double mcc = 0;
    if (ok) {
      // model_cost_change = -(step^T g + 1/2 step^T H step) with step = -y and (H + D) y = g
      //                   = 1/2 (y^T g + y^T D y)
      double yg = 0, yDy = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        step[a] = -y[a];
        yg += y[a] * gs[a];
        yDy += y[a] * y[a] * (s->diag[a] * inv_radius);
        ok = ok && isfinite(y[a]);
      }
      mcc = 0.5 * (yg + yDy);
    }
    if (!ok || !(mcc > 0.0)) {  // HandleInvalidStep
      s->n_unsuccess += 1;
      if (++s->invalid_run >= 5) {
        lm_terminate(s, rep, ILSM_FAILURE);
        return;
      }
      s->radius = s->radius * frcp(s->decrease_factor);
      s->decrease_factor *= 2.0;
      s->reuse_diag = 1;
      continue;
    }
    s->invalid_run = 0;
    s->model_cost_change = mcc;
    double delta[6];
#pragma unroll
    for (int a = 0; a < 6; ++a) delta[a] = step[a] * s->scale[a];
    quat_plus_d(s->xq, delta, s->cq);
#pragma unroll
    for (int i = 0; i < 3; ++i) s->ct[i] = s->xt[i] + delta[3 + i];
    s->phase = 1;
    return;
  }
}

// ---------------------------------------------------------------------------------------------------
// solve_cluster_kernel: the whole ceres::Solve in ONE launch on one thread-block cluster (8 CTAs = 8 SMs).
// Each thread keeps its factor in registers across all evaluations; per evaluation the 30 sums are reduced
// warp -> CTA (shared memory) -> cluster (distributed shared memory), every CTA advances an identical copy of
// the LM state machine (no broadcast needed), one cluster barrier per evaluation (double-buffered partials).
// ---------------------------------------------------------------------------------------------------
// The LM solve runs as ONE thread-block cluster.  16 CTAs x 192 threads (a non-portable cluster size, B200 schedules it)
// when the device can place such a cluster, else 8 x 384: the same 3072 threads, but 6 instead of 12 warps per SM share
// an SM's fp64 pipe during the evaluation (solve 19.8 -> 18.4 us at config 1).
constexpr int kClusterSize = 8, kSolveThreads = 384;
constexpr int kClusterSizeWide = 16, kSolveThreadsWide = 192;
constexpr int kCoreWords = (int)(offsetof(LmState, report) / 8);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// mbarrier / bulk-copy primitives (sm_90+ PTX)
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Push one double into a peer's shared memory; the store completes 8 bytes of the transaction count of the peer's
// mbarrier (release at cluster scope), so the peer learns about the data without a cluster-wide barrier.
__device__ __forceinline__ void dsmem_push_f64(uint32_t remote_addr, double v, uint32_t remote_mbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(remote_addr),
               "l"(__double_as_longlong(v)), "r"(remote_mbar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {  // acquire at cluster scope
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "XWAIT_LOOP:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra XWAIT_DONE;\n"
      "bra XWAIT_LOOP;\n"
      "XWAIT_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}

struct SolveParams {
  int max_iter, pass, arm;
  double huber_a;
  double* d_pose7_out;             // non-null: the pose after this solve is also written here
  ilsm_reg_report* d_report_out;   // non-null: the accumulated report is also written here
};

template <int kCS, int kThr>
__global__ void __cluster_dims__(kCS, 1, 1) __launch_bounds__(kThr, 1)
    solve_cluster_kernel(FactorView fv, int n, LmState* st, SolveParams prm, const int* __restrict__ d_counts) {
  pdl_entry();
  __shared__ double core[kCoreWords];
  if (d_counts) n = d_counts[0] + d_counts[1];
  __shared__ double red[kThr / 32][kSumStride];
  // partial sums of every CTA of the cluster for the current evaluation, pushed by their owners (double-buffered by
  // evaluation parity) + the transaction barriers that count the 8 x 32 x 8 arriving bytes
  __shared__ double recv[2][kCS][kSumStride];
  __shared__ __align__(8) unsigned long long xbar[2];
  __shared__ double tot[kSumStride];
  constexpr uint32_t kXferBytes = kCS * kSumStride * 8;
  const uint32_t rank = cluster_ctarank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // factor i -> CTA (i % 8), thread (i / 8): the edge factors (3 residual rows, the first nc slots) are spread
  // evenly over the CTAs instead of all landing on CTA 0
  const int cl_tid = tid * kCS + (int)rank, cl_n = kCS * kThr;
  LmState* s = reinterpret_cast<LmState*>(core);  // only the fields before `report` exist in this copy

  // factor of the first round stays in registers for every evaluation
  int type0 = 0;
  float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f);
  double4 a0 = make_double4(0, 0, 0, 0), b0 = a0;
  if (cl_tid < n) {
    type0 = fv.type[cl_tid];
    if (type0) {
      p0 = fv.p[cl_tid];
      a0 = fv.a[cl_tid];
      if (type0 == 1) b0 = fv.b[cl_tid];
    }
  }
  {
    const double* src = reinterpret_cast<const double*>(st);
    for (int w = tid; w < kCoreWords; w += kThr) core[w] = src[w];
  }
  if (tid == 0) {
    mbar_init(smem_u32(&xbar[0]), 1), mbar_init(smem_u32(&xbar[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(smem_u32(&xbar[0]), kXferBytes), mbar_expect_tx(smem_u32(&xbar[1]), kXferBytes);  // evaluations 0 and 1
  }
  __syncthreads();
  if (tid == 0 && prm.arm) lm_arm(s, prm.max_iter, prm.huber_a, prm.pass);
  cluster_sync_all();  // every CTA's barriers are armed before any peer pushes into them (also a CTA barrier)
  ilsm_reg_report* rep = rank == 0 ? &st->report : nullptr;

#ifdef ILSM_DEBUG_TIMING
#define STAMP(k) do { if (rank == 0 && tid == 0 && e < 6) st->dbg[e * 8 + (k)] = clock64(); } while (0)
#else
#define STAMP(k) do { } while (0)
#endif
#pragma unroll 1
  for (int e = 0; s->status == 0; ++e) {
    STAMP(0);
    const double q[4] = {s->cq[0], s->cq[1], s->cq[2], s->cq[3]};
    const double t[3] = {s->ct[0], s->ct[1], s->ct[2]};
    const double huber_a = s->huber_a;
    double acc[kSumStride];
#pragma unroll
    for (int i = 0; i < kSumStride; ++i) acc[i] = 0.0;
#pragma unroll 1
    for (int i = cl_tid, it = 0; i < n; i += cl_n, ++it) {  // it > 0: stacks larger than one cluster round
      int ty = type0;
      float4 pf = p0;
      double4 fa = a0, fb = b0;
      if (it > 0) {
        ty = fv.type[i];
        if (ty) pf = fv.p[i], fa = fv.a[i], fb = fv.b[i];
      }
      if (ty) eval_factor(ty, pf, fa, fb, q, t, huber_a, acc);
    }
    STAMP(1);
    const double mine = warp_reduce_transpose(acc, lane);
    red[warp][lane] = mine;
    __syncthreads();
    STAMP(2);
    const int buf = e & 1;
    if (tid < kSumStride) {
      double v = 0;
#pragma unroll
      for (int w = 0; w < kThr / 32; ++w) v += red[w][tid];
      // push this CTA's partial into slot [rank] of every CTA (itself included): no cluster barrier, no remote loads
      const uint32_t slot = smem_u32(&recv[buf][rank][tid]), bar = smem_u32(&xbar[buf]);
#pragma unroll
      for (uint32_t r = 0; r < (uint32_t)kCS; ++r) {
        uint32_t ra, rb;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(slot), "r"(r));
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb) : "r"(bar), "r"(r));
        dsmem_push_f64(ra, v, rb);
      }
      STAMP(3);
      mbar_wait_cluster(bar, (uint32_t)(e >> 1) & 1u);  // all 8 partials have landed here
      double t8 = 0;
#pragma unroll
      for (int r = 0; r < kCS; ++r) t8 += recv[buf][r][tid];  // same order in every CTA: identical totals
      tot[tid] = t8;
    }
    __syncthreads();
    STAMP(4);
    // re-arm this buffer's barrier for evaluation e + 2: a peer can only push that far ahead after it has received this
    // CTA's partial of evaluation e + 1, which is sent after this point
    if (tid == 0) mbar_expect_tx(smem_u32(&xbar[buf]), kXferBytes);
    if (tid == 0) lm_advance<kThr>(s, rep, tot);
    STAMP(5);
    __syncthreads();
    STAMP(6);
  }
  // no trailing cluster barrier: peers only WRITE into this CTA's shared memory, and every such write has been waited
  // for above (all CTAs run the same number of evaluations)
  if (rank == 0) {
    double* dst = reinterpret_cast<double*>(st);
    for (int w = tid; w < kCoreWords; w += kThr) dst[w] = core[w];
    if (prm.d_pose7_out && tid < 7) prm.d_pose7_out[tid] = core[tid];  // xq[4], xt[3] lead the state
    if (prm.d_report_out) {  // written to st->report by thread 0 (lm_terminate) before the barrier that ended the loop
      const int words = (int)(sizeof(ilsm_reg_report) / 4);
      const int32_t* rs = reinterpret_cast<const int32_t*>(&st->report);
      int32_t* rd = reinterpret_cast<int32_t*>(prm.d_report_out);
      for (int w = tid; w < words; w += kThr) rd[w] = rs[w];
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// normal_eq_kernel: one evaluation of (cost, J^T J, J^T r) over all factors with an ordinary grid (the
// "J^T J kernel" of config 3 and of ilsm_eval_normal_eq); deterministic two-stage reduction, last block sums.
// ---------------------------------------------------------------------------------------------------
// 12 warps per SM in ONE block: the same occupancy as 3 x 128 at this register budget, but a third of the per-block
// partial sums, so the last block's cross-block combine is short (<= 148 x 32 doubles, 12 slices).
constexpr int kEvalThreads = 384, kEvalBlocksPerSm = 1;

__global__ void __launch_bounds__(kEvalThreads, kEvalBlocksPerSm)
    normal_eq_kernel(FactorView fv, int n, LmState* st, const double* __restrict__ pose7, double huber_a,
                     double* __restrict__ partials, double* __restrict__ eval_out) {
  pdl_entry();
  __shared__ double red[kEvalThreads / 32][kSumStride];
  __shared__ int is_last;
  double acc[kSumStride];
#pragma unroll
  for (int i = 0; i < kSumStride; ++i) acc[i] = 0.0;
  const double q[4] = {pose7[0], pose7[1], pose7[2], pose7[3]};
  const double t[3] = {pose7[4], pose7[5], pose7[6]};
  // persistent grid-stride loop: the 32 running sums stay in registers across factors, so the reduction cost is paid
  // once per thread; the next factor's record is in flight while the current one is evaluated.  Only the bytes a
  // factor type needs are read: type 0 (gate / fit failed) 4 B, plane 52 B, edge 84 B.
  const int stride = gridDim.x * kEvalThreads;
  int i = blockIdx.x * kEvalThreads + threadIdx.x;
  int ty = i < n ? __ldg(fv.type + i) : 0;
  float4 pf = make_float4(0.f, 0.f, 0.f, 0.f);
  double4 fa = make_double4(0, 0, 0, 0), fb = fa;
  if (ty) {
    pf = fv.p[i], fa = fv.a[i];
    if (ty == 1) fb = fv.b[i];
  }
#pragma unroll 1
  while (i < n) {
    const int ni = i + stride;
    const int nty = ni < n ? __ldg(fv.type + ni) : 0;
    float4 npf = pf;
    double4 nfa = fa, nfb = fb;
    if (nty) {
      npf = fv.p[ni], nfa = fv.a[ni];
      if (nty == 1) nfb = fv.b[ni];
    }
    if (ty) eval_factor(ty, pf, fa, fb, q, t, huber_a, acc);
    ty = nty, pf = npf, fa = nfa, fb = nfb, i = ni;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  red[warp][lane] = warp_reduce_transpose(acc, lane);
  __syncthreads();
  if (threadIdx.x < kSumStride) {
    double v = 0;
#pragma unroll
    for (int w = 0; w < kEvalThreads / 32; ++w) v += red[w][threadIdx.x];
    partials[(size_t)blockIdx.x * kSumStride + threadIdx.x] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned tk = atomicAdd(&st->ticket, 1u);
    is_last = (tk == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // 12 threads per sum, each a strided slice of the blocks (independent loads, 4 in flight), then a fixed-order combine
  __shared__ double slice[kEvalThreads / 32][kSumStride];
  {
    const int c = threadIdx.x & 31, sl = threadIdx.x >> 5;
    constexpr int S = kEvalThreads / 32;
    double v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    unsigned b = sl;
    for (; b + 3 * S < gridDim.x; b += 4 * S) {
      v0 += __ldcg(partials + (size_t)b * kSumStride + c);
      v1 += __ldcg(partials + (size_t)(b + S) * kSumStride + c);
      v2 += __ldcg(partials + (size_t)(b + 2 * S) * kSumStride + c);
      v3 += __ldcg(partials + (size_t)(b + 3 * S) * kSumStride + c);
    }
    for (; b < gridDim.x; b += S) v0 += __ldcg(partials + (size_t)b * kSumStride + c);
    slice[sl][c] = (v0 + v1) + (v2 + v3);
  }
  __syncthreads();
  if (threadIdx.x < kSumStride) {
    double v = 0;
#pragma unroll
    for (int sl = 0; sl < kEvalThreads / 32; ++sl) v += slice[sl][threadIdx.x];
    eval_out[threadIdx.x] = v;
  }
  if (threadIdx.x == 0) st->ticket = 0u;
}

// ---------------------------------------------------------------------------------------------------
// normal_eq_bulk_kernel: the same evaluation for LARGE factor sets (config 3: many frames' correspondences in one
// launch), where the kernel is HBM-bound.  The register-prefetch kernel above keeps one record per thread in flight
// (~32 KB per SM, 37 % of the copy peak).  Here one producer thread streams 352-factor tiles of the four SoA arrays
// into a ring of shared-memory stages with bulk async copies (cp.async.bulk, the 1-D TMA path: UBLKCP) that complete
// on an mbarrier; the 11 consumer warps wait for a stage, pull their factor into registers, release the stage (one
// mbarrier arrive per warp) and evaluate.  Up to kBulkStages x 29 KB are in flight per SM, independent of the
// consumers' register budget.  Tiles that lie entirely in the surf range (i >= nc) never fetch the `b` array
// (plane factors do not use it).  Tile -> CTA assignment is static, sums are combined in a fixed order: deterministic.
// ---------------------------------------------------------------------------------------------------
constexpr int kBulkTile = 352;                  // factors per stage = consumer threads (11 warps)
constexpr int kBulkThreads = kBulkTile + 32;    // + one producer warp = 12 warps, 3 per SM sub-partition
constexpr int kBulkStages = 6;
constexpr int kBulkStageBytes = kBulkTile * (4 + 16 + 32 + 32);
constexpr size_t kBulkSmemBytes = (size_t)kBulkStages * kBulkStageBytes + 2 * kBulkStages * 8 + 128;

// 12 warps and not 13: registers are allocated per SM sub-partition (4 x 16 K), so a 13th warp would cap the kernel at
// 128 registers per thread (spills in the tile loop).
__global__ void __launch_bounds__(kBulkThreads, 1)
    normal_eq_bulk_kernel(FactorView fv, int n, int nc, LmState* st, const double* __restrict__ pose7, double huber_a,
                          double* __restrict__ partials, double* __restrict__ eval_out) {
  pdl_entry();
  extern __shared__ __align__(128) unsigned char bulk_smem[];
  __shared__ double red[kBulkTile / 32][kSumStride];
  __shared__ int is_last;
  // stage layout: a[T] double4 | b[T] double4 | p[T] float4 | type[T] int
  const uint32_t smem0 = smem_u32(bulk_smem);
  const uint32_t bar0 = smem0 + kBulkStages * kBulkStageBytes;  // full[kBulkStages], then empty[kBulkStages]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < kBulkStages; ++s) {
      mbar_init(bar0 + 8 * s, 1);
      mbar_init(bar0 + 8 * (kBulkStages + s), kBulkTile / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int ntiles = (n + kBulkTile - 1) / kBulkTile;
  const int my_tiles = (int)blockIdx.x < ntiles ? (ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

  double acc[kSumStride];
#pragma unroll
  for (int i = 0; i < kSumStride; ++i) acc[i] = 0.0;

  if (warp == kBulkTile / 32) {
    // ---- producer: one thread keeps the ring full
    if (lane == 0) {
#pragma unroll 1
      for (int k = 0; k < my_tiles; ++k) {
        const int s = k % kBulkStages, use = k / kBulkStages;
        if (use > 0) mbar_wait(bar0 + 8 * (kBulkStages + s), (use - 1) & 1);
        const size_t base = (size_t)(blockIdx.x + (size_t)k * gridDim.x) * kBulkTile;
        const uint32_t cnt = (uint32_t)min((size_t)kBulkTile, (size_t)n - base);
        const bool need_b = base < (size_t)nc;
        const uint32_t ty_bytes = ((cnt * 4u) + 15u) & ~15u;  // the type array has >= 64 ints of slack behind n
        const uint32_t full = bar0 + 8 * s, dst = smem0 + s * kBulkStageBytes;
        mbar_expect_tx(full, cnt * 32u + (need_b ? cnt * 32u : 0u) + cnt * 16u + ty_bytes);
        bulk_g2s(dst, fv.a + base, cnt * 32u, full);
        if (need_b) bulk_g2s(dst + kBulkTile * 32, fv.b + base, cnt * 32u, full);
        bulk_g2s(dst + kBulkTile * 64, fv.p + base, cnt * 16u, full);
        bulk_g2s(dst + kBulkTile * 80, fv.type + base, ty_bytes, full);
      }
    }
  } else {
    // ---- consumers
    const double q[4] = {pose7[0], pose7[1], pose7[2], pose7[3]};
    const double t[3] = {pose7[4], pose7[5], pose7[6]};
    // Eigen::Quaterniond::toRotationMatrix of the pose, once per thread (the pose is constant for the launch)
    const double tx = 2.0 * q[0], ty2 = 2.0 * q[1], tz = 2.0 * q[2];
    const double twx = tx * q[3], twy = ty2 * q[3], twz = tz * q[3], txx = tx * q[0], txy = ty2 * q[0], txz = tz * q[0];
    const double tyy = ty2 * q[1], tyz = tz * q[1], tzz = tz * q[2];
    const double R00 = 1.0 - (tyy + tzz), R01 = txy - twz, R02 = txz + twy, R10 = txy + twz, R11 = 1.0 - (txx + tzz),
                 R12 = tyz - twx, R20 = txz - twy, R21 = tyz + twx, R22 = 1.0 - (txx + tyy);
#pragma unroll 1
    for (int k = 0; k < my_tiles; ++k) {
      const int s = k % kBulkStages, use = k / kBulkStages;
      mbar_wait(bar0 + 8 * s, use & 1);
      const unsigned char* stg = bulk_smem + (size_t)s * kBulkStageBytes;
      const size_t i = (size_t)(blockIdx.x + (size_t)k * gridDim.x) * kBulkTile + tid;
      int ty = 0;
      float4 pf = make_float4(0.f, 0.f, 0.f, 0.f);
      double4 fa = make_double4(0, 0, 0, 0), fb = fa;
      if (i < (size_t)n) {
        ty = reinterpret_cast<const int*>(stg + kBulkTile * 80)[tid];
        if (ty) {
          pf = reinterpret_cast<const float4*>(stg + kBulkTile * 64)[tid];
          fa = reinterpret_cast<const double4*>(stg)[tid];
          if (ty == 1) fb = reinterpret_cast<const double4*>(stg + kBulkTile * 32)[tid];
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar0 + 8 * (kBulkStages + s));  // the stage may be refilled while we evaluate
      if (ty) {
        const double px = (double)pf.x, py = (double)pf.y, pz = (double)pf.z;
        eval_factor_rp(ty, d3(R00 * px + R01 * py + R02 * pz, R10 * px + R11 * py + R12 * pz, R20 * px + R21 * py + R22 * pz),
                       fa, fb, t, huber_a, acc);
      }
    }
  }
  const double mine = warp_reduce_transpose(acc, lane);  // the producer warp contributes zeros
  if (warp < kBulkTile / 32) red[warp][lane] = mine;
  __syncthreads();
  if (tid < kSumStride) {
    double v = 0;
#pragma unroll
    for (int w = 0; w < kBulkTile / 32; ++w) v += red[w][tid];
    partials[(size_t)blockIdx.x * kSumStride + tid] = v;
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    unsigned tk = atomicAdd(&st->ticket, 1u);
    is_last = (tk == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (tid < kSumStride) {  // <= 148 blocks: a fixed-order sum per column
    double v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    unsigned b = 0;
    for (; b + 3 < gridDim.x; b += 4) {
      v0 += __ldcg(partials + (size_t)b * kSumStride + tid);
      v1 += __ldcg(partials + (size_t)(b + 1) * kSumStride + tid);
      v2 += __ldcg(partials + (size_t)(b + 2) * kSumStride + tid);
      v3 += __ldcg(partials + (size_t)(b + 3) * kSumStride + tid);
    }
    for (; b < gridDim.x; ++b) v0 += __ldcg(partials + (size_t)b * kSumStride + tid);
    eval_out[tid] = (v0 + v1) + (v2 + v3);
  }
  if (tid == 0) st->ticket = 0u;
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
static FactorView factor_view(FactorBufs& f, bool want_knn) {
  FactorView v;
  v.type = f.type.p;
  v.p = f.p.p;
  v.a = f.a.p;
  v.b = f.b.p;
  v.knn_idx = want_knn ? f.knn_idx.p : nullptr;
  v.knn_d2 = want_knn ? f.knn_d2.p : nullptr;
  return v;
}

// the pose of `src` into the LM state without an association launch to carry it (empty stacks, ilsm_solve_dev)
__global__ void pose_seed_kernel(LmState* st, PoseSrc src) {
  pdl_entry();
  const double* p7 = src.mode == 2 ? src.dptr : src.v;
  if (threadIdx.x < 7) st->xq[threadIdx.x] = p7[threadIdx.x];
}

int Ctx::seed_pose(const PoseSrc& src) {
  ILSM_CUDA(launch_pdl(pose_seed_kernel, dim3(1), dim3(32), 0, stream, lm.p, src));
  count_launches(1);
  return check_launch("pose_seed");
}

int Ctx::associate_dev(Map* mc, Map* ms, const float* d_corner, int nc, const float* d_surf, int ns, int stride_bytes,
                       const ilsm_reg_opts& o, bool want_knn, const PoseSrc* src) {
  const int n = nc + ns;
  int rc;
  if ((rc = fac.type.reserve(n + 4)) || (rc = fac.p.reserve(n + 1)) || (rc = fac.a.reserve(n + 1)) ||
      (rc = fac.b.reserve(n + 1)))
    return rc;
  if (want_knn && ((rc = fac.knn_idx.reserve((size_t)n * 5 + 1)) || (rc = fac.knn_d2.reserve((size_t)n * 5 + 1))))
    return rc;
  fac.n = n;
  fac.nc = nc;
  const PoseSrc ps = src ? *src : PoseSrc();
  if (n == 0) return ps.mode == 0 ? ILSM_OK : seed_pose(ps);
  if ((rc = mc->wait_ready(stream)) || (rc = ms->wait_ready(stream))) return rc;
  AssocParams prm;
  prm.gate_sq = o.knn_gate_sq;
  prm.line_ratio = o.line_eig_ratio;
  prm.plane_tol = o.plane_tol;
  GridView gc = mc->view(), gs = ms->view();
  FactorView fv = factor_view(fac, want_knn);
  const int stride_f = stride_bytes / 4;
  // one warp per stack point when one resident wave (5 blocks x 4 warps per SM at this register budget) covers the
  // stacks, else up to 8 points per warp and chunk.  With device-side sizes n is an upper bound (the clouds before their
  // VoxelGrid): the one-point-per-warp kernel, which loops if it must, unless the bound is far beyond a wave.
  const long long cap = (long long)sm_count * 5;
  const bool multi = d_stack_counts ? (long long)n > cap * 4 * 8 : (long long)n > cap * 4;
  int per_warp = 1;
  long long blocks = std::min(cap, ((long long)n + 3) / 4);
  if (multi) {
    per_warp = (int)std::min<long long>(8, (n + cap * 4 - 1) / (cap * 4));
    blocks = std::min(cap, ((long long)n + 4 * per_warp - 1) / (4 * per_warp));
    ILSM_CUDA(launch_pdl(associate_kernel<true>, dim3((unsigned)blocks), dim3(kAssocThreads), 0, stream, gc, gs, d_corner, nc,
                         d_surf, ns, stride_f, lm.p, prm, fv, d_stack_counts, ps, per_warp));
  } else {
    ILSM_CUDA(launch_pdl(associate_kernel<false>, dim3((unsigned)blocks), dim3(kAssocThreads), 0, stream, gc, gs, d_corner, nc,
                         d_surf, ns, stride_f, lm.p, prm, fv, d_stack_counts, ps, 1));
  }
  count_launches(1);
  return check_launch("associate");
}

int Ctx::odom_associate_dev(Map* mc, Map* ms, const float* d_sharp, int nsh, const float* d_flat, int nfl,
                            int stride_bytes) {
  const int n = nsh + nfl;
  int rc;
  if ((rc = fac.type.reserve(n + 4)) || (rc = fac.p.reserve(n + 1)) || (rc = fac.a.reserve(n + 1)) ||
      (rc = fac.b.reserve(n + 1)))
    return rc;
  fac.n = n;
  fac.nc = nsh;
  if (n == 0) return ILSM_OK;
  if ((rc = mc->wait_ready(stream)) || (rc = ms->wait_ready(stream))) return rc;
  FactorView fv = factor_view(fac, false);
  long long blocks = ((long long)n + 3) / 4, cap = (long long)sm_count * 5;
  if (blocks > cap) blocks = cap;
  ILSM_CUDA(launch_pdl(odom_associate_kernel, dim3((unsigned)blocks), dim3(kAssocThreads), 0, stream, mc->view(), ms->view(),
                       d_sharp, nsh, d_flat, nfl, stride_bytes / 4, (const LmState*)lm.p, fv));
  count_launches(1);
  return check_launch("odom_associate");
}

int Ctx::odometry_dev(Map* mc, Map* ms, const float* d_sharp, int nsh, const float* d_flat, int nfl, int stride_bytes,
                      const ilsm_reg_opts& o) {
  for (int pass = 0; pass < o.outer_iterations; ++pass) {
    int rc = odom_associate_dev(mc, ms, d_sharp, nsh, d_flat, nfl, stride_bytes);
    if (rc) return rc;
    if ((rc = solve_launch(o.max_num_iterations, o.huber_a, pass))) return rc;
  }
  return ILSM_OK;
}

int Ctx::solve_launch(int max_iter, double huber_a, int pass, const PoseDst* dst) {
  SolveParams prm;
  prm.max_iter = max_iter;
  prm.pass = pass;
  prm.arm = 1;
  prm.huber_a = huber_a;
  prm.d_pose7_out = dst ? dst->d_pose7 : nullptr;
  prm.d_report_out = dst ? dst->d_report : nullptr;
  FactorView fv = factor_view(fac, false);
  if (wide_cluster(solve_wide, solve_cluster_kernel<kClusterSizeWide, kSolveThreadsWide>, kClusterSizeWide, kSolveThreadsWide))
    ILSM_CUDA(launch_pdl(solve_cluster_kernel<kClusterSizeWide, kSolveThreadsWide>, dim3(kClusterSizeWide), dim3(kSolveThreadsWide), 0,
                         stream, fv, fac.n, lm.p, prm, d_stack_counts));
  else
    ILSM_CUDA(launch_pdl(solve_cluster_kernel<kClusterSize, kSolveThreads>, dim3(kClusterSize), dim3(kSolveThreads), 0, stream, fv,
                         fac.n, lm.p, prm, d_stack_counts));
  count_launches(1);
  return check_launch("solve");
}

int Ctx::register_dev(Map* mc, Map* ms, const float* d_corner, int nc, const float* d_surf, int ns, int stride_bytes,
                      const ilsm_reg_opts& o, const PoseSrc* src, const PoseDst* dst) {
  for (int pass = 0; pass < o.outer_iterations; ++pass) {
    int rc = associate_dev(mc, ms, d_corner, nc, d_surf, ns, stride_bytes, o, false, pass == 0 ? src : nullptr);
    if (rc) return rc;
    if ((rc = solve_launch(o.max_num_iterations, o.huber_a, pass, pass == o.outer_iterations - 1 ? dst : nullptr))) return rc;
  }
  return ILSM_OK;
}

// stand-alone evaluation (ilsm_eval_normal_eq[_dev]) at the 7 doubles d_pose7 (q then t, on the device) with Huber
// width huber_a
int eval_only_launch(Ctx* c, double* d_out, const double* d_pose7, double huber_a) {
  // bandwidth regime (at least one 352-factor tile per SM): the bulk-copy staged kernel, one persistent CTA per SM
  const long long ntiles = ((long long)c->fac.n + kBulkTile - 1) / kBulkTile;
  if (ntiles >= c->sm_count) {
    if (!c->bulk_attr_set) {
      ILSM_CUDA(cudaFuncSetAttribute(normal_eq_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBulkSmemBytes));
      c->bulk_attr_set = true;
    }
    const int blocks = c->sm_count;
    int rc;
    if ((rc = c->partials.reserve((size_t)blocks * kSumStride + kSumStride))) return rc;
    FactorView fv = factor_view(c->fac, false);
    ILSM_CUDA(launch_pdl(normal_eq_bulk_kernel, dim3((unsigned)blocks), dim3(kBulkThreads), kBulkSmemBytes, c->stream, fv, c->fac.n,
                         c->fac.nc, c->lm.p, d_pose7, huber_a, c->partials.p, d_out));
    count_launches(1);
    return check_launch("normal_eq_bulk");
  }
  long long blocks = ((long long)c->fac.n + kEvalThreads - 1) / kEvalThreads, cap = (long long)c->sm_count * kEvalBlocksPerSm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  int rc;
  if ((rc = c->partials.reserve((size_t)blocks * kSumStride + kSumStride))) return rc;
  FactorView fv = factor_view(c->fac, false);
  ILSM_CUDA(launch_pdl(normal_eq_kernel, dim3((unsigned)blocks), dim3(kEvalThreads), 0, c->stream, fv, c->fac.n, c->lm.p,
                       d_pose7, huber_a, c->partials.p, d_out));
  count_launches(1);
  return check_launch("normal_eq");
}

// copy factor SoA -> AoS records on the device for ilsm_associate's host output
__global__ void factors_export_kernel(FactorView fv, int n, int nc, ilsm_factor* out) {
  pdl_entry();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ilsm_factor f;
  f.type = fv.type[i];
  f.src = i < nc ? i : i - nc;
  float4 p = fv.p[i];
  double4 a = fv.a[i], b = fv.b[i];
  f.p[0] = p.x, f.p[1] = p.y, f.p[2] = p.z;
  f.a[0] = a.x, f.a[1] = a.y, f.a[2] = a.z;
  if (f.type == 2) {
    f.b[0] = a.w, f.b[1] = 0, f.b[2] = 0;
  } else {
    f.b[0] = b.x, f.b[1] = b.y, f.b[2] = b.z;
  }
  out[i] = f;
}

int factors_export(Ctx* c, ilsm_factor* d_out) {
  if (c->fac.n == 0) return ILSM_OK;
  FactorView fv = factor_view(c->fac, false);
  ILSM_CUDA(launch_pdl(factors_export_kernel, dim3((c->fac.n + 255) / 256), dim3(256), 0, c->stream, fv, c->fac.n, c->fac.nc, d_out));
  count_launches(1);
  return check_launch("factors_export");
}

}  // namespace ilsm
