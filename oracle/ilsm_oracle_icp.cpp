// ilsm_oracle_icp.cpp -- CPU ORACLE (TEST INFRASTRUCTURE) for K6, point-to-point ICP loop verification.
//
// PARITY STATUS: RESTATED, UNPINNED against PCL (not in this image; the reference tree does not ship it).  Written from
// PCL 1.10's icp.hpp (IterativeClosestPoint::computeTransformation), correspondence_estimation.hpp (determineCorrespondences:
// 1-NN, kept when d2 <= max_correspondence_distance^2), transformation_estimation_svd.hpp (rigid fit of the kept pairs,
// no scaling) and default_convergence_criteria.hpp (hasConverged with max_iterations_similar_transforms = 0,
// failure_after_max_iter = false), plus Registration::getFitnessScore(max_range):
//
//   P = guess, nr_iterations = 0, prev_mse = DBL_MAX
//   do {
//     S' = P * S                         from the ORIGINAL points (double math, float store)
//     C  = {(i, j, d2): j = 1-NN of S'[i] in T, (double)d2 <= max_corr^2}        exact, ties by (d2, index)
//     if |C| < 3: NO_CORRESPONDENCES, not converged, P unchanged; stop
//     (R, t) = argmin sum |R S'[i] + t - T[j]|^2 over C;  P = (R, t) o P;  ++nr_iterations
//     nr_iterations >= max_iterations                                -> ITERATIONS
//     0.5 (trace R - 1) >= rot_thr && |t|^2 <= transformation_eps    -> TRANSFORM
//     mse = sum_C d2 / |C|;  |mse - prev_mse| < 1e-12                -> ABS_MSE
//     |mse - prev_mse| / prev_mse < euclidean_fitness_eps            -> REL_MSE
//     prev_mse = mse
//   } while (true)
//   converged = every state but NO_CORRESPONDENCES (PCL reports convergence at max iterations too)
//   fitness   = mean d2 over {1-NN of (P S)[i] : d2 <= fitness_max_range}  (PCL compares the SQUARED distance), DBL_MAX if none
//   rot_thr   = transformation_rotation_epsilon if > 0, else 1 - transformation_epsilon
//
// Declared deviations from PCL (DESIGN section 2): P is kept in fp64 and applied to the original points (PCL composes a
// Matrix4f and re-transforms the already transformed cloud); the sums are fp64 in a fixed order; the rotation is Horn's
// closed form (largest eigenvector of the 4x4 quaternion matrix, cyclic Jacobi in fp64) instead of Eigen's float JacobiSVD;
// correspondence ties are broken by (d2, index).
//
// The fixed order, the same as the kernel's (csrc/icp.cu): the per-point terms count, d2, p - o, q - o, (p - o)(q - o)^T,
// with o the guess translation, are summed per 256-point tile as a lane-pair butterfly over each 32-point group followed
// by the 8 groups in order, and the tiles in tile order.  The 1-NN is the oracle's own exact search (orc_knn_kdtree:
// k-d tree == brute force, pinned against the reference's nanoflann).
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#define ORC_API extern "C" __attribute__((visibility("default")))

extern "C" void orc_knn_kdtree(const float* map, int n, int map_stride_bytes, const float* q, int nq, int q_stride_bytes, int k,
                               int32_t* idx, float* d2);

namespace {

constexpr int kTile = 256, kGroup = 32, kSums = 17;
enum { NOT_CONVERGED = 0, ITERATIONS = 1, TRANSFORM = 2, ABS_MSE = 3, REL_MSE = 4, NO_CORRESPONDENCES = 5 };

// Eigen QuaternionBase::_transformVector (q = x, y, z, w): v + w (2 u x v) + u x (2 u x v)
void rotate(const double q[4], const double v[3], double out[3]) {
  const double u[3] = {q[0], q[1], q[2]};
  double uv[3] = {u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]};
  for (int a = 0; a < 3; ++a) uv[a] = uv[a] + uv[a];
  const double c[3] = {u[1] * uv[2] - u[2] * uv[1], u[2] * uv[0] - u[0] * uv[2], u[0] * uv[1] - u[1] * uv[0]};
  for (int a = 0; a < 3; ++a) out[a] = (v[a] + q[3] * uv[a]) + c[a];
}

// Largest-eigenvalue eigenvector of Horn's N(S) by cyclic Jacobi; unit quaternion (x, y, z, w), w >= 0.
void horn_quat(const double S[3][3], double qo[4]) {
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
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
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
  const double nrm = std::sqrt(w * w + x * x + y * y + z * z);
  w = w / nrm, x = x / nrm, y = y / nrm, z = z / nrm;
  if (w < 0) w = -w, x = -x, y = -y, z = -z;
  qo[0] = x, qo[1] = y, qo[2] = z, qo[3] = w;
}

void quat_mat(const double q[4], double R[3][3]) {
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  R[0][0] = 1.0 - 2.0 * (y * y + z * z), R[0][1] = 2.0 * (x * y - w * z), R[0][2] = 2.0 * (x * z + w * y);
  R[1][0] = 2.0 * (x * y + w * z), R[1][1] = 1.0 - 2.0 * (x * x + z * z), R[1][2] = 2.0 * (y * z - w * x);
  R[2][0] = 2.0 * (x * z - w * y), R[2][1] = 2.0 * (y * z + w * x), R[2][2] = 1.0 - 2.0 * (x * x + y * y);
}

struct Pass {
  const float* tgt;
  int nt, tstride_f;
  const float* src;
  int ns, sstride_f;
  std::vector<float> moved;
  std::vector<int32_t> idx;
  std::vector<float> d2;
};

// One pass over the source under (q, t): S[0..nsum) in the fixed tile order; gate on (double) d2.
void pass_sums(Pass& ps, const double q[4], const double t[3], const double o[3], double gate, int nsum, double S[kSums]) {
  const int n = ps.ns;
  ps.moved.resize((size_t)3 * n + 3), ps.idx.resize(n + 1), ps.d2.resize(n + 1);
  for (int i = 0; i < n; ++i) {  // pointAssociateToMap: double math, float store
    const float* s = ps.src + (size_t)i * ps.sstride_f;
    const double v[3] = {(double)s[0], (double)s[1], (double)s[2]};
    double w[3];
    rotate(q, v, w);
    for (int a = 0; a < 3; ++a) ps.moved[3 * (size_t)i + a] = (float)(w[a] + t[a]);
  }
  if (n) orc_knn_kdtree(ps.tgt, ps.nt, ps.tstride_f * 4, ps.moved.data(), n, 12, 1, ps.idx.data(), ps.d2.data());
  for (int k = 0; k < kSums; ++k) S[k] = 0.0;
  for (int tile = 0; tile * kTile < n; ++tile) {
    double grp[kTile / kGroup][kSums];
    for (int g = 0; g < kTile / kGroup; ++g) {
      double lane[kGroup][kSums];
      for (int l = 0; l < kGroup; ++l) {
        double* c = lane[l];
        for (int k = 0; k < kSums; ++k) c[k] = 0.0;
        const int i = tile * kTile + g * kGroup + l;
        if (i >= n || ps.idx[i] < 0 || !((double)ps.d2[i] <= gate)) continue;
        c[0] = 1.0, c[1] = (double)ps.d2[i];
        if (nsum == 2) continue;
        const float* p = &ps.moved[3 * (size_t)i];
        const float* r = ps.tgt + (size_t)ps.idx[i] * ps.tstride_f;
        const double dp[3] = {(double)p[0] - o[0], (double)p[1] - o[1], (double)p[2] - o[2]};
        const double dq[3] = {(double)r[0] - o[0], (double)r[1] - o[1], (double)r[2] - o[2]};
        for (int a = 0; a < 3; ++a) {
          c[2 + a] = dp[a], c[5 + a] = dq[a];
          for (int b = 0; b < 3; ++b) c[8 + 3 * a + b] = dp[a] * dq[b];
        }
      }
      for (int off = kGroup / 2; off > 0; off >>= 1) {  // butterfly: lane l <- lane l + lane (l ^ off)
        double nxt[kGroup][kSums];
        for (int l = 0; l < kGroup; ++l)
          for (int k = 0; k < kSums; ++k) nxt[l][k] = lane[l][k] + lane[l ^ off][k];
        std::memcpy(lane, nxt, sizeof(lane));
      }
      for (int k = 0; k < kSums; ++k) grp[g][k] = lane[0][k];
    }
    for (int k = 0; k < nsum; ++k) {
      double s = grp[0][k];
      for (int g = 1; g < kTile / kGroup; ++g) s = s + grp[g][k];
      S[k] = S[k] + s;
    }
  }
}

}  // namespace

struct OrcIcpOpts {  // = ilsm_icp_opts
  double max_correspondence_distance;
  int max_iterations, pad;
  double transformation_epsilon, transformation_rotation_epsilon, euclidean_fitness_epsilon, fitness_max_range;
};
struct OrcIcpResult {  // = ilsm_icp_result
  double q_xyzw[4], t[3];
  double fitness, mse;
  int iterations, state, converged, n_correspondences;
};

ORC_API void orc_icp_align(const float* tgt, int nt, int tgt_stride_bytes, const float* src, int ns, int src_stride_bytes,
                           const double guess7[7], const OrcIcpOpts* opt, OrcIcpResult* res) {
  Pass ps;
  ps.tgt = tgt, ps.nt = nt, ps.tstride_f = tgt_stride_bytes / 4;
  ps.src = src, ps.ns = ns, ps.sstride_f = src_stride_bytes / 4;
  double q[4] = {guess7[0], guess7[1], guess7[2], guess7[3]}, t[3] = {guess7[4], guess7[5], guess7[6]};
  const double o[3] = {guess7[4], guess7[5], guess7[6]};
  const double max_corr2 = opt->max_correspondence_distance * opt->max_correspondence_distance;
  const double rot_thr = opt->transformation_rotation_epsilon > 0 ? opt->transformation_rotation_epsilon : 1.0 - opt->transformation_epsilon;
  double prev_mse = DBL_MAX, mse = DBL_MAX;
  int iter = 0, state = NOT_CONVERGED, n_corr = 0;
  double S[kSums];
  for (;;) {
    pass_sums(ps, q, t, o, max_corr2, kSums, S);
    const double n = S[0];
    n_corr = (int)n;
    mse = n > 0 ? S[1] / n : DBL_MAX;
    if (n < 3) {
      state = NO_CORRESPONDENCES;
      break;
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
    const double* b = q;
    const double qn[4] = {qi[3] * b[0] + qi[0] * b[3] + qi[1] * b[2] - qi[2] * b[1],
                          qi[3] * b[1] + qi[1] * b[3] + qi[2] * b[0] - qi[0] * b[2],
                          qi[3] * b[2] + qi[2] * b[3] + qi[0] * b[1] - qi[1] * b[0],
                          qi[3] * b[3] - qi[0] * b[0] - qi[1] * b[1] - qi[2] * b[2]};
    const double qnn = std::sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
    double tn[3];
    for (int a = 0; a < 3; ++a) tn[a] = ((R[a][0] * t[0] + R[a][1] * t[1]) + R[a][2] * t[2]) + ti[a];
    for (int k = 0; k < 4; ++k) q[k] = qn[k] / qnn;
    for (int a = 0; a < 3; ++a) t[a] = tn[a];
    ++iter;
    if (iter >= opt->max_iterations) {
      state = ITERATIONS;
      break;
    }
    const double cos_angle = 0.5 * (R[0][0] + R[1][1] + R[2][2] - 1.0);
    const double tr2 = ti[0] * ti[0] + ti[1] * ti[1] + ti[2] * ti[2];
    if (cos_angle >= rot_thr && tr2 <= opt->transformation_epsilon) {
      state = TRANSFORM;
      break;
    }
    const double dm = std::fabs(mse - prev_mse);
    if (dm < 1e-12) {
      state = ABS_MSE;
      break;
    }
    if (dm / prev_mse < opt->euclidean_fitness_epsilon) {
      state = REL_MSE;
      break;
    }
    prev_mse = mse;
  }
  pass_sums(ps, q, t, o, opt->fitness_max_range, 2, S);
  for (int k = 0; k < 4; ++k) res->q_xyzw[k] = q[k];
  for (int a = 0; a < 3; ++a) res->t[a] = t[a];
  res->fitness = S[0] > 0 ? S[1] / S[0] : DBL_MAX;
  res->mse = mse;
  res->iterations = iter, res->state = state, res->n_correspondences = n_corr;
  res->converged = state != NOT_CONVERGED && state != NO_CORRESPONDENCES;
}
