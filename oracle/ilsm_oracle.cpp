// ilsm_oracle.cpp -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE)
//
// A single-threaded CPU restatement of the reference's LOAM scan-to-map hot path, written from the
// reference's published behaviour (file:line citations are into /root/reference).  Only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this library.
// The shipped CUDA path never calls into it.
//
// PARITY STATUS.  Pinned against the reference's OWN code, compiled from /root/reference into oracle/_ref by
// oracle/Makefile (recipes and line-addressed cuts / repairs under oracle/patches, stand-ins under oracle/shims):
//   * k-NN                      -- the vendored nanoflann 1.3.2 (libref_nanoflann.so)
//   * ikd-Tree Build / Nearest_Search / Add_Points / flatten  -- src/ikd-Tree/ikd_Tree.cpp (libref_ikd.so)
//   * residuals + Jacobians     -- the Ceres cost functors on dual numbers (libref_functors.so)
//   * scan-to-scan association  -- laserOdometry.cpp:417-713 with a recording ceres::Problem (libref_laserodom.so)
//   * rolling cube map, transformAssociateToMap / transformUpdate / pointAssociateToMap, insertion, valid-cube order
//                               -- laserMapping.cpp:327-623, 875-945, 984-1004 (libref_lasermapping.so)
//   * ScanContext (ilsm_oracle_sc.cpp) and the front end (ilsm_oracle_frontend.cpp): see those files
//   * scan-to-map association   -- laserMapping.cpp:624-873, same library (5-NN gate, line / plane tests, point_a / point_b,
//                                  unit normal + offset; Eigen's two solvers run on THIS file's eig3 / lstsq5x3 there)
// "Parity unpinned" for what lives in libraries that are absent here and therefore restated from their published
// algorithms: Ceres 1.14's trust-region loop, Eigen 3.3's SelfAdjointEigenSolver / ColPivHouseholderQR / quaternion
// kernels, PCL's VoxelGrid.  The reference ships no tests, golden vectors or fixtures of its own.
//
// Build: see oracle/Makefile (g++ -O3 -std=c++14 -ffp-contract=off, the reference's flags
// CMakeLists.txt:5-6: -O3, no -march, hence no FMA contraction).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <numeric>
#include <vector>
#include <atomic>
#include <thread>

#define ORC_API extern "C" __attribute__((visibility("default")))

namespace {

// ------------------------------------------------------------------------------------------------
// small fixed-size linear algebra (double)
// ------------------------------------------------------------------------------------------------
struct V3 {
  double x, y, z;
};
inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(double s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline double norm(V3 a) { return std::sqrt(dot(a, a)); }

// Quaternion stored Eigen-coefficient order x,y,z,w (laserMapping.cpp:105-107, hpp:211 reads q[3] as w).
struct Quat {
  double x, y, z, w;
};

// Eigen 3.3 QuaternionBase::_transformVector: v + w*(2 u x v) + u x (2 u x v)   (no normalisation).
inline V3 rotate(const Quat& q, V3 v) {
  V3 u{q.x, q.y, q.z};
  V3 uv = cross(u, v);
  uv = uv + uv;
  return (v + q.w * uv) + cross(u, uv);
}

// Eigen quaternion product a*b.
inline Quat qmul(const Quat& a, const Quat& b) {
  return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y, a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
          a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}

// ------------------------------------------------------------------------------------------------
// k-NN: float arithmetic exactly as FLANN L2_Simple / ikd-Tree calc_dist (ikd_Tree.cpp:2224-2230):
// ((dx*dx)+(dy*dy))+(dz*dz) in float, no FMA.  Fixed tie-break: ascending (d2, index).
// ------------------------------------------------------------------------------------------------
inline float dist2f(const float* a, const float* b) {
  float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
  return (dx * dx + dy * dy) + dz * dz;
}

struct Cand {
  float d;
  int32_t i;
};
inline bool cand_less(const Cand& a, const Cand& b) { return a.d < b.d || (a.d == b.d && a.i < b.i); }

struct TopK {
  int k, n = 0;
  Cand c[32];
  explicit TopK(int k_) : k(k_) {}
  inline float worst() const { return n < k ? std::numeric_limits<float>::infinity() : c[k - 1].d; }
  inline void offer(float d, int32_t i) {
    Cand x{d, i};
    if (n == k && !cand_less(x, c[k - 1])) return;
    int j = (n < k) ? n++ : k - 1;
    while (j > 0 && cand_less(x, c[j - 1])) {
      c[j] = c[j - 1];
      --j;
    }
    c[j] = x;
  }
};

inline const float* pt(const float* base, int stride_f, int i) { return base + (size_t)i * stride_f; }
inline bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

// Exact k-d tree (own implementation; median split on widest axis).  Pruning uses only the single-axis
// bound fl((q-split)^2) which is <= the float distance of every point behind the split plane because
// float subtraction, squaring and adding non-negative terms are all monotone under round-to-nearest,
// so results are identical to brute force including ties.
#ifdef ORC_USE_NANOFLANN
// CPU-baseline variant (oracle/_ref/libref_aloam.so, built only where /root/reference exists): the same restatement
// with the k-d tree replaced by the REFERENCE'S OWN vendored nanoflann 1.3.2 (include/nanoflann.hpp) -- the port of
// FLANN's KDTreeSingleIndex that pcl::KdTreeFLANN wraps (laserMapping.cpp:631-634), leaf size 15 like PCL's
// KDTreeSingleIndexParams(15), L2_Simple<float>, NANOFLANN_FIRST_MATCH (lower index wins ties, the tie-break of this
// repository).  Same build / knn interface as the private tree below, same results (tests pin both to each other).
}  // namespace (reopened below)
#define NANOFLANN_FIRST_MATCH 1
#include <nanoflann.hpp>
#include <memory>
namespace {
struct KdTree {
  const float* base = nullptr;
  int stride_f = 0, n = 0;
  struct Cloud {
    const float* base;
    size_t n;
    int stride_f;
    inline size_t kdtree_get_point_count() const { return n; }
    inline float kdtree_get_pt(const size_t idx, const size_t dim) const { return base[idx * stride_f + dim]; }
    template <class BBOX>
    bool kdtree_get_bbox(BBOX&) const { return false; }
  };
  typedef nanoflann::KDTreeSingleIndexAdaptor<nanoflann::L2_Simple_Adaptor<float, Cloud>, Cloud, 3, int32_t> Tree;
  std::unique_ptr<Cloud> cloud;
  std::unique_ptr<Tree> tree;
  void build(const float* b, int n_, int stride_f_) {
    base = b, n = n_, stride_f = stride_f_;
    cloud.reset(new Cloud{b, (size_t)n_, stride_f_});
    tree.reset(new Tree(3, *cloud, nanoflann::KDTreeSingleIndexAdaptorParams(15)));
    tree->buildIndex();
  }
  void knn(const float* q, int k, int32_t* idx, float* d2) const {
    size_t found = 0;
    if (n > 0) {
      nanoflann::KNNResultSet<float, int32_t> rs((size_t)k);
      rs.init(idx, d2);
      tree->findNeighbors(rs, q, nanoflann::SearchParams(10));
      found = rs.size();
    }
    for (int j = (int)found; j < k; ++j) idx[j] = -1, d2[j] = INFINITY;
  }
};
#else
struct KdTree {
  const float* base = nullptr;
  int stride_f = 0, n = 0;
  std::vector<int32_t> ids;
  struct Node {
    int lo, hi, axis;
    float split;
    int left, right;
  };
  std::vector<Node> nodes;
  static constexpr int LEAF = 12;

  int build_rec(int lo, int hi) {
    Node nd{lo, hi, -1, 0.f, -1, -1};
    int me = (int)nodes.size();
    nodes.push_back(nd);
    if (hi - lo <= LEAF) return me;
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = lo; i < hi; ++i) {
      const float* p = pt(base, stride_f, ids[i]);
      for (int a = 0; a < 3; ++a) {
        mn[a] = std::min(mn[a], p[a]);
        mx[a] = std::max(mx[a], p[a]);
      }
    }
    int ax = 0;
    if (mx[1] - mn[1] > mx[ax] - mn[ax]) ax = 1;
    if (mx[2] - mn[2] > mx[ax] - mn[ax]) ax = 2;
    if (!(mx[ax] > mn[ax])) return me;  // all identical -> leaf
    int mid = (lo + hi) / 2;
    std::nth_element(ids.begin() + lo, ids.begin() + mid, ids.begin() + hi, [&](int32_t a, int32_t b) {
      float va = pt(base, stride_f, a)[ax], vb = pt(base, stride_f, b)[ax];
      return va < vb || (va == vb && a < b);
    });
    float split = pt(base, stride_f, ids[mid])[ax];
    int l = build_rec(lo, mid);
    int r = build_rec(mid, hi);
    nodes[me].axis = ax;
    nodes[me].split = split;
    nodes[me].left = l;
    nodes[me].right = r;
    return me;
  }
  // A point with a non-finite coordinate is left out, as the library's map build leaves it out (mapOptimization.cpp:151
  // strips such points before the tree is built); a NaN would otherwise break the median split and, offered first to a
  // search, hold the result slot.
  void build(const float* b, int n_, int stride_f_) {
    base = b;
    stride_f = stride_f_;
    ids.clear();
    for (int i = 0; i < n_; ++i)
      if (finite3(pt(b, stride_f, i))) ids.push_back(i);
    n = (int)ids.size();
    nodes.clear();
    nodes.reserve(2 * (n / LEAF + 2));
    if (n > 0) build_rec(0, n);
  }
  void search(int node, const float* q, TopK& top) const {
    const Node& nd = nodes[node];
    if (nd.axis < 0) {
      for (int i = nd.lo; i < nd.hi; ++i) top.offer(dist2f(q, pt(base, stride_f, ids[i])), ids[i]);
      return;
    }
    float diff = q[nd.axis] - nd.split;
    // left holds values <= split (by nth_element order), right holds values >= split.
    int near = diff < 0.f ? nd.left : nd.right, far = diff < 0.f ? nd.right : nd.left;
    search(near, q, top);
    float bound = diff * diff;
    if (bound <= top.worst()) search(far, q, top);
  }
  void knn(const float* q, int k, int32_t* idx, float* d2) const {
    TopK top(k);
    if (n > 0) search(0, q, top);
    for (int j = 0; j < k; ++j) {
      idx[j] = j < top.n ? top.c[j].i : -1;
      d2[j] = j < top.n ? top.c[j].d : INFINITY;
    }
  }
};

#endif  // ORC_USE_NANOFLANN

// ------------------------------------------------------------------------------------------------
// Fits (laserMapping.cpp:681-722 line; :756-796 plane; mapOptimization.cpp:395-427 plane)
// ------------------------------------------------------------------------------------------------
// Symmetric 3x3 eigen-decomposition, cyclic Jacobi in double; eigenvalues ascending like
// Eigen::SelfAdjointEigenSolver (Eigen itself uses tridiagonal QL; both are backward stable, results
// agree to ~1e-15 relative -- unpinned, no Eigen here).
void eig3(const double A[3][3], double w[3], double V[3][3]) {
  double a[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      a[i][j] = A[i][j];
      V[i][j] = i == j ? 1.0 : 0.0;
    }
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
    double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
    if (off <= 1e-32 * diag || off == 0.0) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {  // A <- A*G
          double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {  // A <- G^T*A
          double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          double vkp = V[k][p], vkq = V[k][q];
          V[k][p] = c * vkp - s * vkq;
          V[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int ord[3] = {0, 1, 2};
  double d[3] = {a[0][0], a[1][1], a[2][2]};
  std::sort(ord, ord + 3, [&](int i, int j) { return d[i] < d[j]; });
  double Vt[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Vt[i][j] = V[i][ord[j]];
  for (int j = 0; j < 3; ++j) w[j] = d[ord[j]];
  std::memcpy(V, Vt, sizeof(Vt));
}

// Least squares  min ||A x - b||, A is 5x3, via Householder QR with column pivoting
// (Eigen::ColPivHouseholderQR::solve semantic for full column rank).
void lstsq5x3(const double Ain[5][3], const double bin[5], double x[3]) {
  double A[5][3], b[5];
  std::memcpy(A, Ain, sizeof(A));
  std::memcpy(b, bin, sizeof(b));
  int perm[3] = {0, 1, 2};
  for (int k = 0; k < 3; ++k) {
    int piv = k;
    double best = -1.0;
    for (int j = k; j < 3; ++j) {
      double s = 0;
      for (int i = k; i < 5; ++i) s += A[i][j] * A[i][j];
      if (s > best) {
        best = s;
        piv = j;
      }
    }
    if (piv != k) {
      for (int i = 0; i < 5; ++i) std::swap(A[i][k], A[i][piv]);
      std::swap(perm[k], perm[piv]);
    }
    double nrm = std::sqrt(best);
    if (nrm == 0.0) continue;
    double alpha = A[k][k] > 0 ? -nrm : nrm;
    double v[5] = {0, 0, 0, 0, 0};
    for (int i = k; i < 5; ++i) v[i] = A[i][k];
    v[k] -= alpha;
    double vtv = 0;
    for (int i = k; i < 5; ++i) vtv += v[i] * v[i];
    if (vtv == 0.0) continue;
    for (int j = k; j < 3; ++j) {
      double s = 0;
      for (int i = k; i < 5; ++i) s += v[i] * A[i][j];
      s = 2.0 * s / vtv;
      for (int i = k; i < 5; ++i) A[i][j] -= s * v[i];
    }
    double s = 0;
    for (int i = k; i < 5; ++i) s += v[i] * b[i];
    s = 2.0 * s / vtv;
    for (int i = k; i < 5; ++i) b[i] -= s * v[i];
  }
  double y[3];
  for (int k = 2; k >= 0; --k) {
    double s = b[k];
    for (int j = k + 1; j < 3; ++j) s -= A[k][j] * y[j];
    y[k] = A[k][k] != 0.0 ? s / A[k][k] : 0.0;
  }
  for (int k = 0; k < 3; ++k) x[perm[k]] = y[k];
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// Public factor record (shared layout with tests via ctypes)
// ------------------------------------------------------------------------------------------------
struct OrcFactor {
  int32_t type;  // 0 none, 1 edge (LidarEdgeFactor), 2 plane (LidarPlaneNormFactor)
  int32_t src;   // index of the stack point that produced it
  double p[3];   // curr_point (sensor frame)
  double a[3];   // edge: point_a ; plane: unit normal
  double b[3];   // edge: point_b ; plane: b[0] = negative_OA_dot_norm
};

// the two dense kernels behind the fits, exported for oracle/ref_lasermapping.cpp: the reference's association block is
// compiled against an Eigen stand-in whose SelfAdjointEigenSolver / ColPivHouseholderQR forward here (Eigen is not installed)
ORC_API void orc_eig3(const double A[9], double w[3], double V[9]) {
  double a[3][3], v[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = A[3 * i + j];
  eig3(a, w, v);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) V[3 * i + j] = v[i][j];
}
ORC_API void orc_lstsq5x3(const double A[15], const double b[5], double x[3]) {
  double a[5][3];
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 3; ++j) a[i][j] = A[3 * i + j];
  lstsq5x3(a, b, x);
}

namespace {

bool fit_line(const float nb[5][3], OrcFactor* f) {
  // laserMapping.cpp:681-722
  V3 c{0, 0, 0};
  V3 p[5];
  for (int j = 0; j < 5; ++j) {
    p[j] = {nb[j][0], nb[j][1], nb[j][2]};
    c = c + p[j];
  }
  c = {c.x / 5.0, c.y / 5.0, c.z / 5.0};
  double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (int j = 0; j < 5; ++j) {
    V3 z = p[j] - c;
    double zz[3] = {z.x, z.y, z.z};
    for (int r = 0; r < 3; ++r)
      for (int s = 0; s < 3; ++s) cov[r][s] = cov[r][s] + zz[r] * zz[s];
  }
  double w[3], V[3][3];
  eig3(cov, w, V);
  if (!(w[2] > 3 * w[1])) return false;
  V3 dir{V[0][2], V[1][2], V[2][2]};
  V3 a = 0.1 * dir + c, b = -0.1 * dir + c;
  f->type = 1;
  f->a[0] = a.x, f->a[1] = a.y, f->a[2] = a.z;
  f->b[0] = b.x, f->b[1] = b.y, f->b[2] = b.z;
  return true;
}

bool fit_plane(const float nb[5][3], OrcFactor* f) {
  // laserMapping.cpp:756-796, mapOptimization.cpp:395-427
  double A[5][3], b[5] = {-1, -1, -1, -1, -1}, n[3];
  for (int j = 0; j < 5; ++j)
    for (int c = 0; c < 3; ++c) A[j][c] = nb[j][c];
  lstsq5x3(A, b, n);
  double nn = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
  double d = 1 / nn;
  n[0] /= nn, n[1] /= nn, n[2] /= nn;
  for (int j = 0; j < 5; ++j)
    if (std::fabs(n[0] * nb[j][0] + n[1] * nb[j][1] + n[2] * nb[j][2] + d) > 0.2) return false;
  if (!(nn > 0.0) || !std::isfinite(d)) return false;
  f->type = 2;
  f->a[0] = n[0], f->a[1] = n[1], f->a[2] = n[2];
  f->b[0] = d, f->b[1] = 0, f->b[2] = 0;
  return true;
}

// pointAssociateToMap (laserMapping.cpp:152-161; mapOptimization.cpp:377-381): double math, float store.
inline void associate_to_map(const Quat& q, const V3& t, const float* pi, float* po) {
  V3 pw = rotate(q, V3{pi[0], pi[1], pi[2]}) + t;
  po[0] = (float)pw.x, po[1] = (float)pw.y, po[2] = (float)pw.z;
}

// ------------------------------------------------------------------------------------------------
// Residuals + analytic tangent-space Jacobians (lidarFeaturePointsFunction.hpp:199-293 with s=1,
// Ceres autodiff replaced by closed forms; EigenQuaternionParameterization: x+ = [sin|d|/|d| d, cos|d|] * x)
//   d(Rp+t)/d delta = -2 [Rp]x ,  d/dt = I
// Robust loss HuberLoss(0.1) through Ceres' corrector (rho''<=0 => scale r and J by sqrt(rho')).
// ------------------------------------------------------------------------------------------------
struct NormalEq {
  double cost;
  double H[21];  // upper triangle row-major: (0,0)(0,1)..(0,5)(1,1)..(5,5)
  double g[6];
};

inline void add_row(NormalEq& ne, const double j[6], double r) {
  int k = 0;
  for (int a = 0; a < 6; ++a) {
    for (int b = a; b < 6; ++b) ne.H[k++] += j[a] * j[b];
    ne.g[a] += j[a] * r;
  }
}

void eval_factor(const OrcFactor& f, const Quat& q, const V3& t, double huber_a, NormalEq& ne, double* res_out) {
  V3 Rp = rotate(q, V3{f.p[0], f.p[1], f.p[2]});
  V3 lp = Rp + t;
  double r[3] = {0, 0, 0}, J[3][6];
  int nres = 0;
  if (f.type == 1) {
    V3 a{f.a[0], f.a[1], f.a[2]}, b{f.b[0], f.b[1], f.b[2]};
    V3 nu = cross(lp - a, lp - b);
    V3 de = a - b;
    double dn = norm(de);
    r[0] = nu.x / dn, r[1] = nu.y / dn, r[2] = nu.z / dn;
    // J_t = [b-a]x / |a-b|
    V3 m = {(b.x - a.x) / dn, (b.y - a.y) / dn, (b.z - a.z) / dn};
    double Jt[3][3] = {{0, -m.z, m.y}, {m.z, 0, -m.x}, {-m.y, m.x, 0}};
    // J_delta = J_t * (-2 [Rp]x)
    double S[3][3] = {{0, 2 * Rp.z, -2 * Rp.y}, {-2 * Rp.z, 0, 2 * Rp.x}, {2 * Rp.y, -2 * Rp.x, 0}};
    for (int i = 0; i < 3; ++i)
      for (int c = 0; c < 3; ++c) {
        J[i][c] = Jt[i][0] * S[0][c] + Jt[i][1] * S[1][c] + Jt[i][2] * S[2][c];
        J[i][3 + c] = Jt[i][c];
      }
    nres = 3;
  } else if (f.type == 2) {
    V3 n{f.a[0], f.a[1], f.a[2]};
    r[0] = dot(n, lp) + f.b[0];
    V3 jr = 2.0 * cross(Rp, n);  // n^T (-2[Rp]x) = 2 (Rp x n)^T
    J[0][0] = jr.x, J[0][1] = jr.y, J[0][2] = jr.z;
    J[0][3] = n.x, J[0][4] = n.y, J[0][5] = n.z;
    nres = 1;
  } else if (f.type == 3) {
    // front_end_residual (lidarFeaturePointsFunction.hpp:21-58): r = q * src + t - dst; a = dst point.
    r[0] = lp.x - f.a[0], r[1] = lp.y - f.a[1], r[2] = lp.z - f.a[2];
    double S[3][3] = {{0, 2 * Rp.z, -2 * Rp.y}, {-2 * Rp.z, 0, 2 * Rp.x}, {2 * Rp.y, -2 * Rp.x, 0}};  // -2 [Rp]x
    for (int i = 0; i < 3; ++i)
      for (int c = 0; c < 3; ++c) {
        J[i][c] = S[i][c];
        J[i][3 + c] = i == c ? 1.0 : 0.0;
      }
    nres = 3;
  } else {
    return;
  }
  double s = 0;
  for (int i = 0; i < nres; ++i) s += r[i] * r[i];
  double rho0 = s, rho1 = 1.0;
  if (huber_a > 0 && s > huber_a * huber_a) {
    double rr = std::sqrt(s);
    rho0 = 2 * huber_a * rr - huber_a * huber_a;
    rho1 = std::max(std::numeric_limits<double>::min(), huber_a / rr);
  }
  double sc = std::sqrt(rho1);
  ne.cost += 0.5 * rho0;
  for (int i = 0; i < nres; ++i) {
    double jr[6];
    for (int c = 0; c < 6; ++c) jr[c] = sc * J[i][c];
    add_row(ne, jr, sc * r[i]);
    if (res_out) res_out[i] = r[i];
  }
}

void eval_all(const OrcFactor* f, int nf, const Quat& q, const V3& t, double huber_a, NormalEq& ne, double* res) {
  std::memset(&ne, 0, sizeof(ne));
  for (int i = 0; i < nf; ++i) eval_factor(f[i], q, t, huber_a, ne, res ? res + 3 * i : nullptr);
}

// EigenQuaternionParameterization::Plus
inline Quat quat_plus(const Quat& x, const double d[3]) {
  double nd = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  if (nd > 0.0) {
    double sbd = std::sin(nd) / nd;
    Quat dq{sbd * d[0], sbd * d[1], sbd * d[2], std::cos(nd)};
    return qmul(dq, x);
  }
  return x;
}

// 6x6 SPD solve by Cholesky; returns false when not positive definite.
bool chol_solve6(const double Ain[6][6], const double b[6], double x[6]) {
  double L[6][6] = {};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = Ain[i][j];
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      if (i == j) {
        if (!(s > 0.0)) return false;
        L[i][i] = std::sqrt(s);
      } else {
        L[i][j] = s / L[j][j];
      }
    }
  double y[6];
  for (int i = 0; i < 6; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
    y[i] = s / L[i][i];
  }
  for (int i = 5; i >= 0; --i) {
    double s = y[i];
    for (int k = i + 1; k < 6; ++k) s -= L[k][i] * x[k];
    x[i] = s / L[i][i];
  }
  return true;
}

}  // namespace

// Solver summary mirrored to Python.
struct OrcSolveSummary {
  int32_t termination;  // 0 CONVERGENCE, 1 NO_CONVERGENCE, 2 FAILURE   (ceres::TerminationType order)
  int32_t iterations;   // iterations.back().iteration
  int32_t num_successful, num_unsuccessful;
  double initial_cost, final_cost;
  int32_t num_evals;  // residual evaluations performed (1 + trial steps)
  int32_t pad;
};

namespace {

// Ceres 1.14 TrustRegionMinimizer + LevenbergMarquardtStrategy + DENSE_QR, restated on the 6-dof tangent
// normal equations (laserMapping.cpp:836-850, mapOptimization.cpp:433-442, laserOdometry.cpp:705-710).
// Ceres defaults: initial radius 1e4, max 1e16, min 1e-32, min_relative_decrease 1e-3, lm diag clamp
// [1e-6,1e32], function_tolerance 1e-6, gradient_tolerance 1e-10, parameter_tolerance 1e-8, jacobi scaling,
// monotonic steps, max_num_consecutive_invalid_steps 5.
void lm_solve(const OrcFactor* f, int nf, double qt[7], int max_iter, double huber_a, OrcSolveSummary* sum) {
  const double function_tolerance = 1e-6, gradient_tolerance = 1e-10, parameter_tolerance = 1e-8;
  const double min_relative_decrease = 1e-3, min_radius = 1e-32, max_radius = 1e16;
  const double min_diag = 1e-6, max_diag = 1e32;
  std::memset(sum, 0, sizeof(*sum));
  int nvalid = 0;
  for (int i = 0; i < nf; ++i) nvalid += f[i].type != 0;
  if (nvalid == 0) {  // Ceres: "No non-constant parameter blocks found." -> CONVERGENCE, x untouched
    sum->termination = 0;
    return;
  }
  Quat q{qt[0], qt[1], qt[2], qt[3]};
  V3 t{qt[4], qt[5], qt[6]};
  NormalEq ne;
  eval_all(f, nf, q, t, huber_a, ne, nullptr);
  sum->num_evals = 1;
  double cost = ne.cost;
  sum->initial_cost = cost;
  double scale[6];
  {
    int k = 0;
    for (int a = 0; a < 6; ++a) {
      scale[a] = 1.0 / (1.0 + std::sqrt(ne.H[k]));
      k += 6 - a;
    }
  }
  double radius = 1e4, decrease_factor = 2.0;
  bool reuse_diagonal = false;
  double diag[6];
  int iteration = 0, invalid_run = 0;
  int termination = 1;

  auto x_vec = [&](const Quat& qq, const V3& tt, double x[7]) {
    x[0] = qq.x, x[1] = qq.y, x[2] = qq.z, x[3] = qq.w, x[4] = tt.x, x[5] = tt.y, x[6] = tt.z;
  };
  auto gradient_max_norm = [&]() {
    // |x - Plus(x, -g)|_inf in the ambient space
    double ng[6];
    for (int a = 0; a < 6; ++a) ng[a] = -ne.g[a];
    Quat qp = quat_plus(q, ng);
    double x0[7], x1[7];
    x_vec(q, t, x0);
    x_vec(qp, V3{t.x + ng[3], t.y + ng[4], t.z + ng[5]}, x1);
    double m = 0;
    for (int i = 0; i < 7; ++i) m = std::max(m, std::fabs(x0[i] - x1[i]));
    return m;
  };

  // iteration 0 bookkeeping happens in FinalizeIterationAndCheckIfMinimizerCanContinue
  while (true) {
    // ---- Finalize checks (order: max iterations, gradient tolerance, min radius)
    if (iteration >= max_iter) {
      termination = 1;
      break;
    }
    if (gradient_max_norm() <= gradient_tolerance) {
      termination = 0;
      break;
    }
    if (radius <= min_radius) {
      termination = 0;
      break;
    }
    ++iteration;
    // ---- ComputeTrustRegionStep
    double Hs[6][6], gs[6];
    {
      int k = 0;
      for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b) {
          Hs[a][b] = Hs[b][a] = ne.H[k++] * scale[a] * scale[b];
        }
      for (int a = 0; a < 6; ++a) gs[a] = ne.g[a] * scale[a];
    }
    if (!reuse_diagonal)
      for (int a = 0; a < 6; ++a) diag[a] = std::min(std::max(Hs[a][a], min_diag), max_diag);
    double A[6][6], y[6], step[6];
    for (int a = 0; a < 6; ++a)
      for (int b = 0; b < 6; ++b) A[a][b] = Hs[a][b] + (a == b ? diag[a] / radius : 0.0);
    bool ok = chol_solve6(A, gs, y);
    reuse_diagonal = true;
    double model_cost_change = 0;
    if (ok) {
      for (int a = 0; a < 6; ++a) step[a] = -y[a];
      double sg = 0, sHs = 0;
      for (int a = 0; a < 6; ++a) {
        sg += step[a] * gs[a];
        double hv = 0;
        for (int b = 0; b < 6; ++b) hv += Hs[a][b] * step[b];
        sHs += step[a] * hv;
      }
      model_cost_change = -(sg + 0.5 * sHs);
      for (int a = 0; a < 6; ++a) ok = ok && std::isfinite(step[a]);
    }
    if (!ok || !(model_cost_change > 0.0)) {
      // HandleInvalidStep
      if (++invalid_run >= 5) {
        termination = 2;
        ++sum->num_unsuccessful;
        break;
      }
      radius = radius / decrease_factor;
      decrease_factor *= 2.0;
      reuse_diagonal = true;
      ++sum->num_unsuccessful;
      continue;
    }
    invalid_run = 0;
    double delta[6];
    for (int a = 0; a < 6; ++a) delta[a] = step[a] * scale[a];
    // ---- candidate
    Quat qc = quat_plus(q, delta);
    V3 tc{t.x + delta[3], t.y + delta[4], t.z + delta[5]};
    NormalEq nc;
    eval_all(f, nf, qc, tc, huber_a, nc, nullptr);
    ++sum->num_evals;
    double x0[7], x1[7];
    x_vec(q, t, x0);
    x_vec(qc, tc, x1);
    double step_norm = 0, x_norm = 0;
    for (int i = 0; i < 7; ++i) {
      step_norm += (x0[i] - x1[i]) * (x0[i] - x1[i]);
      x_norm += x0[i] * x0[i];
    }
    step_norm = std::sqrt(step_norm), x_norm = std::sqrt(x_norm);
    if (step_norm <= parameter_tolerance * (x_norm + parameter_tolerance)) {
      termination = 0;
      break;
    }
    double cost_change = cost - nc.cost;
    if (std::fabs(cost_change) <= function_tolerance * cost) {
      termination = 0;
      break;
    }
    double rho = cost_change / model_cost_change;
    if (rho > min_relative_decrease) {
      q = qc, t = tc, ne = nc, cost = nc.cost;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rho - 1.0, 3));
      radius = std::min(max_radius, radius);
      decrease_factor = 2.0;
      reuse_diagonal = false;
      ++sum->num_successful;
    } else {
      radius = radius / decrease_factor;
      decrease_factor *= 2.0;
      reuse_diagonal = true;
      ++sum->num_unsuccessful;
    }
  }
  sum->termination = termination;
  sum->iterations = iteration;
  sum->final_cost = cost;
  qt[0] = q.x, qt[1] = q.y, qt[2] = q.z, qt[3] = q.w, qt[4] = t.x, qt[5] = t.y, qt[6] = t.z;
}

// One association pass of laserMapping.cpp:665-797 over both stacks.  knn backend is the oracle's
// own exact k-d tree (== brute force).
int associate(const KdTree& corner_map, const KdTree& surf_map, const float* corner, int nc, const float* surf, int ns,
              int stride_f, const double qt[7], OrcFactor* out) {
  Quat q{qt[0], qt[1], qt[2], qt[3]};
  V3 t{qt[4], qt[5], qt[6]};
  int nf = 0;
  for (int pass = 0; pass < 2; ++pass) {
    const KdTree& map = pass == 0 ? corner_map : surf_map;
    const float* st = pass == 0 ? corner : surf;
    int n = pass == 0 ? nc : ns;
    for (int i = 0; i < n; ++i) {
      const float* pi = pt(st, stride_f, i);
      OrcFactor f;
      std::memset(&f, 0, sizeof(f));
      f.src = i;
      f.p[0] = pi[0], f.p[1] = pi[1], f.p[2] = pi[2];
      if (map.n >= 5) {
        float pw[3];
        associate_to_map(q, t, pi, pw);
        int32_t idx[5];
        float d2[5];
        map.knn(pw, 5, idx, d2);
        if (d2[4] < 1.0f) {
          float nb[5][3];
          for (int j = 0; j < 5; ++j) std::memcpy(nb[j], pt(map.base, map.stride_f, idx[j]), 12);
          if (pass == 0)
            fit_line(nb, &f);
          else
            fit_plane(nb, &f);
        }
      }
      out[nf++] = f;
    }
  }
  return nf;
}

}  // namespace

// ================================================================================================
// C entry points (ctypes)
// ================================================================================================
ORC_API void orc_knn_brute(const float* map, int n, int map_stride_bytes, const float* q, int nq, int q_stride_bytes,
                           int k, int32_t* idx, float* d2) {
  int ms = map_stride_bytes / 4, qs = q_stride_bytes / 4;
  for (int i = 0; i < nq; ++i) {
    TopK top(k);
    const float* qq = pt(q, qs, i);
    for (int j = 0; j < n; ++j)
      if (finite3(pt(map, ms, j))) top.offer(dist2f(qq, pt(map, ms, j)), j);
    for (int j = 0; j < k; ++j) {
      idx[(size_t)i * k + j] = j < top.n ? top.c[j].i : -1;
      d2[(size_t)i * k + j] = j < top.n ? top.c[j].d : INFINITY;
    }
  }
}

ORC_API void orc_knn_kdtree(const float* map, int n, int map_stride_bytes, const float* q, int nq, int q_stride_bytes,
                            int k, int32_t* idx, float* d2) {
  KdTree tree;
  tree.build(map, n, map_stride_bytes / 4);
  int qs = q_stride_bytes / 4;
  for (int i = 0; i < nq; ++i) tree.knn(pt(q, qs, i), k, idx + (size_t)i * k, d2 + (size_t)i * k);
}

ORC_API void orc_transform_points(const double qt[7], const float* in, int n, int stride_bytes, float* out_xyz) {
  Quat q{qt[0], qt[1], qt[2], qt[3]};
  V3 t{qt[4], qt[5], qt[6]};
  for (int i = 0; i < n; ++i) associate_to_map(q, t, pt(in, stride_bytes / 4, i), out_xyz + 3 * (size_t)i);
}

// k-NN only, spread over `threads` host threads (<= 0: all hardware threads): the "B-knn-omp" CPU baseline of
// BASELINE.md section 3 (laserMapping.cpp:673,753 queried from a parallel loop; std::thread instead of OpenMP -- this
// image ships libgomp.so.1 without its spec file, so -fopenmp does not link).  build_s / query_s receive the wall time
// of the two phases; returns the number of threads used.
ORC_API int orc_knn_kdtree_omp(const float* map, int n, int map_stride_bytes, const float* q, int nq, int q_stride_bytes, int k,
                               int32_t* idx, float* d2, int threads, double* build_s, double* query_s) {
  const auto t0 = std::chrono::steady_clock::now();
  KdTree tree;
  tree.build(map, n, map_stride_bytes / 4);
  const auto t1 = std::chrono::steady_clock::now();
  if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
  if (threads < 1) threads = 1;
  std::atomic<int> next(0);
  const int chunk = 256, qs = q_stride_bytes / 4;
  auto work = [&]() {
    for (;;) {
      const int lo = next.fetch_add(chunk);
      if (lo >= nq) return;
      const int hi = lo + chunk < nq ? lo + chunk : nq;
      for (int i = lo; i < hi; ++i) tree.knn(q + (size_t)i * qs, k, idx + (size_t)i * k, d2 + (size_t)i * k);
    }
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < threads; ++t) pool.emplace_back(work);
  work();
  for (auto& th : pool) th.join();
  const auto t2 = std::chrono::steady_clock::now();
  if (build_s) *build_s = std::chrono::duration<double>(t1 - t0).count();
  if (query_s) *query_s = std::chrono::duration<double>(t2 - t1).count();
  return threads;
}

ORC_API int orc_fit_line(const float nb[15], OrcFactor* f) {
  float m[5][3];
  std::memcpy(m, nb, sizeof(m));
  std::memset(f, 0, sizeof(*f));
  return fit_line(m, f) ? 1 : 0;
}
ORC_API int orc_fit_plane(const float nb[15], OrcFactor* f) {
  float m[5][3];
  std::memcpy(m, nb, sizeof(m));
  std::memset(f, 0, sizeof(*f));
  return fit_plane(m, f) ? 1 : 0;
}

ORC_API int orc_associate(const float* map_corner, int n_mc, const float* map_surf, int n_ms, int map_stride_bytes,
                          const float* corner, int nc, const float* surf, int ns, int stride_bytes, const double qt[7],
                          OrcFactor* out) {
  KdTree kc, ks;
  kc.build(map_corner, n_mc, map_stride_bytes / 4);
  ks.build(map_surf, n_ms, map_stride_bytes / 4);
  return associate(kc, ks, corner, nc, surf, ns, stride_bytes / 4, qt, out);
}

// cost, H (6x6 full row-major), g (6), optional raw residuals (3 doubles per factor slot)
ORC_API void orc_eval(const OrcFactor* f, int nf, const double qt[7], double huber_a, double* cost, double* H36,
                      double* g6, double* residuals) {
  NormalEq ne;
  eval_all(f, nf, Quat{qt[0], qt[1], qt[2], qt[3]}, V3{qt[4], qt[5], qt[6]}, huber_a, ne, residuals);
  *cost = ne.cost;
  int k = 0;
  for (int a = 0; a < 6; ++a)
    for (int b = a; b < 6; ++b) H36[a * 6 + b] = H36[b * 6 + a] = ne.H[k++];
  for (int a = 0; a < 6; ++a) g6[a] = ne.g[a];
}

ORC_API void orc_solve(const OrcFactor* f, int nf, double qt[7], int max_iter, double huber_a, OrcSolveSummary* sum) {
  lm_solve(f, nf, qt, max_iter, huber_a, sum);
}

// laserMapping.cpp:624-861: guard, 2 x (associate + Solve(max 4)).  Returns number of outer passes run.
// summaries[2], nfactors[4] = {edge0, plane0, edge1, plane1}
ORC_API int orc_register_aloam(const float* map_corner, int n_mc, const float* map_surf, int n_ms,
                               int map_stride_bytes, const float* corner, int nc, const float* surf, int ns,
                               int stride_bytes, double qt[7], int outer, int max_iter, OrcSolveSummary* summaries,
                               int32_t* nfactors) {
  if (!(n_mc > 10 && n_ms > 50)) return 0;  // laserMapping.cpp:624
  KdTree kc, ks;
  kc.build(map_corner, n_mc, map_stride_bytes / 4);
  ks.build(map_surf, n_ms, map_stride_bytes / 4);
  std::vector<OrcFactor> f((size_t)nc + ns);
  for (int it = 0; it < outer; ++it) {
    int nf = associate(kc, ks, corner, nc, surf, ns, stride_bytes / 4, qt, f.data());
    int ne = 0, np = 0;
    for (int i = 0; i < nf; ++i) {
      ne += f[i].type == 1;
      np += f[i].type == 2;
    }
    nfactors[2 * it] = ne, nfactors[2 * it + 1] = np;
    lm_solve(f.data(), nf, qt, max_iter, 0.1, &summaries[it]);
  }
  return outer;
}

// ================================================================================================
// Scan-to-scan odometry (laserOdometry.cpp:147-194, 417-717): correspondence search on the previous frame's
// ring-sorted less-sharp / less-flat clouds, LidarEdgeFactor / LidarPlaneFactor with s = 1 (DISTORTION 0).
// Clouds are xyzi with intensity = scanID + 0.1 * relTime; int(intensity) is the ring id (:461,470).
// LidarPlaneFactor (hpp:143-196) r = (lp - j) . ljm is stored as a plane-norm record: n = ljm, d = -j . ljm.
// ================================================================================================
namespace {

inline int ring_of(const float* p, int ioff) { return int(p[ioff]); }

int odom_associate(const KdTree& kc, const KdTree& ks, int ioff, const float* sharp, int n_sharp, const float* flat,
                   int n_flat, int stride_f, const double qt[7], OrcFactor* out) {
  const double DISTANCE_SQ_THRESHOLD = 25, NEARBY_SCAN = 2.5;
  Quat q{qt[0], qt[1], qt[2], qt[3]};
  V3 t{qt[4], qt[5], qt[6]};
  int nf = 0;
  auto sqd = [](const float* a, const float* sel) {
    // float expression, evaluated left to right, widened to double afterwards (laserOdometry.cpp:478-483)
    return (double)((a[0] - sel[0]) * (a[0] - sel[0]) + (a[1] - sel[1]) * (a[1] - sel[1]) +
                    (a[2] - sel[2]) * (a[2] - sel[2]));
  };
  for (int i = 0; i < n_sharp; ++i) {
    const float* pi = pt(sharp, stride_f, i);
    OrcFactor f;
    std::memset(&f, 0, sizeof(f));
    f.src = i;
    f.p[0] = pi[0], f.p[1] = pi[1], f.p[2] = pi[2];
    float sel[3];
    associate_to_map(q, t, pi, sel);  // TransformToStart with s = 1
    int32_t ci;
    float cd;
    kc.knn(sel, 1, &ci, &cd);
    int closest = -1, min2 = -1;
    if (ci >= 0 && cd < DISTANCE_SQ_THRESHOLD) {
      closest = ci;
      const int cring = ring_of(pt(kc.base, kc.stride_f, closest), ioff);
      double best2 = DISTANCE_SQ_THRESHOLD;
      for (int j = closest + 1; j < kc.n; ++j) {
        const float* pj = pt(kc.base, kc.stride_f, j);
        if (ring_of(pj, ioff) <= cring) continue;
        if (ring_of(pj, ioff) > (cring + NEARBY_SCAN)) break;
        const double d = sqd(pj, sel);
        if (d < best2) best2 = d, min2 = j;
      }
      for (int j = closest - 1; j >= 0; --j) {
        const float* pj = pt(kc.base, kc.stride_f, j);
        if (ring_of(pj, ioff) >= cring) continue;
        if (ring_of(pj, ioff) < (cring - NEARBY_SCAN)) break;
        const double d = sqd(pj, sel);
        if (d < best2) best2 = d, min2 = j;
      }
    }
    if (min2 >= 0) {
      const float* a = pt(kc.base, kc.stride_f, closest);
      const float* b = pt(kc.base, kc.stride_f, min2);
      f.type = 1;
      for (int k = 0; k < 3; ++k) f.a[k] = a[k], f.b[k] = b[k];
    }
    out[nf++] = f;
  }
  for (int i = 0; i < n_flat; ++i) {
    const float* pi = pt(flat, stride_f, i);
    OrcFactor f;
    std::memset(&f, 0, sizeof(f));
    f.src = i;
    f.p[0] = pi[0], f.p[1] = pi[1], f.p[2] = pi[2];
    float sel[3];
    associate_to_map(q, t, pi, sel);
    int32_t ci;
    float cd;
    ks.knn(sel, 1, &ci, &cd);
    int closest = -1, min2 = -1, min3 = -1;
    if (ci >= 0 && cd < DISTANCE_SQ_THRESHOLD) {
      closest = ci;
      const int cring = ring_of(pt(ks.base, ks.stride_f, closest), ioff);
      double best2 = DISTANCE_SQ_THRESHOLD, best3 = DISTANCE_SQ_THRESHOLD;
      for (int j = closest + 1; j < ks.n; ++j) {
        const float* pj = pt(ks.base, ks.stride_f, j);
        if (ring_of(pj, ioff) > (cring + NEARBY_SCAN)) break;
        const double d = sqd(pj, sel);
        if (ring_of(pj, ioff) <= cring && d < best2)
          best2 = d, min2 = j;
        else if (ring_of(pj, ioff) > cring && d < best3)
          best3 = d, min3 = j;
      }
      for (int j = closest - 1; j >= 0; --j) {
        const float* pj = pt(ks.base, ks.stride_f, j);
        if (ring_of(pj, ioff) < (cring - NEARBY_SCAN)) break;
        const double d = sqd(pj, sel);
        if (ring_of(pj, ioff) >= cring && d < best2)
          best2 = d, min2 = j;
        else if (ring_of(pj, ioff) < cring && d < best3)
          best3 = d, min3 = j;
      }
    }
    if (min2 >= 0 && min3 >= 0) {
      const float* pa = pt(ks.base, ks.stride_f, closest);
      const float* pb = pt(ks.base, ks.stride_f, min2);
      const float* pc = pt(ks.base, ks.stride_f, min3);
      V3 j{pa[0], pa[1], pa[2]}, l{pb[0], pb[1], pb[2]}, m{pc[0], pc[1], pc[2]};
      V3 n = cross(j - l, j - m);
      const double nn = norm(n);
      n = {n.x / nn, n.y / nn, n.z / nn};  // ljm_norm.normalize()
      if (std::isfinite(n.x) && std::isfinite(n.y) && std::isfinite(n.z)) {
        f.type = 2;
        f.a[0] = n.x, f.a[1] = n.y, f.a[2] = n.z;
        f.b[0] = -dot(j, n);
      }
    }
    out[nf++] = f;
  }
  return nf;
}
}  // namespace

ORC_API int orc_odom_associate(const float* last_corner, int n_lc, const float* last_surf, int n_ls, int last_stride_bytes,
                               int ioff, const float* sharp, int n_sharp, const float* flat, int n_flat, int stride_bytes,
                               const double qt[7], OrcFactor* out) {
  KdTree kc, ks;
  kc.build(last_corner, n_lc, last_stride_bytes / 4);
  ks.build(last_surf, n_ls, last_stride_bytes / 4);
  return odom_associate(kc, ks, ioff, sharp, n_sharp, flat, n_flat, stride_bytes / 4, qt, out);
}

// laserOdometry.cpp:417-711: 2 x (correspondences + Solve(max 4)); qt = (para_q, para_t) updated in place
ORC_API int orc_odometry(const float* last_corner, int n_lc, const float* last_surf, int n_ls, int last_stride_bytes, int ioff,
                         const float* sharp, int n_sharp, const float* flat, int n_flat, int stride_bytes, double qt[7],
                         int outer, int max_iter, OrcSolveSummary* summaries, int32_t* nfactors) {
  KdTree kc, ks;
  kc.build(last_corner, n_lc, last_stride_bytes / 4);
  ks.build(last_surf, n_ls, last_stride_bytes / 4);
  std::vector<OrcFactor> f((size_t)n_sharp + n_flat);
  for (int it = 0; it < outer; ++it) {
    const int nf = odom_associate(kc, ks, ioff, sharp, n_sharp, flat, n_flat, stride_bytes / 4, qt, f.data());
    int ne = 0, np = 0;
    for (int i = 0; i < nf; ++i) ne += f[i].type == 1, np += f[i].type == 2;
    nfactors[2 * it] = ne, nfactors[2 * it + 1] = np;
    lm_solve(f.data(), nf, qt, max_iter, 0.1, &summaries[it]);
  }
  return outer;
}

// ================================================================================================
// ikd-Tree Add_Points with down-sampling (ikd_Tree.cpp:570-640), literal point-by-point restatement on a flat
// point list (the tree shape, lazy deletion and re-balancing do not change the resulting point SET).
// Storage order of Search_by_range is the tree's traversal order (unspecified here): ties between existing points
// of one box are broken by lower list position.  in/out: packed xyz (3 floats).
// ================================================================================================
ORC_API int orc_ikd_add_points(const float* existing, int n_old, const float* add, int n_add, float ds, int downsample,
                               float* out_xyz, int out_cap) {
  struct P {
    float x, y, z;
  };
  std::vector<P> pts(n_old);
  for (int i = 0; i < n_old; ++i) pts[i] = {existing[3 * i], existing[3 * i + 1], existing[3 * i + 2]};
  auto calc_dist = [](const P& a, const P& b) {
    return (a.x - b.x) * (a.x - b.x) + (a.y - b.y) * (a.y - b.y) + (a.z - b.z) * (a.z - b.z);
  };
  for (int i = 0; i < n_add; ++i) {
    const P p{add[3 * i], add[3 * i + 1], add[3 * i + 2]};
    if (!downsample) {
      pts.push_back(p);
      continue;
    }
    float mn[3], mx[3];
    const float c[3] = {p.x, p.y, p.z};
    for (int a = 0; a < 3; ++a) {
      mn[a] = std::floor(c[a] / ds) * ds;
      mx[a] = mn[a] + ds;
    }
    P mid;
    mid.x = (float)(mn[0] + (mx[0] - mn[0]) / 2.0);
    mid.y = (float)(mn[1] + (mx[1] - mn[1]) / 2.0);
    mid.z = (float)(mn[2] + (mx[2] - mn[2]) / 2.0);
    std::vector<int> storage;  // Search_by_range: min <= x && max > x (ikd_Tree.cpp:1607-1637)
    for (int j = 0; j < (int)pts.size(); ++j) {
      const P& s = pts[j];
      if (mn[0] <= s.x && mx[0] > s.x && mn[1] <= s.y && mx[1] > s.y && mn[2] <= s.z && mx[2] > s.z) storage.push_back(j);
    }
    float min_dist = calc_dist(p, mid);
    P result = p;
    for (int j : storage) {
      const float d = calc_dist(pts[j], mid);
      if (d < min_dist) min_dist = d, result = pts[j];
    }
    const bool same = std::fabs(p.x - result.x) < 1e-6 && std::fabs(p.y - result.y) < 1e-6 && std::fabs(p.z - result.z) < 1e-6;
    if (storage.size() > 1 || same) {
      // Delete_by_range + Add_by_point: the survivor keeps its place when it was already stored, else is appended
      std::vector<P> next;
      next.reserve(pts.size() + 1);
      size_t k = 0;
      bool placed = false;
      for (int j = 0; j < (int)pts.size(); ++j) {
        if (k < storage.size() && storage[k] == j) {
          ++k;
          if (!placed && pts[j].x == result.x && pts[j].y == result.y && pts[j].z == result.z) {
            next.push_back(pts[j]);
            placed = true;
          }
          continue;
        }
        next.push_back(pts[j]);
      }
      if (!placed) next.push_back(result);
      pts.swap(next);
    }
  }
  const int n = (int)pts.size();
  for (int i = 0; i < n && i < out_cap; ++i) out_xyz[3 * i] = pts[i].x, out_xyz[3 * i + 1] = pts[i].y, out_xyz[3 * i + 2] = pts[i].z;
  return n;
}

// ================================================================================================
// laserMapping.cpp process(): rolling 21x21x11 map of 50 m cubes (:330-606), stack VoxelGrid (:608-616),
// guarded registration (:624-875), insertion (:880-940, once -- the fork's duplicated surf insert :951-979 is a
// defect, upstream A-LOAM inserts once) and per-cube VoxelGrid of the valid cubes (:987-1002).
// ================================================================================================
extern "C" int orc_voxelgrid(const float* in, int n, int stride_bytes, int ioff, float leaf, float* out_xyzi);

namespace {
struct CubeMap {
  static constexpr int W = 21, H = 21, D = 11, NUM = W * H * D;
  int cenW = 10, cenH = 10, cenD = 5;
  bool solve = true;  // false: the frame keeps the pose transformAssociateToMap predicts (map-logic comparisons, tests/test_ref_lasermapping_cpu.py)
  float line_res = 0.4f, plane_res = 0.8f;
  std::vector<std::vector<float>> corner, surf;  // per cube, packed xyzi
  Quat q_wmap_wodom{0, 0, 0, 1};
  V3 t_wmap_wodom{0, 0, 0};
  int valid[125], n_valid = 0;
  CubeMap() : corner(NUM), surf(NUM) {}

  static int cube_coord(double v, int cen) {
    int c = int((v + 25.0) / 50.0) + cen;
    if (v + 25.0 < 0) c--;
    return c;
  }
  template <class F>
  void shift(int axis, int dir, F&& at) {
    // dir = +1: contents move towards higher index along `axis` (centre too low), the lowest slab is cleared
    const int n[3] = {W, H, D};
    for (int a = 0; a < n[(axis + 1) % 3]; ++a)
      for (int b = 0; b < n[(axis + 2) % 3]; ++b) {
        auto idx = [&](int m) {
          int ijk[3];
          ijk[axis] = m, ijk[(axis + 1) % 3] = a, ijk[(axis + 2) % 3] = b;
          return at(ijk[0], ijk[1], ijk[2]);
        };
        if (dir > 0) {
          std::vector<float> lastC = std::move(corner[idx(n[axis] - 1)]), lastS = std::move(surf[idx(n[axis] - 1)]);
          for (int m = n[axis] - 1; m >= 1; --m) corner[idx(m)] = std::move(corner[idx(m - 1)]), surf[idx(m)] = std::move(surf[idx(m - 1)]);
          lastC.clear(), lastS.clear();
          corner[idx(0)] = std::move(lastC), surf[idx(0)] = std::move(lastS);
        } else {
          std::vector<float> firstC = std::move(corner[idx(0)]), firstS = std::move(surf[idx(0)]);
          for (int m = 0; m < n[axis] - 1; ++m) corner[idx(m)] = std::move(corner[idx(m + 1)]), surf[idx(m)] = std::move(surf[idx(m + 1)]);
          firstC.clear(), firstS.clear();
          corner[idx(n[axis] - 1)] = std::move(firstC), surf[idx(n[axis] - 1)] = std::move(firstS);
        }
      }
  }
  void roll(const V3& t) {
    auto at = [](int i, int j, int k) { return i + W * j + W * H * k; };
    int cI = cube_coord(t.x, cenW), cJ = cube_coord(t.y, cenH), cK = cube_coord(t.z, cenD);
    while (cI < 3) shift(0, +1, at), cI++, cenW++;
    while (cI >= W - 3) shift(0, -1, at), cI--, cenW--;
    while (cJ < 3) shift(1, +1, at), cJ++, cenH++;
    while (cJ >= H - 3) shift(1, -1, at), cJ--, cenH--;
    while (cK < 3) shift(2, +1, at), cK++, cenD++;
    while (cK >= D - 3) shift(2, -1, at), cK--, cenD--;
    n_valid = 0;
    for (int i = cI - 2; i <= cI + 2; i++)
      for (int j = cJ - 2; j <= cJ + 2; j++)
        for (int k = cK - 1; k <= cK + 1; k++)
          if (i >= 0 && i < W && j >= 0 && j < H && k >= 0 && k < D) valid[n_valid++] = i + W * j + W * H * k;
  }
  void insert(std::vector<std::vector<float>>& arr, const float* pw /*xyzi*/) {
    const int cI = cube_coord(pw[0], cenW), cJ = cube_coord(pw[1], cenH), cK = cube_coord(pw[2], cenD);
    if (cI >= 0 && cI < W && cJ >= 0 && cJ < H && cK >= 0 && cK < D) {
      auto& v = arr[cI + W * cJ + W * H * cK];
      v.insert(v.end(), pw, pw + 4);
    }
  }
  void filter_valid() {
    std::vector<float> tmp;
    for (int v = 0; v < n_valid; ++v)
      for (int pass = 0; pass < 2; ++pass) {
        auto& c = pass == 0 ? corner[valid[v]] : surf[valid[v]];
        if (c.empty()) continue;
        tmp.resize(c.size());
        const int m = orc_voxelgrid(c.data(), (int)c.size() / 4, 16, 3, pass == 0 ? line_res : plane_res, tmp.data());
        c.assign(tmp.begin(), tmp.begin() + 4 * (size_t)m);
      }
  }
};
}  // namespace

struct OrcCubeFrameStats {
  int32_t n_map_corner, n_map_surf, n_stack_corner, n_stack_surf, ran_optimization, n_valid;
  int32_t cen[3];
  int32_t pad;
};

ORC_API void* orc_cubemap_create(float line_res, float plane_res) {
  CubeMap* m = new CubeMap();
  m->line_res = line_res, m->plane_res = plane_res;
  return m;
}
ORC_API void orc_cubemap_destroy(void* h) { delete static_cast<CubeMap*>(h); }

// seed / direct insertion of WORLD-frame points (xyzi packed), then filter the cubes around `centre`
ORC_API void orc_cubemap_insert_world(void* h, const float* corner, int nc, const float* surf, int ns, const double centre[3]) {
  CubeMap& m = *static_cast<CubeMap*>(h);
  m.roll(V3{centre[0], centre[1], centre[2]});
  for (int i = 0; i < nc; ++i) m.insert(m.corner, corner + 4 * (size_t)i);
  for (int i = 0; i < ns; ++i) m.insert(m.surf, surf + 4 * (size_t)i);
  m.filter_valid();
}

// one process() iteration.  corner_last / surf_last: sensor-frame less-sharp / less-flat clouds (xyzi packed);
// qt_odom: q_wodom_curr, t_wodom_curr; qt_out: q_w_curr, t_w_curr after the update.
ORC_API void orc_cubemap_frame(void* h, const float* corner_last, int nc, const float* surf_last, int ns, const double qt_odom[7],
                               double qt_out[7], OrcSolveSummary* summaries, OrcCubeFrameStats* st) {
  CubeMap& m = *static_cast<CubeMap*>(h);
  const Quat q_wodom{qt_odom[0], qt_odom[1], qt_odom[2], qt_odom[3]};
  const V3 t_wodom{qt_odom[4], qt_odom[5], qt_odom[6]};
  // transformAssociateToMap (:138-142)
  Quat q_w = qmul(m.q_wmap_wodom, q_wodom);
  V3 t_w = rotate(m.q_wmap_wodom, t_wodom) + m.t_wmap_wodom;
  m.roll(t_w);
  std::vector<float> map_c, map_s;
  for (int v = 0; v < m.n_valid; ++v) {
    map_c.insert(map_c.end(), m.corner[m.valid[v]].begin(), m.corner[m.valid[v]].end());
    map_s.insert(map_s.end(), m.surf[m.valid[v]].begin(), m.surf[m.valid[v]].end());
  }
  std::vector<float> stack_c((size_t)4 * std::max(nc, 1)), stack_s((size_t)4 * std::max(ns, 1));
  const int nsc = nc ? orc_voxelgrid(corner_last, nc, 16, 3, m.line_res, stack_c.data()) : 0;
  const int nss = ns ? orc_voxelgrid(surf_last, ns, 16, 3, m.plane_res, stack_s.data()) : 0;
  std::memset(st, 0, sizeof(*st));
  st->n_map_corner = (int)map_c.size() / 4, st->n_map_surf = (int)map_s.size() / 4;
  st->n_stack_corner = nsc, st->n_stack_surf = nss, st->n_valid = m.n_valid;
  double qt[7] = {q_w.x, q_w.y, q_w.z, q_w.w, t_w.x, t_w.y, t_w.z};
  if (m.solve && st->n_map_corner > 10 && st->n_map_surf > 50) {
    int32_t nfac[4];
    orc_register_aloam(map_c.data(), st->n_map_corner, map_s.data(), st->n_map_surf, 16, stack_c.data(), nsc, stack_s.data(),
                       nss, 16, qt, 2, 4, summaries, nfac);
    st->ran_optimization = 1;
  }
  q_w = Quat{qt[0], qt[1], qt[2], qt[3]};
  t_w = V3{qt[4], qt[5], qt[6]};
  // transformUpdate (:145-149): q_wmap_wodom = q_w * q_wodom^-1 ; t_wmap_wodom = t_w - q_wmap_wodom * t_wodom
  const double n2 = q_wodom.x * q_wodom.x + q_wodom.y * q_wodom.y + q_wodom.z * q_wodom.z + q_wodom.w * q_wodom.w;
  const Quat q_inv{-q_wodom.x / n2, -q_wodom.y / n2, -q_wodom.z / n2, q_wodom.w / n2};
  m.q_wmap_wodom = qmul(q_w, q_inv);
  m.t_wmap_wodom = t_w - rotate(m.q_wmap_wodom, t_wodom);
  // insertion of the stack points in the world frame (pointAssociateToMap keeps the intensity)
  for (int pass = 0; pass < 2; ++pass) {
    const std::vector<float>& stck = pass == 0 ? stack_c : stack_s;
    const int n = pass == 0 ? nsc : nss;
    for (int i = 0; i < n; ++i) {
      float pw[4];
      associate_to_map(q_w, t_w, &stck[4 * (size_t)i], pw);
      pw[3] = stck[4 * (size_t)i + 3];
      m.insert(pass == 0 ? m.corner : m.surf, pw);
    }
  }
  m.filter_valid();
  for (int i = 0; i < 7; ++i) qt_out[i] = qt[i];
  st->cen[0] = m.cenW, st->cen[1] = m.cenH, st->cen[2] = m.cenD;
}

// map-logic comparisons against the reference's own code run both sides without the registration
ORC_API void orc_cubemap_set_solve(void* h, int enabled) { static_cast<CubeMap*>(h)->solve = enabled != 0; }

// contents of one cube (array index) of the current window; returns the point count
ORC_API int orc_cubemap_cube(void* h, int which /*0 corner, 1 surf*/, int cube_index, float* out_xyzi, int cap) {
  CubeMap& m = *static_cast<CubeMap*>(h);
  const auto& v = which == 0 ? m.corner[cube_index] : m.surf[cube_index];
  const int n = (int)v.size() / 4;
  for (int i = 0; i < n && i < cap; ++i) std::memcpy(out_xyzi + 4 * (size_t)i, &v[4 * (size_t)i], 16);
  return n;
}
