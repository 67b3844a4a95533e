// ilsm.hpp -- C++ host side above the C ABI (include/ilsm.h): header-only objects with the NAMES, argument meaning and
// error behaviour of the library objects the reference nodes call on the registration hot path, so that the node
// bodies of himhan34/Intensity_based_LiDAR_SLAM_for_me- compile against them with a `using` line instead of an edit:
//
//   reference object / call site                                            drop-in here
//   pcl::KdTreeFLANN<PointType>   laserMapping.cpp:98-99, 631-634, 673,753  ilsm::KdTreeFLANN<PointT>
//                                 laserOdometry.cpp:282-283, 452,574, 807
//   pcl::VoxelGrid<PointType>     laserMapping.cpp:170-172, 608-616         ilsm::VoxelGrid<PointT>
//   KD_TREE (ikd-Tree)            mapOptimization.cpp:192, 393, 475, 224    ilsm::KD_TREE
//   SCManager                     Scancontext.h:58-110                      ilsm::SCManager
//   ImageHandler                  image_handler.h_ouster:14-140             ilsm::ImageHandler
//   association + ceres::Solve    laserMapping.cpp:640-861                  ilsm::ScanToMapRegistration
//   laserCloudHandler             scanRegistration.cpp:189-669              ilsm::ScanRegistration
//   process()                     laserMapping.cpp:233-1166                 ilsm::LaserMapping
//   mapOptimizationCallback       mapOptimization.cpp:99-500                ilsm::MapOptimization
//   the three LiDAR nodes chained (/os_cloud_node/points -> poses)           ilsm::LoamPipeline (synchronous or pipelined)
//   callback() (odometry merge)   odom_handler_node.cpp:44-132              ilsm::OdomHandler (host arithmetic only)
//   nh.param / getParam           spot.yaml + spot.launch:4-6               ilsm::Config (load_yaml / load_launch)
//
// Nothing here computes: every method forwards to libilsm_cuda.so (CUDA, sm_100a).  There is no CPU fallback; without a
// GPU the Context constructor throws ilsm::Error(ILSM_ERR_NO_DEVICE).
//
// Types: with PCL present (`__has_include(<pcl/point_types.h>)`) the classes are used with pcl::PointXYZI /
// pcl::PointCloud directly (any PointT whose first three floats are x,y,z and whose size is 16 or 32 bytes).  Without
// PCL (this repository's image) ilsm::PointXYZI / ilsm::PointXYZ / ilsm::PointCloud below have the same memory layout
// (parameters.h_ouster:121-124) and the subset of the interface the reference uses.
// Error behaviour: the reference's call sites are void and report with printf / ROS_WARN.  The methods that mirror a
// reference method keep its signature and return convention (e.g. nearestKSearch returns the number of neighbours
// found, 0 on failure) and print the library's error text on stderr; everything else throws ilsm::Error.
#ifndef ILSM_HPP_
#define ILSM_HPP_

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "ilsm.h"

namespace ilsm {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};
inline void check(int rc, const char* where) {
  if (rc != ILSM_OK) throw Error(rc, std::string(where) + ": " + ilsm_last_error());
}
inline bool warn(int rc, const char* where) {  // the reference's style: report and carry on
  if (rc != ILSM_OK) std::fprintf(stderr, "[ilsm] %s: %s\n", where, ilsm_last_error());
  return rc == ILSM_OK;
}

// ------------------------------------------------------------------------------------------------ point types
struct alignas(16) PointXYZ {  // pcl::PointXYZ: 16 bytes
  float x = 0, y = 0, z = 0, pad_ = 1.f;
};
struct alignas(16) PointXYZI {  // pcl::PointXYZI: 32 bytes, intensity at byte 16
  float x = 0, y = 0, z = 0, pad_ = 1.f;
  float intensity = 0, pad1_[3] = {0, 0, 0};
};
static_assert(sizeof(PointXYZ) == 16 && sizeof(PointXYZI) == 32, "PCL point layout");

template <typename PointT>
struct PointCloud {  // the subset of pcl::PointCloud the reference uses
  typedef std::shared_ptr<PointCloud<PointT>> Ptr;
  typedef std::shared_ptr<const PointCloud<PointT>> ConstPtr;
  std::vector<PointT> points;
  uint32_t width = 0, height = 1;
  bool is_dense = true;
  size_t size() const { return points.size(); }
  bool empty() const { return points.empty(); }
  void clear() { points.clear(), width = 0, height = 1; }
  void resize(size_t n) { points.resize(n), width = (uint32_t)n, height = 1; }
  void push_back(const PointT& p) { points.push_back(p), width = (uint32_t)points.size(), height = 1; }
  PointT& operator[](size_t i) { return points[i]; }
  const PointT& operator[](size_t i) const { return points[i]; }
  PointCloud& operator+=(const PointCloud& o) {
    points.insert(points.end(), o.points.begin(), o.points.end());
    width = (uint32_t)points.size(), height = 1;
    return *this;
  }
};

template <typename CloudT>
inline const float* cloud_ptr(const CloudT& c) {
  return c.points.empty() ? nullptr : reinterpret_cast<const float*>(c.points.data());
}
template <typename PointT>
constexpr int stride_of() {
  static_assert(sizeof(PointT) == 16 || sizeof(PointT) == 32, "PointT must be a 16- or 32-byte PCL point");
  return (int)sizeof(PointT);
}

// ------------------------------------------------------------------------------------------------ context
// One per thread of the reference's mapping loop (laserMapping.cpp:1215); shared by the objects built on it.
class Context {
 public:
  explicit Context(int device = 0) { check(ilsm_create(device, &h_), "ilsm_create"); }
  ~Context() { ilsm_destroy(h_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  ilsm_ctx* get() const { return h_; }
  void sync() const { check(ilsm_sync(h_), "ilsm_sync"); }
  static std::shared_ptr<Context> shared(int device = 0) {  // process-wide default, like the reference's globals
    static std::weak_ptr<Context> w;
    std::shared_ptr<Context> s = w.lock();
    if (!s) w = s = std::make_shared<Context>(device);
    return s;
  }

 private:
  ilsm_ctx* h_ = nullptr;
};
typedef std::shared_ptr<Context> ContextPtr;

// ------------------------------------------------------------------------------------------------ pcl::KdTreeFLANN
template <typename PointT>
class KdTreeFLANN {
 public:
  typedef PointCloud<PointT> Cloud;
  typedef std::shared_ptr<KdTreeFLANN<PointT>> Ptr;
  explicit KdTreeFLANN(ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {
    check(ilsm_map_create(ctx_->get(), &map_), "ilsm_map_create");
  }
  ~KdTreeFLANN() { ilsm_map_destroy(map_); }
  KdTreeFLANN(const KdTreeFLANN&) = delete;
  KdTreeFLANN& operator=(const KdTreeFLANN&) = delete;

  // kdtreeCornerFromMap->setInputCloud(laserCloudCornerFromMap)   laserMapping.cpp:631-634
  template <typename CloudT>
  void setInputCloud(const std::shared_ptr<CloudT>& cloud) { setInputCloud(*cloud); }
  template <typename CloudT>
  void setInputCloud(const CloudT& cloud) {
    typedef typename std::remove_reference<decltype(cloud.points[0])>::type P;
    warn(ilsm_map_build(map_, cloud_ptr(cloud), (int)cloud.points.size(), (int)sizeof(P), 0.f), "setInputCloud");
  }
  // kdtree->nearestKSearch(pointSel, 5, pointSearchInd, pointSearchSqDis)   laserMapping.cpp:673,753
  // returns the number of neighbours found (PCL's convention); vectors are resized to k like PCL does.
  int nearestKSearch(const PointT& p, int k, std::vector<int>& k_indices, std::vector<float>& k_sqr_distances) const {
    k_indices.assign(k, -1);
    k_sqr_distances.assign(k, std::numeric_limits<float>::infinity());
    if (!warn(ilsm_knn(map_, &p.x, 1, stride_of<PointT>(), k, 0.f, k_indices.data(), k_sqr_distances.data()), "nearestKSearch"))
      return 0;
    int found = 0;
    while (found < k && k_indices[found] >= 0) ++found;
    k_indices.resize(found), k_sqr_distances.resize(found);
    return found;
  }
  // Batched form (what a GPU wants): all points of `queries` at once, results nq x k row-major, -1 / +inf padded.
  template <typename CloudT>
  int nearestKSearch(const CloudT& queries, int k, std::vector<int>& k_indices, std::vector<float>& k_sqr_distances,
                     float max_dist = 0.f) const {
    typedef typename std::remove_reference<decltype(queries.points[0])>::type P;
    const int nq = (int)queries.points.size();
    k_indices.assign((size_t)nq * k, -1);
    k_sqr_distances.assign((size_t)nq * k, std::numeric_limits<float>::infinity());
    if (nq == 0) return 0;
    return warn(ilsm_knn(map_, cloud_ptr(queries), nq, (int)sizeof(P), k, max_dist, k_indices.data(), k_sqr_distances.data()),
                "nearestKSearch(batch)") ? nq : 0;
  }
  int size() const { return ilsm_map_size(map_); }
  ilsm_map* handle() const { return map_; }
  const ContextPtr& context() const { return ctx_; }

 private:
  ContextPtr ctx_;
  ilsm_map* map_ = nullptr;
};

// ------------------------------------------------------------------------------------------------ pcl::VoxelGrid
template <typename PointT>
class VoxelGrid {
 public:
  explicit VoxelGrid(ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {}
  // downSizeFilterCorner.setLeafSize(lineRes, lineRes, lineRes)   laserMapping.cpp:1181-1182 (cubic leaves only)
  void setLeafSize(float lx, float ly, float lz) {
    if (lx != ly || ly != lz) throw Error(ILSM_ERR_INVALID_ARG, "VoxelGrid: only cubic leaves (the reference uses no other)");
    leaf_ = lx;
  }
  template <typename CloudT>
  void setInputCloud(const std::shared_ptr<CloudT>& cloud) { in_ = cloud_ptr(*cloud), n_ = (int)cloud->points.size(); }
  // downSizeFilterCorner.filter(*laserCloudCornerStack)   laserMapping.cpp:608-616
  template <typename CloudT>
  void filter(CloudT& out) {
    static_assert(sizeof(PointT) == 32, "VoxelGrid mirrors pcl::VoxelGrid<pcl::PointXYZI>");
    std::vector<float> packed((size_t)(n_ > 0 ? n_ : 1) * 4);
    int n_out = 0;
    if (!warn(ilsm_voxelgrid(ctx_->get(), in_, n_, 32, leaf_, packed.data(), &n_out), "VoxelGrid::filter")) n_out = 0;
    out.points.resize(n_out);
    for (int i = 0; i < n_out; ++i) {
      PointT& p = out.points[i];
      p.x = packed[4 * i], p.y = packed[4 * i + 1], p.z = packed[4 * i + 2], p.intensity = packed[4 * i + 3];
    }
    out.width = (uint32_t)n_out, out.height = 1, out.is_dense = true;
  }

 private:
  ContextPtr ctx_;
  float leaf_ = 0.4f;
  const float* in_ = nullptr;
  int n_ = 0;
};

// ------------------------------------------------------------------------------------------------ ikd-Tree KD_TREE
struct ikdTree_PointType {  // ikd_Tree.h:22-31
  float x, y, z;
  ikdTree_PointType(float px = 0.0f, float py = 0.0f, float pz = 0.0f) : x(px), y(py), z(pz) {}
};
enum delete_point_storage_set { NOT_RECORD, DELETE_POINTS_REC, MULTI_THREAD_REC };  // ikd_Tree.h:42

class KD_TREE {
 public:
  typedef ikdTree_PointType PointType;
  typedef std::vector<PointType> PointVector;
  // KD_TREE(delete_param, balance_param, box_length)   ikd_Tree.h:257 -- the re-balancing criteria have no meaning for
  // the voxel hash and are accepted and ignored; box_length is the down-sampling box of Add_Points.
  explicit KD_TREE(float /*delete_param*/ = 0.5f, float /*balance_param*/ = 0.6f, float box_length = 0.2f,
                   ContextPtr ctx = Context::shared())
      : ctx_(std::move(ctx)), box_(box_length) {
    check(ilsm_map_create(ctx_->get(), &map_), "ilsm_map_create");
  }
  ~KD_TREE() { ilsm_map_destroy(map_); }
  KD_TREE(const KD_TREE&) = delete;
  KD_TREE& operator=(const KD_TREE&) = delete;
  void set_downsample_param(float box_length) { box_ = box_length; }  // ikd_Tree.h:261
  void InitializeKDTree(float = 0.5f, float = 0.7f, float box_length = 0.2f) { box_ = box_length; }
  int size() const { return ilsm_map_size(map_); }
  // ikdtree->Build(points)   mapOptimization.cpp:192
  void Build(const PointVector& pts) {
    flat_valid_ = false;
    warn(ilsm_map_build(map_, pts.empty() ? nullptr : &pts[0].x, (int)pts.size(), 12, 0.f), "KD_TREE::Build");
  }
  // ikdtree->Nearest_Search(point, 5, points_near, pointSearchSqDis)   mapOptimization.cpp:393 -- neighbours as points,
  // ascending distance; fewer than k entries when the tree holds fewer points (ikd_Tree.cpp:495-547).
  void Nearest_Search(PointType point, int k_nearest, PointVector& Nearest_Points, std::vector<float>& Point_Distance,
                      double max_dist = INFINITY) {
    Nearest_Points.clear(), Point_Distance.clear();
    if (k_nearest < 1 || k_nearest > 8) { warn(ILSM_ERR_INVALID_ARG, "Nearest_Search: 1 <= k <= 8"); return; }
    int32_t idx[8];
    float d2[8];
    const float md = std::isfinite(max_dist) ? (float)max_dist : 0.f;
    if (!warn(ilsm_knn(map_, &point.x, 1, 12, k_nearest, md, idx, d2), "Nearest_Search")) return;
    ensure_flat();
    for (int i = 0; i < k_nearest && idx[i] >= 0; ++i) {
      if (md > 0.f && !(d2[i] <= md * md)) break;
      Nearest_Points.push_back(PointType(flat_[4 * (size_t)idx[i]], flat_[4 * (size_t)idx[i] + 1], flat_[4 * (size_t)idx[i] + 2]));
      Point_Distance.push_back(d2[i]);
    }
  }
  // ikdtree->Add_Points(points, true)   mapOptimization.cpp:475 ; returns the number of points handed in, like
  // ikd_Tree.cpp:570-640 returns its loop counter.
  int Add_Points(PointVector& PointToAdd, bool downsample_on) {
    if (PointToAdd.empty()) return 0;
    flat_valid_ = false;
    warn(ilsm_map_insert(map_, &PointToAdd[0].x, (int)PointToAdd.size(), 12,
                         downsample_on ? ILSM_INSERT_NEAREST_TO_CENTRE : ILSM_INSERT_APPEND, box_), "Add_Points");
    return (int)PointToAdd.size();
  }
  // ikdtree->flatten(ikdtree->Root_Node, storage, NOT_RECORD)   mapOptimization.cpp:224 (Root_Node has no counterpart:
  // pass nullptr or use the one-argument form)
  void flatten(const void* /*root*/, PointVector& Storage, delete_point_storage_set /*storage_type*/ = NOT_RECORD) { flatten(Storage); }
  void flatten(PointVector& Storage) {
    ensure_flat();
    Storage.resize(flat_.size() / 4);
    for (size_t i = 0; i < Storage.size(); ++i) Storage[i] = PointType(flat_[4 * i], flat_[4 * i + 1], flat_[4 * i + 2]);
  }
  void* Root_Node = nullptr;  // so that `tree->flatten(tree->Root_Node, ...)` compiles unchanged
  ilsm_map* handle() const { return map_; }

 private:
  void ensure_flat() {
    if (flat_valid_ && (int)(flat_.size() / 4) == size()) return;
    int n = size(), got = 0;
    flat_.resize((size_t)(n > 0 ? n : 1) * 4);
    flat_valid_ = warn(ilsm_map_points(map_, flat_.data(), n, &got), "flatten");
    flat_.resize((size_t)got * 4);
  }
  ContextPtr ctx_;
  ilsm_map* map_ = nullptr;
  float box_;
  std::vector<float> flat_;  // host copy of the map points, refreshed lazily after Build / Add_Points
  bool flat_valid_ = false;
};
// ------------------------------------------------------------------------------------------------ SCManager
// Descriptors are 20 x 60 row-major (ring, sector).  The reference returns Eigen::MatrixXd; without Eigen in the build
// the same numbers come back as std::vector<double> (row-major); with Eigen, wrap them in
// Eigen::Map<Eigen::Matrix<double, 20, 60, Eigen::RowMajor>>.
class SCManager {
 public:
  const double LIDAR_HEIGHT = 2.0;       // Scancontext.h:77-96
  const int PC_NUM_RING = 20, PC_NUM_SECTOR = 60;
  const double PC_MAX_RADIUS = 80.0;
  const double PC_UNIT_SECTORANGLE = 360.0 / 60.0;
  const int NUM_EXCLUDE_RECENT = 50;
  const int NUM_CANDIDATES_FROM_TREE = 10;
  const double SC_DIST_THRES = 0.13;
  const int TREE_MAKING_PERIOD_ = 50;
  int tree_making_period_conter = 0;

  explicit SCManager(ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {
    check(ilsm_sc_create(ctx_->get(), &sc_), "ilsm_sc_create");
  }
  ~SCManager() { ilsm_sc_destroy(sc_); }
  SCManager(const SCManager&) = delete;
  SCManager& operator=(const SCManager&) = delete;

  // SCManager::makeScancontext   Scancontext.cpp:160-204
  template <typename CloudT>
  std::vector<double> makeScancontext(const CloudT& scan_down) {
    typedef typename std::remove_reference<decltype(scan_down.points[0])>::type P;
    std::vector<float> d(1200);
    check(ilsm_sc_make(sc_, cloud_ptr(scan_down), (int)scan_down.points.size(), (int)sizeof(P), d.data()), "makeScancontext");
    return std::vector<double>(d.begin(), d.end());
  }
  // SCManager::makeAndSaveScancontextAndKeys   Scancontext.cpp:237-251
  template <typename CloudT>
  void makeAndSaveScancontextAndKeys(const CloudT& scan_down) {
    typedef typename std::remove_reference<decltype(scan_down.points[0])>::type P;
    last_.resize(1200);
    if (!warn(ilsm_sc_make(sc_, cloud_ptr(scan_down), (int)scan_down.points.size(), (int)sizeof(P), last_.data()),
              "makeAndSaveScancontextAndKeys"))
      return;
    warn(ilsm_sc_add(sc_, last_.data(), 1), "makeAndSaveScancontextAndKeys");
  }
  // SCManager::detectLoopClosureID   Scancontext.cpp:253-344: {loop id or -1, yaw difference in radians}.
  // Reference-exact by default: the search window is entries [0, size - NUM_EXCLUDE_RECENT) as of the last tree rebuild
  // (every TREE_MAKING_PERIOD_ calls, :270-282), the NUM_CANDIDATES_FROM_TREE nearest float ring keys are selected and
  // only those are scored (ilsm_sc_query_candidates), the first strictly smaller candidate distance wins (:299-312),
  // SC_DIST_THRES decides.  exhaustive_search = true scores EVERY entry of the window instead (a superset: it can find
  // a loop the ring-key pre-selection misses, so its answer may differ from the reference's).
  bool exhaustive_search = false;
  std::pair<int, float> detectLoopClosureID() {
    const int n = ilsm_sc_size(sc_);
    if (n < NUM_EXCLUDE_RECENT + 1 || last_.empty()) return std::make_pair(-1, 0.0f);
    if (tree_making_period_conter % TREE_MAKING_PERIOD_ == 0) n_search_ = n - NUM_EXCLUDE_RECENT;
    tree_making_period_conter += 1;
    double min_dist = 10000000;
    int nn_align = 0, nn_idx = 0;
    if (n_search_ <= 0) return std::make_pair(-1, 0.0f);
    if (exhaustive_search) {
      double dist = 0;
      int32_t id = -1, shift = 0;
      if (!warn(ilsm_sc_query_topk(sc_, last_.data(), n_search_, 0, 1, &dist, &id, &shift), "detectLoopClosureID"))
        return std::make_pair(-1, 0.0f);
      if (id >= 0) min_dist = dist, nn_align = shift, nn_idx = id;
    } else {
      int32_t cid[16], csh[16];
      double cd[16];
      if (!warn(ilsm_sc_query_candidates(sc_, last_.data(), n_search_, NUM_CANDIDATES_FROM_TREE, cid, nullptr, cd, csh),
                "detectLoopClosureID"))
        return std::make_pair(-1, 0.0f);
      for (int i = 0; i < NUM_CANDIDATES_FROM_TREE; ++i) {
        if (cid[i] < 0) continue;
        if (cd[i] < min_dist) min_dist = cd[i], nn_align = csh[i], nn_idx = cid[i];
      }
    }
    last_dist_ = min_dist;
    const float yaw_diff_rad = (float)(nn_align * PC_UNIT_SECTORANGLE * M_PI / 180.0);
    return std::make_pair(min_dist < SC_DIST_THRES ? nn_idx : -1, yaw_diff_rad);
  }
  double lastDistance() const { return last_dist_; }
  int size() const { return ilsm_sc_size(sc_); }
  ilsm_sc* handle() const { return sc_; }

 private:
  ContextPtr ctx_;
  ilsm_sc* sc_ = nullptr;
  std::vector<float> last_;
  int n_search_ = 0;
  double last_dist_ = 0;
};

// ------------------------------------------------------------------------------------------------ pcl::IterativeClosestPoint
// Eigen::Matrix4f's layout without Eigen: 16 floats, column-major, m(r, c).
struct Matrix4f {
  float m[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  static Matrix4f Identity() { return Matrix4f(); }
  float& operator()(int r, int c) { return m[c * 4 + r]; }
  float operator()(int r, int c) const { return m[c * 4 + r]; }
};

// Rigid transform (rotation block + translation column) -> (qx, qy, qz, qw, tx, ty, tz), in double.
inline void matrix_to_pose7(const Matrix4f& T, double out[7]) {
  double R[3][3];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) R[r][c] = T(r, c);
  const double tr = R[0][0] + R[1][1] + R[2][2];
  double x, y, z, w;
  if (tr > 0) {
    const double s = std::sqrt(tr + 1.0) * 2;
    w = 0.25 * s, x = (R[2][1] - R[1][2]) / s, y = (R[0][2] - R[2][0]) / s, z = (R[1][0] - R[0][1]) / s;
  } else if (R[0][0] > R[1][1] && R[0][0] > R[2][2]) {
    const double s = std::sqrt(1.0 + R[0][0] - R[1][1] - R[2][2]) * 2;
    w = (R[2][1] - R[1][2]) / s, x = 0.25 * s, y = (R[0][1] + R[1][0]) / s, z = (R[0][2] + R[2][0]) / s;
  } else if (R[1][1] > R[2][2]) {
    const double s = std::sqrt(1.0 + R[1][1] - R[0][0] - R[2][2]) * 2;
    w = (R[0][2] - R[2][0]) / s, x = (R[0][1] + R[1][0]) / s, y = 0.25 * s, z = (R[1][2] + R[2][1]) / s;
  } else {
    const double s = std::sqrt(1.0 + R[2][2] - R[0][0] - R[1][1]) * 2;
    w = (R[1][0] - R[0][1]) / s, x = (R[0][2] + R[2][0]) / s, y = (R[1][2] + R[2][1]) / s, z = 0.25 * s;
  }
  const double n = std::sqrt(x * x + y * y + z * z + w * w);
  out[0] = x / n, out[1] = y / n, out[2] = z / n, out[3] = w / n;
  out[4] = T(0, 3), out[5] = T(1, 3), out[6] = T(2, 3);
}

inline Matrix4f pose7_to_matrix(const double q[4], const double t[3]) {
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  Matrix4f T;
  T(0, 0) = (float)(1 - 2 * (y * y + z * z)), T(0, 1) = (float)(2 * (x * y - w * z)), T(0, 2) = (float)(2 * (x * z + w * y));
  T(1, 0) = (float)(2 * (x * y + w * z)), T(1, 1) = (float)(1 - 2 * (x * x + z * z)), T(1, 2) = (float)(2 * (y * z - w * x));
  T(2, 0) = (float)(2 * (x * z - w * y)), T(2, 1) = (float)(2 * (y * z + w * x)), T(2, 2) = (float)(1 - 2 * (x * x + y * y));
  T(0, 3) = (float)t[0], T(1, 3) = (float)t[1], T(2, 3) = (float)t[2];
  return T;
}

// icp.setInputSource(cur); icp.setInputTarget(submap); icp.align(result, guess);
// if (icp.hasConverged() && icp.getFitnessScore() < threshold) ...   loopClosureThread, intensity_feature_tracker.cpp:195-393
// One align() is a batch of one of ilsm_icp_align_batch; the pose is kept in double (lastResult()) and rounded into the
// Matrix4f of getFinalTransformation().
template <typename PointSource, typename PointTarget>
class IterativeClosestPoint {
 public:
  typedef PointCloud<PointSource> SourceCloud;
  explicit IterativeClosestPoint(ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {
    check(ilsm_map_create(ctx_->get(), &target_), "ilsm_map_create");
    ilsm_icp_opts_default(&opts_);
    res_ = ilsm_icp_result();
  }
  ~IterativeClosestPoint() { ilsm_map_destroy(target_); }
  IterativeClosestPoint(const IterativeClosestPoint&) = delete;
  IterativeClosestPoint& operator=(const IterativeClosestPoint&) = delete;

  template <typename CloudT>
  void setInputSource(const std::shared_ptr<CloudT>& cloud) { setInputSource(*cloud); }
  template <typename CloudT>
  void setInputSource(const CloudT& cloud) {
    src_.resize(cloud.points.size() * 3);
    for (size_t i = 0; i < cloud.points.size(); ++i)
      src_[3 * i] = cloud.points[i].x, src_[3 * i + 1] = cloud.points[i].y, src_[3 * i + 2] = cloud.points[i].z;
  }
  // the target's search structure is built here, once, like PCL's k-d tree
  template <typename CloudT>
  void setInputTarget(const std::shared_ptr<CloudT>& cloud) { setInputTarget(*cloud); }
  template <typename CloudT>
  void setInputTarget(const CloudT& cloud) {
    typedef typename std::remove_reference<decltype(cloud.points[0])>::type P;
    check(ilsm_map_build(target_, cloud_ptr(cloud), (int)cloud.points.size(), stride_of<P>(), 0.f), "setInputTarget");
  }
  void setMaxCorrespondenceDistance(double d) { opts_.max_correspondence_distance = d; }
  void setMaximumIterations(int n) { opts_.max_iterations = n; }
  void setTransformationEpsilon(double e) { opts_.transformation_epsilon = e; }
  void setTransformationRotationEpsilon(double e) { opts_.transformation_rotation_epsilon = e; }
  void setEuclideanFitnessEpsilon(double e) { opts_.euclidean_fitness_epsilon = e; }
  void setRANSACIterations(int n) {  // no correspondence rejector is implemented: only PCL's "none" (0) is honoured
    if (n != 0) std::fprintf(stderr, "[ilsm] IterativeClosestPoint::setRANSACIterations(%d) ignored: no rejector\n", n);
  }

  void align(SourceCloud& output) { align(output, Matrix4f::Identity()); }
  void align(SourceCloud& output, const Matrix4f& guess) {
    double g[7];
    matrix_to_pose7(guess, g);
    const int offs[2] = {0, (int)(src_.size() / 3)};
    ilsm_map* tg = target_;
    check(ilsm_icp_align_batch(ctx_->get(), &tg, 1, src_.empty() ? nullptr : src_.data(), offs, 12, g, &opts_, &res_),
          "IterativeClosestPoint::align");
    final_ = pose7_to_matrix(res_.q_xyzw, res_.t);
    output.resize(src_.size() / 3);
    for (size_t i = 0; i < output.points.size(); ++i) {  // the source under the final transformation
      const float* p = &src_[3 * i];
      PointSource& o = output.points[i];
      o.x = final_(0, 0) * p[0] + final_(0, 1) * p[1] + final_(0, 2) * p[2] + final_(0, 3);
      o.y = final_(1, 0) * p[0] + final_(1, 1) * p[1] + final_(1, 2) * p[2] + final_(1, 3);
      o.z = final_(2, 0) * p[0] + final_(2, 1) * p[1] + final_(2, 2) * p[2] + final_(2, 3);
    }
  }
  bool hasConverged() const { return res_.converged != 0; }
  double getFitnessScore() const { return res_.fitness; }  // PCL's default range: every point
  Matrix4f getFinalTransformation() const { return final_; }
  const ilsm_icp_result& lastResult() const { return res_; }

 private:
  ContextPtr ctx_;
  ilsm_map* target_ = nullptr;
  std::vector<float> src_;
  ilsm_icp_opts opts_;
  ilsm_icp_result res_;
  Matrix4f final_;
};

// ------------------------------------------------------------------------------------------------ loop closure per keyframe
// The body of loopClosureThread (intensity_feature_tracker.cpp:195-393) over ilsm_loop: every keyframe passed in is stored
// on the device and answered with its loop decision (ScanContext detection, ICP verification of the best candidate
// against the world-frame submap of its neighbours).  Give it a Context of its own when the mapping loop runs on another
// thread, as the reference runs loopClosureThread on its own.
class LoopClosure {
 public:
  explicit LoopClosure(ContextPtr ctx = Context::shared(), const ilsm_loop_opts* opts = nullptr) : ctx_(std::move(ctx)) {
    check(ilsm_loop_create(ctx_->get(), opts, &h_), "ilsm_loop_create");
  }
  ~LoopClosure() { ilsm_loop_destroy(h_); }
  LoopClosure(const LoopClosure&) = delete;
  LoopClosure& operator=(const LoopClosure&) = delete;

  // cloud: the keyframe's points (16- or 32-byte PCL points) in its own frame; (q, t): its world pose.  Returns
  // result->accepted.
  template <typename CloudT>
  bool addKeyframe(const CloudT& cloud, const double q_xyzw[4], const double t_xyz[3], ilsm_loop_result* result) {
    typedef typename std::remove_reference<decltype(cloud.points[0])>::type P;
    check(ilsm_loop_add_keyframe(h_, cloud_ptr(cloud), (int)cloud.points.size(), stride_of<P>(), q_xyzw, t_xyz, result),
          "LoopClosure::addKeyframe");
    return result->accepted != 0;
  }
  int size() const { return ilsm_loop_size(h_); }
  ilsm_loop* handle() const { return h_; }

 private:
  ContextPtr ctx_;
  ilsm_loop* h_ = nullptr;
};

// ------------------------------------------------------------------------------------------------ ImageHandler
class ImageHandler {
 public:
  int IMAGE_HEIGHT, IMAGE_WIDTH, NUM_THREADS;
  std::vector<uint8_t> image_range, image_intensity, image_ambient;  // H x W row-major (cv::Mat CV_8UC1 data)
  PointCloud<PointXYZI>::Ptr cloud_track;
  PointCloud<PointXYZ>::Ptr GroundPointOut;
  float ground_coeff[4] = {0, 0, 0, 0};

  // ImageHandler(height, width, threadNum)   image_handler.h_ouster:30-39
  explicit ImageHandler(int height = 128, int width = 1024, int threadNum = 6, ContextPtr ctx = Context::shared())
      : IMAGE_HEIGHT(height), IMAGE_WIDTH(width), NUM_THREADS(threadNum), ctx_(std::move(ctx)) {
    cloud_track.reset(new PointCloud<PointXYZI>());
    cloud_track->resize((size_t)height * width);
    GroundPointOut.reset(new PointCloud<PointXYZ>());
    check(ilsm_ground_create(ctx_->get(), &ground_), "ilsm_ground_create");
  }
  ~ImageHandler() { ilsm_ground_destroy(ground_); }
  ImageHandler(const ImageHandler&) = delete;
  ImageHandler& operator=(const ImageHandler&) = delete;

  // cloud_handler(cloud_msg)   image_handler.h_ouster:103-140, after pcl::fromROSMsg: the organised cloud, u * W + v
  template <typename CloudT>
  void cloud_handler(const CloudT& laser_cloud) {
    typedef typename std::remove_reference<decltype(laser_cloud.points[0])>::type P;
    const size_t hw = (size_t)IMAGE_HEIGHT * IMAGE_WIDTH;
    if (laser_cloud.points.size() != hw) { warn(ILSM_ERR_INVALID_ARG, "cloud_handler: cloud is not IMAGE_HEIGHT x IMAGE_WIDTH"); return; }
    image_range.assign(hw, 0), image_intensity.assign(hw, 0), image_ambient.assign(hw, 0);
    std::vector<float> track(hw * 4);
    if (!warn(ilsm_project(ctx_->get(), cloud_ptr(laser_cloud), IMAGE_HEIGHT, IMAGE_WIDTH, (int)sizeof(P), image_range.data(),
                           image_intensity.data(), track.data()), "cloud_handler"))
      return;
    cloud_track->resize(hw);
    for (size_t i = 0; i < hw; ++i) {
      PointXYZI& p = cloud_track->points[i];
      p.x = track[4 * i], p.y = track[4 * i + 1], p.z = track[4 * i + 2], p.intensity = track[4 * i + 3];
    }
  }
  // groundPlaneExtraction(cloud_msg)   image_handler.h_ouster:41-100: fills GroundPointOut
  template <typename CloudT>
  void groundPlaneExtraction(const CloudT& cloud, const ilsm_ground_opts* opts = nullptr, ilsm_ground_info* info = nullptr) {
    typedef typename std::remove_reference<decltype(cloud.points[0])>::type P;
    const int n = (int)cloud.points.size();
    GroundPointOut->points.clear();
    std::vector<float> out((size_t)(n > 0 ? n : 1) * 4);
    int n_out = 0;
    if (!warn(ilsm_ground_extract(ground_, cloud_ptr(cloud), n, (int)sizeof(P), opts, out.data(), n, &n_out, ground_coeff, info),
              "groundPlaneExtraction"))
      return;
    GroundPointOut->resize(n_out);
    for (int i = 0; i < n_out; ++i) {
      PointXYZ& p = GroundPointOut->points[i];
      p.x = out[4 * i], p.y = out[4 * i + 1], p.z = out[4 * i + 2];
    }
  }

 private:
  ContextPtr ctx_;
  ilsm_ground* ground_ = nullptr;
};

// ------------------------------------------------------------------------------------------------ registration block
// The body of `if (laserCloudCornerFromMapNum > 10 && laserCloudSurfFromMapNum > 50)` (laserMapping.cpp:624-875): two
// kd-trees, 2 x (association + ceres::Solve).  `parameters` is the reference's double[7] = {qx,qy,qz,qw, tx,ty,tz}
// (laserMapping.cpp:105-107), updated in place like Ceres does.
template <typename PointT>
class ScanToMapRegistration {
  ContextPtr ctx_;  // declared first: the kd-trees below are built on it

 public:
  explicit ScanToMapRegistration(ContextPtr ctx = Context::shared())
      : ctx_(ctx), kdtreeCornerFromMap(ctx), kdtreeSurfFromMap(ctx) {
    ilsm_reg_opts_default(&options);
    warn(ilsm_set_async(ctx_->get(), 1), "ilsm_set_async");  // the two setInputCloud replacements overlap
  }
  ilsm_reg_opts options;        // laserMapping values; mapOptimization: outer 1, max_num_iterations 10, min_*_map 0
  ilsm_reg_report report;       // per-pass ceres::Solver::Summary fields + corner_num / surf_num
  KdTreeFLANN<PointT> kdtreeCornerFromMap, kdtreeSurfFromMap;
  // returns false when the guard of laserMapping.cpp:624 skips the optimisation ("Map corner and surf num are not enough")
  template <typename CloudT>
  bool align(const CloudT& cornerFromMap, const CloudT& surfFromMap, const CloudT& cornerStack, const CloudT& surfStack,
             double parameters[7]) {
    kdtreeCornerFromMap.setInputCloud(cornerFromMap);
    kdtreeSurfFromMap.setInputCloud(surfFromMap);
    std::memset(&report, 0, sizeof(report));
    const int rc = ilsm_register(ctx_->get(), kdtreeCornerFromMap.handle(), kdtreeSurfFromMap.handle(), cloud_ptr(cornerStack),
                                 (int)cornerStack.points.size(), cloud_ptr(surfStack), (int)surfStack.points.size(),
                                 stride_of<PointT>(), parameters, parameters + 4, &options, &report);
    if (rc == ILSM_ERR_NOT_ENOUGH_MAP) return false;
    check(rc, "ilsm_register");
    return true;
  }
};

// ------------------------------------------------------------------------------------------------ node bodies
// laserCloudHandler (scanRegistration.cpp:189-669): the five clouds it publishes.
class ScanRegistration {
 public:
  explicit ScanRegistration(float minimum_range = 0.3f, ContextPtr ctx = Context::shared())
      : MINIMUM_RANGE(minimum_range), ctx_(std::move(ctx)) {}
  float MINIMUM_RANGE;  // scanRegistration.cpp:59, `minimum_range` param
  PointCloud<PointXYZI> laserCloud, cornerPointsSharp, cornerPointsLessSharp, surfPointsFlat, surfPointsLessFlat;
  ilsm_feature_counts counts;
  template <typename CloudT>
  void laserCloudHandler(const CloudT& laserCloudIn) {
    typedef typename std::remove_reference<decltype(laserCloudIn.points[0])>::type P;
    const int n = (int)laserCloudIn.points.size();
    const size_t cap = (size_t)(n > 0 ? n : 1);
    std::vector<float> cloud(cap * 4), lflat(cap * 4);
    std::vector<int32_t> sharp(cap), lsharp(cap), flat(cap);
    ilsm_features f;
    std::memset(&f, 0, sizeof(f));
    f.cloud_xyzi = cloud.data(), f.sharp_idx = sharp.data(), f.less_sharp_idx = lsharp.data(), f.flat_idx = flat.data();
    f.less_flat_xyzi = lflat.data();
    check(ilsm_extract_features(ctx_->get(), cloud_ptr(laserCloudIn), n, (int)sizeof(P), MINIMUM_RANGE, &f), "laserCloudHandler");
    counts = f.counts;
    fill(laserCloud, cloud.data(), nullptr, counts.n_cloud);
    fill(cornerPointsSharp, cloud.data(), sharp.data(), counts.n_sharp);
    fill(cornerPointsLessSharp, cloud.data(), lsharp.data(), counts.n_less_sharp);
    fill(surfPointsFlat, cloud.data(), flat.data(), counts.n_flat);
    fill(surfPointsLessFlat, lflat.data(), nullptr, counts.n_less_flat);
  }

 private:
  static void fill(PointCloud<PointXYZI>& out, const float* xyzi, const int32_t* idx, int n) {
    out.resize(n);
    for (int i = 0; i < n; ++i) {
      const float* s = xyzi + 4 * (size_t)(idx ? idx[i] : i);
      out.points[i].x = s[0], out.points[i].y = s[1], out.points[i].z = s[2], out.points[i].intensity = s[3];
    }
  }
  ContextPtr ctx_;
};

// process() of laserMapping.cpp:233-1166 for one frame: the rolling 21 x 21 x 11 cube map lives in HBM.
class LaserMapping {
 public:
  LaserMapping(float lineRes = 0.4f, float planeRes = 0.8f, ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {
    check(ilsm_cubemap_create(ctx_->get(), lineRes, planeRes, 0, &cm_), "ilsm_cubemap_create");
  }
  ~LaserMapping() { ilsm_cubemap_destroy(cm_); }
  LaserMapping(const LaserMapping&) = delete;
  LaserMapping& operator=(const LaserMapping&) = delete;
  double parameters[7] = {0, 0, 0, 1, 0, 0, 0};  // q_w_curr (x,y,z,w), t_w_curr   laserMapping.cpp:105-107
  ilsm_reg_report report;
  ilsm_cubemap_stats stats;
  // q_wodom_curr / t_wodom_curr = the odometry pose of /laser_odom_to_init (laserMapping.cpp:305-311)
  template <typename CloudT>
  void process(const CloudT& laserCloudCornerLast, const CloudT& laserCloudSurfLast, const double q_wodom_curr[4],
               const double t_wodom_curr[3]) {
    typedef typename std::remove_reference<decltype(laserCloudCornerLast.points[0])>::type P;
    check(ilsm_cubemap_frame(cm_, cloud_ptr(laserCloudCornerLast), (int)laserCloudCornerLast.points.size(),
                             cloud_ptr(laserCloudSurfLast), (int)laserCloudSurfLast.points.size(), (int)sizeof(P), q_wodom_curr,
                             t_wodom_curr, parameters, parameters + 4, nullptr, &report, &stats), "LaserMapping::process");
  }
  ilsm_cubemap* handle() const { return cm_; }

 private:
  ContextPtr ctx_;
  ilsm_cubemap* cm_ = nullptr;
};

// mapOptimization::mapOptimizationCallback (mapOptimization.cpp:99-500), LiDAR part.
class MapOptimization {
 public:
  MapOptimization(float voxel_leaf = 0.8f, float downsample_size = 0.4f, ContextPtr ctx = Context::shared()) : ctx_(std::move(ctx)) {
    check(ilsm_mapopt_create(ctx_->get(), voxel_leaf, downsample_size, &mo_), "ilsm_mapopt_create");
  }
  ~MapOptimization() { ilsm_mapopt_destroy(mo_); }
  MapOptimization(const MapOptimization&) = delete;
  MapOptimization& operator=(const MapOptimization&) = delete;
  double parameters[7] = {0, 0, 0, 1, 0, 0, 0};  // mapOptimization.hpp:109
  ilsm_mapopt_stats stats;
  template <typename CloudT, typename PlaneCloudT>
  void mapOptimizationCallback(const CloudT& frame, const PlaneCloudT& pc_plane, const double q_wodom_curr[4],
                               const double t_wodom_curr[3]) {
    typedef typename std::remove_reference<decltype(frame.points[0])>::type P;
    typedef typename std::remove_reference<decltype(pc_plane.points[0])>::type Q;
    check(ilsm_mapopt_frame(mo_, cloud_ptr(frame), (int)frame.points.size(), (int)sizeof(P), cloud_ptr(pc_plane),
                            (int)pc_plane.points.size(), (int)sizeof(Q), q_wodom_curr, t_wodom_curr, parameters, parameters + 4,
                            nullptr, &stats), "mapOptimizationCallback");
  }
  int map_size() const { return ilsm_mapopt_map_size(mo_); }

 private:
  ContextPtr ctx_;
  ilsm_mapopt* mo_ = nullptr;
};

// Loop closure of a full-loop handle (ilsm_slam_enable_loop / ilsm_slam_loop_results), shared by LoamPipeline and
// StagedLoamPipeline: enable before the first frame; collect the decisions of the keyframes answered so far (wait: first
// wait for every keyframe selected so far), appended to `out` in keyframe order.
inline void slam_enable_loop(ilsm_slam* slam, const ilsm_slam_loop_opts& opts) {
  check(ilsm_slam_enable_loop(slam, &opts), "ilsm_slam_enable_loop");
}
inline void slam_loop_results(ilsm_slam* slam, std::vector<ilsm_slam_loop_event>& out, bool wait) {
  ilsm_slam_loop_event buf[32];
  for (int n = 32; n == 32;) {
    check(ilsm_slam_loop_results(slam, wait ? 1 : 0, buf, 32, &n), "ilsm_slam_loop_results");
    out.insert(out.end(), buf, buf + n);
  }
}

// The three LiDAR nodes chained on one GPU (ilsm_slam): scanRegistration -> laserOdometry -> laserMapping, inter-node
// clouds resident in HBM.  pipelined = true runs laserMapping as its own stage (second context + host thread inside the
// handle, like the reference's separate node): frame() then returns the mapped pose of the PREVIOUS frame
// (has_mapped_pose false on the first call) and flush() the last one.
class LoamPipeline {
 public:
  LoamPipeline(float lineRes = 0.4f, float planeRes = 0.8f, float minimum_range = 0.3f, bool pipelined = false,
               int cube_capacity = 0, ContextPtr ctx = Context::shared())
      : ctx_(std::move(ctx)), pipelined_(pipelined) {
    check(pipelined ? ilsm_slam_create_async(ctx_->get(), lineRes, planeRes, minimum_range, cube_capacity, &slam_)
                    : ilsm_slam_create(ctx_->get(), lineRes, planeRes, minimum_range, cube_capacity, &slam_),
          "ilsm_slam_create");
  }
  ~LoamPipeline() { ilsm_slam_destroy(slam_); }
  LoamPipeline(const LoamPipeline&) = delete;
  LoamPipeline& operator=(const LoamPipeline&) = delete;
  double q_odom[4] = {0, 0, 0, 1}, t_odom[3] = {0, 0, 0};  // /laser_odom_to_init of the frame just handed in
  double q_map[4] = {0, 0, 0, 1}, t_map[3] = {0, 0, 0};    // /aft_mapped_to_init (previous frame's in pipelined mode)
  bool has_mapped_pose = false;
  ilsm_slam_stats stats;
  template <typename CloudT>
  void frame(const CloudT& laserCloudIn, bool use_aloam = true) {
    typedef typename std::remove_reference<decltype(laserCloudIn.points[0])>::type P;
    const int n = (int)laserCloudIn.points.size();
    if (pipelined_) {
      int have = 0;
      check(ilsm_slam_frame_async(slam_, cloud_ptr(laserCloudIn), n, (int)sizeof(P), use_aloam ? 1 : 0, q_odom, t_odom, q_map, t_map,
                                  &have, &stats), "ilsm_slam_frame_async");
      has_mapped_pose = have != 0;
    } else {
      check(ilsm_slam_frame(slam_, cloud_ptr(laserCloudIn), n, (int)sizeof(P), use_aloam ? 1 : 0, q_odom, t_odom, q_map, t_map, &stats),
            "ilsm_slam_frame");
      has_mapped_pose = true;
    }
  }
  bool flush() {  // pipelined mode: the mapped pose of the last frame; false when nothing was in flight
    int have = 0;
    check(ilsm_slam_flush(slam_, q_map, t_map, &have, &stats), "ilsm_slam_flush");
    has_mapped_pose = have != 0;
    return has_mapped_pose;
  }
  void enableLoopClosure(const ilsm_slam_loop_opts& opts) { slam_enable_loop(slam_, opts); }
  void loopResults(std::vector<ilsm_slam_loop_event>& out, bool wait) { slam_loop_results(slam_, out, wait); }
  ilsm_slam* handle() const { return slam_; }

 private:
  ContextPtr ctx_;
  ilsm_slam* slam_ = nullptr;
  bool pipelined_;
};

// The same three nodes as three STAGES (ilsm_slam_create_staged): scanRegistration, laserOdometry and laserMapping each on
// its own context and host thread inside the handle, the way the reference runs three processes.  push(cloud) hands frame k
// to the front-end stage and returns what has come out of the other two: the odometry pose of frame k - 1 and the mapped
// pose of frame k - 2 (frame indices in odom_frame / map_frame, -1 while the stages fill); drain() advances the stages
// without a new frame -- two calls after the last push hand out everything.  The cloud handed to push() is read
// asynchronously: the object keeps its own copy until the next call returns.
class StagedLoamPipeline {
 public:
  StagedLoamPipeline(float lineRes = 0.4f, float planeRes = 0.8f, float minimum_range = 0.3f, int cube_capacity = 0,
                     ContextPtr ctx = Context::shared())
      : ctx_(std::move(ctx)) {
    check(ilsm_slam_create_staged(ctx_->get(), lineRes, planeRes, minimum_range, cube_capacity, &slam_), "ilsm_slam_create_staged");
  }
  ~StagedLoamPipeline() { ilsm_slam_destroy(slam_); }
  StagedLoamPipeline(const StagedLoamPipeline&) = delete;
  StagedLoamPipeline& operator=(const StagedLoamPipeline&) = delete;
  int odom_frame = -1, map_frame = -1;
  double q_odom[4] = {0, 0, 0, 1}, t_odom[3] = {0, 0, 0};  // /laser_odom_to_init of frame odom_frame
  double q_map[4] = {0, 0, 0, 1}, t_map[3] = {0, 0, 0};    // /aft_mapped_to_init of frame map_frame
  ilsm_slam_stats stats;
  template <typename CloudT>
  void push(const CloudT& laserCloudIn, bool use_aloam = true) {
    typedef typename std::remove_reference<decltype(laserCloudIn.points[0])>::type P;
    std::vector<float>& keep = held_[turn_ ^= 1];
    const size_t floats = laserCloudIn.points.size() * (sizeof(P) / 4);
    keep.resize(floats);
    if (floats) std::memcpy(keep.data(), laserCloudIn.points.data(), floats * 4);
    check(ilsm_slam_frame_staged(slam_, keep.data(), (int)laserCloudIn.points.size(), (int)sizeof(P), use_aloam ? 1 : 0, q_odom, t_odom,
                                 &odom_frame, q_map, t_map, &map_frame, &stats), "ilsm_slam_frame_staged");
  }
  void drain() {
    check(ilsm_slam_frame_staged(slam_, nullptr, -1, 16, 1, q_odom, t_odom, &odom_frame, q_map, t_map, &map_frame, &stats),
          "ilsm_slam_frame_staged");
  }
  void enableLoopClosure(const ilsm_slam_loop_opts& opts) { slam_enable_loop(slam_, opts); }
  void loopResults(std::vector<ilsm_slam_loop_event>& out, bool wait) { slam_loop_results(slam_, out, wait); }
  ilsm_slam* handle() const { return slam_; }

 private:
  ContextPtr ctx_;
  ilsm_slam* slam_ = nullptr;
  std::vector<float> held_[2];
  int turn_ = 0;
};

// ------------------------------------------------------------------------------------------------ parameters
// The keys the reference's nodes read from the ROS parameter server (config/spot.yaml + launch/spot.launch:4-6), for a build
// without ROS: a two-level "key: value  # comment" reader that accepts the reference's own spot.yaml unchanged, and a
// <param name= value=> reader for its launch file.  Defaults = the reference's nh.param defaults.
struct Config {
  int image_width = 1024;                  // /intensity_feature_tracker/image_width     mapOptimization.cpp:522
  int image_height = 64;                   // /intensity_feature_tracker/image_height    scanRegistration.cpp:692 (N_SCANS)
  double minimum_range = 0.3;              // /map_optimization_parameters/remove_radius scanRegistration.cpp:695
  double mapping_line_resolution = 0.4;    // spot.launch:4  laserMapping.cpp:1181
  double mapping_plane_resolution = 0.8;   // spot.launch:5  laserMapping.cpp:1183
  int mapping_skip_frame = 1;              // spot.launch:6  laserOdometry.cpp:265
  int sliding_window_size = 0;             // mapOptimization.cpp:538
  int ground_plane_window_size = 2;        // mapOptimization.cpp:541
  std::string cloud_topic = "/os_cloud_node/points";

  static std::string trim(std::string v) {
    const size_t h = v.find(" #");
    if (h != std::string::npos) v.erase(h);
    if (!v.empty() && v[0] == '#') v.clear();
    while (!v.empty() && (v.back() == ' ' || v.back() == '\t' || v.back() == '\r' || v.back() == '\n')) v.pop_back();
    size_t b = 0;
    while (b < v.size() && (v[b] == ' ' || v[b] == '\t')) ++b;
    v.erase(0, b);
    if (v.size() >= 2 && (v.front() == '"' || v.front() == '\'') && v.back() == v.front()) v = v.substr(1, v.size() - 2);
    return v;
  }
  void set(const std::string& section, const std::string& key, const std::string& val) {
    if (val.empty()) return;
    const std::string k = section.empty() ? key : section + "/" + key;
    if (k == "intensity_feature_tracker/image_width") image_width = std::atoi(val.c_str());
    else if (k == "intensity_feature_tracker/image_height") image_height = std::atoi(val.c_str());
    else if (k == "intensity_feature_tracker/cloud_topic") cloud_topic = val;
    else if (k == "map_optimization_parameters/remove_radius") minimum_range = std::atof(val.c_str());
    else if (k == "map_optimization_parameters/sliding_window_size") sliding_window_size = std::atoi(val.c_str());
    else if (k == "map_optimization_parameters/ground_plane_window_size") ground_plane_window_size = std::atoi(val.c_str());
    else if (k == "mapping_line_resolution") mapping_line_resolution = std::atof(val.c_str());
    else if (k == "mapping_plane_resolution") mapping_plane_resolution = std::atof(val.c_str());
    else if (k == "mapping_skip_frame") mapping_skip_frame = std::atoi(val.c_str());
  }
  // returns false when the file cannot be opened (the defaults stay)
  bool load_yaml(const std::string& path) {
    FILE* f = std::fopen(path.c_str(), "r");
    if (!f) return false;
    char line[1024];
    std::string section;
    while (std::fgets(line, sizeof(line), f)) {
      std::string l(line);
      size_t indent = 0;
      while (indent < l.size() && l[indent] == ' ') ++indent;
      const size_t colon = l.find(':');
      if (colon == std::string::npos || l[indent] == '#' || l[indent] == '\n') continue;
      const std::string key = trim(l.substr(indent, colon - indent)), val = trim(l.substr(colon + 1));
      if (indent == 0) {
        section = val.empty() ? key : "";
        if (!val.empty()) set("", key, val);
      } else {
        set(section, key, val);
      }
    }
    std::fclose(f);
    return true;
  }
  bool load_launch(const std::string& path) {  // <param name="mapping_line_resolution" type="double" value="0.4"/>
    FILE* f = std::fopen(path.c_str(), "r");
    if (!f) return false;
    char line[2048];
    while (std::fgets(line, sizeof(line), f)) {
      const std::string l(line);
      const size_t p = l.find("<param"), n = l.find("name=\""), v = l.find("value=\"");
      if (p == std::string::npos || n == std::string::npos || v == std::string::npos) continue;
      const size_t ne = l.find('"', n + 6), ve = l.find('"', v + 7);
      if (ne == std::string::npos || ve == std::string::npos) continue;
      set("", l.substr(n + 6, ne - (n + 6)), l.substr(v + 7, ve - (v + 7)));
    }
    std::fclose(f);
    return true;
  }
  void validate() const {
    if (image_height != 64) throw Error(ILSM_ERR_INVALID_ARG, "only the 64-ring branch of scanRegistration.cpp:308-316 is implemented");
    if (image_width <= 0 || !(mapping_line_resolution > 0) || !(mapping_plane_resolution > 0) || !(minimum_range >= 0))
      throw Error(ILSM_ERR_INVALID_ARG, "bad parameter value");
  }
};

// ------------------------------------------------------------------------------------------------ odom_handler_node
// callback() of odom_handler_node.cpp:44-132: merges the A-LOAM and the intensity odometry streams -- the merged pose
// advances by the A-LOAM increment on frames flagged "/odom_skip" (child_frame_id of the intensity odometry), else by the
// intensity increment.  Pure host arithmetic on 4x4 transforms (no GPU work on this node), kept here so that the launched
// graph is complete above the C ABI.  Poses are {qx,qy,qz,qw, tx,ty,tz}.
class OdomHandler {
 public:
  struct Mat4 {
    double m[4][4];
  };
  bool aloam_odom_init = false, intensity_odom_init = false;
  Mat4 odom_cur, aloam_prev, intensity_prev;

  static Mat4 from_pose(const double p[7]) {  // Eigen::Quaterniond::toRotationMatrix + translation
    const double x = p[0], y = p[1], z = p[2], w = p[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z, twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x,
                 tyy = ty * y, tyz = tz * y, tzz = tz * z;
    Mat4 r = {{{1 - (tyy + tzz), txy - twz, txz + twy, p[4]}, {txy + twz, 1 - (txx + tzz), tyz - twx, p[5]},
               {txz - twy, tyz + twx, 1 - (txx + tyy), p[6]}, {0, 0, 0, 1}}};
    return r;
  }
  static Mat4 mul(const Mat4& a, const Mat4& b) {
    Mat4 c;
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) c.m[i][j] = a.m[i][0] * b.m[0][j] + a.m[i][1] * b.m[1][j] + a.m[i][2] * b.m[2][j] + a.m[i][3] * b.m[3][j];
    return c;
  }
  static Mat4 rigid_inverse(const Mat4& a) {  // the inputs are rigid transforms: inverse = [R^T, -R^T t]
    Mat4 c = {{{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 1}}};
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) c.m[i][j] = a.m[j][i];
      c.m[i][3] = -(a.m[0][i] * a.m[0][3] + a.m[1][i] * a.m[1][3] + a.m[2][i] * a.m[2][3]);
    }
    return c;
  }
  // Eigen::Quaterniond(rot): the branch structure of Eigen's quat_product-free conversion (trace > 0, else largest diagonal)
  static void to_pose(const Mat4& a, double p[7]) {
    const double (*m)[4] = a.m;
    double t = m[0][0] + m[1][1] + m[2][2];
    if (t > 0) {
      t = std::sqrt(t + 1.0);
      p[3] = 0.5 * t;
      t = 0.5 / t;
      p[0] = (m[2][1] - m[1][2]) * t, p[1] = (m[0][2] - m[2][0]) * t, p[2] = (m[1][0] - m[0][1]) * t;
    } else {
      int i = 0;
      if (m[1][1] > m[0][0]) i = 1;
      if (m[2][2] > m[i][i]) i = 2;
      const int j = (i + 1) % 3, k = (j + 1) % 3;
      t = std::sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
      p[i] = 0.5 * t;
      t = 0.5 / t;
      p[3] = (m[k][j] - m[j][k]) * t, p[j] = (m[j][i] + m[i][j]) * t, p[k] = (m[k][i] + m[i][k]) * t;
    }
    p[4] = m[0][3], p[5] = m[1][3], p[6] = m[2][3];
  }
  // returns the merged pose published on the merged-odometry topic (odom_handler_node.cpp:113-129)
  void callback(const double aloam_odom[7], const double intensity_odom[7], const std::string& skip_flag, double merged[7]) {
    const Mat4 aloam_odom_cur = from_pose(aloam_odom), intensity_odom_cur = from_pose(intensity_odom);
    if (!aloam_odom_init && !intensity_odom_init) {
      aloam_prev = aloam_odom_cur, intensity_prev = intensity_odom_cur, odom_cur = intensity_odom_cur;
      aloam_odom_init = intensity_odom_init = true;
    } else {
      const Mat4 intensity_odom_diff = mul(rigid_inverse(intensity_prev), intensity_odom_cur);
      const Mat4 aloam_odom_diff = mul(rigid_inverse(aloam_prev), aloam_odom_cur);
      odom_cur = mul(odom_cur, skip_flag == "/odom_skip" ? aloam_odom_diff : intensity_odom_diff);
      aloam_prev = aloam_odom_cur, intensity_prev = intensity_odom_cur;
    }
    to_pose(odom_cur, merged);
  }
};

// ------------------------------------------------------------------------------------------------ messages out (SURVEY 8f f4)
// What the nodes publish, as plain structs a ROS-free caller can forward (and a ROS caller copies field by field into
// sensor_msgs::PointCloud2 / nav_msgs::Odometry / tf::StampedTransform): the wire format and the frame names of the
// reference, nothing computed on the host.
struct Header {
  double stamp = 0.0;  // seconds
  std::string frame_id;
};
struct PointCloud2Msg {  // sensor_msgs/PointCloud2 of a pcl::PointXYZI cloud, as pcl::toROSMsg fills it
  Header header;
  uint32_t height = 1, width = 0, point_step = 32, row_step = 0;
  bool is_bigendian = false, is_dense = true;
  struct Field {
    const char* name;
    uint32_t offset;
    uint8_t datatype;  // sensor_msgs/PointField::FLOAT32 = 7
    uint32_t count;
  } fields[4] = {{"x", 0, 7, 1}, {"y", 4, 7, 1}, {"z", 8, 7, 1}, {"intensity", 16, 7, 1}};
  std::vector<uint8_t> data;
};
struct OdometryMsg {  // nav_msgs/Odometry, the fields the reference sets
  Header header;
  std::string child_frame_id;
  double orientation_xyzw[4] = {0, 0, 0, 1}, position[3] = {0, 0, 0};
};
struct TransformMsg {  // tf::StampedTransform
  double stamp = 0.0;
  std::string frame_id, child_frame_id;
  double rotation_xyzw[4] = {0, 0, 0, 1}, origin[3] = {0, 0, 0};
};

// pcl::toROSMsg + the two header lines every publisher adds (scanRegistration.cpp:593-596 and the like): packed on the GPU
// by ilsm_pc2_pack.  Clouds of the front end are published in "os_sensor" (:595), clouds of the mapping node in "map"
// (laserMapping.cpp:1025,1046,1063).
template <typename CloudT>
inline PointCloud2Msg toROSMsg(const CloudT& cloud, double stamp, const std::string& frame_id, const ContextPtr& ctx = Context::shared()) {
  static_assert(sizeof(cloud.points[0]) == 32, "toROSMsg: a PointXYZI-layout cloud (32-byte points) is expected");
  PointCloud2Msg m;
  m.header.stamp = stamp, m.header.frame_id = frame_id;
  m.width = (uint32_t)cloud.points.size(), m.row_step = m.width * m.point_step, m.is_dense = cloud.is_dense;
  m.data.resize((size_t)m.width * m.point_step);
  if (m.width == 0) return m;
  std::vector<float> packed((size_t)m.width * 4);
  for (size_t i = 0; i < cloud.points.size(); ++i)
    packed[4 * i] = cloud.points[i].x, packed[4 * i + 1] = cloud.points[i].y, packed[4 * i + 2] = cloud.points[i].z, packed[4 * i + 3] = cloud.points[i].intensity;
  ilsm_pc2_layout lay;
  ilsm_pc2_layout_pcl_xyzi(&lay);
  check(ilsm_pc2_pack(ctx->get(), packed.data(), (int)m.width, &lay, m.data.data()), "ilsm_pc2_pack");
  return m;
}

// /aft_mapped_to_init and its transform (laserMapping.cpp:1075-1088, 1129-1146: frame "map", child "/aft_mapped"), and
// /laser_odom_to_init (laserOdometry.cpp:726-735: frame "camera_init", child "/laser_odom"), from a pose {qx,qy,qz,qw, tx,ty,tz}
inline OdometryMsg make_odometry(const double q_xyzw[4], const double t[3], double stamp, const std::string& frame_id,
                                 const std::string& child_frame_id) {
  OdometryMsg m;
  m.header.stamp = stamp, m.header.frame_id = frame_id, m.child_frame_id = child_frame_id;
  for (int i = 0; i < 4; ++i) m.orientation_xyzw[i] = q_xyzw[i];
  for (int i = 0; i < 3; ++i) m.position[i] = t[i];
  return m;
}
inline OdometryMsg odomAftMapped(const double q_w_curr[4], const double t_w_curr[3], double timeLaserOdometry) {
  return make_odometry(q_w_curr, t_w_curr, timeLaserOdometry, "map", "/aft_mapped");
}
inline OdometryMsg laserOdometryMsg(const double q_w_curr[4], const double t_w_curr[3], double timeSurfPointsLessFlat) {
  return make_odometry(q_w_curr, t_w_curr, timeSurfPointsLessFlat, "camera_init", "/laser_odom");
}
inline TransformMsg aftMappedTransform(const OdometryMsg& o) {  // br.sendTransform(StampedTransform(transform, stamp, "map", "/aft_mapped"))
  TransformMsg t;
  t.stamp = o.header.stamp, t.frame_id = o.header.frame_id, t.child_frame_id = o.child_frame_id;
  for (int i = 0; i < 4; ++i) t.rotation_xyzw[i] = o.orientation_xyzw[i];
  for (int i = 0; i < 3; ++i) t.origin[i] = o.position[i];
  return t;
}

}  // namespace ilsm
#endif  // ILSM_HPP_
