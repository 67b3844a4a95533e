/* ilsm.h -- C ABI of libilsm_cuda.so: the B200 (sm_100a) implementation of the LOAM-style scan-to-map
 * registration hot path of himhan34/Intensity_based_LiDAR_SLAM_for_me-.
 *
 * The reference has no FFI layer: its "API" for this path is a set of library call sites inside the node
 * bodies (PCL KdTreeFLANN / ikd-Tree / Ceres / ImageHandler).  Every entry point below replaces one such
 * call site; the citation after each declaration is the reference file:line it stands in for
 * (paths relative to the reference tree).  INTEGRATION.md shows the C++ stub a maintainer adds at each site.
 *
 * Conventions
 *  - plain C types only; the caller owns every host buffer; the library owns device memory inside handles.
 *  - point clouds are arrays of floats with a byte stride: 16 (pcl::PointXYZ / packed xyzi) or 32
 *    (pcl::PointXYZI: x@0 y@4 z@8 intensity@16, parameters.h_ouster:121).  xyz are the first three floats.
 *  - poses are Eigen-ordered: q = {x,y,z,w}, t = {x,y,z}, double (laserMapping.cpp:105-107).
 *  - every function returns ILSM_OK (0) or a negative ilsm_status; ilsm_last_error() gives the text
 *    (thread-local).  There is NO CPU fallback: without a CUDA device ilsm_create fails.
 *  - handles are re-entrant per handle: calls on objects of the same ilsm_ctx are serialised by a mutex
 *    and run on that context's single CUDA stream (the reference runs this path on one thread,
 *    laserMapping.cpp:1215).
 *  - *_dev variants take DEVICE pointers (inputs already resident in HBM) and enqueue on the context
 *    stream without synchronising; call ilsm_sync() before reading results on the host.  A *_dev variant checks its
 *    arguments as its host form does, with the same status; both return an argument error before any CUDA call.
 */
#ifndef ILSM_H_
#define ILSM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ILSM_ABI_VERSION 1

#if defined(__GNUC__)
#define ILSM_API __attribute__((visibility("default")))
#else
#define ILSM_API
#endif

typedef enum ilsm_status {
  ILSM_OK = 0,
  ILSM_ERR_INVALID_ARG = -1,
  ILSM_ERR_CUDA = -2,
  ILSM_ERR_NO_DEVICE = -3,
  ILSM_ERR_NOT_ENOUGH_MAP = -4, /* guard of laserMapping.cpp:624 (corner map <= 10 or surf map <= 50) */
  ILSM_ERR_OUT_OF_MEMORY = -5,
  ILSM_ERR_STATE = -6
} ilsm_status;

/* ceres::TerminationType order (ceres/types.h): the reference gates on it at mapOptimization.cpp:448. */
typedef enum ilsm_termination {
  ILSM_CONVERGENCE = 0,
  ILSM_NO_CONVERGENCE = 1,
  ILSM_FAILURE = 2
} ilsm_termination;

typedef struct ilsm_ctx ilsm_ctx; /* stream + scratch + LM state */
typedef struct ilsm_map ilsm_map; /* voxel-hashed local map (replaces KdTreeFLANN / ikd-Tree search) */

ILSM_API int ilsm_abi_version(void);
ILSM_API const char* ilsm_last_error(void);

/* One context per thread of the reference's mapping loop (laserMapping.cpp:1215 `std::thread mapping_process`). */
ILSM_API int ilsm_create(int device, ilsm_ctx** out);
ILSM_API void ilsm_destroy(ilsm_ctx* ctx);
ILSM_API int ilsm_sync(ilsm_ctx* ctx);
/* on != 0: ilsm_map_build (host pointers) returns as soon as its copy and kernels are enqueued on the map's own
 * stream; the caller must leave the source buffer untouched until the next blocking call that uses the map
 * (ilsm_register / ilsm_knn / ilsm_sync).  laserMapping.cpp keeps laserCloud*FromMap alive until the next
 * frame, so the two setInputCloud replacements can overlap.  Default 0 (blocking, like setInputCloud). */
ILSM_API int ilsm_set_async(ilsm_ctx* ctx, int on);
/* cudaStream_t of the context (for CUDA-event timing by the caller). */
ILSM_API void* ilsm_stream(ilsm_ctx* ctx);

/* Page-lock a caller-owned host buffer (e.g. the storage of a pcl::PointCloud or of a sensor_msgs/PointCloud2 that is
 * reused from frame to frame) so that the host-pointer entry points copy from it by DMA instead of through a staging
 * buffer; unregister before freeing it.  Optional: every entry point also accepts pageable memory. */
ILSM_API int ilsm_host_register(void* ptr, size_t bytes);
ILSM_API int ilsm_host_unregister(void* ptr);

/* ------------------------------------------------------------------ K1: local map + exact k-NN ------- */
ILSM_API int ilsm_map_create(ilsm_ctx* ctx, ilsm_map** out);
ILSM_API void ilsm_map_destroy(ilsm_map* map);
ILSM_API int ilsm_map_size(const ilsm_map* map);

/* (Re)build the search structure over n points.  `cell` = voxel edge in metres (<= 0 selects the default
 * 1.0 m, the reference's d2[4] < 1.0 gate radius).  Non-finite points are skipped (the reference strips
 * NaNs first, mapOptimization.cpp:151).
 * Replaces: kdtreeCornerFromMap->setInputCloud / kdtreeSurfFromMap->setInputCloud  laserMapping.cpp:631-634
 *           kdtreeCornerLast/SurfLast->setInputCloud                               laserOdometry.cpp:807-808
 *           ikdtree->Build(points)                                                mapOptimization.cpp:192 */
ILSM_API int ilsm_map_build(ilsm_map* map, const float* xyz, int n, int stride_bytes, float cell);
ILSM_API int ilsm_map_build_dev(ilsm_map* map, const float* d_xyz, int n, int stride_bytes, float cell);
/* Both search structures of a frame in one call: three launches build the two maps side by side (the reference builds
 * them on consecutive lines).  Same semantics as two ilsm_map_build_dev calls.
 * Replaces: kdtreeCornerFromMap->setInputCloud(...); kdtreeSurfFromMap->setInputCloud(...);  laserMapping.cpp:631-634
 *           kdtreeCornerLast->setInputCloud(...); kdtreeSurfLast->setInputCloud(...);          laserOdometry.cpp:807-808 */
ILSM_API int ilsm_map_build_pair_dev(ilsm_map* map_a, const float* d_xyz_a, int n_a, ilsm_map* map_b, const float* d_xyz_b, int n_b,
                                     int stride_bytes, float cell);
/* Builds run on the map's own stream (the corner and surf structures of a frame are built concurrently); every entry
 * point that uses a map orders itself after its build.  ilsm_map_join makes the CONTEXT stream wait for the build
 * without using the map (for CUDA-event timing of the build on the context stream). */
ILSM_API int ilsm_map_join(ilsm_map* map);

/* Incremental insertion.
 *   ILSM_INSERT_NEAREST_TO_CENTRE: ikd-Tree's down-sampled insertion -- per cubic box of edge `leaf` around each new
 *     point, the point of {box contents, new point} nearest to the box centre survives (strict <: a new point wins
 *     ties against existing ones, a later new point against an earlier one); equivalent to processing the batch
 *     point by point.  Boxes not touched by the batch are left alone (a Build-seeded box may hold several points).
 *   ILSM_INSERT_APPEND: downsample_on = false.
 * The k-NN cell size chosen at build time is kept.  Blocking.
 * Replaces: ikdtree->Add_Points(points, true)  mapOptimization.cpp:475,479 (ikd_Tree.cpp:570-640) */
#define ILSM_INSERT_APPEND 0
#define ILSM_INSERT_NEAREST_TO_CENTRE 1
ILSM_API int ilsm_map_insert(ilsm_map* map, const float* xyz, int n, int stride_bytes, int policy, float leaf);

/* Copy the current map points (packed xyzi, map order) to the host; *n_out = map size (may exceed capacity).
 * Replaces: ikdtree->flatten(Root_Node, storage, NOT_RECORD)  mapOptimization.cpp:224 */
ILSM_API int ilsm_map_points(ilsm_map* map, float* out_xyzi, int capacity, int* n_out);

/* Exact k-NN (1 <= k <= 8), ascending squared distance computed in float as ((dx*dx)+(dy*dy))+(dz*dz) without
 * FMA (FLANN L2_Simple<float>; ikd_Tree.cpp:2224-2230), ties broken by lower point index.  idx/d2 are nq*k;
 * missing neighbours are idx -1 / d2 +inf.  max_dist <= 0 means unbounded (exact for every query);
 * with max_dist > 0 only neighbours closer than max_dist are guaranteed exact (ikd-Tree's max_dist argument,
 * ikd_Tree.h:267).
 * Replaces: nearestKSearch(pointSel, 5, idx, d2)   laserMapping.cpp:673,753
 *           nearestKSearch(pointSel, 1, idx, d2)   laserOdometry.cpp:452,574
 *           ikdtree->Nearest_Search(p, 5, pts, d2) mapOptimization.cpp:393 */
ILSM_API int ilsm_knn(ilsm_map* map, const float* q_xyz, int nq, int stride_bytes, int k, float max_dist, int32_t* idx,
             float* d2);
ILSM_API int ilsm_knn_dev(ilsm_map* map, const float* d_q_xyz, int nq, int stride_bytes, int k, float max_dist,
                 int32_t* d_idx, float* d_d2);

/* ------------------------------------------------- K2+K3: association, fit, residuals, LM solve ------ */
typedef struct ilsm_reg_opts {
  int32_t outer_iterations;   /* re-association passes: 2 (laserMapping.cpp:640), 1 (mapOptimization.cpp:377) */
  int32_t max_num_iterations; /* Ceres max_num_iterations: 4 (laserMapping.cpp:840), 10 (mapOptimization.cpp:435) */
  double huber_a;             /* ceres::HuberLoss(0.1) laserMapping.cpp:644 */
  float knn_gate_sq;          /* pointSearchSqDis[4] < 1.0  laserMapping.cpp:676,758 */
  float reserved0;
  double line_eig_ratio;      /* eigenvalues[2] > 3 * eigenvalues[1]  laserMapping.cpp:708 */
  double plane_tol;           /* fabs(n.p + d) > 0.2 invalidates the plane  laserMapping.cpp:778-788 */
  int32_t min_corner_map;     /* > 10  laserMapping.cpp:624 (0 disables, as in mapOptimization.cpp) */
  int32_t min_surf_map;       /* > 50  laserMapping.cpp:624 */
} ilsm_reg_opts;

ILSM_API void ilsm_reg_opts_default(ilsm_reg_opts* o); /* laserMapping values */

typedef struct ilsm_solve_summary { /* the fields of ceres::Solver::Summary the reference reads or prints */
  int32_t termination; /* ilsm_termination */
  int32_t iterations;
  int32_t num_successful_steps;
  int32_t num_unsuccessful_steps;
  int32_t num_edge_factors;  /* corner_num */
  int32_t num_plane_factors; /* surf_num */
  int32_t num_evaluations;
  int32_t reserved;
  double initial_cost;
  double final_cost;
} ilsm_solve_summary;

#define ILSM_MAX_OUTER 8
typedef struct ilsm_reg_report {
  int32_t passes; /* outer passes actually run */
  int32_t reserved;
  ilsm_solve_summary pass[ILSM_MAX_OUTER];
} ilsm_reg_report;

/* The whole association + solve block.  corner/surf are the SENSOR-frame feature stacks
 * (laserCloudCornerStack / laserCloudSurfStack); q,t are read as the initial guess and overwritten with the
 * optimised pose (Eigen::Map over `parameters`).  Either stack may be empty (ns == 0 gives the
 * mapOptimization.cpp plane-only problem when called with the ground/less-flat cloud as `surf`).
 * Replaces: laserMapping.cpp:640-861 ; mapOptimization.cpp:377-450. */
ILSM_API int ilsm_register(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* corner, int nc,
                  const float* surf, int ns, int stride_bytes, double q_xyzw[4], double t_xyz[3],
                  const ilsm_reg_opts* opts, ilsm_reg_report* report);
/* Device-resident variant: stacks are device pointers, the pose lives in d_pose (7 doubles: q xyzw, t) and is
 * updated in place; the report is written to the device too (d_report may be NULL).  Nothing is copied to
 * the host and the call does not synchronise. */
ILSM_API int ilsm_register_dev(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* d_corner, int nc,
                      const float* d_surf, int ns, int stride_bytes, double* d_pose7, const ilsm_reg_opts* opts,
                      ilsm_reg_report* d_report);

/* One organised LiDAR frame registered against two prebuilt maps -- SURVEY 8d config 1 as the reference pipeline runs it:
 * laserCloudHandler (min-range filter, ring bucketing, curvature, labelling, per-ring VoxelGrid;
 * scanRegistration.cpp:189-669), cornerPointsLessSharp / surfPointsLessFlat become the mapping inputs
 * (laserOdometry.cpp:793-796), downSizeFilterCorner / downSizeFilterSurf with mapping_line_resolution /
 * mapping_plane_resolution (laserMapping.cpp:608-616), then the association + solve block (:640-861) from the initial
 * guess q, t, which is overwritten with the optimised pose.  sizes_out (may be NULL) = {less-sharp points, less-flat
 * points, corner stack, surf stack}.  The feature clouds stay on the device between the stages; the call synchronises
 * once for the feature counts (they size the VoxelGrid sorts) and once for the pose.  The _dev form takes the frame and
 * the pose (7 doubles, updated in place) on the device and returns without the final synchronisation.  Both forms
 * return ILSM_ERR_STATE when a map has not been built and ILSM_ERR_NOT_ENOUGH_MAP under the map-size guard of
 * ilsm_register (opts->min_corner_map / min_surf_map), before any launch. */
ILSM_API int ilsm_register_frame(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* xyzi, int n, int stride_bytes,
                                 float min_range, float line_res, float plane_res, double q_xyzw[4], double t_xyz[3],
                                 const ilsm_reg_opts* opts, ilsm_reg_report* report, int32_t sizes_out[4]);
ILSM_API int ilsm_register_frame_dev(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* d_xyzi, int n,
                                     int stride_bytes, float min_range, float line_res, float plane_res, double* d_pose7,
                                     const ilsm_reg_opts* opts);

/* One correspondence record, in the reference functors' own terms (lidarFeaturePointsFunction.hpp). */
typedef struct ilsm_factor {
  int32_t type; /* 0 none, 1 LidarEdgeFactor (hpp:243-293), 2 LidarPlaneNormFactor (hpp:199-240) */
  int32_t src;  /* index of the stack point */
  double p[3];  /* curr_point (sensor frame) */
  double a[3];  /* edge: last_point_a ; plane: plane_unit_norm */
  double b[3];  /* edge: last_point_b ; plane: b[0] = negative_OA_dot_norm */
} ilsm_factor;

/* One association pass at pose (q,t): k-NN + line/plane fit for every stack point; fills nc+ns records
 * (corner slots first) and keeps them in the context for ilsm_eval_normal_eq / ilsm_solve.
 * knn_idx (5 per slot) / knn_d2 may be NULL.
 * Replaces: laserMapping.cpp:665-797 (one iterCount). */
ILSM_API int ilsm_associate(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* corner, int nc,
                   const float* surf, int ns, int stride_bytes, const double q_xyzw[4], const double t_xyz[3],
                   const ilsm_reg_opts* opts, ilsm_factor* factors, int32_t* knn_idx, float* knn_d2);

/* Device-resident association only (no export, no synchronisation): the k-NN + fit kernel on the context stream,
 * pose read from d_pose7.  Used by bench.py to time the kernel in isolation. */
ILSM_API int ilsm_associate_dev(ilsm_ctx* ctx, ilsm_map* map_corner, ilsm_map* map_surf, const float* d_corner, int nc,
                                const float* d_surf, int ns, int stride_bytes, const double* d_pose7,
                                const ilsm_reg_opts* opts);

/* Number of kernels this library has launched since it was loaded (all contexts). */
ILSM_API long long ilsm_launch_count(void);

/* One evaluation of the robustified problem at (q,t) over the factors held by the context:
 * cost = 1/2 sum rho(|r|^2), JtJ (6x6 row-major, tangent order [rotation(3), translation(3)] of
 * EigenQuaternionParameterization) and Jtr.  This is the single kernel a Gauss-Newton/LM iteration needs.
 * Replaces: one Evaluate() of the ceres::Problem built at laserMapping.cpp:651-797. */
ILSM_API int ilsm_eval_normal_eq(ilsm_ctx* ctx, const double q_xyzw[4], const double t_xyz[3], double huber_a, double* cost,
                        double JtJ[36], double Jtr[6]);

/* Device-resident variant for timing the J^T J kernel alone: pose from d_pose7, the 28 sums {cost, 21 upper-triangle
 * J^T J entries (row-major), 6 J^T r entries} written to d_out32 (32 doubles); no synchronisation. */
ILSM_API int ilsm_eval_normal_eq_dev(ilsm_ctx* ctx, const double* d_pose7, double huber_a, double* d_out32);

/* ceres::Solve(options, &problem, &summary) over the factors held by the context (Levenberg-Marquardt,
 * trust-region loop run on the device, one kernel per iteration).
 * Replaces: laserMapping.cpp:836-850 ; mapOptimization.cpp:433-442 ; laserOdometry.cpp:705-710. */
ILSM_API int ilsm_solve(ilsm_ctx* ctx, double q_xyzw[4], double t_xyz[3], int max_num_iterations, double huber_a,
               ilsm_solve_summary* summary);

/* Device-resident variant for timing the solve kernel alone: the factors held by the context, start pose from
 * d_pose7_in (NULL: continue from the pose in the context); nothing is copied back and the call does not synchronise. */
ILSM_API int ilsm_solve_dev(ilsm_ctx* ctx, const double* d_pose7_in, int max_num_iterations, double huber_a);

/* ---------------------------------------------------------- laserMapping: device-resident rolling cube map ---- */
typedef struct ilsm_cubemap ilsm_cubemap;

typedef struct ilsm_cubemap_stats {
  int32_t n_map_corner;     /* laserCloudCornerFromMapNum */
  int32_t n_map_surf;       /* laserCloudSurfFromMapNum */
  int32_t n_stack_corner;   /* laserCloudCornerStackNum */
  int32_t n_stack_surf;     /* laserCloudSurfStackNum */
  int32_t ran_optimization; /* 0 when the guard of laserMapping.cpp:624 skipped the solve */
  int32_t n_valid;          /* laserCloudValidNum */
  int32_t cen[3];           /* laserCloudCenWidth / Height / Depth after the roll */
  int32_t flags;            /* non-zero: a cube or a stack exceeded its capacity */
} ilsm_cubemap_stats;

/* The 21x21x11 map of 50 m cubes (laserMapping.cpp:70-78), resident in HBM: every cube owns a slab of
 * cube_capacity points (<= 16384; 0 selects 16384).  line_res / plane_res = mapping_line_resolution /
 * mapping_plane_resolution (spot.launch:4-5). */
ILSM_API int ilsm_cubemap_create(ilsm_ctx* ctx, float line_res, float plane_res, int cube_capacity, ilsm_cubemap** out);
ILSM_API void ilsm_cubemap_destroy(ilsm_cubemap* cm);

/* Insert WORLD-frame points (e.g. a prior map) after rolling the window around `centre`, then VoxelGrid the valid
 * cubes (the tail of process(), laserMapping.cpp:880-1002, without a registration). */
ILSM_API int ilsm_cubemap_insert_world(ilsm_cubemap* cm, const float* corner, int nc, const float* surf, int ns,
                                       int stride_bytes, const double centre_xyz[3]);

/* One iteration of process() (laserMapping.cpp:327-1002) for one frame: corner_last / surf_last are the frame's
 * less-sharp / less-flat clouds in the sensor frame, (q_wodom, t_wodom) the odometry pose; returns the mapped pose
 * (q_w, t_w).  transformAssociateToMap, window roll, 5x5x3 gather, stack VoxelGrid, guarded 2 x (associate + Solve),
 * transformUpdate, insertion of the stack at the optimised pose and per-cube VoxelGrid of the valid cubes.  The
 * map and q/t_wmap_wodom persist in the handle.  Feature clouds of any size below 2^24 points (clouds above 16384
 * points take the tiled multi-block VoxelGrid); the DOWN-SAMPLED stacks must fit 16384 points each. */
ILSM_API int ilsm_cubemap_frame(ilsm_cubemap* cm, const float* corner_last, int nc, const float* surf_last, int ns,
                                int stride_bytes, const double q_wodom_xyzw[4], const double t_wodom[3], double q_w_xyzw[4],
                                double t_w[3], const ilsm_reg_opts* opts, ilsm_reg_report* report, ilsm_cubemap_stats* stats);

/* Copy one cube (array index i + 21*j + 441*k of the current window; which = 0 corner, 1 surf) to the host. */
ILSM_API int ilsm_cubemap_cube(ilsm_cubemap* cm, int which, int cube_index, float* out_xyzi, int capacity, int* n_out);

/* --------------------------------------------- full per-frame loop: scanRegistration -> laserOdometry -> laserMapping ---- */
typedef struct ilsm_slam ilsm_slam;

typedef struct ilsm_slam_stats {
  int32_t n_cloud, n_sharp, n_less_sharp, n_flat, n_less_flat; /* sizes of the five clouds scanRegistration publishes */
  int32_t ran_odometry;        /* 0 on the first frame (systemInited) and when use_aloam == 0 */
  ilsm_reg_report odometry;    /* the two ceres::Solve summaries of laserOdometry.cpp:705-710 */
  ilsm_reg_report mapping;     /* those of laserMapping.cpp:836-850 */
  ilsm_cubemap_stats cubemap;
} ilsm_slam_stats;

/* The three LOAM nodes of the reference chained on one GPU with the inter-node topics kept in HBM.  line_res / plane_res
 * = mapping_line_resolution / mapping_plane_resolution (spot.launch:4-5), min_range = MINIMUM_RANGE (scanRegistration),
 * cube_capacity as in ilsm_cubemap_create. */
ILSM_API int ilsm_slam_create(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                              ilsm_slam** out);
/* The same front end and odometry with mapOptimization (ilsm_mapopt) as the mapping stage -- the node spot.launch
 * starts.  In ilsm_slam_stats the mapping summary is pass[0]; cubemap.n_map_surf = ground-map size,
 * cubemap.n_stack_surf = query points after VoxelGrid(0.8), cubemap.n_valid = 1 when the solve CONVERGED. */
ILSM_API int ilsm_slam_create_mapopt(ilsm_ctx* ctx, float voxel_leaf, float downsample_size, float min_range, ilsm_slam** out);
ILSM_API void ilsm_slam_destroy(ilsm_slam* slam);
/* The cube map owned by the pipeline (for ilsm_cubemap_cube / ilsm_cubemap_insert_world). */
ILSM_API ilsm_cubemap* ilsm_slam_cubemap(ilsm_slam* slam);

/* One LiDAR frame through the whole loop: laserCloudHandler (scanRegistration.cpp:189-669), the laserOdometry iteration
 * (laserOdometry.cpp:376-845: 2 x (association + Solve) from the previous q/t_last_curr when use_aloam != 0 -- the
 * fork runs it only on frames flagged "skip_intensity", :406-417 -- then t_w_curr += q_w_curr * t_last_curr,
 * q_w_curr *= q_last_curr and the swap of the "last" clouds / trees), and the laserMapping iteration (ilsm_cubemap_frame
 * with the less-sharp / less-flat clouds).  Returns the odometry pose (/laser_odom_to_init) and the mapped pose
 * (/aft_mapped_to_init).  Replaces: the three node bodies between /os_cloud_node/points and /aft_mapped_to_init. */
ILSM_API int ilsm_slam_frame(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam, double q_odom_xyzw[4],
                             double t_odom[3], double q_map_xyzw[4], double t_map[3], ilsm_slam_stats* stats);

/* The same loop with laserMapping as its own pipeline stage, the way the reference runs it as its own node: the cube map
 * lives on a second context owned by the handle, and the process() iteration of frame k runs there while the caller's
 * next call enqueues the front end and the odometry of frame k + 1.  ilsm_slam_frame_async returns the odometry pose of
 * THIS frame and the mapped pose of the PREVIOUS one (*have_prev = 0 on the first call; stats->mapping / cubemap then
 * also belong to the previous frame); ilsm_slam_flush collects the last frame's.  Pose for pose the results are those
 * of ilsm_slam_frame (same kernels, same order within each stage). */
ILSM_API int ilsm_slam_create_async(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                    ilsm_slam** out);
ILSM_API int ilsm_slam_frame_async(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam, double q_odom_xyzw[4],
                                   double t_odom[3], double q_map_prev_xyzw[4], double t_map_prev[3], int* have_prev,
                                   ilsm_slam_stats* stats);
ILSM_API int ilsm_slam_flush(ilsm_slam* slam, double q_map_xyzw[4], double t_map[3], int* have, ilsm_slam_stats* stats);
/* The same loop as THREE stages, the way the reference runs three nodes (spot.launch: ascanRegistration, alaserOdometry,
 * alaserMapping, each its own process fed by a topic queue): scanRegistration on an owned context with its own host
 * thread, laserOdometry on the caller's context and thread, laserMapping on a second owned context and thread.  One call
 * pushes frame k to the front-end stage, runs the odometry of frame k - 1 (pushed by the previous call) and collects the
 * mapping of frame k - 2:
 *   *odom_frame = index of the frame q_odom / t_odom belong to (-1: none yet), *map_frame likewise for q_map / t_map;
 *   stats: counts and odometry report of *odom_frame, mapping report and cube-map statistics of *map_frame.
 * n < 0 pushes nothing and only advances the stages (drain: two such calls after the last frame hand out everything).
 * `xyzi` is read asynchronously by the front-end stage: it must stay valid until the NEXT call of this function returns.
 * use_aloam travels with the frame.  Pose for pose the results are those of ilsm_slam_frame (same kernels, same order
 * within each stage; the inter-stage clouds rotate through three device slots). */
ILSM_API int ilsm_slam_create_staged(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                     ilsm_slam** out);
ILSM_API int ilsm_slam_frame_staged(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam,
                                    double q_odom_xyzw[4], double t_odom[3], int* odom_frame, double q_map_xyzw[4],
                                    double t_map[3], int* map_frame, ilsm_slam_stats* stats);
/* Profiling aid: host seconds spent per phase of ilsm_slam_frame[_async] since the last call of this function (reset on
 * read): [0] upload + front-end launches, [1] wait for the previous frame's mapping (pipelined mode), [2] wait for the front
 * end, [3] gathers / VoxelGrid / odometry launches, [4] wait for the odometry, [5] tree builds + mapping stage; pipelined mode:
 * [6] launches and [7] waits of the mapping stage's own thread.  Staged mode: [2] wait for the front-end stage, [0] hand-over to it,
 * [3] odometry launches, [1] wait for the mapping stage, [4] wait for the odometry, [5] tree builds + hand-over to the mapping stage,
 * [6] and [7] as in pipelined mode.  [6] and [7] of a frame are counted by the call that hands out its mapped pose, not
 * while the frame runs: over a run they add up to the mapping stage's time for every frame whose pose was handed out. */
ILSM_API int ilsm_slam_host_phases(ilsm_slam* slam, double out8[8]);

/* ------------------------------------------------------------------- scan-to-scan odometry (laserOdometry) ---- */

/* One frame of the A-LOAM odometry optimisation.  last_corner / last_surf are maps built (ilsm_map_build) over the
 * PREVIOUS frame's cornerPointsLessSharp / surfPointsLessFlat clouds, xyzi with intensity = scanID + 0.1*relTime and
 * ring-sorted as scanRegistration emits them; sharp / flat are the CURRENT frame's cornerPointsSharp /
 * surfPointsFlat.  q,t = para_q / para_t (q_last_curr, t_last_curr): read as the initial value, overwritten with
 * the optimised one.  Per pass: TransformToStart (s = 1), 1-NN (d2 < 25), second/third point on the neighbouring
 * rings (+-2.5), LidarEdgeFactor / LidarPlaneFactor, ceres::Solve (max 4 iterations, Huber 0.1); 2 passes.
 * If `factors` is non-NULL only the association at (q,t) is run and the nsh+nfl records are returned (plane factors
 * as unit normal + offset: r = n.lp + d == (lp - j).ljm).
 * Replaces: laserOdometry.cpp:417-711 (TransformToStart :147-170, edge search :446-565, plane search :568-689). */
ILSM_API int ilsm_odometry(ilsm_ctx* ctx, ilsm_map* last_corner, ilsm_map* last_surf, const float* sharp, int nsh,
                           const float* flat, int nfl, int stride_bytes, double q_xyzw[4], double t_xyz[3],
                           const ilsm_reg_opts* opts, ilsm_reg_report* report, ilsm_factor* factors);

/* ------------------------------------------------------------- K4: front end (projection + features) ---- */

/* Organised H x W cloud -> image_range (u8, min(range*20,255)), image_intensity (u8, min(I,255)) and cloud_track
 * (H*W packed xyzi floats; zeroed where range < 0.1).  Intensity is read at byte 16 for 32-byte PCL points and at
 * byte 12 for 16-byte packed points.  image_ambient of the reference stays all-zero and is not produced.
 * Replaces: ImageHandler::cloud_handler(msg)  image_handler.h_ouster:103-140 (called at scanRegistration.cpp:195,
 *           mapOptimization.cpp:145). */
ILSM_API int ilsm_project(ilsm_ctx* ctx, const float* xyzi, int H, int W, int stride_bytes, uint8_t* range_img,
                          uint8_t* inten_img, float* cloud_track_xyzi);
ILSM_API int ilsm_project_dev(ilsm_ctx* ctx, const float* d_xyzi, int H, int W, int stride_bytes, uint8_t* d_range_img,
                              uint8_t* d_inten_img, float* d_cloud_track_xyzi);

typedef struct ilsm_feature_counts {
  int32_t n_cloud;      /* ring-ordered cloud size (laserCloud) */
  int32_t n_sharp;      /* cornerPointsSharp */
  int32_t n_less_sharp; /* cornerPointsLessSharp */
  int32_t n_flat;       /* surfPointsFlat */
  int32_t n_less_flat;  /* surfPointsLessFlat (after the per-ring 0.2 m VoxelGrid) */
  int32_t flags;        /* non-zero: a ring segment exceeded the supported size */
  int32_t ring_start[64]; /* scanStartInd */
  int32_t ring_end[64];   /* scanEndInd */
} ilsm_feature_counts;

/* Caller-provided output arrays, each sized for n input points (any pointer may be NULL to skip that output). */
typedef struct ilsm_features {
  float* cloud_xyzi;       /* n x 4: ring-ordered cloud, intensity = scanID + 0.1 * relTime */
  float* curvature;        /* n     : cloudCurvature */
  int32_t* label;          /* n     : cloudLabel {2, 1, 0, -1} */
  int32_t* src_index;      /* n     : index of each ring-ordered point in the input cloud */
  int32_t* sharp_idx;      /* indices into the ring-ordered cloud, reference push order */
  int32_t* less_sharp_idx;
  int32_t* flat_idx;
  float* less_flat_xyzi;   /* n x 4 */
  ilsm_feature_counts counts;
} ilsm_features;

/* The numeric body of laserCloudHandler for a 64-ring sensor: min-range filter, ring (scanID) bucketing, curvature,
 * per-ring 6-segment sort (ties broken by point index) and sharp / less-sharp / flat / less-flat selection with
 * neighbour suppression, per-ring VoxelGrid(0.2) of the less-flat points.
 * Replaces: scanRegistration.cpp:235-589 (removeClosedPointCloud :152-186, ring/time tagging :277-374,
 *           curvature :397-412, labelling :427-577, VoxelGrid :580-589). */
ILSM_API int ilsm_extract_features(ilsm_ctx* ctx, const float* xyzi, int n, int stride_bytes, float min_range,
                                   ilsm_features* out);

/* pcl::VoxelGrid<PointXYZI>::filter with a cubic leaf: centroid of every field per voxel, output in ascending
 * voxel index; points of one voxel are accumulated in input order.  Up to 16384 points are handled by one block (one
 * launch); larger clouds (< 2^24 points) by a tiled multi-block sort.
 * Replaces: downSizeFilterCorner/Surf.filter  laserMapping.cpp:608-616 ; voxel_grid_.filter mapOptimization.cpp:368-370 */
ILSM_API int ilsm_voxelgrid(ilsm_ctx* ctx, const float* xyzi, int n, int stride_bytes, float leaf, float* out_xyzi,
                            int* n_out);

/* --------------------------------------------------- sensor_msgs/PointCloud2 wire format -> packed points ---- */

/* Where the fields the path reads sit inside one point of a sensor_msgs/PointCloud2 `data` blob (the message's
 * `fields[]`: name, offset, datatype).  x, y, z must be FLOAT32 (PCL's field map accepts nothing else for PointXYZI);
 * intensity may be FLOAT32 (what pcl::fromROSMsg maps) or, as an extension, UINT8 / UINT16 / UINT32 / FLOAT64
 * (converted to float); off_intensity < 0 = no such field (intensity 0).  Big-endian blobs are rejected. */
typedef struct ilsm_pc2_layout {
  int32_t point_step;         /* bytes per point (>= 12) */
  int32_t off_x, off_y, off_z;
  int32_t off_intensity;
  int32_t intensity_datatype; /* sensor_msgs/PointField: 2 UINT8, 4 UINT16, 6 UINT32, 7 FLOAT32, 8 FLOAT64 */
  int32_t is_bigendian;
  int32_t reserved;
} ilsm_pc2_layout;

/* Ouster OS0/OS1 driver layout: point_step 48, x 0, y 4, z 8, intensity FLOAT32 at 16. */
ILSM_API void ilsm_pc2_layout_ouster(ilsm_pc2_layout* l);

/* `data` (n_points * point_step bytes, row padding already skipped) -> n_points packed xyzi floats, on the device.
 * The blob is uploaded as it is and unpacked by a kernel: the host-side repacking loop of pcl::fromROSMsg disappears.
 * Replaces: pcl::fromROSMsg(*laserCloudMsg, laserCloudIn)  scanRegistration.cpp:235 ; image_handler.h_ouster:44,106 */
ILSM_API int ilsm_pc2_unpack(ilsm_ctx* ctx, const uint8_t* data, int n_points, const ilsm_pc2_layout* layout, float* out_xyzi);
ILSM_API int ilsm_pc2_unpack_dev(ilsm_ctx* ctx, const uint8_t* d_data, int n_points, const ilsm_pc2_layout* layout,
                                 float* d_out_xyzi);

/* The other direction: packed xyzi points -> the `data` blob of a sensor_msgs/PointCloud2 (n_points * point_step bytes;
 * x / y / z / intensity as FLOAT32 at the layout's 4-byte-aligned offsets, every other byte zero), for the clouds the nodes
 * publish.  ilsm_pc2_layout_pcl_xyzi = what pcl::toROSMsg emits for pcl::PointXYZI (point_step 32: x 0, y 4, z 8,
 * intensity 16).  The _dev form reads and writes device memory and does not synchronise.
 * Replaces: pcl::toROSMsg(...)  scanRegistration.cpp:593,599,622,630,638 ; laserMapping.cpp:1023,1043,1061 */
ILSM_API void ilsm_pc2_layout_pcl_xyzi(ilsm_pc2_layout* l);
ILSM_API int ilsm_pc2_pack(ilsm_ctx* ctx, const float* xyzi, int n_points, const ilsm_pc2_layout* layout, uint8_t* data_out);
ILSM_API int ilsm_pc2_pack_dev(ilsm_ctx* ctx, const float* d_xyzi, int n_points, const ilsm_pc2_layout* layout, uint8_t* d_data_out);

/* ilsm_slam_frame fed with the raw message blob (same outputs). */
ILSM_API int ilsm_slam_frame_pc2(ilsm_slam* slam, const uint8_t* data, int n_points, const ilsm_pc2_layout* layout, int use_aloam,
                                 double q_odom_xyzw[4], double t_odom[3], double q_map_xyzw[4], double t_map[3],
                                 ilsm_slam_stats* stats);

/* ------------------------------------------------------- ground-plane extraction (feeds mapOptimization) ---- */
typedef struct ilsm_ground ilsm_ground;

typedef struct ilsm_ground_opts {
  double z_min, z_max;        /* screening band: -2.0 <= z <= -0.45   image_handler.h_ouster:50 */
  double distance_threshold;  /* seg.setDistanceThreshold(0.01)       :60 */
  double probability;         /* pcl::SACSegmentation default 0.99 */
  int32_t max_iterations;     /* pcl::SACSegmentation default 50 (at most 62 here) */
  int32_t seed;               /* seed of the declared sampler (PCL's rand() is unpinned) */
  double band;                /* height <= 0.03                        :85 */
  double max_angle_deg;       /* plane_normal . z > cos(15 deg)        :75 */
} ilsm_ground_opts;

typedef struct ilsm_ground_info {
  int32_t n_band;           /* points in the screening band */
  int32_t best_hypothesis;  /* index of the winning sample triple (-1: none) */
  int32_t n_best_inliers;
  int32_t iterations;       /* RANSAC iterations the adaptive loop ran */
  int32_t accepted;         /* the refitted plane passed the 15-degree test */
  int32_t reserved;
} ilsm_ground_info;

ILSM_API void ilsm_ground_opts_default(ilsm_ground_opts* o);
ILSM_API int ilsm_ground_create(ilsm_ctx* ctx, ilsm_ground** out);
ILSM_API void ilsm_ground_destroy(ilsm_ground* g);

/* z-band screening, RANSAC plane (PCL 1.10 RandomSampleConsensus loop: best-so-far, adaptive k, all 64 candidate
 * planes scored in parallel on the device), least-squares refit of the winner's inliers, 15-degree acceptance, then
 * the points of the WHOLE input within `band` of the plane and z < 0, in input order, as 16-byte pcl::PointXYZ
 * (out_xyz capacity in points; *n_out = number found).  coeff_abcd = the refitted plane (float, normal oriented up).
 * Replaces: ImageHandler::groundPlaneExtraction  image_handler.h_ouster:41-100 (called at mapOptimization.cpp:136). */
ILSM_API int ilsm_ground_extract(ilsm_ground* g, const float* xyz, int n, int stride_bytes, const ilsm_ground_opts* opts,
                                 float* out_xyz, int capacity, int* n_out, float coeff_abcd[4], ilsm_ground_info* info);

/* ----------------------------------------------- mapOptimization: the mapping node spot.launch starts ---- */
typedef struct ilsm_mapopt ilsm_mapopt;

typedef struct ilsm_mapopt_stats {
  ilsm_ground_info ground;
  float ground_coeff[4];
  int32_t n_ground;          /* RANSAC ground points of the frame */
  int32_t n_plane_in;        /* pc_plane points appended */
  int32_t n_query;           /* points after VoxelGrid(0.8) */
  int32_t ran_optimization;  /* 0 on the first callback (tree build only) */
  int32_t converged;         /* summary.termination_type == ceres::CONVERGENCE  mapOptimization.cpp:448 */
  int32_t map_size;          /* points in the ground map after Add_Points */
  ilsm_solve_summary solve;
  double q_key[4], t_key[3]; /* cur_keyframe pose used for the insertion: optimised if converged, else predicted */
  double reserved;
} ilsm_mapopt_stats;

/* voxel_leaf = voxel_grid_ leaf (0.8, mapOptimization.cpp:578), downsample_size = ikd-Tree box (0.4, :504);
 * <= 0 selects those defaults. */
ILSM_API int ilsm_mapopt_create(ilsm_ctx* ctx, float voxel_leaf, float downsample_size, ilsm_mapopt** out);
ILSM_API void ilsm_mapopt_destroy(ilsm_mapopt* mo);
ILSM_API int ilsm_mapopt_map_size(const ilsm_mapopt* mo);
/* ikdtree->flatten: the ground map in map order (packed xyz0). */
ILSM_API int ilsm_mapopt_map_points(ilsm_mapopt* mo, float* out_xyz0, int capacity, int* n_out);

/* One mapOptimizationCallback iteration (mapOptimization.cpp:99-500, LiDAR part): ground extraction from the organised
 * frame, + pc_plane (the less-flat cloud of scanRegistration), first call: tree build at the predicted pose; afterwards
 * VoxelGrid(0.8), 5-NN plane association against the ground map, LidarPlaneNormFactor solve (one pass, 10 iterations,
 * Huber 0.1), transformUpdate only on CONVERGENCE, Add_Points(0.4 m boxes) at the keyframe pose.  q_w / t_w return the
 * parameter block after the solve (Ceres writes it in place whatever the termination type); stats->q_key / t_key the
 * pose the map was extended with.  Replaces: mapOptimization::mapOptimizationCallback, LiDAR residuals only (the ORB
 * point-to-point blocks are dead code in the reference: `&& false` at :251, sliding window size 0). */
ILSM_API int ilsm_mapopt_frame(ilsm_mapopt* mo, const float* frame_xyz, int n, int stride_bytes, const float* plane_xyz, int n_plane,
                               int plane_stride_bytes, const double q_wodom_xyzw[4], const double t_wodom[3], double q_w_xyzw[4],
                               double t_w[3], const ilsm_ground_opts* gopts, ilsm_mapopt_stats* stats);

/* --------------------------------------- intensity-image feature back end (ORB matching + 3D-3D alignment) ---- */

/* cv::DMatch layout (queryIdx, trainIdx, imgIdx, distance): a std::vector<cv::DMatch> can be filled in place. */
typedef struct ilsm_dmatch {
  int32_t queryIdx;
  int32_t trainIdx;
  int32_t imgIdx;
  float distance;
} ilsm_dmatch;

/* Brute-force Hamming matching of 256-bit ORB descriptors (rows of cv::Mat CV_8U, 32 bytes each): every query row
 * takes its nearest train row, first minimum wins; with cross_check != 0 a pair survives only if it is mutual.
 * matches: the surviving pairs in query order (capacity n_cur); good: the same pairs sorted by (distance, queryIdx),
 * truncated to ceil(n_matches * keep_fraction) (capacity n_cur).  At most 16384 query descriptors.
 * Replaces: cv::BFMatcher(cv::NORM_HAMMING, true).match(cur, prev, matches); std::sort(matches); first 30 % / 20 %
 *           intensity_feature_tracker.cpp:631-648, 678-686. */
ILSM_API int ilsm_orb_match(ilsm_ctx* ctx, const uint8_t* cur_desc, int n_cur, const uint8_t* prev_desc, int n_prev, int desc_bytes,
                            int cross_check, double keep_fraction, ilsm_dmatch* matches, int* n_matches, ilsm_dmatch* good,
                            int* n_good);

/* 3D-3D alignment of matched points: minimise sum rho(|q * src_i + t - dst_i|^2), HuberLoss(huber_a),
 * EigenQuaternionParameterization, Levenberg-Marquardt on the device (the same solver as ilsm_solve); q, t are read
 * as the initial value ({0,0,0,1},{0,0,0} in the reference) and overwritten.  Points are 3 floats with a byte stride
 * (12 for cv::Point3f).  summary->num_edge_factors counts the point pairs.
 * Replaces: feature_tracker::p2p_calculateRandT  intensity_feature_tracker.cpp:880-928 (front_end_residual,
 *           lidarFeaturePointsFunction.hpp:21-58; max_num_iterations 20). */
ILSM_API int ilsm_align_points(ilsm_ctx* ctx, const float* src_xyz, const float* dst_xyz, int n, int stride_bytes, double q_xyzw[4],
                               double t_xyz[3], int max_num_iterations, double huber_a, ilsm_solve_summary* summary);

/* ------------------------------------------------------ K5: ScanContext loop-closure candidate scoring ---- */
typedef struct ilsm_sc ilsm_sc; /* keyframe descriptor database (one shard when split across ranks) */

ILSM_API int ilsm_sc_create(ilsm_ctx* ctx, ilsm_sc** out);
ILSM_API void ilsm_sc_destroy(ilsm_sc* sc);
ILSM_API int ilsm_sc_size(const ilsm_sc* sc);

/* Points -> 20x60 polar max-height descriptor, row-major float (ring, sector); empty bins 0.
 * Replaces: SCManager::makeScancontext  Scancontext.cpp:160-204 */
ILSM_API int ilsm_sc_make(ilsm_sc* sc, const float* xyz, int n, int stride_bytes, float* desc_20x60);

/* Append `count` descriptors (ring/sector keys are recomputed on the fly when scoring).
 * Replaces: the push_backs of makeAndSaveScancontextAndKeys  Scancontext.cpp:237-251 */
ILSM_API int ilsm_sc_add(ilsm_sc* sc, const float* desc_20x60, int count);
ILSM_API int ilsm_sc_add_dev(ilsm_sc* sc, const float* d_desc_20x60, int count);

/* Score the query against database entries [0, n_search) (n_search < 0: all; the caller excludes the most recent
 * NUM_EXCLUDE_RECENT = 50 entries like Scancontext.cpp:270-275) with distanceBtnScanContext -- sector-key alignment
 * over 60 shifts, column-cosine distance on the 7 shifts around it, first minimum wins -- and return the k <= 16
 * best by (distance, id).  id_offset is added to the returned ids (global id of this shard's first entry).
 * Replaces: Scancontext.cpp:79-157 and the candidate loop :299-312, scored over EVERY entry: a superset of the
 *           reference's 10 ring-key candidates, so it can report a closer entry than the reference finds -- the
 *           reference-exact search is ilsm_sc_query_candidates below. */
ILSM_API int ilsm_sc_query_topk(ilsm_sc* sc, const float* desc_20x60, int n_search, int id_offset, int k, double* dist,
                                int32_t* id, int32_t* shift);
ILSM_API int ilsm_sc_query_topk_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_search, int id_offset, int k,
                                    double* d_dist, int32_t* d_id, int32_t* d_shift);

/* Host-side deterministic merge of gathered per-shard top-k lists (n_entries = shards * k). */
ILSM_API int ilsm_sc_merge_topk(const double* dist, const int32_t* id, const int32_t* shift, int n_entries, int k,
                                double* out_dist, int32_t* out_id, int32_t* out_shift);

/* The same merge on the device, for the all-gathered buffer of a sharded query (no host round trip between the
 * scoring kernels, the NCCL all-gather and the merge).  Packed layout per shard and for the output:
 * k x f64 distance | k x i32 id | k x i32 shift (16 k bytes); ilsm_sc_query_topk_dev can write it directly with
 * d_dist = base, d_id = base + 8 k, d_shift = base + 12 k. */
ILSM_API int ilsm_sc_merge_topk_dev(ilsm_sc* sc, const void* d_packed, int shards, int k, void* d_out_packed);

/* detectLoopClosureID's own two steps over database entries [0, n_search) (n_search < 0: all; the caller passes the
 * size of the ring-key tree at its last refresh, i.e. it excludes the most recent NUM_EXCLUDE_RECENT = 50 entries and
 * applies TREE_MAKING_PERIOD_ like Scancontext.cpp:270-282):
 *   1. the num_candidates (<= 16; NUM_CANDIDATES_FROM_TREE = 10) nearest FLOAT ring keys -- polarcontext_invkeys_mat_,
 *      row means cast to float -- under the L2 metric as nanoflann's L2_Adaptor<float> evaluates it (groups of four,
 *      no FMA), ascending (distance, index): the result set of polarcontext_tree_->index->findNeighbors (:289-295);
 *   2. distanceBtnScanContext (:126-157) for exactly those entries.
 * cand_id / cand_key_d2 / cand_dist / cand_shift receive num_candidates entries in candidate order (id -1, distance
 * +inf when the database is smaller); the caller's `candidate_dist < min_dist` loop and SC_DIST_THRES test (:299-323)
 * then give the reference's loop id and yaw difference.  cand_key_d2 may be NULL.
 * Replaces: SCManager::detectLoopClosureID  Scancontext.cpp:283-312 (same candidates, same result). */
ILSM_API int ilsm_sc_query_candidates(ilsm_sc* sc, const float* desc_20x60, int n_search, int num_candidates, int32_t* cand_id,
                                      float* cand_key_d2, double* cand_dist, int32_t* cand_shift);

/* n_queries descriptors (contiguous, 1200 floats each) scored against entries [0, n_search) in one call; outputs are
 * [n_queries][k].  The _dev form takes device descriptors and writes n_queries packed records (16 k bytes each, the
 * layout of ilsm_sc_merge_topk_dev) without synchronising.  Both forms take 1 <= n_queries <= 4096 and 1 <= k <= 16,
 * else ILSM_ERR_INVALID_ARG. */
ILSM_API int ilsm_sc_query_topk_batch(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                      double* dist, int32_t* id, int32_t* shift);
ILSM_API int ilsm_sc_query_topk_batch_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                          void* d_packed);

/* Large shards (>= 4096 entries) are scored in two steps: an approximate distance of every (query, entry) pair on the
 * tensor cores (f16 operands, fp32 accumulation, 8 queries per staged entry), then the exact fp64 scorer on the entries
 * whose approximate distance is within a proven error bound of the k-th best (and on every pair whose sector-key
 * alignment the approximation could not decide).  The reported top-k is the one an exact scan of every entry gives.
 * ilsm_sc_prefilter_debug exposes the first step for tests: approx[q * n_search + c] (-1 = pair flagged for exact
 * rescoring; <= -2 = the alignment is one of two, the value is -2 - the smaller of the two distances, a lower bound of the
 * exact one) and the aligned shift it used; n_queries <= 8. */
ILSM_API int ilsm_sc_prefilter_debug(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, float* approx,
                                     uint8_t* aligned_shift);

/* The keyframe database sharded over n_ranks processes (one per GPU), contiguous id ranges: every rank holds its
 * shard in its own ilsm_sc and the ranks share an NCCL communicator.  ilsm_sc_init_nccl adopts a communicator the
 * host already owns (ncclComm_t passed as void*; it is not destroyed with the handle); ilsm_sc_nccl_unique_id +
 * ilsm_sc_init_nccl_rank create one (rank 0 makes the 128-byte id, the host distributes it by its own means, every
 * rank calls init_nccl_rank -- a collective call).  NCCL is loaded with dlopen at the first of these calls. */
ILSM_API int ilsm_sc_nccl_unique_id(char id_out[128]);
ILSM_API int ilsm_sc_init_nccl_rank(ilsm_sc* sc, const char id[128], int n_ranks, int rank);
ILSM_API int ilsm_sc_init_nccl(ilsm_sc* sc, void* nccl_comm, int n_ranks, int rank);
ILSM_API int ilsm_sc_nccl_version(int* version);

/* A sharded query batch -- a COLLECTIVE call, every rank passes the same descriptors: the local shard is scored
 * (entries [0, n_search) of this rank, ids reported as id_offset + local index), the per-rank packed top-k records of
 * the whole batch are exchanged with ONE ncclAllGather (n_queries x 16 k bytes per rank) and merged by the same
 * deterministic kernel on every rank (ascending (distance, id)); nothing visits the host in between.  Every rank
 * receives the global top-k.  Without a communicator (n_ranks 1) it degenerates to ilsm_sc_query_topk_batch.
 * n_queries and k have the bounds of ilsm_sc_query_topk_batch in both forms.
 * Replaces: the candidate scoring of Scancontext.cpp:299-312 over a database split across GPUs (BASELINE configs[4]). */
ILSM_API int ilsm_sc_query_topk_sharded(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                        double* dist, int32_t* id, int32_t* shift);
ILSM_API int ilsm_sc_query_topk_sharded_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                            void* d_packed_out);

/* ------------------------------------------------ K6: loop-closure verification, point-to-point ICP ---- */
/* pcl::IterativeClosestPoint<PointXYZI, PointXYZI> (PCL 1.10) for a batch of (source, target) pairs.  Per pair, starting
 * from the guess P: every iteration maps the ORIGINAL source points by P (double math, float store), takes the exact 1-NN
 * of each in the target (ties by (d2, index)), keeps the pairs with d2 <= max_correspondence_distance^2, fits the rigid
 * transform of those pairs in closed form (fp64 sums, Horn's quaternion method) and composes it onto P, until
 * DefaultConvergenceCriteria stops it.  The fitness is getFitnessScore(fitness_max_range) of the final pose: the mean 1-NN
 * d2 over the points with d2 <= fitness_max_range -- PCL compares the SQUARED distance with the range; kept.
 * Replaces: the pcl::IterativeClosestPoint of loopClosureThread  intensity_feature_tracker.cpp:195-393. */
typedef enum ilsm_icp_state { /* pcl::registration::DefaultConvergenceCriteria::ConvergenceState, same order */
  ILSM_ICP_NOT_CONVERGED = 0,
  ILSM_ICP_ITERATIONS = 1,
  ILSM_ICP_TRANSFORM = 2,
  ILSM_ICP_ABS_MSE = 3,
  ILSM_ICP_REL_MSE = 4,
  ILSM_ICP_NO_CORRESPONDENCES = 5
} ilsm_icp_state;

typedef struct ilsm_icp_opts {
  double max_correspondence_distance; /* metres; sqrt(DBL_MAX) = no gate */
  int max_iterations;                 /* the loop is a do-while: 0 still runs one iteration */
  int pad;
  double transformation_epsilon;          /* on |t|^2 of one iteration's increment */
  double transformation_rotation_epsilon; /* on cos(angle) of the increment; <= 0: 1 - transformation_epsilon */
  double euclidean_fitness_epsilon;       /* on the relative change of the correspondence MSE */
  double fitness_max_range;               /* compared with the 1-NN d2 of the fitness score */
} ilsm_icp_opts;

/* PCL 1.10's defaults: sqrt(DBL_MAX), 10, 0, 0, -DBL_MAX, DBL_MAX. */
ILSM_API void ilsm_icp_opts_default(ilsm_icp_opts* o);

typedef struct ilsm_icp_result {
  double q_xyzw[4], t[3]; /* final transformation, source -> target */
  double fitness;         /* getFitnessScore(fitness_max_range); DBL_MAX when no point is in range */
  double mse;             /* the last correspondence search's mean d2; DBL_MAX when it found none */
  int iterations;         /* nr_iterations_ */
  int state;              /* ilsm_icp_state */
  int converged;          /* hasConverged(): every state but NOT_CONVERGED and NO_CORRESPONDENCES */
  int n_correspondences;  /* of the last correspondence search */
} ilsm_icp_result;

/* Pair p aligns source points [src_offsets[p], src_offsets[p+1]) (3 floats with a byte stride) to targets[p] (a built
 * ilsm_map of this context), starting from guess7[7p..7p+6] = (qx,qy,qz,qw,tx,ty,tz), a unit quaternion, or the identity
 * when guess7 is NULL.  opts NULL: the defaults.  One kernel launch for the whole batch; returns when results[0..n_pairs)
 * are filled.  A pair with fewer than 3 source points or an empty target ends in ILSM_ICP_NO_CORRESPONDENCES with 0
 * iterations and the guess as its pose.  The _dev form reads the points from device memory (offsets, guesses and results
 * stay on the host). */
ILSM_API int ilsm_icp_align_batch(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* src_xyz,
                                  const int* src_offsets, int stride_bytes, const double* guess7,
                                  const ilsm_icp_opts* opts, ilsm_icp_result* results);
ILSM_API int ilsm_icp_align_batch_dev(ilsm_ctx* ctx, ilsm_map* const* targets, int n_pairs, const float* d_src_xyz,
                                      const int* src_offsets, int stride_bytes, const double* guess7,
                                      const ilsm_icp_opts* opts, ilsm_icp_result* results);

/* ------------------------------------------- K7: loop closure per keyframe against a resident keyframe store ---- */
/* One handle per loop-closure thread (give it its own ilsm_ctx, the way the reference runs loopClosureThread on its own
 * thread).  Every keyframe passed in is stored on the device -- its ScanContext descriptor, VoxelGrid(leaf) of its cloud and
 * its pose -- and answered with that keyframe's loop decision; choosing which frames are keyframes stays with the caller.
 * Replaces: the body of loopClosureThread (intensity_feature_tracker.cpp:195-393) around SCManager::
 *           makeAndSaveScancontextAndKeys + detectLoopClosureID (Scancontext.cpp:237-344) and the ICP check. */
typedef struct ilsm_loop ilsm_loop;

typedef struct ilsm_loop_opts {
  int32_t exclude_recent;     /* NUM_EXCLUDE_RECENT = 50; >= 1 */
  int32_t tree_period;        /* TREE_MAKING_PERIOD_ = 50; >= 1 */
  int32_t num_candidates;     /* NUM_CANDIDATES_FROM_TREE = 10; 1..16 */
  int32_t submap_half;        /* target = keyframes c-h .. c+h; 0..7 (2) */
  double sc_dist_threshold;   /* SC_DIST_THRES = 0.13: a loop iff min_dist < this */
  float leaf;                 /* VoxelGrid leaf of the stored keyframes and of the submap (0.4); > 0 */
  float cell;                 /* k-NN cell of the submap's map (1.0); > 0 */
  double fitness_threshold;   /* accepted iff the ICP converged && fitness < this (0.3) */
  ilsm_icp_opts icp;          /* 2.0 m, 50 iterations, transformation_epsilon 1e-8, euclidean_fitness_epsilon 1e-6 */
} ilsm_loop_opts;

typedef struct ilsm_loop_result {
  int32_t keyframe_id;   /* id of this keyframe (0, 1, 2, ... in call order) */
  int32_t loop_id;       /* detectLoopClosureID's loop id, -1: none */
  int32_t nn_id;         /* best candidate, -1: early return (fewer than exclude_recent + 1 keyframes) */
  int32_t shift;         /* its aligning column shift (sectors of 6 degrees) */
  double sc_dist;        /* its distance (min_dist) */
  double yaw_diff_rad;   /* deg2rad(shift * 6) as the reference returns it (a float) */
  int32_t verified;      /* 1 when loop_id >= 0: the ICP ran */
  int32_t accepted;      /* verified && icp.converged && icp.fitness < fitness_threshold */
  int32_t submap_first, submap_last; /* the target's keyframes: [loop_id - h, loop_id + h] within [0, size - exclude_recent) */
  int32_t submap_points; /* VoxelGrid(leaf) size of the world-frame target */
  int32_t reserved;
  double q_rel_xyzw[4], t_rel[3]; /* when accepted: T_loop^-1 * T_icp, this keyframe in the frame of keyframe loop_id */
  ilsm_icp_result icp;   /* when verified: the world pose of this keyframe ICP found (source = this keyframe's stored
                            cloud, guess = (q_loop * Rz(-yaw_diff_rad), t_loop)) */
} ilsm_loop_result;

/* The values above. */
ILSM_API void ilsm_loop_opts_default(ilsm_loop_opts* o);
/* opts NULL: the defaults; options outside the ranges above: ILSM_ERR_INVALID_ARG.  ILSM_ERR_NO_DEVICE without a GPU. */
ILSM_API int ilsm_loop_create(ilsm_ctx* ctx, const ilsm_loop_opts* opts, ilsm_loop** out);
ILSM_API void ilsm_loop_destroy(ilsm_loop* loop);
/* keyframes stored */
ILSM_API int ilsm_loop_size(const ilsm_loop* loop);
/* Store one keyframe (n xyzi points, stride_bytes >= 16, intensity at the fourth float, or the fifth from 32 bytes; n < 2^24)
 * with its world pose (q unit within 1e-6, else ILSM_ERR_INVALID_ARG) and return its loop decision in *result:
 *   detect  SCManager's state machine -- fewer than exclude_recent + 1 keyframes: early return, the refresh counter stays;
 *           every tree_period-th search the searchable size becomes size - exclude_recent; the num_candidates nearest
 *           ring keys are scored (ilsm_sc_query_candidates), the first strict minimum wins, min_dist < sc_dist_threshold;
 *   verify  with a loop: keyframes [c-h, c+h] of the store to the world frame (double math, float store), VoxelGrid(leaf),
 *           a map with cell `cell`, one ICP pair (ilsm_icp_align_batch) from the guess above.
 * One host synchronisation per call; two more for a verified keyframe.  The _dev form reads the points from device memory.
 * Argument errors come back before any CUDA call. */
ILSM_API int ilsm_loop_add_keyframe(ilsm_loop* loop, const float* xyz, int n, int stride_bytes, const double q_xyzw[4],
                                    const double t_xyz[3], ilsm_loop_result* result);
ILSM_API int ilsm_loop_add_keyframe_dev(ilsm_loop* loop, const float* d_xyz, int n, int stride_bytes, const double q_xyzw[4],
                                        const double t_xyz[3], ilsm_loop_result* result);

/* ---------------------------------------------- the full loop with loop closure as its own stage ---- */
/* A full-loop handle (ilsm_slam, every kind) can run loop closure beside mapping, the way the reference runs
 * loopClosureThread beside its mapping loop.  Every mapped pose the handle hands out is checked against the keyframe rule:
 * frame k is a keyframe when it is the first frame handed out, or when ||t_k - t_kf|| >= keyframe_dist, or when
 * 2 atan2(||v||, |w|) >= keyframe_angle_rad for (v, w) = q_kf^-1 * q_k, where (q_kf, t_kf) is the mapped pose of the last
 * keyframe (fp64 on the host; DESIGN section 2 gives the order of operations).  Both thresholds 0: every frame is one.
 * A keyframe's cloud never leaves the device: the front end's ring-ordered cloud (/velodyne_cloud_2, what
 * ilsm_extract_features returns as cloud_xyzi, n_cloud points of 16 bytes, after the range filter) is copied into one of
 * max_pending device buffers and handed, with the mapped pose, to an ilsm_loop on a context and host thread the handle
 * owns.  The cloud's fourth float is scanID + 0.1 relTime, not intensity; neither ScanContext nor the ICP reads it.
 * Loop closure only reads: every odometry and mapped pose is bit-identical to the same handle without it. */
typedef struct ilsm_slam_loop_opts {
  double keyframe_dist;       /* m (1.0); finite, >= 0 */
  double keyframe_angle_rad;  /* (0.2); finite, >= 0 */
  int32_t max_pending;        /* keyframes handed to the loop stage and not yet answered before a frame call waits (8); >= 1 */
  int32_t reserved;
  ilsm_loop_opts loop;        /* the loop handle's options (ilsm_loop_opts_default) */
} ilsm_slam_loop_opts;

typedef struct ilsm_slam_loop_event {
  int64_t frame;              /* index of the frame that became the keyframe, 0-based in hand-in order */
  double q_xyzw[4], t[3];     /* its mapped pose, as stored */
  ilsm_loop_result result;    /* its loop decision; result.keyframe_id = 0, 1, 2, ... */
} ilsm_slam_loop_event;

/* keyframe_dist 1.0, keyframe_angle_rad 0.2, max_pending 8, loop = ilsm_loop_opts_default */
ILSM_API void ilsm_slam_loop_opts_default(ilsm_slam_loop_opts* o);
/* Turn loop closure on.  opts NULL: the defaults.  Call before the first frame (ILSM_ERR_STATE after it, or when it is
 * already on).  Options outside the ranges above, including those of ilsm_loop_create: ILSM_ERR_INVALID_ARG, before any
 * CUDA call; ILSM_ERR_NO_DEVICE without a GPU.  The slot and pending buffers are reserved here, at 65 536 points.
 * A frame call waits for loop closure only when a new keyframe finds all max_pending buffers in flight: it then waits
 * for the oldest answer and queues it for ilsm_slam_loop_results. */
ILSM_API int ilsm_slam_enable_loop(ilsm_slam* slam, const ilsm_slam_loop_opts* opts);
/* The decisions of the keyframes answered so far, in keyframe order, at most `capacity` of them into out[0 .. *n_out).
 * wait != 0: first wait until every keyframe selected so far has been answered.  The rest stay queued for the next call.
 * Call it from the thread that hands in the frames, not during a frame call; it takes no context lock.  ILSM_ERR_STATE on a
 * handle without loop closure.  A keyframe that failed (on the loop stage, or while being handed over) is reported here
 * and only here, in keyframe order: the call that reaches it with nothing handed out before it returns its status and
 * error text and drops it; later keyframes stay queued.  Frame calls never return loop-closure errors. */
ILSM_API int ilsm_slam_loop_results(ilsm_slam* slam, int wait, ilsm_slam_loop_event* out, int capacity, int* n_out);

#ifdef __cplusplus
}
#endif
#endif /* ILSM_H_ */
