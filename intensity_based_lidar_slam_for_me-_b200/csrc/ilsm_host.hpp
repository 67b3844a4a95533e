// ilsm_host.hpp -- host-side objects behind the opaque C handles (ilsm_ctx, ilsm_map).
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <memory>
#include <mutex>
#include <string>

#include "../../include/ilsm.h"
#include "ilsm_internal.cuh"

namespace ilsm {

int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int fail_cuda(cudaError_t e, const char* where);
int check_launch(const char* where);
void count_launches(int k);

// A point stride the entry points accept: x, y, z as floats on 4-byte boundaries.
inline bool valid_stride(int stride_bytes) { return stride_bytes >= 12 && (stride_bytes % 4) == 0; }
// Float index of a point's intensity: the fifth word of a 32-byte-or-wider record (PCL's PointXYZI), else the fourth.
inline int intensity_word(int stride_bytes) { return stride_bytes >= 32 ? 4 : 3; }

#define ILSM_CUDA(call)                                        \
  do {                                                         \
    cudaError_t e__ = (call);                                  \
    if (e__ != cudaSuccess) return ::ilsm::fail_cuda(e__, #call); \
  } while (0)

// Launch with programmatic stream serialization: the kernel's launch latency overlaps the tail of its predecessor
// (the short kernels of a registration are launch-latency-bound).  The kernel must start with pdl_entry().
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr, cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Cluster size of the kernels that run a whole iterative solve in one thread-block cluster (the LM solve, ICP): `wide`
// CTAs, a non-portable size, where the device can place one cluster of `kernel` with `threads` threads per CTA, else the
// portable 8; ILSM_SOLVE_CLUSTER=8 forces 8.  Probed once per context and kernel: `cached` is -1 until then, then 1 or 0.
template <typename... KArgs>
bool wide_cluster(int& cached, void (*kernel)(KArgs...), int wide, int threads) {
  if (cached < 0) {
    cached = 0;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(wide), cfg.blockDim = dim3(threads);
      cudaLaunchAttribute at;
      at.id = cudaLaunchAttributeClusterDimension;
      at.val.clusterDim.x = wide, at.val.clusterDim.y = 1, at.val.clusterDim.z = 1;
      cfg.attrs = &at, cfg.numAttrs = 1;
      int n_clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&n_clusters, kernel, &cfg) == cudaSuccess && n_clusters >= 1) cached = 1;
    }
    (void)cudaGetLastError();
    if (const char* e = getenv("ILSM_SOLVE_CLUSTER"))
      if (atoi(e) == 8) cached = 0;
  }
  return cached != 0;
}

// Bytes held by all device [0] and pinned [1] buffers of the process (ilsm_debug_live_bytes): a test can check that
// closing a handle frees everything it allocated, which cudaMemGetInfo cannot show on a GPU other processes use too.
extern std::atomic<long long> g_live_bytes[2];

struct DeviceMem {
  static constexpr int kind = 0;
  static constexpr const char* what = "cudaMalloc failed";
  static cudaError_t alloc(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
  static void dealloc(void* p) { cudaFree(p); }  // implicit device sync
};
struct PinnedMem {
  static constexpr int kind = 1;
  static constexpr const char* what = "cudaMallocHost failed";
  static cudaError_t alloc(void** p, size_t bytes) { return cudaMallocHost(p, bytes); }
  static void dealloc(void* p) { cudaFreeHost(p); }
};

// Grow-only buffer that owns its memory (HBM is plentiful: 180 GB; reallocation would serialise the stream).  Freed
// when the buffer is destroyed: its owner's teardown must have synchronised every stream that still reads it.
template <typename T, typename Mem>
struct Buf {
  T* p = nullptr;
  size_t cap = 0;
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  Buf(Buf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr, o.cap = 0; }
  Buf& operator=(Buf&& o) noexcept {
    if (this != &o) release(), p = o.p, cap = o.cap, o.p = nullptr, o.cap = 0;
    return *this;
  }
  ~Buf() { release(); }
  int reserve(size_t n) {
    if (n <= cap) return ILSM_OK;
    size_t want = n + n / 2 + 64;
    void* np = nullptr;
    if (Mem::alloc(&np, want * sizeof(T)) != cudaSuccess) {
      cudaGetLastError();
      return fail(ILSM_ERR_OUT_OF_MEMORY, "%s", Mem::what);
    }
    release();  // only on growth
    p = static_cast<T*>(np);
    cap = want;
    g_live_bytes[Mem::kind].fetch_add((long long)(cap * sizeof(T)), std::memory_order_relaxed);
    return ILSM_OK;
  }

 private:
  void release() {
    if (!p) return;
    Mem::dealloc(p);
    g_live_bytes[Mem::kind].fetch_sub((long long)(cap * sizeof(T)), std::memory_order_relaxed);
    p = nullptr;
    cap = 0;
  }
};
template <typename T>
using DevBuf = Buf<T, DeviceMem>;
template <typename T>
using PinnedBuf = Buf<T, PinnedMem>;

// CUDA events, streams and graph execs held by all owners of the process (ilsm_debug_live_handles), for the same check.
extern std::atomic<long long> g_live_handles;

// how each kind of handle is made and released: events without timing, non-blocking streams
inline cudaError_t create_handle(cudaEvent_t* h) { return cudaEventCreateWithFlags(h, cudaEventDisableTiming); }
inline cudaError_t create_handle(cudaStream_t* h) { return cudaStreamCreateWithFlags(h, cudaStreamNonBlocking); }
inline cudaError_t create_handle(cudaGraphExec_t* h, cudaGraph_t g) { return cudaGraphInstantiate(h, g, 0); }
inline void destroy_handle(cudaEvent_t h) { cudaEventDestroy(h); }
inline void destroy_handle(cudaStream_t h) { cudaStreamDestroy(h); }
inline void destroy_handle(cudaGraphExec_t h) { cudaGraphExecDestroy(h); }

// Move-only owner of one CUDA handle, released when the owner is destroyed: its owner's teardown must have synchronised
// every stream that still uses it.  Converts to the raw handle (nullptr while empty).
template <typename Raw>
class Owned {
 public:
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  Owned(Owned&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  ~Owned() { reset(); }
  operator Raw() const { return h_; }
  // releases the handle held, then makes a new one: ILSM_OK, or ILSM_ERR_CUDA through fail_cuda (the owner is left empty)
  template <typename... Args>
  int create(Args... args) {
    reset();
    Raw h = nullptr;
    const cudaError_t e = create_handle(&h, args...);
    if (e != cudaSuccess) return fail_cuda(e, "Owned::create");
    h_ = h;
    g_live_handles.fetch_add(1, std::memory_order_relaxed);
    return ILSM_OK;
  }
  void reset() {
    if (!h_) return;
    destroy_handle(h_);
    g_live_handles.fetch_sub(1, std::memory_order_relaxed);
    h_ = nullptr;
  }

 private:
  Raw h_ = nullptr;
};
using Event = Owned<cudaEvent_t>;
using Stream = Owned<cudaStream_t>;
using GraphExec = Owned<cudaGraphExec_t>;

// Levenberg-Marquardt state that lives in HBM for the duration of a registration: the trust-region loop of
// ceres::Solve runs on the device, one evaluation kernel per iteration, no host round trip.
struct LmState {
  double xq[4], xt[3];  // accepted pose (q = x,y,z,w)
  double cq[4], ct[3];  // candidate pose: what the next evaluation kernel evaluates
  double cost;          // cost at x
  double H[21], g[6];   // unscaled J^T J (upper triangle, row-major) and J^T r at x
  double scale[6];      // Jacobi scaling fixed at iteration 0
  double diag[6];       // LM diagonal (of the scaled J^T J) kept while reuse_diagonal
  double radius, decrease_factor, model_cost_change;
  double huber_a;
  double initial_cost;
  int status;  // 0 running, 1 + ilsm_termination when finished
  int phase;   // 0: next evaluation is the initial one, 1: trial step
  int iteration, max_iter, invalid_run, reuse_diag;
  int n_success, n_unsuccess, n_evals;
  int n_edge, n_plane;
  int pass;  // which report slot the running solve fills
  unsigned ticket;
  int pad;
  ilsm_reg_report report;
  long long dbg[64];  // clock64() phase stamps written when ILSM_DEBUG_TIMING is compiled in (profiling aid)
};
constexpr size_t kLmHostBytes = offsetof(LmState, report) + sizeof(ilsm_reg_report);  // what a solve reads back of the LM state

// Where the association kernel of the FIRST pass takes the pose from, and where the solve kernel of the LAST pass
// leaves the result: folding these into the two kernels removes the 1-warp pose upload / download launches.
struct PoseSrc {
  const double* dptr = nullptr;  // mode 2: 7 doubles on the device
  double v[7] = {0, 0, 0, 1, 0, 0, 0};  // mode 1: by value (host-pointer entry points)
  int mode = 0;                  // 0: the accepted pose already in the LM state
};
struct PoseDst {
  double* d_pose7 = nullptr;           // pose after the last pass (nullptr: stays in the LM state only)
  ilsm_reg_report* d_report = nullptr;  // the whole report (nullptr: stays in the LM state only)
};

struct Ctx;
struct Map;
int build_pair_dev(Map* a, const float* d_a, int na, Map* b, const float* d_b, int nb, int stride_bytes, float cell_size);

struct Map {
  Ctx* ctx = nullptr;
  int n = 0;
  float cell = 1.f, inv_cell = 1.f;
  uint32_t table_size = 0;
  int log2_size = 0;
  DevBuf<GridCell> cells;
  DevBuf<float4> sorted, orig;
  DevBuf<uint32_t> slot_of, rank_of, counters;
  // Two hash tables, occupied-slot lists, counter sets and boxes per map, used alternately: build g fills table g & 1
  // while its scatter launch empties the other one (the slots listed by the build before), so no clear pass is ever on
  // the critical path.  Table t = cells.p + t * table_cap, list t = occ.p + t * occ_cap, set t = counters.p + 8 t,
  // box t = bbox.p + 8 t.
  DevBuf<uint32_t> occ;
  uint32_t table_cap = 0;    // slots allocated per table
  size_t occ_cap = 0;        // entries allocated per list
  int gen = 0;               // build generation
  int cur = 0;               // table of the last build (what view() shows)
  size_t clean_size[2] = {0, 0};  // table t is EMPTY in [0, clean_size[t]) ...
  int filled_n[2] = {0, 0};       // ... unless filled_n[t] != 0: it still holds a build of (at most) that many voxels
  DevBuf<int> bbox;
  DevBuf<float> raw;  // staging of caller bytes for the host-pointer entry points
  // Each map builds on its own stream so that the corner and surf structures of a frame are built concurrently
  // (and their H2D copies overlap); users on the context stream wait on `ready`.
  Stream stream;
  // builds run in line on the context's stream, with no fork / join events: for callers whose builds have nothing to
  // overlap with (the cube map's two search structures sit on the mapping stage's critical path, and every event call is
  // host time there)
  bool in_line = false;
  Event ready, ctx_done;
  bool pending = false;

  // Add_Points scratch (ikdmap.cu)
  DevBuf<u64> vox_table;
  DevBuf<float4> ins_new, ins_out;
  DevBuf<uint32_t> ins_slot_new, ins_slot_old, ins_keep, ins_pos, ins_bsum;
  int insert_dev(const float* d_src, int n_new, int stride_bytes, int policy, float ds);

  int init(Ctx* c);
  int wait_ready(cudaStream_t user);
  int build_dev(const float* d_src, int n_pts, int stride_bytes, float cell_size);
  int prepare_build(const float* d_src, int n_pts, int stride_bytes, float cell_size, cudaStream_t s, void* job_out);
  // allocate for builds of up to n_pts points now (a buffer that grows later costs a device-wide synchronisation); only
  // while no build is in flight
  int reserve_points(int n_pts);
  const GridCell* cur_cells() const { return cells.p + (size_t)cur * table_cap; }
  const uint32_t* cur_occ() const { return occ.p + (size_t)cur * occ_cap; }
  const uint32_t* cur_counters() const { return counters.p + 8 * cur; }
  int knn_dev(const float* d_q, int nq, int stride_bytes, int k, float max_dist, int32_t* d_idx, float* d_d2);
  GridView view() const;
  ~Map();  // synchronises the map's stream
};

// Device-side factor storage (SoA), one slot per stack point (corner slots first).
struct FactorBufs {
  DevBuf<int> type;
  DevBuf<float4> p;    // curr_point (sensor frame), w unused
  DevBuf<double4> a;   // edge: point_a        ; plane: unit normal, w = negative_OA_dot_norm
  DevBuf<double4> b;   // edge: point_b
  DevBuf<int32_t> knn_idx;  // 5 per slot (debug / parity output)
  DevBuf<float> knn_d2;
  int n = 0, nc = 0;
};

struct VgState {      // device-resident scalars of one multi-block VoxelGrid
  int mn[3], mx[3];   // ordered-int encoded float min / max of the finite points
  int n_out;
  int pad;
};

// Front-end scratch and outputs (device-resident between the front end and the registration).
struct FeBufs {
  DevBuf<unsigned char> scanid, picked;
  DevBuf<float> ori, curv;
  DevBuf<int> stats, src_index, label, sort_ind, ring_sharp, ring_lsharp, ring_flat, sharp, lsharp, flat, counts;
  DevBuf<u64> vg_keys;            // multi-block VoxelGrid: sort keys, state, per-chunk head counts / bases
  DevBuf<VgState> vg_state;
  DevBuf<int> vg_chunk;
  DevBuf<uint32_t> vg_hash;         // hash-based block VoxelGrid: global scratch of the (at most two) blocks of a launch
  DevBuf<int> chunk_hist, chunk_base;  // ring counts per 256-point chunk of the frame and their per-ring prefix
  DevBuf<float4> cloud, ring_pts, ring_out, lflat, vox_packed;
  DevBuf<float> raw;                 // staged caller frame
  DevBuf<unsigned char> pc2;         // staged sensor_msgs/PointCloud2 blob (ilsm_pc2_unpack, ilsm_slam_frame_pc2)
  DevBuf<unsigned char> img;         // projection outputs (range | intensity)
  DevBuf<float4> track;
  DevBuf<float4> vox_out;
  DevBuf<int> vox_n;
  int n_in = 0, ring_cap = 0;
};

struct Ctx {
  int device = 0;
  int sm_count = 148;
  Stream stream;
  Stream aux;  // side stream: work of a frame that does not depend on the odometry
  Event ev_fork, ev_join;
  std::mutex mu;
  DevBuf<LmState> lm;
  DevBuf<double> partials;  // [blocks][32]
  DevBuf<float> stack_raw;  // staged caller stacks
  DevBuf<int32_t> out_idx;
  DevBuf<float> out_d2;
  PinnedBuf<unsigned char> pinned;
  FactorBufs fac;
  FeBufs fe;
  const int* d_stack_counts = nullptr;  // when set, associate/solve read {nc, ns} from the device (cube-map path)
  int solve_wide = -1;                  // LM solve as a 16-CTA cluster (1) or the portable 8 (0); -1: not probed yet
  DevBuf<float4> rf_lsharp, rf_stack_c, rf_stack_s;  // ilsm_register_frame: less-sharp cloud and the two down-sampled stacks
  DevBuf<int> rf_stack_n;
  std::unique_ptr<Map> qbin;  // query binning of the throughput k-NN path (knn_binned.cu): the query cloud grouped by voxel
  DevBuf<int> qwork;          // its work items (4 ints each) + the item counter
  int knn_group = 8;          // queries per group of the binned search (ILSM_KNN_GROUP: 1, 2, 4, 8, 16 or 32)
  int knn_binned_min = 8192;  // query sets at least this large take the binned path (ILSM_KNN_BINNED_MIN overrides)
  size_t partial_blocks = 0;
  bool bulk_attr_set = false;
  // ICP verification batches (icp.cu): staged source points, per-pair records, tile partials, results
  DevBuf<float> icp_src;
  DevBuf<unsigned char> icp_pairs;
  DevBuf<double> icp_part;
  DevBuf<ilsm_icp_result> icp_res;
  PinnedBuf<unsigned char> icp_pin;
  int icp_wide = -1;  // ICP as 16-CTA clusters (1) or 8 (0); -1: not probed yet  // normal_eq_bulk_kernel's dynamic shared-memory opt-in done on this device

  int init(int dev);
  ~Ctx();  // the caller has made `device` current
  // LM pose staging in `pinned`: the LM state prefix (pose and report, xq first) comes back to offset 0 in one copy, a
  // pose goes up from kPinPoseIn.  [kPinSite, kPinPoseIn) is left to a call site's own read-back in the same synchronise.
  static constexpr size_t kPinSite = 1024, kPinPoseIn = 2048;
  static_assert(offsetof(LmState, xq) == 0 && offsetof(LmState, xt) == 4 * sizeof(double) && kLmHostBytes <= kPinSite,
                "the LM read-back overlaps the call sites' area");
  int upload_pose(const double q[4], const double t[3], cudaStream_t s) {  // -> lm.p->xq, xt
    double* p = reinterpret_cast<double*>(pinned.p + kPinPoseIn);
    for (int i = 0; i < 4; ++i) p[i] = q[i];
    for (int i = 0; i < 3; ++i) p[4 + i] = t[i];
    ILSM_CUDA(cudaMemcpyAsync(lm.p->xq, p, 7 * sizeof(double), cudaMemcpyHostToDevice, s));
    return ILSM_OK;
  }
  int read_back_lm(cudaStream_t s) {
    ILSM_CUDA(cudaMemcpyAsync(pinned.p, lm.p, kLmHostBytes, cudaMemcpyDeviceToHost, s));
    return ILSM_OK;
  }
  // after the caller has synchronised with read_back_lm's stream: the accepted pose and the report
  void lm_result(double q[4], double t[3], ilsm_reg_report* report) const {
    const double* x = reinterpret_cast<const double*>(pinned.p);
    for (int i = 0; i < 4; ++i) q[i] = x[i];
    for (int i = 0; i < 3; ++i) t[i] = x[4 + i];
    if (report) memcpy(report, pinned.p + offsetof(LmState, report), sizeof(*report));
  }
  // the whole LM tail of a host-pointer entry point: read back, synchronise, then the pose and the report (`passes`:
  // the outer passes that ran)
  int lm_finish(double q[4], double t[3], ilsm_reg_report* report, int passes) {
    int rc = read_back_lm(stream);
    if (rc) return rc;
    ILSM_CUDA(cudaStreamSynchronize(stream));
    lm_result(q, t, report);
    if (report) report->passes = passes;
    return ILSM_OK;
  }
  bool async_build = false;  // ilsm_set_async: host-pointer map builds return without synchronising
  int seed_pose(const PoseSrc& src);  // src's pose -> lm.p->xq, xt, one 1-warp launch
  int associate_dev(Map* mc, Map* ms, const float* d_corner, int nc, const float* d_surf, int ns, int stride_bytes,
                    const ilsm_reg_opts& o, bool want_knn, const PoseSrc* src = nullptr);
  int solve_launch(int max_iter, double huber_a, int pass, const PoseDst* dst = nullptr);  // the whole LM solve, one cluster launch
  int odom_associate_dev(Map* mc, Map* ms, const float* d_sharp, int nsh, const float* d_flat, int nfl, int stride_bytes);
  int odometry_dev(Map* mc, Map* ms, const float* d_sharp, int nsh, const float* d_flat, int nfl, int stride_bytes,
                   const ilsm_reg_opts& o);
  // front end (frontend.cu)
  int project_dev(const float* d_cloud, int n, int stride_bytes, unsigned char* d_range, unsigned char* d_inten,
                  float* d_track);
  int features_dev(const float* d_in, int n, int stride_bytes, float min_range);
  int features_launch(const float* d_in, int n, int stride_bytes, float min_range, int ring_cap);  // the 10 plain launches
  GraphExec fe_graph_exec;  // the captured front-end chain and the parameter hash it was captured for
  unsigned long long fe_graph_key = 0;
  bool fe_graphs_ok = true;  // false after a failed capture: plain launches from then on
  int pc2_unpack_dev(const unsigned char* d_data, int n, const ilsm_pc2_layout& l, float4* d_out);
  int pc2_pack_dev(const float4* d_in, int n, const ilsm_pc2_layout& l, unsigned char* d_out);
  // VoxelGrid of 1 or 2 clouds on stream s; d_err: the error word the kernels OR their flags into (nullptr: the front
  // end's)
  struct VgCloud {
    const float* in;
    int n;
    float leaf;
    float4* out;
    int* n_out;  // device slot of the voxel count
  };
  int voxelgrid(const VgCloud* clouds, int count, int stride_bytes, int ioff, cudaStream_t s, int* d_err = nullptr);
  int voxelgrid_large_dev(const float* d_in, int n, int stride_bytes, int ioff, float leaf, float4* d_out, int* d_n_out,
                          cudaStream_t s, int* d_err);
  int gather_dev(const float4* d_cloud, const int* d_idx, const int* d_counts, int slot, int max_n, float4* d_out);
  int register_dev(Map* mc, Map* ms, const float* d_corner, int nc, const float* d_surf, int ns, int stride_bytes,
                   const ilsm_reg_opts& o, const PoseSrc* src = nullptr, const PoseDst* dst = nullptr);
};

// The way into a context: holds its mutex and makes its device current.  `rc` is ILSM_OK, or the cudaSetDevice error
// through fail_cuda.  ILSM_ENTER(c) is the form for a function that returns that error at once.
struct CtxGuard {
  std::lock_guard<std::mutex> lk;
  int rc;
  explicit CtxGuard(Ctx& c) : lk(c.mu) {
    const cudaError_t e = cudaSetDevice(c.device);
    rc = e == cudaSuccess ? ILSM_OK : fail_cuda(e, "cudaSetDevice");
  }
};
#define ILSM_ENTER(c)               \
  ::ilsm::CtxGuard ilsm_guard__(c); \
  if (ilsm_guard__.rc) return ilsm_guard__.rc

// ScanContext keyframe database (one shard when the database is split across ranks).
struct ScQuery;
struct ScDb {
  Ctx* ctx = nullptr;
  int count = 0;
  DevBuf<float> db;        // [count][20][60] float32
  DevBuf<int> bins;        // makeScancontext scratch
  DevBuf<ScQuery> query;
  DevBuf<double> out_dist;
  DevBuf<int> out_id, out_shift;
  DevBuf<u64> part_d;      // per-block top-k lists of the scoring kernel
  DevBuf<int> part_id, part_sh;
  DevBuf<float> stage;     // staged caller descriptors / points
  DevBuf<float> ringkey;   // [count][20] float ring keys (polarcontext_invkeys_mat_, Scancontext.cpp:243,249)
  DevBuf<u64> rk_part;     // ring-key candidate selection: per-block lists + the selected list
  DevBuf<unsigned char> cand_out;  // candidate query outputs (ids | key d2 | distances | shifts)
  // sharded queries (ilsm_sc_init_nccl): per-rank packed top-k records, the all-gathered buffer, the merged result
  void* nccl_comm = nullptr;
  bool nccl_owned = false;
  int nccl_ranks = 1, nccl_rank = 0;
  DevBuf<unsigned char> pk_local, pk_all, pk_out;
  DevBuf<float> qbatch;
  int append_dev(const float* desc, int n_add, bool from_host);
  int query_batch_dev(const float* d_qdesc, int B, int n_search, int id_offset, int k, unsigned char* d_packed);
  // tensor-core prefilter + exact rescoring (scancontext_tc.cu); shards smaller than tc_min keep the plain exact scan
  int tc_min = 4096;
  DevBuf<unsigned char> pf_query;   // PfQuery records of the batch in flight
  DevBuf<float> pf_dist, pf_thr;    // approximate distances [8][n], thresholds [8]
  DevBuf<u64> pf_part, pf_list;     // selection scratch, rescoring lists [8][n]
  DevBuf<int> pf_list_n;
  int query_batch_tc_dev(const float* d_qdesc, int B, int n_search, int id_offset, int k, unsigned char* d_packed, unsigned char* d_shift_dbg);
  int candidates_dev(const float* d_qdesc, int n_search, int num_cand, int* d_id, float* d_key_d2, double* d_dist, int* d_shift);
  int make_dev(const float* d_pts, int n, int stride_bytes, float* d_desc);
  int query_dev(const float* d_qdesc, int n_search, int id_offset, int k, double* d_dist, int* d_id, int* d_shift);
  // the entries a query scans: the first n_search, every entry when n_search < 0
  int searched(int n_search) const { return n_search < 0 ? count : n_search; }
  ScDb();  // both in scancontext.cu, where ScQuery is complete
  ~ScDb();
};

}  // namespace ilsm

// the opaque handles of include/ilsm.h
struct ilsm_ctx {
  ilsm::Ctx c;
};
struct ilsm_map {
  ilsm::Map m;
};
struct ilsm_sc {
  ilsm::ScDb d;
};
