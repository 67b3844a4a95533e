// pipeline.cu -- the full per-frame loop of the reference's three LOAM nodes chained on one GPU (BASELINE config 2):
//   scanRegistration  laserCloudHandler          scanRegistration.cpp:189-669   -> Ctx::features_dev
//   laserOdometry     main loop                  laserOdometry.cpp:256-845      -> Ctx::odometry_dev + pose composition
//   laserMapping      process()                  laserMapping.cpp:233-1166      -> cubemap_frame_enqueue / _collect
// The topics between the nodes (/laser_cloud_sharp, /laser_cloud_less_sharp, /laser_cloud_flat, /laser_cloud_less_flat,
// /laser_cloud_corner_last, /laser_cloud_surf_last, /laser_odom_to_init) become device buffers: the organised frame is
// the only upload, the two poses and a few counters the only downloads.  Host synchronisation points per frame: the
// feature counts (sizes of the next launches), the odometry pose (the host owns q_w_curr / t_w_curr and the cube
// window indices, as the reference nodes do) and the mapped pose.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <deque>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "ilsm_cubemap.hpp"
#include "ilsm_keyframe.hpp"
#include "ilsm_stage.hpp"

struct ilsm_mapopt;
int check_loop_opts(const ilsm_loop_opts& o);  // loop.cu

namespace ilsm {

int mapopt_frame_core(ilsm_mapopt* mo, const float* frame_xyz, int n, int stride_bytes, const float* plane_xyz, int n_plane,
                      int plane_stride_bytes, bool from_host, const double q_wodom[4], const double t_wodom[3], double q_w[4],
                      double t_w[3], const ilsm_ground_opts* gopts, ilsm_mapopt_stats* stats);  // mapopt.cu

// voxel edge of the "last frame" search structures: the odometry gate is 5 m (DISTANCE_SQ_THRESHOLD 25,
// laserOdometry.cpp:31), the clouds are sparse (a few thousand points)
constexpr float kOdomCell = 1.0f;
// points of one OS0-64 frame (64 x 1024): the size the loop-closure buffers are reserved at
constexpr int kFramePoints = 65536;

// The host phase clocks.  The first eight are those of ilsm_slam_host_phases, in the order include/ilsm.h documents;
// the rest are the stage threads' detail that ILSM_STAGE_TRACE prints.
enum Phase {
  kFeLaunch, kWaitMapping, kWaitFrontEnd, kOdomLaunch, kWaitOdom, kMapping, kMapLaunch, kMapWait,
  kMapTailWait, kFeStageLaunch, kFeStageWait, kFeStageGather, kNumPhases
};

static int fail_text(int code, const char* text) { return fail(code, "%s", text); }

// A sub-handle created through the C ABI and released through its destroy function.
template <typename T>
using Owner = std::unique_ptr<T, void (*)(T*)>;

// Runs `create`, a C entry point that returns a new T through its last argument, and hands the result to `o`.
template <typename T, typename... P, typename... A>
static int create_into(Owner<T>& o, int (*create)(P...), A... args) {
  T* p = nullptr;
  const int rc = create(args..., &p);
  o.reset(p);
  return rc;
}

// Members are declared in dependency order, so that the destructor releases them in the right one: each context before
// the handles that live on it, and the stage threads last, so that they are joined first.
struct SlamH {
  Ctx* ctx = nullptr;  // the caller's
  // asynchronous mapping (ilsm_slam_create_async, ilsm_slam_create_staged): the cube map lives on a second, owned context;
  // the mapping of frame k runs there while the front end and the odometry of frame k + 1 run on other contexts
  Owner<ilsm_ctx> ctx2{nullptr, ilsm_destroy};
  bool async = false;
  // staged mode (ilsm_slam_create_staged): the three nodes as three stages, each with its own context (streams, scratch)
  // and host thread like the reference's three processes -- scanRegistration on ctx0 + `frontend`, laserOdometry on the
  // caller's context and thread, laserMapping on ctx2 + `mapping`.  Frame k's front end, frame k-1's odometry and frame
  // k-2's / k-1's mapping are in flight together.
  Owner<ilsm_ctx> ctx0{nullptr, ilsm_destroy};
  bool staged = false;
  Owner<ilsm_cubemap> cube{nullptr, ilsm_cubemap_destroy};  // mapping = laserMapping (rolling cube map)
  Owner<ilsm_mapopt> mapopt{nullptr, ilsm_mapopt_destroy};  // mapping = mapOptimization (ground map), the node spot.launch starts
  Map last_corner, last_surf;  // kdtreeCornerLast / kdtreeSurfLast (laserOdometry.cpp:807-808)
  bool inited = false;        // systemInited (laserOdometry.cpp:384)
  double para_q[4] = {0, 0, 0, 1}, para_t[3] = {0, 0, 0};  // q_last_curr / t_last_curr, kept between frames (:51-52)
  QuatH q_w_curr{0, 0, 0, 1};
  double t_w_curr[3] = {0, 0, 0};
  float min_range = 0.3f;
  long long frames = 0;
  long long pushed = 0;
  // The clouds between the nodes live in three rotating slots (frame % 3), so that the stage after the front end can
  // still read frame k while frame k + 1 or k + 2 is produced: a slot is rewritten by the front end of frame k + 3, after
  // the mapped pose of frame k has been handed out.
  struct FeSlot {
    DevBuf<float4> sharp, flat, lsharp, lflat;
    const float4* lf = nullptr;  // this frame's less-flat cloud: lflat, or the front end's own fe.lflat (synchronous loop)
    Event ev;                    // recorded once the slot is written
    // loop closure in the pipelined and staged loops: the front end's cloud, kept until the frame's mapped pose is known
    DevBuf<float4> cloud;
    int n_cloud = 0;
    Event ev_read;              // recorded after a keyframe's copy read `cloud`
    bool read_pending = false;  // the next front end into this slot waits for ev_read
  } fslot[3];
  // the two mapping stacks (VoxelGrid of the less-sharp / less-flat clouds, laserMapping.cpp:608-616), double-buffered:
  // the odometry stage's side stream writes set k & 1 for frame k under its solve while the mapping of frame k - 1 (solve
  // and deferred insertion) still reads the other one
  struct StackSet {
    DevBuf<float4> c, s;
    DevBuf<int> n;
    Event ev_ready, ev_free;  // stacks written / last reader (deferred insertion) enqueued
    bool free_recorded = false;
  } stk[2];
  // host-side phase clock (profiling aid, ilsm_slam_host_phases): seconds per phase, written by the caller's thread only
  double phase_s[kNumPhases] = {};
  // loop closure (ilsm_slam_enable_loop): an ilsm_loop on its own context (ctx3) and host thread, like the reference's
  // loopClosureThread.  Each keyframe's cloud is copied on the device into one of the buffers; a buffer is used again only
  // after the job that read it has been answered.
  struct LoopJob {
    int buf = 0, n = 0;
    long long frame = -1;
    double q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
  };
  struct LoopDone {
    ilsm_slam_loop_event ev = {};
    double seconds = 0;  // the stage's time on this keyframe
  };
  struct LoopBuf {
    DevBuf<float4> cloud;
    Event ev;  // recorded once the keyframe's cloud is copied in
  };
  struct LoopAnswer {
    ilsm_slam_loop_event ev = {};
    int rc = 0;  // a keyframe that failed: its status and error text, reported by ilsm_slam_loop_results in its turn
    std::string err;
  };
  struct LoopStage {
    Owner<ilsm_ctx> ctx3{nullptr, ilsm_destroy};
    Owner<ilsm_loop> loop{nullptr, ilsm_loop_destroy};
    ilsm_slam_loop_opts opts = {};
    std::vector<LoopBuf> bufs;  // opts.max_pending of them
    bool kf_have = false;       // (kf_q, kf_t): the mapped pose of the last keyframe
    double kf_q[4] = {0, 0, 0, 1}, kf_t[3] = {0, 0, 0};
    long long keyframes = 0;          // selected so far
    std::deque<LoopAnswer> answered;  // taken from the loop stage, not yet handed out
    double loop_s = 0;                // the loop stage's time over the answered keyframes
    Stage<LoopJob, LoopDone> looper{ilsm_last_error, fail_text};
  };
  std::unique_ptr<LoopStage> loop;
  // The mapping stage has its own host thread, like the reference's laserMapping node has its own process: its ~25
  // launches per frame (3-4 us of host time each) are issued while the caller's thread launches the next front end.
  // At most two jobs queue: the staged loop posts frame k before it collects frame k - 1, so the mapping thread goes
  // from one frame to the next without a round trip through the caller.
  struct MapJob {
    int n_lsharp = 0, n_lflat = 0;
    const float4 *d_lsharp = nullptr, *d_lflat = nullptr;  // this frame's slot
    cudaEvent_t ev_in = nullptr;                           // recorded once the slot is written
    int stack_set = 0;  // which of the two stack sets (SlamH::stk) holds this frame's down-sampled stacks
    double q_odom[4] = {0, 0, 0, 1}, t_odom[3] = {0, 0, 0};
    long long frame = -1;
  };
  struct MapResult {
    double q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
    ilsm_reg_report report = {};
    ilsm_cubemap_stats cstats = {};
    long long frame = -1;
    double phase_s[kNumPhases] = {};  // the stage's own phases, added to SlamH::phase_s when the result is taken
  };
  Stage<MapJob, MapResult> mapping{ilsm_last_error, fail_text};
  struct FeJob {
    const float* xyzi = nullptr;
    int n = 0, stride = 16, use_aloam = 1;
    long long frame = 0;
  };
  struct FeResult {
    int use_aloam = 1;
    int counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long frame = 0;
    double phase_s[kNumPhases] = {};
  };
  Stage<FeJob, FeResult> frontend{ilsm_last_error, fail_text};
};

// a stage's oldest result, with the phase times it took added to the handle's
template <typename Job, typename Result>
static int take_result(SlamH& s, Stage<Job, Result>& stage, Result& r) {
  const int rc = stage.take(r);
  for (int i = 0; i < kNumPhases; ++i) s.phase_s[i] += r.phase_s[i];
  return rc;
}

struct PhaseClock {
  double* acc;
  std::chrono::steady_clock::time_point t;
  explicit PhaseClock(double* a) : acc(a), t(std::chrono::steady_clock::now()) {}
  void lap(Phase k) {
    const auto n = std::chrono::steady_clock::now();
    acc[k] += std::chrono::duration<double>(n - t).count();
    t = n;
  }
};

// ---- the steps of one frame, shared by the synchronous, pipelined and staged loops

// scanRegistration's laserCloudHandler (scanRegistration.cpp:189-669) up to the feature counts, the sizes of the next
// launches: uploads the frame -- a sensor_msgs/PointCloud2 blob as it is when `pc2` is set, pcl::fromROSMsg's repacking
// (:235) then runs as a kernel -- runs the front end on f.stream and waits for the counts.
static int frontend_counts(Ctx& f, const float* xyzi, int n, int stride_bytes, const ilsm_pc2_layout* pc2, float min_range,
                           int cnt[8], PhaseClock& clk, Phase lap_launch, Phase lap_wait) {
  const size_t bytes = (size_t)n * stride_bytes;
  int rc;
  if ((rc = f.fe.raw.reserve((pc2 ? (size_t)n * 4 : bytes / 4) + 4))) return rc;
  if (pc2) {
    if ((rc = f.fe.pc2.reserve(bytes + 16))) return rc;
    if (bytes) ILSM_CUDA(cudaMemcpyAsync(f.fe.pc2.p, xyzi, bytes, cudaMemcpyHostToDevice, f.stream));
    if ((rc = f.pc2_unpack_dev(f.fe.pc2.p, n, *pc2, reinterpret_cast<float4*>(f.fe.raw.p)))) return rc;
    stride_bytes = 16;
  } else if (bytes) {
    ILSM_CUDA(cudaMemcpyAsync(f.fe.raw.p, xyzi, bytes, cudaMemcpyHostToDevice, f.stream));
  }
  if ((rc = f.features_dev(f.fe.raw.p, n, stride_bytes, min_range))) return rc;
  int* pin = reinterpret_cast<int*>(f.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, f.fe.counts.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, f.stream));
  clk.lap(lap_launch);
  ILSM_CUDA(cudaStreamSynchronize(f.stream));
  clk.lap(lap_wait);
  if (pin[5]) return fail(ILSM_ERR_INVALID_ARG, "slam_frame: a ring segment exceeds the supported size");
  for (int i = 0; i < 8; ++i) cnt[i] = pin[i];
  return ILSM_OK;
}

// The front end's sharp, less-sharp and flat clouds gathered into slot `o`.  Less-flat is copied there when `copy_lflat`
// (a later front end on `f` may rewrite fe.lflat before this frame's last reader has run); otherwise o.lf is fe.lflat.
// With `copy_cloud` (loop closure, under the same condition) the ring-ordered cloud is copied there too, for the keyframe
// copy that follows once the frame's mapped pose is known; it waits for that copy of the slot's previous frame.
static int frontend_gather(Ctx& f, const int cnt[8], SlamH::FeSlot& o, bool copy_lflat, bool copy_cloud) {
  const int n_sharp = cnt[1], n_lsharp = cnt[2], n_flat = cnt[3], n_lflat = cnt[4];
  int rc;
  if ((rc = o.sharp.reserve(n_sharp + 4)) || (rc = o.flat.reserve(n_flat + 4)) || (rc = o.lsharp.reserve(n_lsharp + 4)) ||
      (copy_lflat && (rc = o.lflat.reserve(n_lflat + 4))) || (copy_cloud && (rc = o.cloud.reserve((size_t)cnt[0] + 4))))
    return rc;
  o.n_cloud = cnt[0];
  if (copy_cloud) {
    if (o.read_pending) ILSM_CUDA(cudaStreamWaitEvent(f.stream, o.ev_read, 0));
    o.read_pending = false;
    if (cnt[0])
      ILSM_CUDA(cudaMemcpyAsync(o.cloud.p, f.fe.cloud.p, (size_t)cnt[0] * sizeof(float4), cudaMemcpyDeviceToDevice, f.stream));
  }
  if ((rc = f.gather_dev(f.fe.cloud.p, f.fe.sharp.p, f.fe.counts.p, 1, n_sharp, o.sharp.p)) ||
      (rc = f.gather_dev(f.fe.cloud.p, f.fe.lsharp.p, f.fe.counts.p, 2, n_lsharp, o.lsharp.p)) ||
      (rc = f.gather_dev(f.fe.cloud.p, f.fe.flat.p, f.fe.counts.p, 3, n_flat, o.flat.p)))
    return rc;
  o.lf = copy_lflat ? o.lflat.p : f.fe.lflat.p;
  if (copy_lflat && n_lflat)
    ILSM_CUDA(cudaMemcpyAsync(o.lflat.p, f.fe.lflat.p, (size_t)n_lflat * sizeof(float4), cudaMemcpyDeviceToDevice, f.stream));
  ILSM_CUDA(cudaEventRecord(o.ev, f.stream));
  return ILSM_OK;
}

static void feature_stats(ilsm_slam_stats* stats, const int cnt[8]) {
  if (stats)
    stats->n_cloud = cnt[0], stats->n_sharp = cnt[1], stats->n_less_sharp = cnt[2], stats->n_flat = cnt[3], stats->n_less_flat = cnt[4];
}

// The mapping stacks of slot `o` (VoxelGrid of the less-sharp / less-flat clouds, laserMapping.cpp:608-616) into `set`, on
// c's side stream: they depend only on the front end and run under the odometry solve.  They wait for the slot and for
// the set's last reader.  Clouds above 16384 points take the tiled multi-block VoxelGrid (no size limit below 2^24
// points, like the reference); the VoxelGrid reports into the cube map's error word.
static int stack_voxelgrid(Ctx& c, const CubeMapH& cm, const SlamH::FeSlot& o, const int cnt[8], SlamH::StackSet& set) {
  const int n_lsharp = cnt[2], n_lflat = cnt[4];
  int rc;
  if ((rc = set.c.reserve(n_lsharp + 4)) || (rc = set.s.reserve(n_lflat + 4))) return rc;
  ILSM_CUDA(cudaStreamWaitEvent(c.aux, o.ev, 0));
  if (set.free_recorded) ILSM_CUDA(cudaStreamWaitEvent(c.aux, set.ev_free, 0));  // frame - 2's insertion read this set
  ILSM_CUDA(cudaMemsetAsync(set.n.p, 0, 4 * sizeof(int), c.aux));
  const Ctx::VgCloud vc[2] = {{reinterpret_cast<const float*>(o.lsharp.p), n_lsharp, cm.line_res, set.c.p, set.n.p},
                              {reinterpret_cast<const float*>(o.lf), n_lflat, cm.plane_res, set.s.p, set.n.p + 1}};
  if ((rc = c.voxelgrid(vc, 2, 16, 3, c.aux, cm.err))) return rc;
  ILSM_CUDA(cudaEventRecord(set.ev_ready, c.aux));
  return ILSM_OK;
}

static ilsm_reg_opts odometry_opts() {  // 2 passes x max 4 iterations, Huber 0.1 (laserOdometry.cpp:417,644,705-710)
  ilsm_reg_opts o;
  ilsm_reg_opts_default(&o);
  return o;
}

// laserOdometry, first half: the solve of q/t_last_curr against the "last" trees and the read-back of its result.  The
// fork optimises only on frames flagged "skip_intensity" (use_aloam, laserOdometry.cpp:406-417), never on the first.
static int odometry_launch(SlamH& s, Ctx& c, const SlamH::FeSlot& o, const int cnt[8], bool solve) {
  if (!solve) return ILSM_OK;
  int rc;
  if ((rc = c.upload_pose(s.para_q, s.para_t, c.stream)) ||
      (rc = c.odometry_dev(&s.last_corner, &s.last_surf, reinterpret_cast<const float*>(o.sharp.p), cnt[1],
                           reinterpret_cast<const float*>(o.flat.p), cnt[3], 16, odometry_opts())) ||
      (rc = c.read_back_lm(c.stream)))
    return rc;
  return ILSM_OK;
}

// laserOdometry, second half: wait for the solve, compose the world pose (also when the solve was skipped: the stale
// q/t_last_curr is composed; the first frame only sets systemInited) and rebuild both "last" trees from this frame.
static int odometry_finish(SlamH& s, Ctx& c, const SlamH::FeSlot& o, const int cnt[8], bool solve, double q_odom[4],
                           double t_odom[3], ilsm_slam_stats* stats, PhaseClock& clk) {
  clk.lap(kOdomLaunch);
  if (solve) {
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
    c.lm_result(s.para_q, s.para_t, stats ? &stats->odometry : nullptr);
    if (stats) stats->odometry.passes = odometry_opts().outer_iterations, stats->ran_odometry = 1;
  }
  clk.lap(kWaitOdom);
  if (!s.inited) {
    s.inited = true;
  } else {  // t_w_curr = t_w_curr + q_w_curr * t_last_curr;  q_w_curr = q_w_curr * q_last_curr   (laserOdometry.cpp:716-717)
    double r[3];
    qrot_h(s.q_w_curr, s.para_t, r);
    for (int i = 0; i < 3; ++i) s.t_w_curr[i] = s.t_w_curr[i] + r[i];
    s.q_w_curr = qmul_h(s.q_w_curr, QuatH{s.para_q[0], s.para_q[1], s.para_q[2], s.para_q[3]});
  }
  q_odom[0] = s.q_w_curr.x, q_odom[1] = s.q_w_curr.y, q_odom[2] = s.q_w_curr.z, q_odom[3] = s.q_w_curr.w;
  for (int i = 0; i < 3; ++i) t_odom[i] = s.t_w_curr[i];
  // laserCloudCornerLast = cornerPointsLessSharp, laserCloudSurfLast = surfPointsLessFlat; rebuild both trees (:793-808)
  return build_pair_dev(&s.last_corner, reinterpret_cast<const float*>(o.lsharp.p), cnt[2], &s.last_surf,
                        reinterpret_cast<const float*>(o.lf), cnt[4], 16, kOdomCell);
}

// laserMapping's process() for one frame up to its deferred insertion, on the stacks the odometry stage wrote into
// `set`.  The map reads them only in the launches enqueued here; afterwards it is back on its own stacks, which
// ilsm_cubemap_frame and ilsm_cubemap_insert_world on it stage into.
static int mapping_enqueue(CubeMapH& cm, const SlamH::StackSet& set, const float4* lsharp, int n_lsharp, const float4* lflat,
                           int n_lflat, const double q_odom[4], const double t_odom[3]) {
  ilsm_reg_opts mo;
  ilsm_reg_opts_default(&mo);
  cm.ext_c = set.c.p, cm.ext_s = set.s.p, cm.ext_n = set.n.p;
  const int rc = cubemap_frame_enqueue(cm, reinterpret_cast<const float*>(lsharp), n_lsharp, reinterpret_cast<const float*>(lflat),
                                       n_lflat, 16, q_odom, t_odom, mo, true, true, set.ev_ready);
  cm.ext_c = cm.ext_s = nullptr, cm.ext_n = nullptr;
  return rc;
}

// one process() iteration of the mapping stage: enqueue + collect on the second context
static int mapping_job(SlamH& s, const SlamH::MapJob& j, SlamH::MapResult& r) {
  Ctx& c2 = s.ctx2->c;
  std::lock_guard<std::mutex> lk(c2.mu);
  r.frame = j.frame;
  cudaError_t e = cudaStreamWaitEvent(c2.stream, j.ev_in, 0);
  if (e != cudaSuccess) return fail_cuda(e, "cudaStreamWaitEvent(mapping stage)");
  PhaseClock clk(r.phase_s);
  CubeMapH& cm = s.cube->m;
  SlamH::StackSet& set = s.stk[j.stack_set];
  int rc;
  if ((rc = cm.wait_tail())) return rc;
  clk.lap(kMapTailWait);
  if ((rc = mapping_enqueue(cm, set, j.d_lsharp, j.n_lsharp, j.d_lflat, j.n_lflat, j.q_odom, j.t_odom))) return rc;
  e = cudaEventRecord(set.ev_free, c2.aux);  // the deferred insertion (side stream) is the set's last reader
  set.free_recorded = true;
  if (e != cudaSuccess) return fail_cuda(e, "cudaEventRecord(stack set)");
  clk.lap(kMapLaunch);
  if ((rc = cubemap_frame_collect(cm, r.q, r.t, &r.report, &r.cstats))) return rc;
  clk.lap(kMapWait);
  return ILSM_OK;
}

// hand frame `frame`, written into slot `o` and stack set frame & 1, to the mapping stage
static void post_mapping_job(SlamH& s, const SlamH::FeSlot& o, const int cnt[8], long long frame, const double q_odom[4],
                             const double t_odom[3]) {
  SlamH::MapJob j;
  j.n_lsharp = cnt[2], j.n_lflat = cnt[4], j.frame = frame;
  j.d_lsharp = o.lsharp.p, j.d_lflat = o.lf, j.ev_in = o.ev, j.stack_set = (int)(frame & 1);
  for (int i = 0; i < 4; ++i) j.q_odom[i] = q_odom[i];
  for (int i = 0; i < 3; ++i) j.t_odom[i] = t_odom[i];
  s.mapping.post(j);
}

// ---- loop closure: the keyframe rule on every mapped pose handed out, the keyframe's cloud to the loop stage

// The loop stage's answer to its oldest keyframe, queued for ilsm_slam_loop_results.  A failed keyframe is queued too, with
// its error: it is reported there, in keyframe order, and never by a frame call.
static void take_loop_result(SlamH::LoopStage& L) {
  SlamH::LoopDone d;
  SlamH::LoopAnswer a;
  if ((a.rc = L.looper.take(d))) a.err = ilsm_last_error();
  a.ev = d.ev;
  L.loop_s += d.seconds;
  L.answered.push_back(std::move(a));
}

// hand keyframe `frame` to the loop stage (loop_offer)
static int loop_post(Ctx& c, SlamH::LoopStage& L, long long frame, SlamH::FeSlot* o, const float4* cloud, int n, const double q[4],
                     const double t[3]) {
  const int max_pending = (int)L.bufs.size();
  // every buffer in flight: wait for the oldest answer, which frees the buffer this keyframe takes
  if (L.looper.in_flight() >= max_pending) take_loop_result(L);
  int rc;
  SlamH::LoopJob j;
  j.buf = (int)(L.keyframes % max_pending), j.n = n, j.frame = frame;
  for (int i = 0; i < 4; ++i) j.q[i] = q[i];
  for (int i = 0; i < 3; ++i) j.t[i] = t[i];
  SlamH::LoopBuf& b = L.bufs[j.buf];
  if ((rc = b.cloud.reserve((size_t)n + 4))) return rc;
  if (o) ILSM_CUDA(cudaStreamWaitEvent(c.stream, o->ev, 0));
  if (n) ILSM_CUDA(cudaMemcpyAsync(b.cloud.p, cloud, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, c.stream));
  if (o) {
    ILSM_CUDA(cudaEventRecord(o->ev_read, c.stream));
    o->read_pending = true;
  }
  ILSM_CUDA(cudaEventRecord(b.ev, c.stream));
  L.looper.post(j);
  L.keyframes++;
  return ILSM_OK;
}

// Frame `frame`'s mapped pose is being handed out: when it is a keyframe, copy its cloud (n points of 16 bytes at `cloud`,
// on c's stream: the front end's own buffer in the synchronous loop, slot `o` otherwise) into a free loop buffer and post
// it to the loop stage.  The copy is ordered after the slot's event, and the next front end into the slot after the copy.
// Nothing here fails the frame call: the frame's odometry and mapping have already advanced the handle.  A keyframe that
// cannot be handed over is queued as a failed answer behind every keyframe before it.
static void loop_offer(SlamH& s, long long frame, SlamH::FeSlot* o, const float4* cloud, int n, const double q[4], const double t[3]) {
  if (!s.loop) return;
  SlamH::LoopStage& L = *s.loop;
  if (L.kf_have && !keyframe_due(L.kf_q, L.kf_t, q, t, L.opts.keyframe_dist, L.opts.keyframe_angle_rad)) return;
  L.kf_have = true;
  for (int i = 0; i < 4; ++i) L.kf_q[i] = q[i];
  for (int i = 0; i < 3; ++i) L.kf_t[i] = t[i];
  SlamH::LoopAnswer a;
  if (!(a.rc = loop_post(*s.ctx, L, frame, o, cloud, n, q, t))) return;
  a.err = ilsm_last_error();
  a.ev.frame = frame;
  for (int i = 0; i < 4; ++i) a.ev.q_xyzw[i] = q[i];
  for (int i = 0; i < 3; ++i) a.ev.t[i] = t[i];
  while (L.looper.in_flight() > 0) take_loop_result(L);
  L.answered.push_back(std::move(a));
}

// one keyframe on the loop stage: ilsm_loop_add_keyframe_dev on ctx3, after the copy into its buffer
static int loop_job(SlamH::LoopStage& L, const SlamH::LoopJob& j, SlamH::LoopDone& r) {
  const auto t0 = std::chrono::steady_clock::now();
  r.ev.frame = j.frame;
  for (int i = 0; i < 4; ++i) r.ev.q_xyzw[i] = j.q[i];
  for (int i = 0; i < 3; ++i) r.ev.t[i] = j.t[i];
  const SlamH::LoopBuf& b = L.bufs[j.buf];
  {
    Ctx& l = L.ctx3->c;
    std::lock_guard<std::mutex> lk(l.mu);
    const cudaError_t e = cudaStreamWaitEvent(l.stream, b.ev, 0);
    if (e != cudaSuccess) return fail_cuda(e, "cudaStreamWaitEvent(loop stage)");
  }
  const int rc = ilsm_loop_add_keyframe_dev(L.loop.get(), reinterpret_cast<const float*>(b.cloud.p), j.n, 16, j.q, j.t, &r.ev.result);
  r.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

// wait for the mapping stage's answer to its oldest job and hand it out
static int take_mapping_result(SlamH& s, double q_map[4], double t_map[3], ilsm_slam_stats* stats, int* frame = nullptr) {
  SlamH::MapResult r;
  int rc = take_result(s, s.mapping, r);
  if (rc) return rc;
  if (frame) *frame = (int)r.frame;
  for (int i = 0; i < 4; ++i) q_map[i] = r.q[i];
  for (int i = 0; i < 3; ++i) t_map[i] = r.t[i];
  if (stats) stats->mapping = r.report, stats->cubemap = r.cstats;
  SlamH::FeSlot& o = s.fslot[r.frame % 3];
  loop_offer(s, r.frame, &o, o.cloud.p, o.n_cloud, r.q, r.t);
  return ILSM_OK;
}

// ---- staged mode: scanRegistration as its own stage, on ctx0
static int frontend_job(SlamH& s, const SlamH::FeJob& j, SlamH::FeResult& r) {
  Ctx& f = s.ctx0->c;
  std::lock_guard<std::mutex> lk(f.mu);
  r.frame = j.frame, r.use_aloam = j.use_aloam;
  PhaseClock clk(r.phase_s);
  int rc;
  if ((rc = frontend_counts(f, j.xyzi, j.n, j.stride, nullptr, s.min_range, r.counts, clk, kFeStageLaunch, kFeStageWait)) ||
      (rc = frontend_gather(f, r.counts, s.fslot[j.frame % 3], true, s.loop != nullptr)))
    return rc;
  clk.lap(kFeStageGather);
  return ILSM_OK;
}

}  // namespace ilsm

using namespace ilsm;

struct ilsm_slam {
  SlamH s;
};

// the mapping stage on its own context and host thread (pipelined and staged handles)
static int slam_create_mapping_stage(SlamH& s, float line_res, float plane_res, int cube_capacity) {
  int rc;
  if ((rc = create_into(s.ctx2, ilsm_create, s.ctx->device)) ||
      (rc = create_into(s.cube, ilsm_cubemap_create, s.ctx2.get(), line_res, plane_res, cube_capacity)))
    return rc;
  s.mapping.start([&s] { cudaSetDevice(s.ctx2->c.device); },
                  [&s](const SlamH::MapJob& j, SlamH::MapResult& r) { return mapping_job(s, j, r); });
  return ILSM_OK;
}

// The one creation path of the four ilsm_slam_create* entry points: the parts every handle has, then `mode(s)`, the
// mode's own.  The handle is held here until it is complete, so that it releases itself on any failure.
template <typename Mode>
static int slam_create(ilsm_ctx* ctx, float min_range, ilsm_slam** out, Mode mode) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "slam_create: null argument");
  std::unique_ptr<ilsm_slam> h(new (std::nothrow) ilsm_slam());
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  SlamH& s = h->s;
  s.ctx = &ctx->c;
  s.min_range = min_range > 0.f ? min_range : 0.3f;
  int rc;
  {
    CtxGuard g(ctx->c);
    if ((rc = g.rc) || (rc = s.last_corner.init(&ctx->c)) || (rc = s.last_surf.init(&ctx->c)) ||
        (rc = s.last_corner.reserve_points(16384)) || (rc = s.last_surf.reserve_points(65536)))
      return rc;
    // the slots and stack sets at typical 16-ring sizes up front: a growing buffer costs a device-wide synchronisation
    for (SlamH::FeSlot& o : s.fslot)
      if ((rc = o.ev.create()) || (rc = o.ev_read.create()) || (rc = o.sharp.reserve(1024)) || (rc = o.flat.reserve(4096)) ||
          (rc = o.lsharp.reserve(8192)) || (rc = o.lflat.reserve(32768)))
        return rc;
    for (SlamH::StackSet& set : s.stk)
      if ((rc = set.ev_ready.create()) || (rc = set.ev_free.create()) || (rc = set.c.reserve(8192)) || (rc = set.s.reserve(32768)) ||
          (rc = set.n.reserve(4)))
        return rc;
  }
  if ((rc = mode(s))) return rc;  // after the guard: the mode's creates, and a failed handle's release, take the lock
  *out = h.release();
  return ILSM_OK;
}

extern "C" {

ILSM_API int ilsm_slam_create(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                              ilsm_slam** out) {
  return slam_create(ctx, min_range, out, [&](SlamH& s) {
    return create_into(s.cube, ilsm_cubemap_create, ctx, line_res, plane_res, cube_capacity);
  });
}

ILSM_API int ilsm_slam_create_mapopt(ilsm_ctx* ctx, float voxel_leaf, float downsample_size, float min_range, ilsm_slam** out) {
  return slam_create(ctx, min_range, out, [&](SlamH& s) {
    return create_into(s.mapopt, ilsm_mapopt_create, ctx, voxel_leaf, downsample_size);
  });
}

ILSM_API int ilsm_slam_create_async(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                    ilsm_slam** out) {
  return slam_create(ctx, min_range, out, [&](SlamH& s) {
    s.async = true;
    return slam_create_mapping_stage(s, line_res, plane_res, cube_capacity);
  });
}

ILSM_API int ilsm_slam_create_staged(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                     ilsm_slam** out) {
  return slam_create(ctx, min_range, out, [&](SlamH& s) -> int {
    s.staged = true;
    s.last_corner.in_line = s.last_surf.in_line = true;  // nothing follows the tree builds on this stage's stream
    int rc;
    if ((rc = create_into(s.ctx0, ilsm_create, ctx->c.device)) || (rc = slam_create_mapping_stage(s, line_res, plane_res, cube_capacity)))
      return rc;
    s.frontend.start([&s] { cudaSetDevice(s.ctx0->c.device); },
                     [&s](const SlamH::FeJob& j, SlamH::FeResult& r) { return frontend_job(s, j, r); });
    return ILSM_OK;
  });
}

// Drains the stages in order, each before anything it reads goes away; then the handle releases what it owns.
ILSM_API void ilsm_slam_destroy(ilsm_slam* slam) {
  if (!slam) return;
  SlamH& s = slam->s;
  s.frontend.stop();
  const double us = 1e6 / (s.frames ? s.frames : 1);  // per frame
  if (getenv("ILSM_STAGE_TRACE"))
    fprintf(stderr, "[ilsm stage trace] frames %lld  mapping: tail-wait %.1f us  enqueue %.1f us  collect %.1f us   front end: launches %.1f us  "
                    "wait %.1f us  gathers %.1f us per frame\n", s.frames,
            us * s.phase_s[kMapTailWait], us * s.phase_s[kMapLaunch], us * s.phase_s[kMapWait], us * s.phase_s[kFeStageLaunch],
            us * s.phase_s[kFeStageWait], us * s.phase_s[kFeStageGather]);
  if (s.ctx0) {
    CtxGuard g(s.ctx0->c);
    cudaStreamSynchronize(s.ctx0->c.stream);
  }
  s.mapping.stop();
  if (s.ctx2) {  // let the mapping stage drain before anything it reads goes away
    CtxGuard g(s.ctx2->c);
    cudaStreamSynchronize(s.ctx2->c.stream);
    cudaStreamSynchronize(s.ctx2->c.aux);
  }
  if (s.loop) {
    SlamH::LoopStage& L = *s.loop;
    if (getenv("ILSM_STAGE_TRACE")) {
      const long long taken = L.keyframes - L.looper.in_flight();  // the answers the caller collected, with their stage times
      fprintf(stderr, "[ilsm stage trace] loop: keyframes %lld  collected %lld  stage %.1f us per collected keyframe\n", L.keyframes,
              taken, 1e6 * L.loop_s / (taken ? taken : 1));
    }
    L.looper.stop();  // every posted keyframe is answered; the loop handle's destroy synchronises its stream
  }
  {
    CtxGuard g(*s.ctx);
    cudaStreamSynchronize(s.ctx->stream);
  }
  delete slam;  // outside the context's lock (ilsm_mapopt_destroy takes it), with the handle's device current
}

ILSM_API void ilsm_slam_loop_opts_default(ilsm_slam_loop_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->keyframe_dist = 1.0;
  o->keyframe_angle_rad = 0.2;
  o->max_pending = 8;
  ilsm_loop_opts_default(&o->loop);
}

ILSM_API int ilsm_slam_enable_loop(ilsm_slam* slam, const ilsm_slam_loop_opts* opts) {
  if (!slam) return fail(ILSM_ERR_INVALID_ARG, "slam_enable_loop: null handle");
  ilsm_slam_loop_opts o;
  if (opts)
    o = *opts;
  else
    ilsm_slam_loop_opts_default(&o);
  if (!(o.keyframe_dist >= 0.0) || !(o.keyframe_angle_rad >= 0.0) || !isfinite(o.keyframe_dist) || !isfinite(o.keyframe_angle_rad))
    return fail(ILSM_ERR_INVALID_ARG, "slam_enable_loop: keyframe_dist and keyframe_angle_rad must be finite and >= 0");
  if (o.max_pending < 1) return fail(ILSM_ERR_INVALID_ARG, "slam_enable_loop: max_pending must be >= 1");
  int rc = check_loop_opts(o.loop);
  if (rc) return rc;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return fail(ILSM_ERR_NO_DEVICE, "slam_enable_loop: no CUDA device available (libilsm_cuda has no CPU fallback)");
  }
  SlamH& s = slam->s;
  if (s.loop) return fail(ILSM_ERR_STATE, "slam_enable_loop: loop closure is already on");
  if (s.frames > 0 || s.pushed > 0) return fail(ILSM_ERR_STATE, "slam_enable_loop: call it before the first frame");
  // built complete before it is installed: on a failure it releases itself and the handle stays as it was
  std::unique_ptr<SlamH::LoopStage> L(new (std::nothrow) SlamH::LoopStage());
  if (!L) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  L->opts = o;
  if ((rc = create_into(L->ctx3, ilsm_create, s.ctx->device)) || (rc = create_into(L->loop, ilsm_loop_create, L->ctx3.get(), &o.loop)))
    return rc;
  {
    CtxGuard g(*s.ctx);
    if ((rc = g.rc)) return rc;
    try {
      L->bufs.resize(o.max_pending);
    } catch (const std::bad_alloc&) {
      return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
    // the frame's size up front: a growing buffer costs a device-wide synchronisation (slam_create)
    for (SlamH::LoopBuf& b : L->bufs)
      if ((rc = b.ev.create()) || (rc = b.cloud.reserve(kFramePoints + 4))) return rc;
    for (SlamH::FeSlot& sl : s.fslot)
      if (s.ctx2 && (rc = sl.cloud.reserve(kFramePoints + 4))) return rc;
  }
  L->looper.start([lp = L.get()] { cudaSetDevice(lp->ctx3->c.device); },
                  [lp = L.get()](const SlamH::LoopJob& j, SlamH::LoopDone& r) { return loop_job(*lp, j, r); });
  s.loop = std::move(L);
  return ILSM_OK;
}

ILSM_API int ilsm_slam_loop_results(ilsm_slam* slam, int wait, ilsm_slam_loop_event* out, int capacity, int* n_out) {
  if (!slam || !n_out || (capacity > 0 && !out)) return fail(ILSM_ERR_INVALID_ARG, "slam_loop_results: null argument");
  if (capacity < 0) return fail(ILSM_ERR_INVALID_ARG, "slam_loop_results: capacity < 0");
  *n_out = 0;
  if (!slam->s.loop) return fail(ILSM_ERR_STATE, "slam_loop_results: loop closure is not on (ilsm_slam_enable_loop)");
  SlamH::LoopStage& L = *slam->s.loop;
  // no context lock: the queue and the stage's in-flight count belong to the thread that hands in the frames, and a drain
  // must not hold up other users of the caller's context
  while (L.looper.in_flight() > 0 && (wait || L.looper.ready())) take_loop_result(L);
  int k = 0;
  for (; k < capacity && !L.answered.empty() && !L.answered.front().rc; ++k) {
    out[k] = L.answered.front().ev;
    L.answered.pop_front();
  }
  *n_out = k;
  if (k == 0 && capacity > 0 && !L.answered.empty()) {  // a failed keyframe is next in order: report it
    const SlamH::LoopAnswer a = std::move(L.answered.front());
    L.answered.pop_front();
    return fail(a.rc, "slam_loop_results: keyframe of frame %lld: %s", (long long)a.ev.frame, a.err.c_str());
  }
  return ILSM_OK;
}

ILSM_API ilsm_cubemap* ilsm_slam_cubemap(ilsm_slam* slam) { return slam ? slam->s.cube.get() : nullptr; }
ILSM_API ilsm_mapopt* ilsm_slam_mapopt(ilsm_slam* slam) { return slam ? slam->s.mapopt.get() : nullptr; }

}  // extern "C"
namespace ilsm {
int check_pc2_layout(const ilsm_pc2_layout* l);  // api.cu
}
// pc2 != nullptr: `xyzi` is a sensor_msgs/PointCloud2 data blob, unpacked on the device into packed points
static int slam_frame_impl(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, const ilsm_pc2_layout* pc2, int use_aloam,
                           double q_odom[4], double t_odom[3], double q_map[4], double t_map[3], ilsm_slam_stats* stats,
                           int* have_prev = nullptr);
extern "C" {

ILSM_API int ilsm_slam_frame(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam, double q_odom[4],
                             double t_odom[3], double q_map[4], double t_map[3], ilsm_slam_stats* stats) {
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "slam_frame: bad n/stride");
  return slam_frame_impl(slam, xyzi, n, stride_bytes, nullptr, use_aloam, q_odom, t_odom, q_map, t_map, stats);
}

ILSM_API int ilsm_slam_frame_pc2(ilsm_slam* slam, const uint8_t* data, int n_points, const ilsm_pc2_layout* layout, int use_aloam,
                                 double q_odom[4], double t_odom[3], double q_map[4], double t_map[3], ilsm_slam_stats* stats) {
  if (n_points < 0) return fail(ILSM_ERR_INVALID_ARG, "slam_frame_pc2: bad n_points");
  int rc = check_pc2_layout(layout);
  if (rc) return rc;
  return slam_frame_impl(slam, reinterpret_cast<const float*>(data), n_points, layout->point_step, layout, use_aloam, q_odom, t_odom,
                         q_map, t_map, stats);
}

ILSM_API int ilsm_slam_frame_async(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam, double q_odom[4],
                                   double t_odom[3], double q_map_prev[4], double t_map_prev[3], int* have_prev,
                                   ilsm_slam_stats* stats) {
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "slam_frame_async: bad n/stride");
  if (!have_prev) return fail(ILSM_ERR_INVALID_ARG, "slam_frame_async: null have_prev");
  return slam_frame_impl(slam, xyzi, n, stride_bytes, nullptr, use_aloam, q_odom, t_odom, q_map_prev, t_map_prev, stats, have_prev);
}

ILSM_API int ilsm_slam_flush(ilsm_slam* slam, double q_map[4], double t_map[3], int* have, ilsm_slam_stats* stats) {
  if (!slam || !q_map || !t_map || !have) return fail(ILSM_ERR_INVALID_ARG, "slam_flush: null argument");
  SlamH& s = slam->s;
  *have = 0;
  if (s.staged) return fail(ILSM_ERR_STATE, "slam_flush: staged handles drain with ilsm_slam_frame_staged(n = -1)");
  if (!s.async || s.mapping.in_flight() == 0) return ILSM_OK;
  std::lock_guard<std::mutex> lk(s.ctx->mu);
  int rc = take_mapping_result(s, q_map, t_map, stats);
  if (rc) return rc;
  *have = 1;
  return ILSM_OK;
}

}  // extern "C"

static int slam_frame_impl(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, const ilsm_pc2_layout* pc2, int use_aloam,
                           double q_odom[4], double t_odom[3], double q_map[4], double t_map[3], ilsm_slam_stats* stats,
                           int* have_prev) {
  if (!slam || (n > 0 && !xyzi) || !q_odom || !t_odom || !q_map || !t_map)
    return fail(ILSM_ERR_INVALID_ARG, "slam_frame: null argument");
  SlamH& s = slam->s;
  if (s.staged) return fail(ILSM_ERR_STATE, "slam_frame: ilsm_slam_create_staged handles take ilsm_slam_frame_staged");
  if (s.async != (have_prev != nullptr))
    return fail(ILSM_ERR_STATE, "slam_frame: ilsm_slam_create_async handles take ilsm_slam_frame_async (and only those)");
  if (have_prev) *have_prev = 0;
  Ctx& c = *s.ctx;
  ILSM_ENTER(c);
  if (stats) memset(stats, 0, sizeof(*stats));
  int rc;
  PhaseClock clk(s.phase_s);
  // ---- scanRegistration: the frame is the only upload
  // the previous frame's tree builds (on the maps' own streams, overlapping its mapping step) read its clouds: order this
  // frame's front end after them
  if ((rc = s.last_corner.wait_ready(c.stream)) || (rc = s.last_surf.wait_ready(c.stream))) return rc;
  int cnt[8];
  if ((rc = frontend_counts(c, xyzi, n, stride_bytes, pc2, s.min_range, cnt, clk, kFeLaunch, kWaitFrontEnd))) return rc;
  if (s.async && s.mapping.in_flight() > 0) {
    // the previous frame's mapped pose: the mapping stage's thread has had this frame's upload and front end to finish
    if ((rc = take_mapping_result(s, q_map, t_map, stats))) return rc;
    *have_prev = 1;
  }
  clk.lap(kWaitMapping);  // (pipelined)
  feature_stats(stats, cnt);
  SlamH::FeSlot& o = s.fslot[s.frames % 3];
  SlamH::StackSet& set = s.stk[s.frames & 1];
  CubeMapH* cmp = s.cube ? &s.cube->m : nullptr;
  // With the mapping stage on its own context nothing orders the next call's front end, which rewrites fe.lflat, after
  // this frame's stack VoxelGrid: that reads a copy in the slot.
  if ((rc = frontend_gather(c, cnt, o, s.ctx2 != nullptr, s.ctx2 != nullptr && s.loop != nullptr))) return rc;
  if (cmp && (rc = stack_voxelgrid(c, *cmp, o, cnt, set))) return rc;
  // ---- laserOdometry
  // the previous frame's deferred map insertion (side stream) reads the mapped pose from the LM state the odometry is
  // about to overwrite when the map shares this context: order the main stream after it (long finished by now -- it
  // overlapped this frame's front end)
  if (cmp && cmp->ctx == &c && cmp->tail_pending) ILSM_CUDA(cudaStreamWaitEvent(c.stream, cmp->ev_tail, 0));
  const bool solve = s.inited && use_aloam;
  if ((rc = odometry_launch(s, c, o, cnt, solve)) || (rc = odometry_finish(s, c, o, cnt, solve, q_odom, t_odom, stats, clk)))
    return rc;
  // ---- mapping (mapping_skip_frame = 1: every frame is published, laserOdometry.cpp:810-833)
  if (s.async) {
    // laserMapping as its own stage (the reference runs it as its own node): hand this frame to the mapping thread and
    // return; its mapped pose is collected by the next call (or by ilsm_slam_flush)
    post_mapping_job(s, o, cnt, s.frames, q_odom, t_odom);
  } else if (cmp) {  // laserMapping: rolling cube map
    rc = mapping_enqueue(*cmp, set, o.lsharp.p, cnt[2], o.lf, cnt[4], q_odom, t_odom);
    if (!rc) rc = cubemap_frame_collect(*cmp, q_map, t_map, stats ? &stats->mapping : nullptr, stats ? &stats->cubemap : nullptr);
  } else {    // mapOptimization: ground extraction from the frame already on the device + the less-flat cloud
    ilsm_mapopt_stats ms;
    rc = mapopt_frame_core(s.mapopt.get(), c.fe.raw.p, n, pc2 ? 16 : stride_bytes, reinterpret_cast<const float*>(o.lf), cnt[4], 16,
                           false, q_odom, t_odom, q_map, t_map, nullptr, &ms);
    if (!rc && stats) {
      stats->mapping.passes = ms.ran_optimization;
      stats->mapping.pass[0] = ms.solve;
      stats->cubemap.ran_optimization = ms.ran_optimization;
      stats->cubemap.n_map_surf = ms.map_size;
      stats->cubemap.n_stack_surf = ms.n_query;
      stats->cubemap.n_valid = ms.converged;
    }
  }
  // the synchronous loops hand out this frame's mapped pose now, while the front end's cloud is still this frame's
  if (!rc && !s.async) loop_offer(s, s.frames, nullptr, c.fe.cloud.p, cnt[0], q_map, t_map);
  clk.lap(kMapping);  // synchronous: enqueue and wait; pipelined: enqueue only
  if (rc) return rc;
  s.frames++;
  return ILSM_OK;
}

// Staged mode, one call: collect the front end of the frame pushed by the previous call, push this frame to the front-end
// stage, run the odometry of the collected frame here, collect the mapping of the frame before it, post the collected
// frame to the mapping stage.  n < 0: nothing is pushed (drain).
extern "C" ILSM_API int ilsm_slam_frame_staged(ilsm_slam* slam, const float* xyzi, int n, int stride_bytes, int use_aloam,
                                               double q_odom[4], double t_odom[3], int* odom_frame, double q_map[4],
                                               double t_map[3], int* map_frame, ilsm_slam_stats* stats) {
  if (!slam || (n > 0 && !xyzi) || !q_odom || !t_odom || !q_map || !t_map || !odom_frame || !map_frame)
    return fail(ILSM_ERR_INVALID_ARG, "slam_frame_staged: null argument");
  if (n >= 0 && !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "slam_frame_staged: bad stride");
  SlamH& s = slam->s;
  if (!s.staged) return fail(ILSM_ERR_STATE, "slam_frame_staged: not an ilsm_slam_create_staged handle");
  *odom_frame = *map_frame = -1;
  Ctx& c = *s.ctx;
  ILSM_ENTER(c);
  if (stats) memset(stats, 0, sizeof(*stats));
  int rc;
  PhaseClock clk(s.phase_s);
  SlamH::FeResult fr;
  const bool have_fe = s.frontend.in_flight() > 0;
  if (have_fe && (rc = take_result(s, s.frontend, fr))) return rc;
  clk.lap(kWaitFrontEnd);
  if (n >= 0) s.frontend.post({xyzi, n, stride_bytes, use_aloam, s.pushed++});
  clk.lap(kFeLaunch);  // hand-over to the front-end stage
  if (!have_fe) {  // nothing for the odometry: first call, or the pipeline is draining
    if (s.mapping.in_flight() > 0 && (rc = take_mapping_result(s, q_map, t_map, stats, map_frame))) return rc;
    clk.lap(kWaitMapping);
    return ILSM_OK;
  }
  const int* cnt = fr.counts;
  feature_stats(stats, cnt);
  SlamH::FeSlot& o = s.fslot[fr.frame % 3];
  ILSM_CUDA(cudaStreamWaitEvent(c.stream, o.ev, 0));
  // ---- laserOdometry of frame fr.frame
  const bool solve = s.inited && fr.use_aloam;
  if ((rc = odometry_launch(s, c, o, cnt, solve))) return rc;
  // ---- the mapping stacks of frame fr.frame, enqueued after the odometry solve: the solve is the longer of the two and
  // the odometry pose is what this stage's caller waits for
  if ((rc = stack_voxelgrid(c, s.cube->m, o, cnt, s.stk[fr.frame & 1]))) return rc;
  if ((rc = odometry_finish(s, c, o, cnt, solve, q_odom, t_odom, stats, clk))) return rc;
  *odom_frame = (int)fr.frame;
  // this frame goes to the mapping stage BEFORE the previous frame's result is collected: the mapping thread moves on to
  // it the moment it has finished the previous one
  const bool collect_prev = s.mapping.in_flight() > 0;
  post_mapping_job(s, o, cnt, fr.frame, q_odom, t_odom);
  clk.lap(kMapping);  // tree builds + hand-over to the mapping stage
  if (collect_prev && (rc = take_mapping_result(s, q_map, t_map, stats, map_frame))) return rc;
  clk.lap(kWaitMapping);  // the frame before
  s.frames++;
  return ILSM_OK;
}

extern "C" ILSM_API int ilsm_slam_host_phases(ilsm_slam* slam, double out8[8]) {
  if (!slam || !out8) return fail(ILSM_ERR_INVALID_ARG, "slam_host_phases: null argument");
  for (int i = 0; i < 8; ++i) out8[i] = slam->s.phase_s[i], slam->s.phase_s[i] = 0;
  return ILSM_OK;
}
