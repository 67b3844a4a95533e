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
#include <atomic>
#include <condition_variable>
#include <deque>
#include <new>
#include <thread>

#include "ilsm_cubemap.hpp"

struct ilsm_mapopt;

namespace ilsm {

int mapopt_frame_core(ilsm_mapopt* mo, const float* frame_xyz, int n, int stride_bytes, const float* plane_xyz, int n_plane,
                      int plane_stride_bytes, bool from_host, const double q_wodom[4], const double t_wodom[3], double q_w[4],
                      double t_w[3], const ilsm_ground_opts* gopts, ilsm_mapopt_stats* stats);  // mapopt.cu

// voxel edge of the "last frame" search structures: the odometry gate is 5 m (DISTANCE_SQ_THRESHOLD 25,
// laserOdometry.cpp:31), the clouds are sparse (a few thousand points)
constexpr float kOdomCell = 1.0f;

struct SlamH {
  Ctx* ctx = nullptr;
  ilsm_cubemap* cube = nullptr;   // mapping = laserMapping (rolling cube map)
  ilsm_mapopt* mapopt = nullptr;  // mapping = mapOptimization (ground map), the node spot.launch starts
  Map last_corner, last_surf;  // kdtreeCornerLast / kdtreeSurfLast (laserOdometry.cpp:807-808)
  bool inited = false;        // systemInited (laserOdometry.cpp:384)
  double para_q[4] = {0, 0, 0, 1}, para_t[3] = {0, 0, 0};  // q_last_curr / t_last_curr, kept between frames (:51-52)
  QuatH q_w_curr{0, 0, 0, 1};
  double t_w_curr[3] = {0, 0, 0};
  float min_range = 0.3f;
  long long frames = 0;
  // The clouds between the nodes live in three rotating slots (frame % 3), so that the stage after the front end can
  // still read frame k while frame k + 1 or k + 2 is produced: a slot is rewritten by the front end of frame k + 3, after
  // the mapped pose of frame k has been handed out.
  struct FeSlot {
    DevBuf<float4> sharp, flat, lsharp, lflat;
    const float4* lf = nullptr;  // this frame's less-flat cloud: lflat, or the front end's own fe.lflat (synchronous loop)
    cudaEvent_t ev = nullptr;    // recorded once the slot is written
  } fslot[3];
  // the two mapping stacks (VoxelGrid of the less-sharp / less-flat clouds, laserMapping.cpp:608-616), double-buffered:
  // the odometry stage's side stream writes set k & 1 for frame k under its solve while the mapping of frame k - 1 (solve
  // and deferred insertion) still reads the other one
  struct StackSet {
    DevBuf<float4> c, s;
    DevBuf<int> n;
    cudaEvent_t ev_ready = nullptr, ev_free = nullptr;  // stacks written / last reader (deferred insertion) enqueued
    bool free_recorded = false;
  } stk[2];
  // asynchronous mapping (ilsm_slam_create_async, ilsm_slam_create_staged): the cube map lives on a second, owned context;
  // the mapping of frame k runs there while the front end and the odometry of frame k + 1 run on other contexts
  ilsm_ctx* ctx2 = nullptr;
  bool async = false;
  // The mapping stage has its own host thread, like the reference's laserMapping node has its own process: its ~25
  // launches per frame (3-4 us of host time each) are issued while the caller's thread launches the next front end.
  struct MapJob {
    int n_lsharp = 0, n_lflat = 0;
    const float4 *d_lsharp = nullptr, *d_lflat = nullptr;  // this frame's slot
    cudaEvent_t ev_in = nullptr;                           // recorded once the slot is written
    int stack_set = 0;  // which of the two stack sets (SlamH::stk) holds this frame's down-sampled stacks
    double q_odom[4] = {0, 0, 0, 1}, t_odom[3] = {0, 0, 0};
    long long frame = -1;
  };
  struct MapResult {
    int rc = 0;
    char err[256] = "";
    double q[4] = {0, 0, 0, 1}, t[3] = {0, 0, 0};
    ilsm_reg_report report;
    ilsm_cubemap_stats cstats;
    long long frame = -1;
  };
  // jobs and results queue up (at most two of each: the staged loop posts frame k before it collects frame k - 1, so the
  // mapping thread goes from one frame to the next without a round trip through the caller)
  std::deque<MapJob> jobs;
  std::deque<MapResult> results;
  std::thread worker;
  std::mutex wmu;
  std::condition_variable wcv;
  bool stop = false;
  int maps_in_flight = 0;
  // queue / mailbox occupancy mirrored in atomics: a stage that finds its input empty SPINS on these for up to ~100 us
  // before it sleeps on the condition variable -- a futex wake-up costs 10-50 us, a third of a stage's time per frame
  std::atomic<int> n_jobs{0}, n_results{0}, n_fjobs{0}, n_fres{0};
  // staged mode (ilsm_slam_create_staged): the three nodes as three stages, each with its own context (streams, scratch)
  // and host thread like the reference's three processes -- scanRegistration on ctx0 + fworker, laserOdometry on the
  // caller's context and thread, laserMapping on ctx2 + worker.  Frame k's front end, frame k-1's odometry and frame
  // k-2's / k-1's mapping are in flight together.
  ilsm_ctx* ctx0 = nullptr;
  bool staged = false, fe_in_flight = false;
  struct FeJob {
    const float* xyzi = nullptr;
    int n = 0, stride = 16, use_aloam = 1;
    long long frame = 0;
  } fjob;
  struct FeResult {
    int rc = 0, use_aloam = 1;
    char err[256] = "";
    int counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long frame = 0;
  } fres;
  std::thread fworker;
  std::mutex fmu;
  std::condition_variable fcv;
  bool fjob_posted = false, fres_ready = false, fstop = false;
  long long pushed = 0;
  // host-side phase clock (profiling aid, read with ilsm_slam_host_phases): seconds accumulated per phase
  double phase_s[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // [8..] mapping-stage detail (ILSM_STAGE_TRACE)
};

static inline void spin_until_nonzero(const std::atomic<int>& a, const bool* stop = nullptr) {
  for (int i = 0; i < 4000 && a.load(std::memory_order_acquire) == 0 && !(stop && *stop); ++i) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
}

struct PhaseClock {
  double* acc;
  std::chrono::steady_clock::time_point t;
  explicit PhaseClock(double* a) : acc(a), t(std::chrono::steady_clock::now()) {}
  void lap(int k) {
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
                           int cnt[8], PhaseClock& clk, int lap_launch, int lap_wait) {
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
static int frontend_gather(Ctx& f, const int cnt[8], SlamH::FeSlot& o, bool copy_lflat) {
  const int n_sharp = cnt[1], n_lsharp = cnt[2], n_flat = cnt[3], n_lflat = cnt[4];
  int rc;
  if ((rc = o.sharp.reserve(n_sharp + 4)) || (rc = o.flat.reserve(n_flat + 4)) || (rc = o.lsharp.reserve(n_lsharp + 4)) ||
      (copy_lflat && (rc = o.lflat.reserve(n_lflat + 4))))
    return rc;
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
  clk.lap(3);  // odometry launches
  if (solve) {
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
    c.lm_result(s.para_q, s.para_t, stats ? &stats->odometry : nullptr);
    if (stats) stats->odometry.passes = odometry_opts().outer_iterations, stats->ran_odometry = 1;
  }
  clk.lap(4);  // wait for the odometry
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

// body of the mapping stage's thread: one process() iteration per posted job, enqueue + collect on the second context
static void mapping_worker(SlamH* sp) {
  SlamH& s = *sp;
  Ctx& c2 = s.ctx2->c;
  cudaSetDevice(c2.device);
  for (;;) {
    SlamH::MapJob j;
    spin_until_nonzero(s.n_jobs, &s.stop);
    {
      std::unique_lock<std::mutex> lk(s.wmu);
      s.wcv.wait(lk, [&] { return !s.jobs.empty() || s.stop; });
      if (s.jobs.empty()) return;  // (stop is only raised once the queue has drained)
      j = s.jobs.front();
      s.jobs.pop_front();
      s.n_jobs.fetch_sub(1, std::memory_order_relaxed);
    }
    SlamH::MapResult r;
    r.frame = j.frame;
    {
      std::lock_guard<std::mutex> lk2(c2.mu);
      memset(&r.report, 0, sizeof(r.report)), memset(&r.cstats, 0, sizeof(r.cstats));
      cudaError_t e = cudaStreamWaitEvent(c2.stream, j.ev_in, 0);
      r.rc = e == cudaSuccess ? ILSM_OK : fail_cuda(e, "cudaStreamWaitEvent(mapping stage)");
      PhaseClock wclk(s.phase_s);  // [6] mapping-stage launches, [7] wait for the mapped pose (written by this thread only)
      CubeMapH& cm = s.cube->m;
      SlamH::StackSet& set = s.stk[j.stack_set];
      if (!r.rc) r.rc = cm.wait_tail();
      wclk.lap(8);  // wait for the previous frame's deferred insertion
      if (!r.rc) r.rc = mapping_enqueue(cm, set, j.d_lsharp, j.n_lsharp, j.d_lflat, j.n_lflat, j.q_odom, j.t_odom);
      if (!r.rc) {  // the deferred insertion (side stream) is the set's last reader
        e = cudaEventRecord(set.ev_free, c2.aux);
        if (e != cudaSuccess) r.rc = fail_cuda(e, "cudaEventRecord(stack set)");
        set.free_recorded = true;
      }
      wclk.lap(6);
      if (!r.rc) r.rc = cubemap_frame_collect(cm, r.q, r.t, &r.report, &r.cstats);
      wclk.lap(7);
      if (r.rc) snprintf(r.err, sizeof(r.err), "%s", ilsm_last_error());  // the error text is thread-local: carry it over
    }
    {
      std::lock_guard<std::mutex> lk(s.wmu);
      s.results.push_back(r);
      s.n_results.fetch_add(1, std::memory_order_release);
    }
    s.wcv.notify_all();
  }
}

// hand frame `frame`, written into slot `o` and stack set frame & 1, to the mapping thread
static void post_mapping_job(SlamH& s, const SlamH::FeSlot& o, const int cnt[8], long long frame, const double q_odom[4],
                             const double t_odom[3]) {
  SlamH::MapJob j;
  j.n_lsharp = cnt[2], j.n_lflat = cnt[4], j.frame = frame;
  j.d_lsharp = o.lsharp.p, j.d_lflat = o.lf, j.ev_in = o.ev, j.stack_set = (int)(frame & 1);
  for (int i = 0; i < 4; ++i) j.q_odom[i] = q_odom[i];
  for (int i = 0; i < 3; ++i) j.t_odom[i] = t_odom[i];
  {
    std::lock_guard<std::mutex> lk(s.wmu);
    s.jobs.push_back(j);
    s.n_jobs.fetch_add(1, std::memory_order_release);
  }
  s.maps_in_flight++;
  s.wcv.notify_all();
}

// wait for the mapping stage's answer to its oldest job and hand it out
static int take_mapping_result(SlamH& s, double q_map[4], double t_map[3], ilsm_slam_stats* stats, long long* frame = nullptr) {
  spin_until_nonzero(s.n_results);
  std::unique_lock<std::mutex> lk(s.wmu);
  s.wcv.wait(lk, [&] { return !s.results.empty(); });
  const SlamH::MapResult r = s.results.front();
  s.results.pop_front();
  s.n_results.fetch_sub(1, std::memory_order_relaxed);
  lk.unlock();
  s.maps_in_flight--;
  if (frame) *frame = r.frame;
  if (r.rc) return fail(r.rc, r.err);
  for (int i = 0; i < 4; ++i) q_map[i] = r.q[i];
  for (int i = 0; i < 3; ++i) t_map[i] = r.t[i];
  if (stats) stats->mapping = r.report, stats->cubemap = r.cstats;
  return ILSM_OK;
}

// ---- staged mode: scanRegistration as its own stage
static int frontend_stage(SlamH& s, Ctx& f, const SlamH::FeJob& j, SlamH::FeResult& r) {
  PhaseClock fclk(s.phase_s);  // [9] upload + front-end launches, [10] wait for the feature counts, [11] gathers (this thread only)
  int rc;
  if ((rc = frontend_counts(f, j.xyzi, j.n, j.stride, nullptr, s.min_range, r.counts, fclk, 9, 10)) ||
      (rc = frontend_gather(f, r.counts, s.fslot[j.frame % 3], true)))
    return rc;
  fclk.lap(11);
  return ILSM_OK;
}

static void frontend_worker(SlamH* sp) {
  SlamH& s = *sp;
  Ctx& f = s.ctx0->c;
  cudaSetDevice(f.device);
  for (;;) {
    SlamH::FeJob j;
    spin_until_nonzero(s.n_fjobs, &s.fstop);
    {
      std::unique_lock<std::mutex> lk(s.fmu);
      s.fcv.wait(lk, [&] { return s.fjob_posted || s.fstop; });
      if (s.fstop) return;
      j = s.fjob;
      s.fjob_posted = false;
      s.n_fjobs.store(0, std::memory_order_relaxed);
    }
    SlamH::FeResult r;
    r.frame = j.frame, r.use_aloam = j.use_aloam;
    {
      std::lock_guard<std::mutex> lk2(f.mu);
      r.rc = frontend_stage(s, f, j, r);
      if (r.rc) snprintf(r.err, sizeof(r.err), "%s", ilsm_last_error());
    }
    {
      std::lock_guard<std::mutex> lk(s.fmu);
      s.fres = r;
      s.fres_ready = true;
      s.n_fres.store(1, std::memory_order_release);
    }
    s.fcv.notify_all();
  }
}

static int take_frontend_result(SlamH& s, SlamH::FeResult* out) {
  spin_until_nonzero(s.n_fres);
  std::unique_lock<std::mutex> lk(s.fmu);
  s.fcv.wait(lk, [&] { return s.fres_ready; });
  s.fres_ready = false;
  s.n_fres.store(0, std::memory_order_relaxed);
  s.fe_in_flight = false;
  *out = s.fres;
  if (out->rc) return fail(out->rc, out->err);
  return ILSM_OK;
}

}  // namespace ilsm

using namespace ilsm;

struct ilsm_slam {
  SlamH s;
};

extern "C" {

// the slots and stack sets (SlamH::fslot, SlamH::stk) at typical 16-ring sizes up front: a growing buffer costs a
// device-wide synchronisation
static int reserve_frame_buffers(SlamH& s) {
  int rc;
  for (SlamH::FeSlot& o : s.fslot) {
    if (cudaEventCreateWithFlags(&o.ev, cudaEventDisableTiming) != cudaSuccess)
      return fail(ILSM_ERR_CUDA, "slam_create: event creation failed");
    if ((rc = o.sharp.reserve(1024)) || (rc = o.flat.reserve(4096)) || (rc = o.lsharp.reserve(8192)) || (rc = o.lflat.reserve(32768)))
      return rc;
  }
  for (SlamH::StackSet& set : s.stk) {
    if (cudaEventCreateWithFlags(&set.ev_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&set.ev_free, cudaEventDisableTiming) != cudaSuccess)
      return fail(ILSM_ERR_CUDA, "slam_create: event creation failed");
    if ((rc = set.c.reserve(8192)) || (rc = set.s.reserve(32768)) || (rc = set.n.reserve(4))) return rc;
  }
  return ILSM_OK;
}

static int slam_create_common(ilsm_ctx* ctx, float min_range, ilsm_slam** out, ilsm_slam** h_out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "slam_create: null argument");
  ilsm_slam* h = new (std::nothrow) ilsm_slam();
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  h->s.ctx = &ctx->c;
  h->s.min_range = min_range > 0.f ? min_range : 0.3f;
  int rc;
  {
    std::lock_guard<std::mutex> lk(ctx->c.mu);
    cudaSetDevice(ctx->c.device);
    if (!(rc = h->s.last_corner.init(&ctx->c))) rc = h->s.last_surf.init(&ctx->c);
    if (!rc && !(rc = h->s.last_corner.reserve_points(16384))) rc = h->s.last_surf.reserve_points(65536);
    if (!rc) rc = reserve_frame_buffers(h->s);
  }
  if (rc) {
    ilsm_slam_destroy(h);
    return rc;
  }
  *h_out = h;
  return ILSM_OK;
}

// the mapping stage on its own context and host thread (pipelined and staged handles)
static int slam_create_mapping_stage(ilsm_slam* h, float line_res, float plane_res, int cube_capacity) {
  int rc;
  if ((rc = ilsm_create(h->s.ctx->device, &h->s.ctx2)) ||
      (rc = ilsm_cubemap_create(h->s.ctx2, line_res, plane_res, cube_capacity, &h->s.cube)))
    return rc;
  h->s.worker = std::thread(mapping_worker, &h->s);
  return ILSM_OK;
}

ILSM_API int ilsm_slam_create(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                              ilsm_slam** out) {
  ilsm_slam* h = nullptr;
  int rc = slam_create_common(ctx, min_range, out, &h);
  if (rc) return rc;
  if ((rc = ilsm_cubemap_create(ctx, line_res, plane_res, cube_capacity, &h->s.cube))) {
    ilsm_slam_destroy(h);
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API int ilsm_slam_create_mapopt(ilsm_ctx* ctx, float voxel_leaf, float downsample_size, float min_range, ilsm_slam** out) {
  ilsm_slam* h = nullptr;
  int rc = slam_create_common(ctx, min_range, out, &h);
  if (rc) return rc;
  if ((rc = ilsm_mapopt_create(ctx, voxel_leaf, downsample_size, &h->s.mapopt))) {
    ilsm_slam_destroy(h);
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API int ilsm_slam_create_async(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                    ilsm_slam** out) {
  ilsm_slam* h = nullptr;
  int rc = slam_create_common(ctx, min_range, out, &h);
  if (rc) return rc;
  h->s.async = true;
  if ((rc = slam_create_mapping_stage(h, line_res, plane_res, cube_capacity))) {
    ilsm_slam_destroy(h);
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API int ilsm_slam_create_staged(ilsm_ctx* ctx, float line_res, float plane_res, float min_range, int cube_capacity,
                                     ilsm_slam** out) {
  ilsm_slam* h = nullptr;
  int rc = slam_create_common(ctx, min_range, out, &h);
  if (rc) return rc;
  h->s.staged = true;
  h->s.last_corner.in_line = h->s.last_surf.in_line = true;  // nothing follows the tree builds on this stage's stream
  if ((rc = ilsm_create(ctx->c.device, &h->s.ctx0)) || (rc = slam_create_mapping_stage(h, line_res, plane_res, cube_capacity))) {
    ilsm_slam_destroy(h);
    return rc;
  }
  h->s.fworker = std::thread(frontend_worker, &h->s);
  *out = h;
  return ILSM_OK;
}

ILSM_API void ilsm_slam_destroy(ilsm_slam* slam) {
  if (!slam) return;
  SlamH& s = slam->s;
  if (s.fworker.joinable()) {
    {
      std::unique_lock<std::mutex> lk(s.fmu);
      s.fcv.wait(lk, [&] { return !s.fjob_posted; });
      s.fstop = true;
    }
    s.fcv.notify_all();
    s.fworker.join();
  }
  if (getenv("ILSM_STAGE_TRACE"))
    fprintf(stderr, "[ilsm stage trace] frames %lld  mapping: tail-wait %.1f us  enqueue %.1f us  collect %.1f us   front end: launches %.1f us  "
                    "wait %.1f us  gathers %.1f us per frame\n", s.frames,
            1e6 * s.phase_s[8] / (s.frames ? s.frames : 1), 1e6 * s.phase_s[6] / (s.frames ? s.frames : 1),
            1e6 * s.phase_s[7] / (s.frames ? s.frames : 1), 1e6 * s.phase_s[9] / (s.frames ? s.frames : 1),
            1e6 * s.phase_s[10] / (s.frames ? s.frames : 1), 1e6 * s.phase_s[11] / (s.frames ? s.frames : 1));
  if (s.ctx0) {
    std::lock_guard<std::mutex> lk0(s.ctx0->c.mu);
    cudaSetDevice(s.ctx0->c.device);
    cudaStreamSynchronize(s.ctx0->c.stream);
  }
  if (s.worker.joinable()) {
    {
      std::unique_lock<std::mutex> lk(s.wmu);
      s.wcv.wait(lk, [&] { return s.jobs.empty(); });  // posted jobs are taken (and finished) before the thread is told to stop
      s.stop = true;
    }
    s.wcv.notify_all();
    s.worker.join();
  }
  if (s.ctx2) {  // let the mapping stage drain before anything it reads goes away
    std::lock_guard<std::mutex> lk2(s.ctx2->c.mu);
    cudaSetDevice(s.ctx2->c.device);
    cudaStreamSynchronize(s.ctx2->c.stream);
    cudaStreamSynchronize(s.ctx2->c.aux);
  }
  {
    std::lock_guard<std::mutex> lk(s.ctx->mu);
    cudaSetDevice(s.ctx->device);
    cudaStreamSynchronize(s.ctx->stream);
    for (SlamH::FeSlot& o : s.fslot)
      if (o.ev) cudaEventDestroy(o.ev);
    for (SlamH::StackSet& set : s.stk) {
      if (set.ev_ready) cudaEventDestroy(set.ev_ready);
      if (set.ev_free) cudaEventDestroy(set.ev_free);
    }
  }
  if (s.cube) ilsm_cubemap_destroy(s.cube);
  if (s.mapopt) ilsm_mapopt_destroy(s.mapopt);
  if (s.ctx2) ilsm_destroy(s.ctx2);
  if (s.ctx0) ilsm_destroy(s.ctx0);
  cudaSetDevice(s.ctx->device);
  delete slam;  // frees the slots, stack sets and last-frame maps: no stage reads them any more
}

ILSM_API ilsm_cubemap* ilsm_slam_cubemap(ilsm_slam* slam) { return slam ? slam->s.cube : nullptr; }
ILSM_API ilsm_mapopt* ilsm_slam_mapopt(ilsm_slam* slam) { return slam ? slam->s.mapopt : nullptr; }

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
  if (!s.async || s.maps_in_flight == 0) return ILSM_OK;
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
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (stats) memset(stats, 0, sizeof(*stats));
  int rc;
  PhaseClock clk(s.phase_s);
  // ---- scanRegistration: the frame is the only upload
  // the previous frame's tree builds (on the maps' own streams, overlapping its mapping step) read its clouds: order this
  // frame's front end after them
  if ((rc = s.last_corner.wait_ready(c.stream)) || (rc = s.last_surf.wait_ready(c.stream))) return rc;
  int cnt[8];
  if ((rc = frontend_counts(c, xyzi, n, stride_bytes, pc2, s.min_range, cnt, clk, 0, 2))) return rc;
  if (s.async && s.maps_in_flight > 0) {
    // the previous frame's mapped pose: the mapping stage's thread has had this frame's upload and front end to finish
    if ((rc = take_mapping_result(s, q_map, t_map, stats))) return rc;
    *have_prev = 1;
  }
  clk.lap(1);  // (pipelined) wait for the previous frame's mapping
  feature_stats(stats, cnt);
  SlamH::FeSlot& o = s.fslot[s.frames % 3];
  SlamH::StackSet& set = s.stk[s.frames & 1];
  CubeMapH* cmp = s.cube ? &s.cube->m : nullptr;
  // With the mapping stage on its own context nothing orders the next call's front end, which rewrites fe.lflat, after
  // this frame's stack VoxelGrid: that reads a copy in the slot.
  if ((rc = frontend_gather(c, cnt, o, s.ctx2 != nullptr))) return rc;
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
    rc = mapopt_frame_core(s.mapopt, c.fe.raw.p, n, pc2 ? 16 : stride_bytes, reinterpret_cast<const float*>(o.lf), cnt[4], 16,
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
  clk.lap(5);  // tree builds + mapping stage (synchronous: enqueue and wait; pipelined: enqueue only)
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
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (stats) memset(stats, 0, sizeof(*stats));
  int rc;
  PhaseClock clk(s.phase_s);
  SlamH::FeResult fr;
  const bool have_fe = s.fe_in_flight;
  if (have_fe && (rc = take_frontend_result(s, &fr))) return rc;
  clk.lap(2);  // wait for the front-end stage
  if (n >= 0) {
    {
      std::lock_guard<std::mutex> lkf(s.fmu);
      s.fjob.xyzi = xyzi, s.fjob.n = n, s.fjob.stride = stride_bytes, s.fjob.use_aloam = use_aloam, s.fjob.frame = s.pushed;
      s.fjob_posted = true;
      s.n_fjobs.store(1, std::memory_order_release);
    }
    s.fcv.notify_all();
    s.fe_in_flight = true;
    s.pushed++;
  }
  clk.lap(0);  // hand-over to the front-end stage
  if (!have_fe) {  // nothing for the odometry: first call, or the pipeline is draining
    if (s.maps_in_flight > 0) {
      long long mf = -1;
      if ((rc = take_mapping_result(s, q_map, t_map, stats, &mf))) return rc;
      *map_frame = (int)mf;
    }
    clk.lap(1);
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
  const bool collect_prev = s.maps_in_flight > 0;
  post_mapping_job(s, o, cnt, fr.frame, q_odom, t_odom);
  clk.lap(5);  // tree builds + hand-over to the mapping stage
  if (collect_prev) {
    long long mf = -1;
    if ((rc = take_mapping_result(s, q_map, t_map, stats, &mf))) return rc;
    *map_frame = (int)mf;
  }
  clk.lap(1);  // wait for the mapping stage (the frame before)
  s.frames++;
  return ILSM_OK;
}

extern "C" ILSM_API int ilsm_slam_host_phases(ilsm_slam* slam, double out8[8]) {
  if (!slam || !out8) return fail(ILSM_ERR_INVALID_ARG, "slam_host_phases: null argument");
  for (int i = 0; i < 8; ++i) out8[i] = slam->s.phase_s[i], slam->s.phase_s[i] = 0;
  return ILSM_OK;
}
