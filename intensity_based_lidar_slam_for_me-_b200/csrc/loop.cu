// loop.cu -- K7: loop closure per keyframe on the device, the body of the reference's loopClosureThread
// (intensity_feature_tracker.cpp:195-393 around SCManager::detectLoopClosureID, Scancontext.cpp:253-344).
//
// One ilsm_loop_add_keyframe call:
//   store   ScanContext descriptor of the cloud as passed (ScDb::make_dev, append_dev) and VoxelGrid(leaf) of it into a
//           device keyframe pool (float4 xyzi, keyframes back to back, grown by doubling with its contents kept), the
//           pose on the host;
//   detect  SCManager's state machine: early return below exclude_recent + 1 keyframes, the searchable size refreshed
//           every tree_period-th search, candidates_dev over it, the first strict minimum, the threshold;
//   verify  (only with a loop) loop_gather_kernel moves keyframes [c-h, c+h] of the pool to the world frame in ONE launch
//           (the keyframe items are kernel parameters), VoxelGrid(leaf) of the concatenation, a map build on the context
//           stream and one icp_align pair: source = this keyframe's stored cloud, guess = (q_c * Rz(-yaw_diff), t_c).
// Host synchronisations: one per call (candidate records and the keyframe's voxel count), two more for a verified
// keyframe (the submap's voxel count before the build, the ICP result).
#include <float.h>
#include <math.h>

#include <new>
#include <vector>

#include "ilsm_cubemap.hpp"

namespace ilsm {
int icp_align(Ctx& c, ilsm_map* const* targets, int n_pairs, const float* d_src, const int* offs, int stride_bytes,
              const double* guess7, const ilsm_icp_opts& o, ilsm_icp_result* results);

namespace {

constexpr int kLoopMaxItems = 15;  // 2 * submap_half + 1 keyframes, submap_half <= 7

struct LoopItem {
  double q[4], t[3];    // keyframe pose (world <- keyframe)
  long long src;        // first point in the pool
  int count, dst;       // points; first slot in the gathered submap
};
struct LoopItems {  // kernel parameters, like GatherItems: no staging copy before the launch
  LoopItem it[kLoopMaxItems];
};

// grid (x, n_items): item blockIdx.y's points under its pose, pointAssociateToMap's order (quat_rotate then dadd: double
// math, float store) -- the same steps as icp_tile's transform; intensity carried
__global__ void loop_gather_kernel(const float4* __restrict__ pool, const __grid_constant__ LoopItems items, float4* __restrict__ out) {
  pdl_entry();
  const LoopItem& it = items.it[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < it.count; i += gridDim.x * blockDim.x) {
    const float4 p = pool[it.src + i];
    const D3 w = quat_rotate(it.q, d3((double)p.x, (double)p.y, (double)p.z));
    out[it.dst + i] = make_float4(__double2float_rn(dadd(w.x, it.t[0])), __double2float_rn(dadd(w.y, it.t[1])),
                                  __double2float_rn(dadd(w.z, it.t[2])), p.w);
  }
}

// device layout of the per-call read-back (one copy): 16 x f64 distances | 16 x i32 ids | 16 x i32 shifts | 16 x f32 key
// distances | i32 keyframe voxel count | i32 submap voxel count
constexpr size_t kOffDist = 0, kOffId = 128, kOffShift = 192, kOffKey = 256, kOffKfN = 320, kOffSubN = 324, kOutBytes = 336;

}  // namespace

struct LoopDb {
  Ctx* ctx = nullptr;
  ilsm_loop_opts o;
  ScDb sc;
  ilsm_map submap;            // the submap's search structure, built in line on the context stream
  DevBuf<float4> pool;        // stored keyframes, VoxelGrid(leaf) of each, back to back
  long long pool_n = 0;
  std::vector<long long> kf_off;
  std::vector<int> kf_n;
  std::vector<double> kf_pose;  // 7 per keyframe: qx qy qz qw tx ty tz
  DevBuf<float> stage;          // the caller's cloud (host form)
  DevBuf<float> desc;           // this keyframe's descriptor
  DevBuf<unsigned char> out;    // kOutBytes
  PinnedBuf<unsigned char> pin;
  DevBuf<float4> sub, sub_vox;  // gathered submap, its VoxelGrid
  int tree_counter = 0, n_search = 0;

  int add(const float* d_xyz, int n, int stride_bytes, const double q[4], const double t[3], ilsm_loop_result* r);
  int verify(int cand, double yaw, ilsm_loop_result* r);
};

// 1. store
static int loop_store(LoopDb& L, const float* d_xyz, int n, int stride_bytes) {
  Ctx& c = *L.ctx;
  int rc;
  if ((rc = L.desc.reserve(1200)) || (rc = L.out.reserve(kOutBytes)) || (rc = L.pin.reserve(kOutBytes))) return rc;
  if ((rc = L.sc.make_dev(d_xyz, n, stride_bytes, L.desc.p)) || (rc = L.sc.append_dev(L.desc.p, 1, false))) return rc;
  const size_t need = (size_t)L.pool_n + (size_t)n + 1;
  if (need > L.pool.cap) {  // grow and keep the contents
    DevBuf<float4> bigger;
    if ((rc = bigger.reserve(2 * need))) return rc;
    if (L.pool_n > 0)
      ILSM_CUDA(cudaMemcpyAsync(bigger.p, L.pool.p, (size_t)L.pool_n * sizeof(float4), cudaMemcpyDeviceToDevice, c.stream));
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
    L.pool = std::move(bigger);
  }
  int* d_kfn = reinterpret_cast<int*>(L.out.p + kOffKfN);
  if (n == 0) {
    ILSM_CUDA(cudaMemsetAsync(d_kfn, 0, sizeof(int), c.stream));
    return ILSM_OK;
  }
  // the VoxelGrid dispatch of ilsm_voxelgrid: the same voxels, in the same order, as that entry point gives
  const Ctx::VgCloud vc = {d_xyz, n, L.o.leaf, L.pool.p + L.pool_n, d_kfn};
  return c.voxelgrid(&vc, 1, stride_bytes, intensity_word(stride_bytes), c.stream);
}

int LoopDb::add(const float* d_xyz, int n, int stride_bytes, const double q[4], const double t[3], ilsm_loop_result* r) {
  Ctx& c = *ctx;
  memset(r, 0, sizeof(*r));
  r->loop_id = r->nn_id = -1, r->submap_first = r->submap_last = -1;
  int rc;
  if ((rc = loop_store(*this, d_xyz, n, stride_bytes))) return rc;
  const int size = sc.count;
  r->keyframe_id = size - 1;
  // 2. detect (Scancontext.cpp:265-323)
  const bool early = size < o.exclude_recent + 1;  // the refresh counter does not advance
  if (!early) {
    if (tree_counter % o.tree_period == 0) n_search = size - o.exclude_recent;
    tree_counter += 1;
    unsigned char* d = out.p;
    if ((rc = sc.candidates_dev(desc.p, n_search, o.num_candidates, reinterpret_cast<int*>(d + kOffId),
                                reinterpret_cast<float*>(d + kOffKey), reinterpret_cast<double*>(d + kOffDist),
                                reinterpret_cast<int*>(d + kOffShift))))
      return rc;
  }
  ILSM_CUDA(cudaMemcpyAsync(pin.p, out.p, kOutBytes, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  int kn;
  memcpy(&kn, pin.p + kOffKfN, sizeof(int));
  kf_off.push_back(pool_n), kf_n.push_back(kn), kf_pose.insert(kf_pose.end(), q, q + 4), kf_pose.insert(kf_pose.end(), t, t + 3);
  pool_n += kn;
  if (early) return ILSM_OK;
  double min_dist = 10000000;
  int nn_align = 0, nn_idx = 0;
  for (int i = 0; i < o.num_candidates; ++i) {
    int id, sh;
    double dist;
    memcpy(&id, pin.p + kOffId + 4 * i, 4), memcpy(&sh, pin.p + kOffShift + 4 * i, 4), memcpy(&dist, pin.p + kOffDist + 8 * i, 8);
    if (id >= 0 && dist < min_dist) min_dist = dist, nn_align = sh, nn_idx = id;
  }
  r->nn_id = nn_idx, r->shift = nn_align, r->sc_dist = min_dist;
  r->yaw_diff_rad = (float)(nn_align * (360.0 / 60.0) * M_PI / 180.0);  // deg2rad returns a float
  if (!(min_dist < o.sc_dist_threshold)) return ILSM_OK;
  r->loop_id = nn_idx;
  return verify(nn_idx, r->yaw_diff_rad, r);
}

// 3. verify
int LoopDb::verify(int cand, double yaw, ilsm_loop_result* r) {
  Ctx& c = *ctx;
  const int size = sc.count, k = size - 1;
  const int lo = cand - o.submap_half < 0 ? 0 : cand - o.submap_half;
  const int lim = size - o.exclude_recent;  // [0, size - exclude_recent): keyframes the tree may hold
  const int hi = cand + o.submap_half < lim - 1 ? cand + o.submap_half : lim - 1;
  LoopItems items;
  memset(&items, 0, sizeof(items));
  int raw = 0, n_items = 0, most = 0;
  for (int j = lo; j <= hi; ++j) {
    LoopItem& it = items.it[n_items++];
    for (int a = 0; a < 4; ++a) it.q[a] = kf_pose[7 * (size_t)j + a];
    for (int a = 0; a < 3; ++a) it.t[a] = kf_pose[7 * (size_t)j + 4 + a];
    it.src = kf_off[j], it.count = kf_n[j], it.dst = raw;
    raw += kf_n[j];
    most = kf_n[j] > most ? kf_n[j] : most;
  }
  r->verified = 1, r->submap_first = lo, r->submap_last = hi;
  int rc;
  if ((rc = sub.reserve((size_t)raw + 4)) || (rc = sub_vox.reserve((size_t)raw + 4))) return rc;
  int n_vox = 0;
  if (raw > 0) {
    ILSM_CUDA(launch_pdl(loop_gather_kernel, dim3((unsigned)((most + 255) / 256), (unsigned)n_items), dim3(256), 0, c.stream,
                         (const float4*)pool.p, items, sub.p));
    count_launches(1);
    if ((rc = check_launch("loop_gather"))) return rc;
    int* d_subn = reinterpret_cast<int*>(out.p + kOffSubN);
    const Ctx::VgCloud vc = {reinterpret_cast<const float*>(sub.p), raw, o.leaf, sub_vox.p, d_subn};
    if ((rc = c.voxelgrid(&vc, 1, 16, 3, c.stream))) return rc;
    ILSM_CUDA(cudaMemcpyAsync(pin.p + kOffSubN, d_subn, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
    memcpy(&n_vox, pin.p + kOffSubN, sizeof(int));
  }
  r->submap_points = n_vox;
  if ((rc = submap.m.build_dev(reinterpret_cast<const float*>(sub_vox.p), n_vox, 16, o.cell))) return rc;
  // the guess: the candidate's pose turned by the aligning shift, q_c * Rz(-yaw_diff_rad)
  const double* pc = &kf_pose[7 * (size_t)cand];
  const QuatH qc = {pc[0], pc[1], pc[2], pc[3]};
  const double h = -yaw * 0.5;
  const QuatH g = qmul_h(qc, QuatH{0.0, 0.0, sin(h), cos(h)});
  const double guess[7] = {g.x, g.y, g.z, g.w, pc[4], pc[5], pc[6]};
  const int offs[2] = {0, kf_n[k]};
  ilsm_map* target = &submap;
  if ((rc = icp_align(c, &target, 1, reinterpret_cast<const float*>(pool.p + kf_off[k]), offs, 16, guess, o.icp, &r->icp))) return rc;
  r->accepted = r->icp.converged && r->icp.fitness < o.fitness_threshold;
  if (r->accepted) {  // T_loop^-1 * T_icp
    const QuatH qi = {-pc[0], -pc[1], -pc[2], pc[3]};
    const QuatH qr = qmul_h(qi, QuatH{r->icp.q_xyzw[0], r->icp.q_xyzw[1], r->icp.q_xyzw[2], r->icp.q_xyzw[3]});
    const double dt[3] = {r->icp.t[0] - pc[4], r->icp.t[1] - pc[5], r->icp.t[2] - pc[6]};
    qrot_h(qi, dt, r->t_rel);
    r->q_rel_xyzw[0] = qr.x, r->q_rel_xyzw[1] = qr.y, r->q_rel_xyzw[2] = qr.z, r->q_rel_xyzw[3] = qr.w;
  }
  return ILSM_OK;
}

}  // namespace ilsm

struct ilsm_loop {
  ilsm::LoopDb l;
};

using namespace ilsm;

// also the check of ilsm_slam_enable_loop's loop options (pipeline.cu)
int check_loop_opts(const ilsm_loop_opts& o) {
  if (o.exclude_recent < 1 || o.tree_period < 1 || o.num_candidates < 1 || o.num_candidates > 16 || o.submap_half < 0 ||
      o.submap_half > 7)
    return fail(ILSM_ERR_INVALID_ARG, "loop_create: exclude_recent >= 1, tree_period >= 1, num_candidates in [1,16], submap_half in [0,7]");
  if (!(o.leaf > 0.f) || !(o.cell > 0.f) || !isfinite(o.leaf) || !isfinite(o.cell))
    return fail(ILSM_ERR_INVALID_ARG, "loop_create: leaf and cell must be positive and finite");
  if (isnan(o.sc_dist_threshold) || isnan(o.fitness_threshold)) return fail(ILSM_ERR_INVALID_ARG, "loop_create: NaN threshold");
  if (o.icp.max_iterations < 0) return fail(ILSM_ERR_INVALID_ARG, "loop_create: icp.max_iterations < 0");
  return ILSM_OK;
}

// the argument check of ilsm_loop_add_keyframe[_dev]
static int check_keyframe_args(const ilsm_loop* loop, const float* xyz, int n, int stride_bytes, const double* q, const double* t,
                               const ilsm_loop_result* result, const char* who) {
  if (!loop || !result || !q || !t || (n > 0 && !xyz)) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (n < 0 || n >= (1 << 24) || !valid_stride(stride_bytes) || stride_bytes < 16)
    return fail(ILSM_ERR_INVALID_ARG, "%s: bad n/stride (0 <= n < 2^24 xyzi points, stride >= 16)", who);
  const double nq = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (!(fabs(nq - 1.0) <= 1e-6)) return fail(ILSM_ERR_INVALID_ARG, "%s: the quaternion is not unit (|q| = %.9g)", who, nq);
  if (!isfinite(t[0]) || !isfinite(t[1]) || !isfinite(t[2])) return fail(ILSM_ERR_INVALID_ARG, "%s: non-finite translation", who);
  return ILSM_OK;
}

extern "C" {

ILSM_API void ilsm_loop_opts_default(ilsm_loop_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->exclude_recent = 50;
  o->tree_period = 50;
  o->num_candidates = 10;
  o->submap_half = 2;
  o->sc_dist_threshold = 0.13;
  o->leaf = 0.4f;
  o->cell = 1.0f;
  o->fitness_threshold = 0.3;
  ilsm_icp_opts_default(&o->icp);
  o->icp.max_correspondence_distance = 2.0;
  o->icp.max_iterations = 50;
  o->icp.transformation_epsilon = 1e-8;
  o->icp.euclidean_fitness_epsilon = 1e-6;
}

ILSM_API int ilsm_loop_create(ilsm_ctx* ctx, const ilsm_loop_opts* opts, ilsm_loop** out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "loop_create: null argument");
  *out = nullptr;
  ilsm_loop_opts o;
  if (opts)
    o = *opts;
  else
    ilsm_loop_opts_default(&o);
  int rc = check_loop_opts(o);
  if (rc) return rc;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return fail(ILSM_ERR_NO_DEVICE, "loop_create: no CUDA device available (libilsm_cuda has no CPU fallback)");
  }
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  ilsm_loop* h = new (std::nothrow) ilsm_loop();
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  LoopDb& L = h->l;
  L.ctx = &c, L.o = o, L.sc.ctx = &c;
  L.submap.m.in_line = true;
  if ((rc = L.submap.m.init(&c))) {
    delete h;
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API void ilsm_loop_destroy(ilsm_loop* loop) {
  if (!loop) return;
  Ctx& c = *loop->l.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  cudaSetDevice(c.device);
  cudaStreamSynchronize(c.stream);
  delete loop;
}

ILSM_API int ilsm_loop_size(const ilsm_loop* loop) { return loop ? loop->l.sc.count : 0; }

ILSM_API int ilsm_loop_add_keyframe(ilsm_loop* loop, const float* xyz, int n, int stride_bytes, const double q_xyzw[4],
                                    const double t_xyz[3], ilsm_loop_result* result) {
  int rc = check_keyframe_args(loop, xyz, n, stride_bytes, q_xyzw, t_xyz, result, "loop_add_keyframe");
  if (rc) return rc;
  LoopDb& L = loop->l;
  ILSM_ENTER(*L.ctx);
  const size_t bytes = (size_t)n * stride_bytes;
  if ((rc = L.stage.reserve(bytes / 4 + 4))) return rc;
  if (bytes) ILSM_CUDA(cudaMemcpyAsync(L.stage.p, xyz, bytes, cudaMemcpyHostToDevice, L.ctx->stream));
  return L.add(L.stage.p, n, stride_bytes, q_xyzw, t_xyz, result);
}

ILSM_API int ilsm_loop_add_keyframe_dev(ilsm_loop* loop, const float* d_xyz, int n, int stride_bytes, const double q_xyzw[4],
                                        const double t_xyz[3], ilsm_loop_result* result) {
  int rc = check_keyframe_args(loop, d_xyz, n, stride_bytes, q_xyzw, t_xyz, result, "loop_add_keyframe_dev");
  if (rc) return rc;
  LoopDb& L = loop->l;
  ILSM_ENTER(*L.ctx);
  return L.add(d_xyz, n, stride_bytes, q_xyzw, t_xyz, result);
}

}  // extern "C"
