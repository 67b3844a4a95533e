// api.cu -- the C ABI (include/ilsm.h) over the kernels: handle management, staging of caller buffers, errors.
// No CPU fallback anywhere: without a CUDA device ilsm_create fails and nothing else can be called.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <new>

#include "ilsm_host.hpp"

namespace ilsm {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int fail_cuda(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), where);
  cudaGetLastError();
  return ILSM_ERR_CUDA;
}
static std::atomic<long long> g_launches{0};
void count_launches(int k) { g_launches.fetch_add(k, std::memory_order_relaxed); }
std::atomic<long long> g_live_bytes[2] = {{0}, {0}};
std::atomic<long long> g_live_handles{0};

int check_launch(const char* where) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(e, where);
  return ILSM_OK;
}

int eval_only_launch(Ctx* c, double* d_out, const double* d_pose7, double huber_a);
int factors_export(Ctx* c, ilsm_factor* d_out);
int sc_merge_dev(Ctx* ctx, const void* d_packed, int shards, int k, void* d_out, int batch = 1, size_t shard_stride = 0);
void sc_nccl_release(ScDb& d);  // scancontext_api.cu

int Ctx::init(int dev) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return fail(ILSM_ERR_NO_DEVICE, "no CUDA device available (libilsm_cuda has no CPU fallback)");
  }
  if (dev < 0 || dev >= count) return fail(ILSM_ERR_INVALID_ARG, "ilsm_create: device index out of range");
  device = dev;
  ILSM_CUDA(cudaSetDevice(dev));
  cudaDeviceProp prop;
  ILSM_CUDA(cudaGetDeviceProperties(&prop, dev));
  sm_count = prop.multiProcessorCount;
  int rc;
  if ((rc = stream.create()) || (rc = aux.create()) || (rc = ev_fork.create()) || (rc = ev_join.create()) || (rc = lm.reserve(1)))
    return rc;
  ILSM_CUDA(cudaMemsetAsync(lm.p, 0, sizeof(LmState), stream));
  if ((rc = pinned.reserve(4096))) return rc;
  ILSM_CUDA(cudaStreamSynchronize(stream));
  if (const char* e2 = getenv("ILSM_KNN_BINNED_MIN")) knn_binned_min = atoi(e2) > 0 ? atoi(e2) : 0x7fffffff;
  if (const char* e3 = getenv("ILSM_KNN_GROUP")) {
    const int gsz = atoi(e3);
    if (gsz == 1 || gsz == 2 || gsz == 4 || gsz == 8 || gsz == 16 || gsz == 32) knn_group = gsz;
  }
  return ILSM_OK;
}

Ctx::~Ctx() {
  if (stream) cudaStreamSynchronize(stream);
  if (aux) cudaStreamSynchronize(aux);
}

Map::~Map() {
  if (stream) cudaStreamSynchronize(stream);
}

// the LM iteration budget the solve kernel accepts
static int clamp_iterations(int n) { return n < 0 ? 0 : (n > 200 ? 200 : n); }

static ilsm_reg_opts sanitize(const ilsm_reg_opts* o) {
  ilsm_reg_opts r;
  if (o)
    r = *o;
  else
    ilsm_reg_opts_default(&r);
  if (r.outer_iterations < 1) r.outer_iterations = 1;
  if (r.outer_iterations > ILSM_MAX_OUTER) r.outer_iterations = ILSM_MAX_OUTER;
  r.max_num_iterations = clamp_iterations(r.max_num_iterations);
  return r;
}

}  // namespace ilsm

using namespace ilsm;



extern "C" {

ILSM_API int ilsm_abi_version(void) { return ILSM_ABI_VERSION; }
ILSM_API long long ilsm_launch_count(void) { return g_launches.load(); }
ILSM_API const char* ilsm_last_error(void) { return g_err; }

ILSM_API void ilsm_reg_opts_default(ilsm_reg_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->outer_iterations = 2;
  o->max_num_iterations = 4;
  o->huber_a = 0.1;
  o->knn_gate_sq = 1.0f;
  o->line_eig_ratio = 3.0;
  o->plane_tol = 0.2;
  o->min_corner_map = 10;
  o->min_surf_map = 50;
}

ILSM_API int ilsm_create(int device, ilsm_ctx** out) {
  if (!out) return fail(ILSM_ERR_INVALID_ARG, "ilsm_create: out is null");
  *out = nullptr;
  ilsm_ctx* h = new (std::nothrow) ilsm_ctx();
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  int rc = h->c.init(device);
  if (rc) {
    delete h;
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API void ilsm_destroy(ilsm_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->c.device);
  delete ctx;
}

ILSM_API int ilsm_sync(ilsm_ctx* ctx) {
  if (!ctx) return fail(ILSM_ERR_INVALID_ARG, "null ctx");
  ILSM_CUDA(cudaStreamSynchronize(ctx->c.stream));
  return ILSM_OK;
}

ILSM_API void* ilsm_stream(ilsm_ctx* ctx) { return ctx ? (void*)ctx->c.stream : nullptr; }

// profiling aid (not in include/ilsm.h): copy the 64 clock64() stamps of the last kernels to the host
ILSM_API int ilsm_debug_stamps(ilsm_ctx* ctx, long long* out64) {
  if (!ctx || !out64) return fail(ILSM_ERR_INVALID_ARG, "null");
  ILSM_ENTER(ctx->c);
  ILSM_CUDA(cudaStreamSynchronize(ctx->c.stream));
  ILSM_CUDA(cudaMemcpy(out64, ctx->c.lm.p->dbg, 64 * sizeof(long long), cudaMemcpyDeviceToHost));
  return ILSM_OK;
}

// testing aid (not in include/ilsm.h): bytes held by the device and the pinned buffers of every handle of the process;
// makes no CUDA call
ILSM_API void ilsm_debug_live_bytes(long long* device, long long* pinned) {
  if (device) *device = g_live_bytes[0].load();
  if (pinned) *pinned = g_live_bytes[1].load();
}

// testing aid (not in include/ilsm.h): CUDA events, streams and graph execs held by every handle of the process; makes
// no CUDA call
ILSM_API void ilsm_debug_live_handles(long long* handles) {
  if (handles) *handles = g_live_handles.load();
}

ILSM_API int ilsm_set_async(ilsm_ctx* ctx, int on) {
  if (!ctx) return fail(ILSM_ERR_INVALID_ARG, "null ctx");
  std::lock_guard<std::mutex> lk(ctx->c.mu);
  ctx->c.async_build = on != 0;
  return ILSM_OK;
}

ILSM_API int ilsm_map_create(ilsm_ctx* ctx, ilsm_map** out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "ilsm_map_create: null argument");
  ILSM_ENTER(ctx->c);
  ilsm_map* m = new (std::nothrow) ilsm_map();
  if (!m) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  int rc = m->m.init(&ctx->c);
  if (rc) {
    delete m;
    return rc;
  }
  *out = m;
  return ILSM_OK;
}

ILSM_API void ilsm_map_destroy(ilsm_map* map) {
  if (!map) return;
  std::lock_guard<std::mutex> lk(map->m.ctx->mu);
  cudaSetDevice(map->m.ctx->device);
  cudaStreamSynchronize(map->m.ctx->stream);
  delete map;
}

ILSM_API int ilsm_map_size(const ilsm_map* map) { return map ? map->m.n : 0; }

// the argument check of ilsm_map_build[_dev] (and, per map, of ilsm_map_build_pair_dev)
static int check_build_args(const ilsm_map* map, const float* xyz, int n, int stride_bytes, const char* who) {
  if (!map || (n > 0 && !xyz)) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "%s: bad n/stride", who);
  return ILSM_OK;
}

ILSM_API int ilsm_map_build_dev(ilsm_map* map, const float* d_xyz, int n, int stride_bytes, float cell) {
  int rc = check_build_args(map, d_xyz, n, stride_bytes, "ilsm_map_build_dev");
  if (rc) return rc;
  ILSM_ENTER(*map->m.ctx);
  return map->m.build_dev(d_xyz, n, stride_bytes, cell);
}

ILSM_API int ilsm_map_build_pair_dev(ilsm_map* map_a, const float* d_xyz_a, int n_a, ilsm_map* map_b, const float* d_xyz_b, int n_b,
                                     int stride_bytes, float cell) {
  int rc;
  if ((rc = check_build_args(map_a, d_xyz_a, n_a, stride_bytes, "map_build_pair_dev")) ||
      (rc = check_build_args(map_b, d_xyz_b, n_b, stride_bytes, "map_build_pair_dev")))
    return rc;
  ILSM_ENTER(*map_a->m.ctx);
  return build_pair_dev(&map_a->m, d_xyz_a, n_a, &map_b->m, d_xyz_b, n_b, stride_bytes, cell);
}

ILSM_API int ilsm_map_join(ilsm_map* map) {
  if (!map) return fail(ILSM_ERR_INVALID_ARG, "map_join: null map");
  ILSM_ENTER(*map->m.ctx);
  return map->m.wait_ready(map->m.ctx->stream);
}

ILSM_API int ilsm_map_build(ilsm_map* map, const float* xyz, int n, int stride_bytes, float cell) {
  int rc = check_build_args(map, xyz, n, stride_bytes, "ilsm_map_build");
  if (rc) return rc;
  Map& m = map->m;
  ILSM_ENTER(*m.ctx);
  size_t bytes = (size_t)n * stride_bytes;
  if ((rc = m.raw.reserve(bytes / 4 + 4))) return rc;
  // the staging buffer may still be read by users of the previous build on the context stream
  ILSM_CUDA(cudaEventRecord(m.ctx_done, m.ctx->stream));
  ILSM_CUDA(cudaStreamWaitEvent(m.stream, m.ctx_done, 0));
  if (bytes) ILSM_CUDA(cudaMemcpyAsync(m.raw.p, xyz, bytes, cudaMemcpyHostToDevice, m.stream));
  if ((rc = m.build_dev(m.raw.p, n, stride_bytes, cell))) return rc;
  if (!m.ctx->async_build) ILSM_CUDA(cudaStreamSynchronize(m.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_map_insert(ilsm_map* map, const float* xyz, int n, int stride_bytes, int policy, float leaf) {
  if (!map || (n > 0 && !xyz)) return fail(ILSM_ERR_INVALID_ARG, "ilsm_map_insert: null argument");
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "ilsm_map_insert: bad n/stride");
  Map& m = map->m;
  ILSM_ENTER(*m.ctx);
  if (m.table_size == 0) {  // Add_Points on an empty tree behaves like Build
    int rc0 = m.build_dev(nullptr, 0, 16, m.cell);
    if (rc0) return rc0;
  }
  size_t bytes = (size_t)n * stride_bytes;
  int rc;
  if ((rc = m.raw.reserve(bytes / 4 + 4))) return rc;
  ILSM_CUDA(cudaEventRecord(m.ctx_done, m.ctx->stream));
  ILSM_CUDA(cudaStreamWaitEvent(m.stream, m.ctx_done, 0));
  if (bytes) ILSM_CUDA(cudaMemcpyAsync(m.raw.p, xyz, bytes, cudaMemcpyHostToDevice, m.stream));
  if ((rc = m.insert_dev(m.raw.p, n, stride_bytes, policy, leaf))) return rc;
  ILSM_CUDA(cudaStreamSynchronize(m.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_map_points(ilsm_map* map, float* out_xyzi, int capacity, int* n_out) {
  if (!map || !n_out || (capacity > 0 && !out_xyzi)) return fail(ILSM_ERR_INVALID_ARG, "ilsm_map_points: null argument");
  Map& m = map->m;
  ILSM_ENTER(*m.ctx);
  *n_out = m.n;
  const int k = m.n < capacity ? m.n : capacity;
  if (k > 0) {
    ILSM_CUDA(cudaStreamSynchronize(m.stream));
    ILSM_CUDA(cudaMemcpy(out_xyzi, m.orig.p, (size_t)k * 16, cudaMemcpyDeviceToHost));
  }
  return ILSM_OK;
}

// the argument check of ilsm_knn[_dev]
static int check_knn_args(const ilsm_map* map, const float* q, int nq, int stride_bytes, int k, const int32_t* idx, const float* d2,
                          const char* who) {
  if (!map || (nq > 0 && (!q || !idx || !d2))) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (nq < 0 || !valid_stride(stride_bytes) || k < 1 || k > 8) return fail(ILSM_ERR_INVALID_ARG, "%s: bad nq/k/stride", who);
  return ILSM_OK;
}

ILSM_API int ilsm_knn_dev(ilsm_map* map, const float* d_q, int nq, int stride_bytes, int k, float max_dist, int32_t* d_idx,
                 float* d_d2) {
  int rc = check_knn_args(map, d_q, nq, stride_bytes, k, d_idx, d_d2, "ilsm_knn_dev");
  if (rc) return rc;
  ILSM_ENTER(*map->m.ctx);
  return map->m.knn_dev(d_q, nq, stride_bytes, k, max_dist, d_idx, d_d2);
}

ILSM_API int ilsm_knn(ilsm_map* map, const float* q, int nq, int stride_bytes, int k, float max_dist, int32_t* idx, float* d2) {
  int rc = check_knn_args(map, q, nq, stride_bytes, k, idx, d2, "ilsm_knn");
  if (rc) return rc;
  Map& m = map->m;
  Ctx& c = *m.ctx;
  ILSM_ENTER(c);
  if (nq == 0) return ILSM_OK;
  size_t bytes = (size_t)nq * stride_bytes;
  if ((rc = c.stack_raw.reserve(bytes / 4 + 4)) || (rc = c.out_idx.reserve((size_t)nq * k)) ||
      (rc = c.out_d2.reserve((size_t)nq * k)))
    return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.stack_raw.p, q, bytes, cudaMemcpyHostToDevice, c.stream));
  if ((rc = m.knn_dev(c.stack_raw.p, nq, stride_bytes, k, max_dist, c.out_idx.p, c.out_d2.p))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(idx, c.out_idx.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(d2, c.out_d2.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

// the argument check of ilsm_register[_dev], ilsm_associate[_dev] and ilsm_odometry; `has_pose`: the pose pointers
// are not null
static int check_reg_args(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* corner, int nc, const float* surf,
                          int ns, int stride_bytes, bool has_pose, const char* who) {
  if (!ctx || !mc || !ms) return fail(ILSM_ERR_INVALID_ARG, "%s: null handle", who);
  if (mc->m.ctx != &ctx->c || ms->m.ctx != &ctx->c) return fail(ILSM_ERR_INVALID_ARG, "%s: map belongs to another context", who);
  if (nc < 0 || ns < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "%s: bad counts/stride", who);
  if ((nc > 0 && !corner) || (ns > 0 && !surf)) return fail(ILSM_ERR_INVALID_ARG, "%s: null stack", who);
  if (mc->m.table_size == 0 || ms->m.table_size == 0) return fail(ILSM_ERR_STATE, "%s: map not built", who);
  if (!has_pose) return fail(ILSM_ERR_INVALID_ARG, "%s: null pose", who);
  return ILSM_OK;
}

static int check_map_size(const ilsm_reg_opts& o, const ilsm_map* mc, const ilsm_map* ms) {
  if ((o.min_corner_map > 0 && !(mc->m.n > o.min_corner_map)) || (o.min_surf_map > 0 && !(ms->m.n > o.min_surf_map)))
    return fail(ILSM_ERR_NOT_ENOUGH_MAP, "time Map corner and surf num are not enough");
  return ILSM_OK;
}

// the initial guess of a host-pointer entry point, carried by the first association launch
static PoseSrc host_pose(const double q[4], const double t[3]) {
  PoseSrc src;
  src.mode = 1;
  for (int i = 0; i < 4; ++i) src.v[i] = q[i];
  for (int i = 0; i < 3; ++i) src.v[4 + i] = t[i];
  return src;
}

// the factor records of the last association to the caller's host buffer (nullptr: none wanted), through the out_idx
// scratch (reinterpreted) to keep allocations few; the caller synchronises
static int export_factors(Ctx& c, ilsm_factor* factors) {
  const int n = c.fac.n;
  if (!factors || n == 0) return ILSM_OK;
  size_t words = ((size_t)n * sizeof(ilsm_factor) + 3) / 4;
  int rc;
  if ((rc = c.out_idx.reserve(words + 8))) return rc;
  ilsm_factor* d_f = reinterpret_cast<ilsm_factor*>(c.out_idx.p);
  if ((rc = factors_export(&c, d_f))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(factors, d_f, (size_t)n * sizeof(ilsm_factor), cudaMemcpyDeviceToHost, c.stream));
  return ILSM_OK;
}

// stage both stacks into ctx.stack_raw; returns device pointers
static int stage_stacks(Ctx& c, const float* corner, int nc, const float* surf, int ns, int stride_bytes,
                        const float** d_corner, const float** d_surf) {
  size_t bc = (size_t)nc * stride_bytes, bs = (size_t)ns * stride_bytes;
  size_t off_s = (bc + 255) & ~(size_t)255;
  int rc;
  if ((rc = c.stack_raw.reserve((off_s + bs) / 4 + 64))) return rc;
  char* base = reinterpret_cast<char*>(c.stack_raw.p);
  if (bc) ILSM_CUDA(cudaMemcpyAsync(base, corner, bc, cudaMemcpyHostToDevice, c.stream));
  if (bs) ILSM_CUDA(cudaMemcpyAsync(base + off_s, surf, bs, cudaMemcpyHostToDevice, c.stream));
  *d_corner = reinterpret_cast<const float*>(base);
  *d_surf = reinterpret_cast<const float*>(base + off_s);
  return ILSM_OK;
}

ILSM_API int ilsm_register_dev(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* d_corner, int nc, const float* d_surf,
                      int ns, int stride_bytes, double* d_pose7, const ilsm_reg_opts* opts, ilsm_reg_report* d_report) {
  int rc = check_reg_args(ctx, mc, ms, d_corner, nc, d_surf, ns, stride_bytes, d_pose7 != nullptr, "register_dev");
  if (rc) return rc;
  ilsm_reg_opts o = sanitize(opts);
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  if ((rc = check_map_size(o, mc, ms))) return rc;
  // the first association reads the pose straight from d_pose7 (and seeds the LM state), the last solve writes the
  // result and the report back: no separate pose upload / download launches
  PoseSrc src;
  src.mode = 2, src.dptr = d_pose7;
  PoseDst dst;
  dst.d_pose7 = d_pose7, dst.d_report = d_report;
  return c.register_dev(&mc->m, &ms->m, d_corner, nc, d_surf, ns, stride_bytes, o, &src, &dst);
}

ILSM_API int ilsm_associate_dev(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* d_corner, int nc,
                                const float* d_surf, int ns, int stride_bytes, const double* d_pose7,
                                const ilsm_reg_opts* opts) {
  int rc = check_reg_args(ctx, mc, ms, d_corner, nc, d_surf, ns, stride_bytes, d_pose7 != nullptr, "associate_dev");
  if (rc) return rc;
  ilsm_reg_opts o = sanitize(opts);
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  PoseSrc src;
  src.mode = 2, src.dptr = d_pose7;
  return c.associate_dev(&mc->m, &ms->m, d_corner, nc, d_surf, ns, stride_bytes, o, false, &src);
}

ILSM_API int ilsm_register(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* corner, int nc, const float* surf, int ns,
                  int stride_bytes, double q[4], double t[3], const ilsm_reg_opts* opts, ilsm_reg_report* report) {
  int rc = check_reg_args(ctx, mc, ms, corner, nc, surf, ns, stride_bytes, q && t, "register");
  if (rc) return rc;
  ilsm_reg_opts o = sanitize(opts);
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  if (report) memset(report, 0, sizeof(*report));
  if ((rc = check_map_size(o, mc, ms))) return rc;
  const float *d_corner, *d_surf;
  if ((rc = stage_stacks(c, corner, nc, surf, ns, stride_bytes, &d_corner, &d_surf))) return rc;
  const PoseSrc src = host_pose(q, t);
  if ((rc = c.register_dev(&mc->m, &ms->m, d_corner, nc, d_surf, ns, stride_bytes, o, &src, nullptr))) return rc;
  return c.lm_finish(q, t, report, o.outer_iterations);
}

// Front end + stacks + registration of one organised frame against two prebuilt maps, the frame already on the device.
// One host synchronisation in the middle (the feature counts size the VoxelGrid sorts, as in the full loop).
// min_range <= 0 takes the default 0.3 m.
static int register_frame_core(Ctx& c, Map* mc, Map* ms, const float* d_frame, int n, int stride_bytes, float min_range, float line_res,
                               float plane_res, const ilsm_reg_opts& o, const PoseSrc* src, const PoseDst* dst, int counts_out[8]) {
  int rc;
  if ((rc = c.features_dev(d_frame, n, stride_bytes, min_range > 0.f ? min_range : 0.3f))) return rc;
  int* pin = reinterpret_cast<int*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, c.fe.counts.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  for (int i = 0; i < 8; ++i) counts_out[i] = pin[i];
  if (pin[5]) return fail(ILSM_ERR_INVALID_ARG, "register_frame: a ring segment exceeds the supported size");
  const int n_lsharp = pin[2], n_lflat = pin[4];
  if ((rc = c.rf_lsharp.reserve(n_lsharp + 4)) || (rc = c.rf_stack_c.reserve(n_lsharp + 4)) || (rc = c.rf_stack_s.reserve(n_lflat + 4)) ||
      (rc = c.rf_stack_n.reserve(4)))
    return rc;
  // laserCloudCornerLast = cornerPointsLessSharp, laserCloudSurfLast = surfPointsLessFlat (laserOdometry.cpp:793-796)
  if ((rc = c.gather_dev(c.fe.cloud.p, c.fe.lsharp.p, c.fe.counts.p, 2, n_lsharp, c.rf_lsharp.p))) return rc;
  // downSizeFilterCorner / downSizeFilterSurf (laserMapping.cpp:608-616)
  ILSM_CUDA(cudaMemsetAsync(c.rf_stack_n.p, 0, 4 * sizeof(int), c.stream));
  const Ctx::VgCloud vc[2] = {{reinterpret_cast<const float*>(c.rf_lsharp.p), n_lsharp, line_res, c.rf_stack_c.p, c.rf_stack_n.p},
                              {reinterpret_cast<const float*>(c.fe.lflat.p), n_lflat, plane_res, c.rf_stack_s.p, c.rf_stack_n.p + 1}};
  if ((rc = c.voxelgrid(vc, 2, 16, 3, c.stream))) return rc;
  // the association / solve block with the stack sizes read on the device (laserMapping.cpp:640-861)
  c.d_stack_counts = c.rf_stack_n.p;
  rc = c.register_dev(mc, ms, reinterpret_cast<const float*>(c.rf_stack_c.p), n_lsharp, reinterpret_cast<const float*>(c.rf_stack_s.p), n_lflat,
                      16, o, src, dst);
  c.d_stack_counts = nullptr;
  return rc;
}

// the argument check of ilsm_register_frame[_dev], the built maps and the map-size guard included
static int check_frame_args(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* xyzi, int n, bool has_pose, int stride_bytes,
                            float line_res, float plane_res, const ilsm_reg_opts& o, const char* who) {
  if (!ctx || !mc || !ms || (n > 0 && !xyzi) || !has_pose) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (mc->m.ctx != &ctx->c || ms->m.ctx != &ctx->c) return fail(ILSM_ERR_INVALID_ARG, "%s: map belongs to another context", who);
  if (n < 0 || !valid_stride(stride_bytes) || stride_bytes < 16 || !(line_res > 0.f) || !(plane_res > 0.f))
    return fail(ILSM_ERR_INVALID_ARG, "%s: bad n/stride/resolution", who);
  if (mc->m.table_size == 0 || ms->m.table_size == 0) return fail(ILSM_ERR_STATE, "%s: map not built", who);
  return check_map_size(o, mc, ms);
}

ILSM_API int ilsm_register_frame(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* xyzi, int n, int stride_bytes, float min_range,
                                 float line_res, float plane_res, double q[4], double t[3], const ilsm_reg_opts* opts,
                                 ilsm_reg_report* report, int32_t sizes_out[4]) {
  if (report) memset(report, 0, sizeof(*report));
  const ilsm_reg_opts o = sanitize(opts);
  int rc = check_frame_args(ctx, mc, ms, xyzi, n, q && t, stride_bytes, line_res, plane_res, o, "register_frame");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const size_t bytes = (size_t)n * stride_bytes;
  if ((rc = c.fe.raw.reserve(bytes / 4 + 4))) return rc;
  if (bytes) ILSM_CUDA(cudaMemcpyAsync(c.fe.raw.p, xyzi, bytes, cudaMemcpyHostToDevice, c.stream));
  const PoseSrc src = host_pose(q, t);
  int counts[8];
  if ((rc = register_frame_core(c, &mc->m, &ms->m, c.fe.raw.p, n, stride_bytes, min_range, line_res, plane_res, o, &src, nullptr,
                                counts)))
    return rc;
  int* sn = reinterpret_cast<int*>(c.pinned.p + Ctx::kPinSite);  // the down-sampled stack sizes
  if ((rc = c.read_back_lm(c.stream))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(sn, c.rf_stack_n.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  c.lm_result(q, t, report);
  if (report) report->passes = o.outer_iterations;
  if (sizes_out) {
    sizes_out[0] = counts[2], sizes_out[1] = counts[4], sizes_out[2] = sn[0], sizes_out[3] = sn[1];
  }
  return ILSM_OK;
}

ILSM_API int ilsm_register_frame_dev(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* d_xyzi, int n, int stride_bytes,
                                     float min_range, float line_res, float plane_res, double* d_pose7, const ilsm_reg_opts* opts) {
  const ilsm_reg_opts o = sanitize(opts);
  int rc = check_frame_args(ctx, mc, ms, d_xyzi, n, d_pose7 != nullptr, stride_bytes, line_res, plane_res, o, "register_frame_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  PoseSrc src;
  src.mode = 2, src.dptr = d_pose7;
  PoseDst dst;
  dst.d_pose7 = d_pose7;
  int counts[8];
  return register_frame_core(c, &mc->m, &ms->m, d_xyzi, n, stride_bytes, min_range, line_res, plane_res, o, &src, &dst, counts);
}

ILSM_API int ilsm_associate(ilsm_ctx* ctx, ilsm_map* mc, ilsm_map* ms, const float* corner, int nc, const float* surf, int ns,
                   int stride_bytes, const double q[4], const double t[3], const ilsm_reg_opts* opts,
                   ilsm_factor* factors, int32_t* knn_idx, float* knn_d2) {
  int rc = check_reg_args(ctx, mc, ms, corner, nc, surf, ns, stride_bytes, q && t, "associate");
  if (rc) return rc;
  ilsm_reg_opts o = sanitize(opts);
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const float *d_corner, *d_surf;
  if ((rc = stage_stacks(c, corner, nc, surf, ns, stride_bytes, &d_corner, &d_surf))) return rc;
  if ((rc = c.upload_pose(q, t, c.stream))) return rc;
  const bool want_knn = knn_idx != nullptr && knn_d2 != nullptr;
  if ((rc = c.associate_dev(&mc->m, &ms->m, d_corner, nc, d_surf, ns, stride_bytes, o, want_knn)) || (rc = export_factors(c, factors)))
    return rc;
  const int n = nc + ns;
  if (want_knn && n > 0) {
    ILSM_CUDA(cudaMemcpyAsync(knn_idx, c.fac.knn_idx.p, (size_t)n * 5 * 4, cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaMemcpyAsync(knn_d2, c.fac.knn_d2.p, (size_t)n * 5 * 4, cudaMemcpyDeviceToHost, c.stream));
  }
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

// ------------------------------------------------------------------------------------------------ odometry
ILSM_API int ilsm_odometry(ilsm_ctx* ctx, ilsm_map* last_corner, ilsm_map* last_surf, const float* sharp, int nsh,
                           const float* flat, int nfl, int stride_bytes, double q[4], double t[3],
                           const ilsm_reg_opts* opts, ilsm_reg_report* report, ilsm_factor* factors) {
  int rc = check_reg_args(ctx, last_corner, last_surf, sharp, nsh, flat, nfl, stride_bytes, q && t, "odometry");
  if (rc) return rc;
  ilsm_reg_opts o = sanitize(opts);
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  if (report) memset(report, 0, sizeof(*report));
  const float *d_sharp, *d_flat;
  if ((rc = stage_stacks(c, sharp, nsh, flat, nfl, stride_bytes, &d_sharp, &d_flat))) return rc;
  if ((rc = c.upload_pose(q, t, c.stream))) return rc;
  if (factors) {
    // association only at the given pose (parity aid): export the factor records, no solve
    if ((rc = c.odom_associate_dev(&last_corner->m, &last_surf->m, d_sharp, nsh, d_flat, nfl, stride_bytes)) ||
        (rc = export_factors(c, factors)))
      return rc;
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
    return ILSM_OK;
  }
  if ((rc = c.odometry_dev(&last_corner->m, &last_surf->m, d_sharp, nsh, d_flat, nfl, stride_bytes, o))) return rc;
  return c.lm_finish(q, t, report, o.outer_iterations);
}

// ------------------------------------------------------------------------------------------------ front end
// the argument check of ilsm_project[_dev]
static int check_project_args(const ilsm_ctx* ctx, const float* xyzi, int H, int W, int stride_bytes, const uint8_t* range_img,
                              const uint8_t* inten_img, const float* track, const char* who) {
  if (!ctx || !xyzi || !range_img || !inten_img || !track) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (H <= 0 || W <= 0 || !valid_stride(stride_bytes) || stride_bytes < 16) return fail(ILSM_ERR_INVALID_ARG, "%s: bad H/W/stride", who);
  return ILSM_OK;
}

ILSM_API int ilsm_project(ilsm_ctx* ctx, const float* xyzi, int H, int W, int stride_bytes, uint8_t* range_img,
                          uint8_t* inten_img, float* cloud_track_xyzi) {
  int rc = check_project_args(ctx, xyzi, H, W, stride_bytes, range_img, inten_img, cloud_track_xyzi, "project");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const int n = H * W;
  const size_t bytes = (size_t)n * stride_bytes;
  if ((rc = c.fe.raw.reserve(bytes / 4 + 4)) || (rc = c.fe.img.reserve((size_t)2 * n + 8)) || (rc = c.fe.track.reserve(n + 4)))
    return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.fe.raw.p, xyzi, bytes, cudaMemcpyHostToDevice, c.stream));
  unsigned char* d_r = c.fe.img.p;
  unsigned char* d_i = c.fe.img.p + (((size_t)n + 3) & ~(size_t)3);
  if ((rc = c.project_dev(c.fe.raw.p, n, stride_bytes, d_r, d_i, reinterpret_cast<float*>(c.fe.track.p)))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(range_img, d_r, n, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(inten_img, d_i, n, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(cloud_track_xyzi, c.fe.track.p, (size_t)n * 16, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_project_dev(ilsm_ctx* ctx, const float* d_xyzi, int H, int W, int stride_bytes, uint8_t* d_range_img,
                              uint8_t* d_inten_img, float* d_cloud_track_xyzi) {
  int rc = check_project_args(ctx, d_xyzi, H, W, stride_bytes, d_range_img, d_inten_img, d_cloud_track_xyzi, "project_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  return c.project_dev(d_xyzi, H * W, stride_bytes, d_range_img, d_inten_img, d_cloud_track_xyzi);
}

ILSM_API int ilsm_host_register(void* ptr, size_t bytes) {
  if (!ptr || bytes == 0) return fail(ILSM_ERR_INVALID_ARG, "host_register: null / empty buffer");
  ILSM_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
  return ILSM_OK;
}
ILSM_API int ilsm_host_unregister(void* ptr) {
  if (!ptr) return fail(ILSM_ERR_INVALID_ARG, "host_unregister: null buffer");
  ILSM_CUDA(cudaHostUnregister(ptr));
  return ILSM_OK;
}

ILSM_API void ilsm_pc2_layout_ouster(ilsm_pc2_layout* l) {
  if (!l) return;
  memset(l, 0, sizeof(*l));
  l->point_step = 48, l->off_x = 0, l->off_y = 4, l->off_z = 8, l->off_intensity = 16, l->intensity_datatype = 7;
}

}  // extern "C"
namespace ilsm {
int check_pc2_layout(const ilsm_pc2_layout* l) {
  if (!l) return fail(ILSM_ERR_INVALID_ARG, "pc2: null layout");
  if (l->is_bigendian) return fail(ILSM_ERR_INVALID_ARG, "pc2: big-endian blobs are not supported");
  const int ps = l->point_step;
  auto in = [ps](int off, int size) { return off >= 0 && off + size <= ps; };
  if (ps < 12 || !in(l->off_x, 4) || !in(l->off_y, 4) || !in(l->off_z, 4)) return fail(ILSM_ERR_INVALID_ARG, "pc2: bad point_step / xyz offsets");
  if (l->off_intensity >= 0) {
    int sz = 0;
    switch (l->intensity_datatype) {
      case 2: sz = 1; break;
      case 4: sz = 2; break;
      case 6: case 7: sz = 4; break;
      case 8: sz = 8; break;
      default: return fail(ILSM_ERR_INVALID_ARG, "pc2: unsupported intensity datatype");
    }
    if (!in(l->off_intensity, sz)) return fail(ILSM_ERR_INVALID_ARG, "pc2: bad intensity offset");
  }
  return ILSM_OK;
}
}  // namespace ilsm
extern "C" {

ILSM_API void ilsm_pc2_layout_pcl_xyzi(ilsm_pc2_layout* l) {
  if (!l) return;
  memset(l, 0, sizeof(*l));
  l->point_step = 32, l->off_x = 0, l->off_y = 4, l->off_z = 8, l->off_intensity = 16, l->intensity_datatype = 7;
}

// a layout a blob can be WRITTEN with: FLOAT32 fields on 4-byte offsets that do not overlap
static int check_pc2_pack_layout(const ilsm_pc2_layout* l) {
  int rc = check_pc2_layout(l);
  if (rc) return rc;
  if (l->point_step % 4 || l->off_x % 4 || l->off_y % 4 || l->off_z % 4) return fail(ILSM_ERR_INVALID_ARG, "pc2_pack: fields must sit on 4-byte offsets");
  if (l->off_intensity >= 0 && (l->intensity_datatype != 7 || l->off_intensity % 4))
    return fail(ILSM_ERR_INVALID_ARG, "pc2_pack: intensity is written as FLOAT32 on a 4-byte offset");
  const int o[4] = {l->off_x, l->off_y, l->off_z, l->off_intensity};
  for (int a = 0; a < 4; ++a)
    for (int b = a + 1; b < 4; ++b)
      if (o[a] >= 0 && o[a] == o[b]) return fail(ILSM_ERR_INVALID_ARG, "pc2_pack: overlapping fields");
  return ILSM_OK;
}

// the argument check of ilsm_pc2_pack[_dev] (`pack`: the layout must be writable) and ilsm_pc2_unpack[_dev]
static int check_pc2_args(const ilsm_ctx* ctx, const void* in, int n_points, const ilsm_pc2_layout* layout, const void* out, bool pack,
                          const char* who) {
  if (!ctx || (n_points > 0 && (!in || !out))) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (n_points < 0) return fail(ILSM_ERR_INVALID_ARG, "%s: bad n_points", who);
  return pack ? check_pc2_pack_layout(layout) : check_pc2_layout(layout);
}

ILSM_API int ilsm_pc2_pack_dev(ilsm_ctx* ctx, const float* d_xyzi, int n_points, const ilsm_pc2_layout* layout, uint8_t* d_data_out) {
  int rc = check_pc2_args(ctx, d_xyzi, n_points, layout, d_data_out, true, "pc2_pack_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  return c.pc2_pack_dev(reinterpret_cast<const float4*>(d_xyzi), n_points, *layout, d_data_out);
}

ILSM_API int ilsm_pc2_pack(ilsm_ctx* ctx, const float* xyzi, int n_points, const ilsm_pc2_layout* layout, uint8_t* data_out) {
  int rc = check_pc2_args(ctx, xyzi, n_points, layout, data_out, true, "pc2_pack");
  if (rc) return rc;
  if (n_points == 0) return ILSM_OK;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const size_t bytes = (size_t)n_points * layout->point_step;
  if ((rc = c.fe.pc2.reserve(bytes + 16)) || (rc = c.fe.raw.reserve((size_t)n_points * 4 + 4))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.fe.raw.p, xyzi, (size_t)n_points * 16, cudaMemcpyHostToDevice, c.stream));
  if ((rc = c.pc2_pack_dev(reinterpret_cast<const float4*>(c.fe.raw.p), n_points, *layout, c.fe.pc2.p))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(data_out, c.fe.pc2.p, bytes, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_pc2_unpack_dev(ilsm_ctx* ctx, const uint8_t* d_data, int n_points, const ilsm_pc2_layout* layout, float* d_out_xyzi) {
  int rc = check_pc2_args(ctx, d_data, n_points, layout, d_out_xyzi, false, "pc2_unpack_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  return c.pc2_unpack_dev(d_data, n_points, *layout, reinterpret_cast<float4*>(d_out_xyzi));
}

ILSM_API int ilsm_pc2_unpack(ilsm_ctx* ctx, const uint8_t* data, int n_points, const ilsm_pc2_layout* layout, float* out_xyzi) {
  int rc = check_pc2_args(ctx, data, n_points, layout, out_xyzi, false, "pc2_unpack");
  if (rc) return rc;
  if (n_points == 0) return ILSM_OK;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const size_t bytes = (size_t)n_points * layout->point_step;
  if ((rc = c.fe.pc2.reserve(bytes + 16)) || (rc = c.fe.raw.reserve((size_t)n_points * 4 + 4))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.fe.pc2.p, data, bytes, cudaMemcpyHostToDevice, c.stream));
  if ((rc = c.pc2_unpack_dev(c.fe.pc2.p, n_points, *layout, reinterpret_cast<float4*>(c.fe.raw.p)))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(out_xyzi, c.fe.raw.p, (size_t)n_points * 16, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_extract_features(ilsm_ctx* ctx, const float* xyzi, int n, int stride_bytes, float min_range,
                                   ilsm_features* out) {
  if (!ctx || !out || (n > 0 && !xyzi)) return fail(ILSM_ERR_INVALID_ARG, "extract_features: null argument");
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "extract_features: bad n/stride");
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const size_t bytes = (size_t)n * stride_bytes;
  int rc;
  if ((rc = c.fe.raw.reserve(bytes / 4 + 4))) return rc;
  if (bytes) ILSM_CUDA(cudaMemcpyAsync(c.fe.raw.p, xyzi, bytes, cudaMemcpyHostToDevice, c.stream));
  if ((rc = c.features_dev(c.fe.raw.p, n, stride_bytes, min_range))) return rc;
  // counts + ring histogram first, then exactly the produced amounts
  int* pin = reinterpret_cast<int*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, c.fe.counts.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(pin + 8, c.fe.stats.p + 4, 64 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  ilsm_feature_counts& k = out->counts;
  memset(&k, 0, sizeof(k));
  k.n_cloud = pin[0], k.n_sharp = pin[1], k.n_less_sharp = pin[2], k.n_flat = pin[3], k.n_less_flat = pin[4];
  k.flags = pin[5];
  int off = 0;
  for (int r = 0; r < 64; ++r) {
    k.ring_start[r] = off + 5;
    off += pin[8 + r];
    k.ring_end[r] = off - 6;
  }
  if (k.flags) return fail(ILSM_ERR_INVALID_ARG, "extract_features: a ring segment exceeds the supported size");
  const int N = k.n_cloud;
  auto d2h = [&](void* dst, const void* src, size_t nbytes) -> cudaError_t {
    if (!dst || nbytes == 0) return cudaSuccess;
    return cudaMemcpyAsync(dst, src, nbytes, cudaMemcpyDeviceToHost, c.stream);
  };
  ILSM_CUDA(d2h(out->cloud_xyzi, c.fe.cloud.p, (size_t)N * 16));
  ILSM_CUDA(d2h(out->curvature, c.fe.curv.p, (size_t)N * 4));
  ILSM_CUDA(d2h(out->label, c.fe.label.p, (size_t)N * 4));
  ILSM_CUDA(d2h(out->src_index, c.fe.src_index.p, (size_t)N * 4));
  ILSM_CUDA(d2h(out->sharp_idx, c.fe.sharp.p, (size_t)k.n_sharp * 4));
  ILSM_CUDA(d2h(out->less_sharp_idx, c.fe.lsharp.p, (size_t)k.n_less_sharp * 4));
  ILSM_CUDA(d2h(out->flat_idx, c.fe.flat.p, (size_t)k.n_flat * 4));
  ILSM_CUDA(d2h(out->less_flat_xyzi, c.fe.lflat.p, (size_t)k.n_less_flat * 16));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_voxelgrid(ilsm_ctx* ctx, const float* xyzi, int n, int stride_bytes, float leaf, float* out_xyzi,
                            int* n_out) {
  if (!ctx || !n_out || (n > 0 && (!xyzi || !out_xyzi))) return fail(ILSM_ERR_INVALID_ARG, "voxelgrid: null argument");
  if (n < 0 || !valid_stride(stride_bytes) || stride_bytes < 16 || !(leaf > 0.f)) return fail(ILSM_ERR_INVALID_ARG, "voxelgrid: bad n/stride/leaf");
  *n_out = 0;
  if (n == 0) return ILSM_OK;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  const size_t bytes = (size_t)n * stride_bytes;
  int rc;
  if ((rc = c.fe.raw.reserve(bytes / 4 + 4)) || (rc = c.fe.vox_out.reserve(n + 4)) || (rc = c.fe.vox_n.reserve(4))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.fe.raw.p, xyzi, bytes, cudaMemcpyHostToDevice, c.stream));
  const Ctx::VgCloud vc = {c.fe.raw.p, n, leaf, c.fe.vox_out.p, c.fe.vox_n.p};
  if ((rc = c.voxelgrid(&vc, 1, stride_bytes, intensity_word(stride_bytes), c.stream))) return rc;
  int* pin = reinterpret_cast<int*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, c.fe.vox_n.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  *n_out = pin[0];
  if (pin[0] > 0) {
    ILSM_CUDA(cudaMemcpyAsync(out_xyzi, c.fe.vox_out.p, (size_t)pin[0] * 16, cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
  }
  return ILSM_OK;
}

// ------------------------------------------------------------------------------------------------ ScanContext
ILSM_API int ilsm_sc_create(ilsm_ctx* ctx, ilsm_sc** out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "sc_create: null argument");
  ilsm_sc* h = new (std::nothrow) ilsm_sc();
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  h->d.ctx = &ctx->c;
  *out = h;
  return ILSM_OK;
}

ILSM_API void ilsm_sc_destroy(ilsm_sc* sc) {
  if (!sc) return;
  std::lock_guard<std::mutex> lk(sc->d.ctx->mu);
  cudaSetDevice(sc->d.ctx->device);
  cudaStreamSynchronize(sc->d.ctx->stream);
  sc_nccl_release(sc->d);
  delete sc;
}

ILSM_API int ilsm_sc_size(const ilsm_sc* sc) { return sc ? sc->d.count : 0; }

ILSM_API int ilsm_sc_make(ilsm_sc* sc, const float* xyz, int n, int stride_bytes, float* desc_20x60) {
  if (!sc || !desc_20x60 || (n > 0 && !xyz)) return fail(ILSM_ERR_INVALID_ARG, "sc_make: null argument");
  if (n < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "sc_make: bad n/stride");
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  ILSM_ENTER(c);
  const size_t words = (size_t)n * stride_bytes / 4;
  int rc;
  if ((rc = d.stage.reserve(words + 1200 + 8))) return rc;
  float* d_desc = d.stage.p;
  float* d_pts = d.stage.p + 1200;
  if (n) ILSM_CUDA(cudaMemcpyAsync(d_pts, xyz, (size_t)n * stride_bytes, cudaMemcpyHostToDevice, c.stream));
  if ((rc = d.make_dev(d_pts, n, stride_bytes, d_desc))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(desc_20x60, d_desc, 1200 * sizeof(float), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

// the argument check of ilsm_sc_add[_dev]
static int check_sc_add_args(const ilsm_sc* sc, const float* desc, int count, const char* who) {
  if (!sc || (count > 0 && !desc) || count < 0) return fail(ILSM_ERR_INVALID_ARG, "%s: bad argument", who);
  return ILSM_OK;
}

ILSM_API int ilsm_sc_add(ilsm_sc* sc, const float* desc_20x60, int count) {
  int rc = check_sc_add_args(sc, desc_20x60, count, "sc_add");
  if (rc) return rc;
  Ctx& c = *sc->d.ctx;
  ILSM_ENTER(c);
  if ((rc = sc->d.append_dev(desc_20x60, count, true))) return rc;
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

ILSM_API int ilsm_sc_add_dev(ilsm_sc* sc, const float* d_desc_20x60, int count) {
  int rc = check_sc_add_args(sc, d_desc_20x60, count, "sc_add_dev");
  if (rc) return rc;
  Ctx& c = *sc->d.ctx;
  ILSM_ENTER(c);
  return sc->d.append_dev(d_desc_20x60, count, false);
}

// the argument check of ilsm_sc_query_topk[_dev]; n_search is checked against the database by ScDb::query_dev
static int check_sc_query_args(const ilsm_sc* sc, const float* desc, int k, const double* dist, const int32_t* id, const int32_t* shift,
                               const char* who) {
  if (!sc || !desc || !dist || !id || !shift) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  if (k < 1 || k > 16) return fail(ILSM_ERR_INVALID_ARG, "%s: k must be in [1,16]", who);
  return ILSM_OK;
}

ILSM_API int ilsm_sc_query_topk_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_search, int id_offset, int k,
                                    double* d_dist, int32_t* d_id, int32_t* d_shift) {
  int rc = check_sc_query_args(sc, d_desc_20x60, k, d_dist, d_id, d_shift, "sc_query_dev");
  if (rc) return rc;
  Ctx& c = *sc->d.ctx;
  ILSM_ENTER(c);
  return sc->d.query_dev(d_desc_20x60, n_search, id_offset, k, d_dist, d_id, d_shift);
}

ILSM_API int ilsm_sc_query_topk(ilsm_sc* sc, const float* desc_20x60, int n_search, int id_offset, int k, double* dist,
                                int32_t* id, int32_t* shift) {
  int rc = check_sc_query_args(sc, desc_20x60, k, dist, id, shift, "sc_query");
  if (rc) return rc;
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  ILSM_ENTER(c);
  if ((rc = d.stage.reserve(1200 + 8)) || (rc = d.out_dist.reserve(16)) || (rc = d.out_id.reserve(16)) ||
      (rc = d.out_shift.reserve(16)))
    return rc;
  ILSM_CUDA(cudaMemcpyAsync(d.stage.p, desc_20x60, 1200 * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  if ((rc = d.query_dev(d.stage.p, n_search, id_offset, k, d.out_dist.p, d.out_id.p, d.out_shift.p))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(dist, d.out_dist.p, k * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(id, d.out_id.p, k * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaMemcpyAsync(shift, d.out_shift.p, k * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  return ILSM_OK;
}

// Deterministic merge of per-shard top-k lists (what every rank does after the all-gather): ascending
// (distance, id); entries with id < 0 are padding.  Pure host code, no device work.
ILSM_API int ilsm_sc_merge_topk(const double* dist, const int32_t* id, const int32_t* shift, int n_entries, int k,
                                double* out_dist, int32_t* out_id, int32_t* out_shift) {
  if (!dist || !id || !shift || !out_dist || !out_id || !out_shift || n_entries < 0 || k < 1)
    return fail(ILSM_ERR_INVALID_ARG, "sc_merge: bad argument");
  for (int j = 0; j < k; ++j) {
    int best = -1;
    for (int i = 0; i < n_entries; ++i) {
      if (id[i] < 0) continue;
      bool taken = false;
      for (int t = 0; t < j; ++t) taken = taken || out_id[t] == id[i];
      if (taken) continue;
      if (best < 0 || dist[i] < dist[best] || (dist[i] == dist[best] && id[i] < id[best])) best = i;
    }
    if (best < 0) {
      out_dist[j] = 1.0 / 0.0, out_id[j] = -1, out_shift[j] = 0;
    } else {
      out_dist[j] = dist[best], out_id[j] = id[best], out_shift[j] = shift[best];
    }
  }
  return ILSM_OK;
}

ILSM_API int ilsm_sc_merge_topk_dev(ilsm_sc* sc, const void* d_packed, int shards, int k, void* d_out_packed) {
  if (!sc || !d_packed || !d_out_packed || shards < 1 || k < 1 || k > 16)
    return fail(ILSM_ERR_INVALID_ARG, "sc_merge_dev: bad argument");
  Ctx& c = *sc->d.ctx;
  ILSM_ENTER(c);
  return sc_merge_dev(&c, d_packed, shards, k, d_out_packed);
}

// the argument check of ilsm_eval_normal_eq[_dev] and ilsm_solve[_dev]; `have`: every pointer the form needs is set
static int check_lm_args(const ilsm_ctx* ctx, bool have, const char* who) {
  if (!ctx || !have) return fail(ILSM_ERR_INVALID_ARG, "%s: null argument", who);
  return ILSM_OK;
}

ILSM_API int ilsm_eval_normal_eq(ilsm_ctx* ctx, const double q[4], const double t[3], double huber_a, double* cost, double JtJ[36],
                        double Jtr[6]) {
  int rc = check_lm_args(ctx, q && t && cost && JtJ && Jtr, "eval");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  // the pose is evaluated where upload_pose leaves it (xq, xt: 7 contiguous doubles); the 32 sums go to out_d2 scratch
  if ((rc = c.upload_pose(q, t, c.stream)) || (rc = c.out_d2.reserve(128))) return rc;
  double* d_out = reinterpret_cast<double*>(c.out_d2.p);
  if ((rc = eval_only_launch(&c, d_out, c.lm.p->xq, huber_a))) return rc;
  double* pin = reinterpret_cast<double*>(c.pinned.p);
  ILSM_CUDA(cudaMemcpyAsync(pin, d_out, 32 * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  *cost = pin[0];
  int k = 1;
  for (int a = 0; a < 6; ++a)
    for (int b = a; b < 6; ++b) {
      JtJ[a * 6 + b] = pin[k];
      JtJ[b * 6 + a] = pin[k];
      ++k;
    }
  for (int a = 0; a < 6; ++a) Jtr[a] = pin[22 + a];
  return ILSM_OK;
}

ILSM_API int ilsm_eval_normal_eq_dev(ilsm_ctx* ctx, const double* d_pose7, double huber_a, double* d_out32) {
  int rc = check_lm_args(ctx, d_pose7 && d_out32, "eval_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  return eval_only_launch(&c, d_out32, d_pose7, huber_a);  // the kernel reads the pose straight from d_pose7
}

ILSM_API int ilsm_solve_dev(ilsm_ctx* ctx, const double* d_pose7_in, int max_num_iterations, double huber_a) {
  int rc = check_lm_args(ctx, true, "solve_dev");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  if (d_pose7_in) {
    PoseSrc src;
    src.mode = 2, src.dptr = d_pose7_in;
    if ((rc = c.seed_pose(src))) return rc;
  }
  return c.solve_launch(clamp_iterations(max_num_iterations), huber_a, 0);
}

ILSM_API int ilsm_solve(ilsm_ctx* ctx, double q[4], double t[3], int max_num_iterations, double huber_a,
               ilsm_solve_summary* summary) {
  int rc = check_lm_args(ctx, q && t, "solve");
  if (rc) return rc;
  Ctx& c = ctx->c;
  ILSM_ENTER(c);
  ilsm_reg_report rep;
  if ((rc = c.upload_pose(q, t, c.stream)) || (rc = c.solve_launch(clamp_iterations(max_num_iterations), huber_a, 0)) || (rc = c.lm_finish(q, t, &rep, 1)))
    return rc;
  if (summary) *summary = rep.pass[0];
  return ILSM_OK;
}

}  // extern "C"
