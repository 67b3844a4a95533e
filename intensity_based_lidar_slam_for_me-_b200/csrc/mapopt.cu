// mapopt.cu -- the mapping node spot.launch actually starts (`<project>_mapping_node`, mapOptimization.cpp): one
// mapOptimizationCallback iteration per frame with every cloud resident on the GPU.
//
//   groundPlaneExtraction(frame)                      mapOptimization.cpp:136   -> ground_extract_core (ground.cu)
//   GroundPointOut += pc_plane ; removeNaN            :147-151                  -> pack kernel (non-finite points dropped
//                                                                                  by the VoxelGrid / build kernels)
//   first callback: ikdtree->Build(transformed cloud) :186-195                  -> Map::build_dev
//   voxel_grid_(0.8).filter(GroundPointOut)           :368-370, 578             -> Ctx::voxelgrid
//   Nearest_Search(5) + plane fit + LidarPlaneNormFactor, Solve (10 it.)  :377-442  -> Ctx::register_dev (planes only)
//   CONVERGENCE gate: transformUpdate / keyframe pose :448-457                  -> host (pose algebra)
//   ikdtree->Add_Points(transformed cloud, true)      :471-475                  -> Map::insert_dev (0.4 m boxes)
// The corner tree of the reference is write-only (never queried, SURVEY 8c) and is not maintained.
#include <string.h>

#include <new>

#include "ilsm_cubemap.hpp"

struct ilsm_ground;
namespace ilsm {
int ground_extract_core(ilsm_ground* g, const float* xyz, bool from_host, int n, int stride_bytes, const ilsm_ground_opts& o,
                        int* n_out, float coeff_abcd[4], ilsm_ground_info* info);
const float4* ground_points_dev(ilsm_ground* g);

// dst[off + i] = {x, y, z, 0} of a strided cloud
__global__ void mo_pack_kernel(const float* __restrict__ in, int n, int stride_f, float4* __restrict__ dst) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = in + (size_t)i * stride_f;
  dst[i] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), 0.f);
}

struct Mat34 {
  double r[3][3], t[3];
};
// pcl::transformPointCloud(cloud, out, Eigen::Matrix4d): double math, float store, rows summed left to right
__global__ void mo_transform_kernel(const float4* __restrict__ in, const int* __restrict__ n_ptr, int n_host, Mat34 T,
                                    float4* __restrict__ out) {
  pdl_entry();
  const int n = n_ptr ? *n_ptr : n_host;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = in[i];
  const double x = p.x, y = p.y, z = p.z;
  float o[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    o[a] = __double2float_rn(dadd(dadd(dadd(dmul(T.r[a][0], x), dmul(T.r[a][1], y)), dmul(T.r[a][2], z)), T.t[a]));
  out[i] = make_float4(o[0], o[1], o[2], 0.f);
}

struct MapOptH {
  Ctx* ctx = nullptr;
  ilsm_ground* ground = nullptr;
  Map map, empty;            // ikdtree (ground map); `empty` stands in for the unused corner map of register_dev
  bool built = false;        // first callback only builds the tree (mapOptimization.cpp:173-196)
  float leaf = 0.8f, ds = 0.4f;
  QuatH q_wmap_wodom{0, 0, 0, 1};
  double t_wmap_wodom[3] = {0, 0, 0};
  DevBuf<float4> merged, stack, world;
  DevBuf<float> plane_raw;
  DevBuf<int> counts;  // {0, n_stack}: the device-side stack sizes register_dev reads
};

// Eigen::Quaterniond::toRotationMatrix()
static void quat_to_mat_h(const QuatH& q, double R[3][3]) {
  const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const double txx = tx * q.x, txy = ty * q.x, txz = tz * q.x, tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  R[0][0] = 1 - (tyy + tzz), R[0][1] = txy - twz, R[0][2] = txz + twy;
  R[1][0] = txy + twz, R[1][1] = 1 - (txx + tzz), R[1][2] = tyz - twx;
  R[2][0] = txz - twy, R[2][1] = tyz + twx, R[2][2] = 1 - (txx + tyy);
}

}  // namespace ilsm

using namespace ilsm;

struct ilsm_mapopt {
  MapOptH m;
};

extern "C" {

ILSM_API int ilsm_mapopt_create(ilsm_ctx* ctx, float voxel_leaf, float downsample_size, ilsm_mapopt** out) {
  if (!ctx || !out) return fail(ILSM_ERR_INVALID_ARG, "mapopt_create: null argument");
  ilsm_mapopt* h = new (std::nothrow) ilsm_mapopt();
  if (!h) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
  MapOptH& m = h->m;
  m.ctx = &ctx->c;
  m.leaf = voxel_leaf > 0.f ? voxel_leaf : 0.8f;   // voxel_grid_.setLeafSize(0.8)  mapOptimization.cpp:578
  m.ds = downsample_size > 0.f ? downsample_size : 0.4f;  // KD_TREE(0.3, 0.6, 0.4)  :504
  int rc = ilsm_ground_create(ctx, &m.ground);
  if (rc == ILSM_OK) {
    CtxGuard g(ctx->c);
    if (!(rc = g.rc) && !(rc = m.map.init(&ctx->c))) rc = m.empty.init(&ctx->c);
    // the stand-in corner map must be a valid (empty) structure: the association kernel reads its bounding box
    if (!rc) rc = m.empty.build_dev(nullptr, 0, 16, 0.f);
    if (!rc) rc = m.empty.wait_ready(ctx->c.stream);
    if (!rc && cudaStreamSynchronize(ctx->c.stream) != cudaSuccess) rc = fail(ILSM_ERR_CUDA, "mapopt_create: sync failed");
  }
  if (rc) {
    if (m.ground) ilsm_ground_destroy(m.ground);
    delete h;
    return rc;
  }
  *out = h;
  return ILSM_OK;
}

ILSM_API void ilsm_mapopt_destroy(ilsm_mapopt* mo) {
  if (!mo) return;
  ilsm_ground* ground = mo->m.ground;
  {
    Ctx& c = *mo->m.ctx;
    std::lock_guard<std::mutex> lk(c.mu);
    cudaSetDevice(c.device);
    cudaStreamSynchronize(c.stream);
    delete mo;
  }
  ilsm_ground_destroy(ground);  // takes the context's mutex itself
}

ILSM_API int ilsm_mapopt_map_size(const ilsm_mapopt* mo) { return mo ? mo->m.map.n : 0; }

ILSM_API int ilsm_mapopt_map_points(ilsm_mapopt* mo, float* out_xyzi, int capacity, int* n_out) {
  if (!mo || !n_out) return fail(ILSM_ERR_INVALID_ARG, "mapopt_map_points: null argument");
  MapOptH& m = mo->m;
  ILSM_ENTER(*m.ctx);
  *n_out = m.map.n;
  const int k = m.map.n < capacity ? m.map.n : capacity;
  if (k > 0 && out_xyzi) {
    int rc = m.map.wait_ready(m.ctx->stream);
    if (rc) return rc;
    ILSM_CUDA(cudaMemcpyAsync(out_xyzi, m.map.orig.p, (size_t)k * 16, cudaMemcpyDeviceToHost, m.ctx->stream));
    ILSM_CUDA(cudaStreamSynchronize(m.ctx->stream));
  }
  return ILSM_OK;
}

}  // extern "C"

namespace ilsm {
// one callback iteration; frame / plane clouds on the host (from_host) or already on the device.  Caller holds the mutex.
int mapopt_frame_core(ilsm_mapopt* mo, const float* frame_xyz, int n, int stride_bytes, const float* plane_xyz, int n_plane,
                      int plane_stride_bytes, bool from_host, const double q_wodom[4], const double t_wodom[3], double q_w[4],
                      double t_w[3], const ilsm_ground_opts* gopts, ilsm_mapopt_stats* stats) {
  MapOptH& m = mo->m;
  Ctx& c = *m.ctx;
  if (stats) memset(stats, 0, sizeof(*stats));
  ilsm_ground_opts go;
  if (gopts) go = *gopts; else ilsm_ground_opts_default(&go);
  if (go.max_iterations < 1 || go.max_iterations > 62) return fail(ILSM_ERR_INVALID_ARG, "mapopt_frame: max_iterations must be in [1, 62]");
  int rc, n_ground = 0;
  ilsm_ground_info ginfo;
  float coeff[4];
  if ((rc = ground_extract_core(m.ground, frame_xyz, from_host, n, stride_bytes, go, &n_ground, coeff, &ginfo))) return rc;
  // GroundPointOut += pc_plane
  const int n_all = n_ground + n_plane;
  const size_t pbytes = (size_t)n_plane * plane_stride_bytes;
  if ((rc = m.merged.reserve(n_all + 4)) || (rc = m.stack.reserve(n_all + 4)) || (rc = m.world.reserve(n_all + 4)) ||
      (rc = m.plane_raw.reserve(pbytes / 4 + 4)) || (rc = m.counts.reserve(4)))
    return rc;
  cudaStream_t s = c.stream;
  if (n_ground > 0)
    ILSM_CUDA(cudaMemcpyAsync(m.merged.p, ground_points_dev(m.ground), (size_t)n_ground * 16, cudaMemcpyDeviceToDevice, s));
  if (n_plane > 0) {
    const float* d_plane = plane_xyz;
    if (from_host) {
      ILSM_CUDA(cudaMemcpyAsync(m.plane_raw.p, plane_xyz, pbytes, cudaMemcpyHostToDevice, s));
      d_plane = m.plane_raw.p;
    }
    ILSM_CUDA(launch_pdl(mo_pack_kernel, dim3((n_plane + 255) / 256), dim3(256), 0, s, d_plane, n_plane, plane_stride_bytes / 4,
                         m.merged.p + n_ground));
    count_launches(1);
  }
  // transformAssociateToMap (mapOptimization.cpp:730-735)
  const QuatH qo{q_wodom[0], q_wodom[1], q_wodom[2], q_wodom[3]};
  QuatH qw = qmul_h(m.q_wmap_wodom, qo);
  double tw[3], r[3];
  qrot_h(m.q_wmap_wodom, t_wodom, r);
  for (int i = 0; i < 3; ++i) tw[i] = r[i] + m.t_wmap_wodom[i];
  if (stats) {
    stats->ground = ginfo;
    stats->n_ground = n_ground, stats->n_plane_in = n_plane;
    for (int i = 0; i < 4; ++i) stats->ground_coeff[i] = coeff[i];
  }
  Mat34 T;
  if (!m.built) {
    // first callback: Build from the un-downsampled cloud at the predicted pose, no solve (:173-196)
    quat_to_mat_h(qw, T.r);
    for (int i = 0; i < 3; ++i) T.t[i] = tw[i];
    if (n_all > 0) {
      ILSM_CUDA(launch_pdl(mo_transform_kernel, dim3((n_all + 255) / 256), dim3(256), 0, s, (const float4*)m.merged.p,
                           (const int*)nullptr, n_all, T, m.world.p));
      count_launches(1);
    }
    if ((rc = m.map.build_dev(reinterpret_cast<const float*>(m.world.p), n_all, 16, 0.f))) return rc;
    if ((rc = m.map.wait_ready(s))) return rc;
    ILSM_CUDA(cudaStreamSynchronize(s));
    m.built = n_all > 0;
    q_w[0] = qw.x, q_w[1] = qw.y, q_w[2] = qw.z, q_w[3] = qw.w;
    for (int i = 0; i < 3; ++i) t_w[i] = tw[i];
    if (stats) stats->map_size = m.map.n;
    return ILSM_OK;
  }
  // VoxelGrid(0.8) of the merged cloud; the stack size stays on the device (counts[1])
  ILSM_CUDA(cudaMemsetAsync(m.counts.p, 0, 4 * sizeof(int), s));
  if (n_all > 0) {
    const Ctx::VgCloud vc = {reinterpret_cast<const float*>(m.merged.p), n_all, m.leaf, m.stack.p, m.counts.p + 1};
    if ((rc = c.voxelgrid(&vc, 1, 16, 3, c.stream))) return rc;
  }
  // association (5-NN in the ground map, plane fit) + ceres::Solve (planes only, one pass, 10 iterations)
  const double qw4[4] = {qw.x, qw.y, qw.z, qw.w};
  if ((rc = c.upload_pose(qw4, tw, s))) return rc;
  ilsm_reg_opts o;
  ilsm_reg_opts_default(&o);
  o.outer_iterations = 1, o.max_num_iterations = 10, o.min_corner_map = 0, o.min_surf_map = 0;
  c.d_stack_counts = m.counts.p;
  rc = c.register_dev(&m.empty, &m.map, nullptr, 0, reinterpret_cast<const float*>(m.stack.p), n_all, 16, o);
  c.d_stack_counts = nullptr;
  if (rc) return rc;
  int* pin_counts = reinterpret_cast<int*>(c.pinned.p + Ctx::kPinSite);
  if ((rc = c.read_back_lm(s))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(pin_counts, m.counts.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
  ILSM_CUDA(cudaStreamSynchronize(s));
  double out[7];
  ilsm_reg_report rep;
  c.lm_result(out, out + 4, &rep);
  const int n_stack = pin_counts[1];
  const bool converged = rep.pass[0].termination == ILSM_CONVERGENCE;  // mapOptimization.cpp:448
  QuatH qk = qw;       // cur_keyframe.q_map_cur_k_ / t_map_cur_k_: the predicted pose unless the solve converged
  double tk[3] = {tw[0], tw[1], tw[2]};
  if (converged) {
    qk = QuatH{out[0], out[1], out[2], out[3]};
    for (int i = 0; i < 3; ++i) tk[i] = out[4 + i];
    // transformUpdate (:738-742)
    const double n2 = qo.x * qo.x + qo.y * qo.y + qo.z * qo.z + qo.w * qo.w;
    const QuatH qinv{-qo.x / n2, -qo.y / n2, -qo.z / n2, qo.w / n2};
    m.q_wmap_wodom = qmul_h(qk, qinv);
    qrot_h(m.q_wmap_wodom, t_wodom, r);
    for (int i = 0; i < 3; ++i) m.t_wmap_wodom[i] = tk[i] - r[i];
  }
  // the parameter block itself (q_w_curr / t_w_curr map Ceres' array) holds the optimised values either way
  for (int i = 0; i < 4; ++i) q_w[i] = out[i];
  for (int i = 0; i < 3; ++i) t_w[i] = out[4 + i];
  // Add_Points(transformed filtered cloud, downsample on)
  quat_to_mat_h(qk, T.r);
  for (int i = 0; i < 3; ++i) T.t[i] = tk[i];
  if (n_stack > 0) {
    ILSM_CUDA(launch_pdl(mo_transform_kernel, dim3((n_stack + 255) / 256), dim3(256), 0, s, (const float4*)m.stack.p,
                         (const int*)nullptr, n_stack, T, m.world.p));
    count_launches(1);
    if ((rc = m.map.insert_dev(reinterpret_cast<const float*>(m.world.p), n_stack, 16, 1, m.ds))) return rc;
    if ((rc = m.map.wait_ready(s))) return rc;
    ILSM_CUDA(cudaStreamSynchronize(s));
  }
  if (stats) {
    stats->n_query = n_stack;
    stats->ran_optimization = 1;
    stats->converged = converged ? 1 : 0;
    stats->solve = rep.pass[0];
    stats->map_size = m.map.n;
    stats->q_key[0] = qk.x, stats->q_key[1] = qk.y, stats->q_key[2] = qk.z, stats->q_key[3] = qk.w;
    for (int i = 0; i < 3; ++i) stats->t_key[i] = tk[i];
  }
  return ILSM_OK;
}
}  // namespace ilsm

extern "C" {

ILSM_API int ilsm_mapopt_frame(ilsm_mapopt* mo, const float* frame_xyz, int n, int stride_bytes, const float* plane_xyz, int n_plane,
                               int plane_stride_bytes, const double q_wodom[4], const double t_wodom[3], double q_w[4],
                               double t_w[3], const ilsm_ground_opts* gopts, ilsm_mapopt_stats* stats) {
  if (!mo || !q_wodom || !t_wodom || !q_w || !t_w || (n > 0 && !frame_xyz) || (n_plane > 0 && !plane_xyz))
    return fail(ILSM_ERR_INVALID_ARG, "mapopt_frame: null argument");
  if (n < 0 || n_plane < 0 || !valid_stride(stride_bytes) || !valid_stride(plane_stride_bytes))
    return fail(ILSM_ERR_INVALID_ARG, "mapopt_frame: bad n/stride");
  ILSM_ENTER(*mo->m.ctx);
  return mapopt_frame_core(mo, frame_xyz, n, stride_bytes, plane_xyz, n_plane, plane_stride_bytes, true, q_wodom, t_wodom, q_w, t_w,
                           gopts, stats);
}

}  // extern "C"
