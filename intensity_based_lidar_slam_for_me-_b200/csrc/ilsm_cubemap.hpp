// ilsm_cubemap.hpp -- host-side object behind ilsm_cubemap (the device-resident rolling cube map of laserMapping.cpp),
// shared by cubemap.cu (the map itself) and pipeline.cu (the full odometry + mapping loop).
#pragma once
#include <vector>

#include "ilsm_host.hpp"

namespace ilsm {

constexpr int kCW = 21, kCH = 21, kCD = 11, kCNum = kCW * kCH * kCD;

struct GatherItem {
  int slab, offset, count;
};
// Launch parameters passed BY VALUE (kernel parameter space): the 2 x 125 gather items and the valid-cube list of a frame used
// to be staged in pinned memory and copied to the device before their kernels -- one API call each on the mapping stage's
// host-bound critical path.
struct GatherItems {
  GatherItem it[250];  // [0, 125): corner cubes, [125, 250): surf cubes
};
struct ValidSlabs {
  int slab[125];
};

struct QuatH {
  double x, y, z, w;
};
static inline QuatH qmul_h(const QuatH& a, const QuatH& b) {
  return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y, a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
          a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
static inline void qrot_h(const QuatH& q, const double v[3], double o[3]) {  // Eigen _transformVector
  const double ux = q.x, uy = q.y, uz = q.z;
  double cx = uy * v[2] - uz * v[1], cy = uz * v[0] - ux * v[2], cz = ux * v[1] - uy * v[0];
  cx += cx, cy += cy, cz += cz;
  o[0] = (v[0] + q.w * cx) + (uy * cz - uz * cy);
  o[1] = (v[1] + q.w * cy) + (uz * cx - ux * cz);
  o[2] = (v[2] + q.w * cz) + (ux * cy - uy * cx);
}

struct CubeMapH {
  Ctx* ctx = nullptr;
  Map map_c, map_s;
  int cap = 0;
  float line_res = 0.4f, plane_res = 0.8f;
  int cenW = 10, cenH = 10, cenD = 5;
  QuatH q_wmap_wodom{0, 0, 0, 1};
  double t_wmap_wodom[3] = {0, 0, 0};
  std::vector<int> slab_of;           // array index -> slab id
  std::vector<int> cnt_c_h, cnt_s_h;  // host mirror of the per-slab counts
  int valid[125], n_valid = 0;
  DevBuf<float4> slabs_c, slabs_s, from_c, from_s, stack_c, stack_s, scratch, world_tmp;
  DevBuf<uint32_t> hscratch;  // hash-based VoxelGrid scratch, one slice per cube_filter block
  DevBuf<int> cnt_all;              // cnt_c | cnt_s | err, contiguous
  int *cnt_c = nullptr, *cnt_s = nullptr, *err = nullptr;  // views into cnt_all
  DevBuf<int> slab_of_d, stack_n, zero_list;
  // per slab and cloud kind: [0, 2 kCNum) the last VoxelGrid pass left the cube unchanged and nothing was inserted since;
  // [2 kCNum, 4 kCNum) how many leading points of the cube are the output of its last pass (merge precondition)
  DevBuf<int> clean;
  bool vg_merge = true;
  // stacks produced outside (full loop: two sets, alternating by frame, written on the odometry stage's side stream):
  // when set, the frame being enqueued -- solve and deferred insertion -- reads these instead of stack_*
  const float4 *ext_c = nullptr, *ext_s = nullptr;
  const int* ext_n = nullptr;
  const float4* cur_stack_c() const { return ext_c ? ext_c : stack_c.p; }
  const float4* cur_stack_s() const { return ext_s ? ext_s : stack_s.p; }
  const int* cur_stack_n() const { return ext_n ? ext_n : stack_n.p; }
  DevBuf<float> raw;
  PinnedBuf<int> pin;

  int init(Ctx* c, float lres, float pres, int cube_cap);
  ~CubeMapH();  // synchronises the context's streams
  int roll(const double t[3]);
  int gather(int* n_mc, int* n_ms);
  int insert(const int* d_counts, int nc_host, int ns_host, int world_frame, cudaStream_t s = nullptr);
  int filter_valid(cudaStream_t s = nullptr);
  int fetch_counts(cudaStream_t s = nullptr);
  int adopt_counts();
  int wait_tail();
  PinnedBuf<int> pin_counts;
  Event ev_tail;
  bool tail_pending = false, counts_in_flight = false;
  int tail_flags = 0;
  struct Pending {  // a frame enqueued by cubemap_frame_enqueue and not yet collected
    bool active = false, optimise = false, defer_tail = false;
    QuatH qo{0, 0, 0, 1};
    double t_wodom[3] = {0, 0, 0};
    int n_mc = 0, n_ms = 0, outer = 2;
  } pend;
};


// One iteration of process() (laserMapping.cpp:327-1002) with the feature clouds already on the device
// (cubemap_frame_core = enqueue + collect).
int cubemap_frame_enqueue(CubeMapH& m, const float* d_corner_last, int nc, const float* d_surf_last, int ns, int stride_bytes,
                          const double q_wodom[4], const double t_wodom[3], const ilsm_reg_opts& o, bool stacks_ready,
                          bool defer_tail, cudaEvent_t stacks_event = nullptr);
int cubemap_frame_collect(CubeMapH& m, double q_w[4], double t_w[3], ilsm_reg_report* report, ilsm_cubemap_stats* stats);
int cubemap_frame_core(CubeMapH& m, const float* d_corner_last, int nc, const float* d_surf_last, int ns, int stride_bytes,
                       const double q_wodom[4], const double t_wodom[3], double q_w[4], double t_w[3],
                       const ilsm_reg_opts& o, ilsm_reg_report* report, ilsm_cubemap_stats* stats, bool stacks_ready, bool defer_tail,
                       cudaEvent_t stacks_event = nullptr);  // stacks_event: recorded after the caller's stack VoxelGrid

}  // namespace ilsm

struct ilsm_cubemap {
  ilsm::CubeMapH m;
};
