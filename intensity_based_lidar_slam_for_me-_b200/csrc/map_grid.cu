// map_grid.cu -- K1: voxel-hashed local map (build) and the stand-alone exact k-NN kernel.
//
// Replaces pcl::KdTreeFLANN::setInputCloud/nearestKSearch (laserMapping.cpp:631-634,673,753;
// laserOdometry.cpp:452,574,807-808) and ikd-Tree Build/Nearest_Search (mapOptimization.cpp:192,393).
//
// Build = 4 short kernels, no sort:
//   clear   : the slots the PREVIOUS build occupied <- EMPTY (its occupied-slot list), counters <- 0; a full clear of
//             the table only when the table grew or was reallocated
//   count   : every point claims its voxel slot with atomicCAS and takes a rank with atomicAdd; slots claimed for the
//             first time are appended to the occupied-slot list (one atomicAdd per block)
//   alloc   : every occupied slot (the list, not the table) gets a contiguous range (one atomicAdd per block)
//   scatter : points are written as float4 {x,y,z,bits(index)} into their voxel's range
// The table has >= 2 N slots (the only safe bound before the points are seen) but only the occupied voxels -- a few
// per cent of it for a dense map -- are ever touched again: at N = 2 M the full clear + full-table alloc pass moved
// 190 MB of the build's 480 MB.
// The memory order of voxels/points is not deterministic, the k-NN result is: selection uses the total
// order (d2, original index).
#include "ilsm_host.hpp"

namespace ilsm {

// One build job = one map.  A launch serves one or two jobs (the corner and surf structures of a frame): blocks
// [0, nb0) work for job 0, the rest for job 1.
struct BuildJob {
  const float* src;
  int n, stride_f, ioff;
  float inv_cell;
  GridCell* cells;       // the table this build fills (EMPTY on entry)
  uint32_t mask;
  int log2_size;
  float4* orig;
  float4* sorted;
  uint32_t *slot_of, *rank_of;
  uint32_t* counters;    // this build's set: [0] range cursor, [2] skipped points, [4] occupied voxels, [6] scatter ticket
  uint32_t* occ;         // slots claimed by this build
  int* bbox;             // this build's bounding box of occupied voxels
  // the OTHER table of the map (filled two builds ago, searched until this build started): cleaned while this build
  // scatters, so that the next build finds it empty -- no clear pass on anybody's critical path
  GridCell* o_cells;
  const uint32_t* o_occ;
  uint32_t* o_counters;
  int* o_bbox;
  int o_cover;           // upper bound of the other table's occupied-slot count (its build's point count), 0: nothing to clean
  int blocks;            // blocks of this job in the count / alloc / scatter launches
};
struct BuildJobs {
  BuildJob j[2];
  int nb0;
};

__global__ void grid_clear_kernel(GridCell* cells, uint32_t size, int* bbox, uint32_t* counters) {
  pdl_entry();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < size) {
    uint4 e;
    e.x = 0xFFFFFFFFu, e.y = 0xFFFFFFFFu, e.z = 0u, e.w = 0u;
    reinterpret_cast<uint4*>(cells)[i] = e;
  }
  if (i < 3) bbox[i] = INT_MAX;
  if (i >= 3 && i < 6) bbox[i] = INT_MIN;
  if (i < 8) counters[i] = 0;
}

__device__ __forceinline__ bool load_point(const float* src, int stride_f, int i, float& x, float& y, float& z) {
  const float* p = src + (size_t)i * stride_f;
  x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
  return isfinite(x) && isfinite(y) && isfinite(z);
}

__global__ void __launch_bounds__(256) grid_count_kernel(BuildJobs jobs) {
  pdl_entry();
  __shared__ uint32_t s_wnew[8];
  __shared__ uint32_t s_obase;
  const int w = (int)blockIdx.x >= jobs.nb0;
  const BuildJob& jb = jobs.j[w];
  const int i = ((int)blockIdx.x - (w ? jobs.nb0 : 0)) * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool in = i < jb.n;
  float x = 0.f, y = 0.f, z = 0.f;
  bool ok = in && load_point(jb.src, jb.stride_f, i, x, y, z);
  // w keeps the caller's intensity channel (LOAM clouds carry scanID + 0.1*relTime there, laserOdometry.cpp:461)
  if (in) jb.orig[i] = make_float4(x, y, z, jb.ioff >= 0 ? __ldg(jb.src + (size_t)i * jb.stride_f + jb.ioff) : 0.f);
  int cx = 0, cy = 0, cz = 0;
  if (ok) {
    float ux = __fmul_rn(x, jb.inv_cell), uy = __fmul_rn(y, jb.inv_cell), uz = __fmul_rn(z, jb.inv_cell);
    ok = fabsf(ux) < (float)kCoordLim && fabsf(uy) < (float)kCoordLim && fabsf(uz) < (float)kCoordLim;
    cx = __float2int_rd(ux), cy = __float2int_rd(uy), cz = __float2int_rd(uz);
  }
  if (in && !ok) {
    jb.slot_of[i] = 0xFFFFFFFFu;
    atomicAdd(&jb.counters[2], 1u);
  }
  // warp-aggregated claim: map clouds arrive voxel-ordered (VoxelGrid output, cube by cube), so the lanes of a warp
  // mostly share a handful of voxels -- one atomicCAS + one atomicAdd per distinct voxel of the warp instead of one
  // per point.  All 32 lanes take part in the match; lanes without a point carry a key nobody shares.
  const u64 key = ok ? pack_voxel(cx, cy, cz) : (kEmptyKey - 1ull - (u64)lane);
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  bool created = false;  // this lane claimed a slot nobody had claimed before
  uint32_t my_slot = 0;
  if (ok) {
    const int leader = __ffs(peers) - 1;
    uint32_t slot = 0, base = 0;
    if (lane == leader) {
      slot = hash_voxel(key, jb.log2_size);
      for (;;) {
        u64 prev = atomicCAS(&jb.cells[slot].key, kEmptyKey, key);
        if (prev == kEmptyKey) created = true;
        if (prev == kEmptyKey || prev == key) break;
        slot = (slot + 1) & jb.mask;
      }
      base = atomicAdd(&jb.cells[slot].count, (uint32_t)__popc(peers));
      my_slot = slot;
    }
    slot = __shfl_sync(peers, slot, leader);
    base = __shfl_sync(peers, base, leader);
    jb.slot_of[i] = slot;
    jb.rank_of[i] = base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
  }
  // occupied-slot list: block-wide count of newly claimed slots, ONE atomicAdd on the list cursor per block
  const unsigned newb = __ballot_sync(0xffffffffu, created);
  const int warp = threadIdx.x >> 5;
  if (lane == 0) s_wnew[warp] = (uint32_t)__popc(newb);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += s_wnew[k];
    s_obase = tot ? atomicAdd(&jb.counters[4], tot) : 0u;
  }
  __syncthreads();
  if (created) {
    uint32_t wb = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (k < warp) wb += s_wnew[k];
    jb.occ[s_obase + wb + (uint32_t)__popc(newb & ((1u << lane) - 1u))] = my_slot;
  }
}

// Every occupied slot gets a contiguous range of the sorted array (one atomicAdd on the cursor per block) and the
// bounding box of occupied voxels is reduced per block (6 atomics per block instead of 6 per voxel).
__global__ void __launch_bounds__(256) grid_alloc_kernel(BuildJobs jobs) {
  pdl_entry();
  const int w = (int)blockIdx.x >= jobs.nb0;
  const BuildJob& jb = jobs.j[w];
  const uint32_t li = ((uint32_t)blockIdx.x - (w ? (uint32_t)jobs.nb0 : 0u)) * blockDim.x + threadIdx.x;
  const uint32_t size = jb.counters[4];  // occupied voxels of this build; the grid covers the upper bound n
  uint32_t cnt = 0;
  int lo[3] = {INT_MAX, INT_MAX, INT_MAX}, hi[3] = {INT_MIN, INT_MIN, INT_MIN};
  const uint32_t i = li < size ? jb.occ[li] : 0u;
  if (li < size) {
    uint4 e = *reinterpret_cast<const uint4*>(jb.cells + i);
    cnt = e.w;
    if (cnt) {
      u64 key = ((u64)e.y << 32) | e.x;
      int c[3] = {(int)((key >> 42) & 0x1FFFFF) - kCoordOff, (int)((key >> 21) & 0x1FFFFF) - kCoordOff,
                  (int)(key & 0x1FFFFF) - kCoordOff};
#pragma unroll
      for (int a = 0; a < 3; ++a) lo[a] = hi[a] = c[a];
    }
  }
  // block-wide exclusive prefix of the counts, ONE atomicAdd on the cursor per block
  __shared__ uint32_t s_wsum[8];
  __shared__ uint32_t s_base;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = cnt;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    uint32_t v = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= (uint32_t)off) inc += v;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
  if (lane == 31) s_wsum[warp] = inc;
  __syncthreads();
  uint32_t wbase = 0, btotal = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (k < (int)warp) wbase += s_wsum[k];
    btotal += s_wsum[k];
  }
  if (threadIdx.x == 0) s_base = btotal ? atomicAdd(&jb.counters[0], btotal) : 0u;
  __syncthreads();
  if (li < size && cnt) jb.cells[i].start = s_base + wbase + inc - cnt;
  // bounding box
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      lo[a] = min(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], off));
      hi[a] = max(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], off));
    }
  }
  __shared__ int s_lo[3], s_hi[3];
  if (threadIdx.x < 3) s_lo[threadIdx.x] = INT_MAX, s_hi[threadIdx.x] = INT_MIN;
  __syncthreads();
  if (lane == 0 && total) {
#pragma unroll
    for (int a = 0; a < 3; ++a) atomicMin(&s_lo[a], lo[a]), atomicMax(&s_hi[a], hi[a]);
  }
  __syncthreads();
  if (threadIdx.x < 3 && s_lo[threadIdx.x] != INT_MAX) {
    atomicMin(&jb.bbox[threadIdx.x], s_lo[threadIdx.x]);
    atomicMax(&jb.bbox[3 + threadIdx.x], s_hi[threadIdx.x]);
  }
}

// Points into their voxel's range -- and, with the spare parallelism of the same launch, the map's OTHER table is
// emptied (only the slots its build occupied); the job's last block then resets that table's counters and box.
__global__ void __launch_bounds__(256) grid_scatter_kernel(BuildJobs jobs) {
  pdl_entry();
  __shared__ int s_last;
  const int w = (int)blockIdx.x >= jobs.nb0;
  const BuildJob& jb = jobs.j[w];
  const int i = ((int)blockIdx.x - (w ? jobs.nb0 : 0)) * blockDim.x + threadIdx.x;
  if (i < jb.n) {
    const uint32_t slot = jb.slot_of[i];
    if (slot != 0xFFFFFFFFu) {
      float4 p = jb.orig[i];
      p.w = __uint_as_float((uint32_t)i);
      jb.sorted[jb.cells[slot].start + jb.rank_of[i]] = p;
    }
  }
  if (jb.o_cover > 0) {
    const uint32_t n_old = jb.o_counters[4];
    for (uint32_t k = (uint32_t)i; k < n_old; k += (uint32_t)jb.blocks * blockDim.x) {
      uint4 e;
      e.x = 0xFFFFFFFFu, e.y = 0xFFFFFFFFu, e.z = 0u, e.w = 0u;
      reinterpret_cast<uint4*>(jb.o_cells)[jb.o_occ[k]] = e;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      s_last = atomicAdd(&jb.counters[6], 1u) == (uint32_t)jb.blocks - 1u;
    }
    __syncthreads();
    if (s_last) {  // every block of the job has read o_counters[4]: the other set can be reset for its next build
      if (threadIdx.x < 8) jb.o_counters[threadIdx.x] = 0;
      if (threadIdx.x < 3) jb.o_bbox[threadIdx.x] = INT_MAX;
      if (threadIdx.x >= 3 && threadIdx.x < 6) jb.o_bbox[threadIdx.x] = INT_MIN;
      if (threadIdx.x == 0) jb.counters[6] = 0;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// stand-alone k-NN kernel: one G-lane group per query
// ---------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(128) knn_kernel(GridView g, const float* __restrict__ q, int nq, int stride_f, int k_out,
                                                  float max_d2, int32_t* __restrict__ idx, float* __restrict__ d2) {
  pdl_entry();
  __shared__ WarpScratch scratch[4];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int bb[6];
  load_bbox(g, bb);
  const int nwarps = gridDim.x * 4;
  for (int gid = blockIdx.x * 4 + warp; gid < nq; gid += nwarps) {
    const float* qp = q + (size_t)gid * stride_f;
    const float qx = __ldg(qp), qy = __ldg(qp + 1), qz = __ldg(qp + 2);
    KnnResult<K, false> res;
    knn_search<K, false>(g, bb, qx, qy, qz, max_d2, lane, scratch[warp], res);
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (k < k_out) {
          bool have = res.key[k] != kSentinel;
          idx[(size_t)gid * k_out + k] = have ? cand_idx(res.key[k]) : -1;
          d2[(size_t)gid * k_out + k] = have ? cand_d2(res.key[k]) : __int_as_float(0x7f800000);
        }
      }
    }
  }
}

int knn_binned_dev(Ctx* ctx, Map* m, const float* d_q, int nq, int stride_bytes, int k, float max_dist, int32_t* d_idx, float* d_d2);

static inline int ilog2_ceil(uint32_t v) {
  int l = 0;
  while ((1u << l) < v) ++l;
  return l;
}

int Map::init(Ctx* c) {
  ctx = c;
  ILSM_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  ILSM_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
  ILSM_CUDA(cudaEventCreateWithFlags(&ctx_done, cudaEventDisableTiming));
  return ILSM_OK;
}

int Map::wait_ready(cudaStream_t user) {
  if (pending) {
    ILSM_CUDA(cudaStreamWaitEvent(user, ready, 0));
    if (user == ctx->stream) pending = false;
  }
  return ILSM_OK;
}

// Sizes, allocations and table hygiene of one map for a build of n_pts points; fills the job.  The map keeps TWO hash
// tables and alternates between them: build g fills table g & 1, which build g - 1 emptied while it scattered.
int Map::prepare_build(const float* d_src, int n_pts, int stride_bytes, float cell_size, cudaStream_t s, void* job_out) {
  BuildJob& jb = *static_cast<BuildJob*>(job_out);
  if (n_pts < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "map_build: bad n/stride");
  if (!(cell_size > 0.f)) cell_size = 1.0f;
  int want_log2 = ilog2_ceil((uint32_t)(n_pts > 0 ? 2u * (uint32_t)n_pts : 2u));
  if (want_log2 < 10) want_log2 = 10;
  const uint32_t want_size = 1u << want_log2;
  const GridCell* cells_before = cells.p;
  const uint32_t *occ_before = occ.p, *counters_before = counters.p;
  const int* bbox_before = bbox.p;
  const uint32_t cap_before = table_cap;
  // both tables / lists live back to back in one allocation each; growing one regrows both
  uint32_t new_cap = table_cap;
  if (want_size > new_cap) new_cap = want_size;
  size_t new_occ_cap = occ_cap;
  if ((size_t)n_pts + 1 > new_occ_cap) new_occ_cap = (size_t)n_pts + (size_t)n_pts / 2 + 64;
  int rc;
  if ((rc = cells.reserve((size_t)2 * new_cap)) || (rc = sorted.reserve(n_pts + 1)) || (rc = orig.reserve(n_pts + 1)) ||
      (rc = slot_of.reserve(n_pts + 1)) || (rc = rank_of.reserve(n_pts + 1)) || (rc = bbox.reserve(16)) ||
      (rc = counters.reserve(16)) || (rc = occ.reserve(2 * new_occ_cap)))
    return rc;
  const bool moved = cells.p != cells_before || occ.p != occ_before || counters.p != counters_before || bbox.p != bbox_before ||
                     new_cap != cap_before || new_occ_cap != occ_cap;
  table_cap = new_cap, occ_cap = new_occ_cap;
  if (moved) clean_size[0] = clean_size[1] = 0, filled_n[0] = filled_n[1] = 0;  // nothing is known about the new memory
  const int t = gen & 1, o = t ^ 1;
  n = n_pts;
  cell = cell_size;
  inv_cell = 1.0f / cell_size;
  log2_size = want_log2;
  table_size = want_size;
  cur = t;
  GridCell* tab = cells.p + (size_t)t * table_cap;
  // Invariant: slots [0, clean_size[t]) of table t are EMPTY and its counters / box are reset -- unless filled_n[t] != 0,
  // i.e. the table still holds a build nobody cleaned (the first builds, or a build whose successor was not run).
  if (filled_n[t] != 0 || (size_t)table_size > clean_size[t]) {
    const int T = 256;
    ILSM_CUDA(launch_pdl(grid_clear_kernel, dim3((table_size + T - 1) / T), dim3(T), 0, s, tab, table_size, bbox.p + 8 * t, counters.p + 8 * t));
    count_launches(1);
    clean_size[t] = table_size;
    filled_n[t] = 0;
  }
  jb.src = d_src, jb.n = n_pts, jb.stride_f = stride_bytes / 4;
  jb.ioff = stride_bytes >= 32 ? 4 : (stride_bytes >= 16 ? 3 : -1);
  jb.inv_cell = inv_cell;
  jb.cells = tab, jb.mask = table_size - 1, jb.log2_size = log2_size;
  jb.orig = orig.p, jb.sorted = sorted.p, jb.slot_of = slot_of.p, jb.rank_of = rank_of.p;
  jb.counters = counters.p + 8 * t, jb.occ = occ.p + (size_t)t * occ_cap, jb.bbox = bbox.p + 8 * t;
  jb.o_cells = cells.p + (size_t)o * table_cap, jb.o_occ = occ.p + (size_t)o * occ_cap;
  jb.o_counters = counters.p + 8 * o, jb.o_bbox = bbox.p + 8 * o;
  jb.o_cover = filled_n[o];  // 0 when the other table is already clean
  jb.blocks = n_pts > 0 ? (n_pts + 255) / 256 : 0;
  if (n_pts > 0 && filled_n[o] != 0) {
    // this build's scatter launch empties the other table: from the next build on it is clean up to the size it had
    filled_n[o] = 0;
  } else if (filled_n[o] != 0) {
    jb.o_cover = 0;  // no launch to piggyback on (empty cloud): the other table stays dirty and is cleared when needed
  }
  filled_n[t] = n_pts > 0 ? (n_pts > 8 ? n_pts : 8) : 0;
  gen += 1;
  return ILSM_OK;
}

int Map::reserve_points(int n_pts) {
  if (n_pts <= 0) return ILSM_OK;
  int want_log2 = ilog2_ceil(2u * (uint32_t)n_pts);
  if (want_log2 < 10) want_log2 = 10;
  const uint32_t want_size = 1u << want_log2;
  const uint32_t new_cap = want_size > table_cap ? want_size : table_cap;
  const size_t new_occ_cap = (size_t)n_pts + 1 > occ_cap ? (size_t)n_pts + (size_t)n_pts / 2 + 64 : occ_cap;
  if (new_cap == table_cap && new_occ_cap == occ_cap && sorted.cap >= (size_t)n_pts + 1) return ILSM_OK;
  int rc;
  if ((rc = cells.reserve((size_t)2 * new_cap)) || (rc = sorted.reserve(n_pts + 1)) || (rc = orig.reserve(n_pts + 1)) ||
      (rc = slot_of.reserve(n_pts + 1)) || (rc = rank_of.reserve(n_pts + 1)) || (rc = bbox.reserve(16)) ||
      (rc = counters.reserve(16)) || (rc = occ.reserve(2 * new_occ_cap)))
    return rc;
  table_cap = new_cap, occ_cap = new_occ_cap;
  clean_size[0] = clean_size[1] = 0, filled_n[0] = filled_n[1] = 0;  // nothing is known about the new memory
  return ILSM_OK;
}

static int launch_build(BuildJobs& jobs, int n_jobs, cudaStream_t s) {
  const int b0 = jobs.j[0].blocks, b1 = n_jobs > 1 ? jobs.j[1].blocks : 0;
  jobs.nb0 = n_jobs > 1 ? b0 : 0x7fffffff;  // a single job owns every block
  if (b0 + b1 == 0) return ILSM_OK;
  if (n_jobs > 1 && b0 == 0) {  // only the second map has points: make it the only job
    jobs.j[0] = jobs.j[1];
    jobs.nb0 = 0x7fffffff;
  }
  ILSM_CUDA(launch_pdl(grid_count_kernel, dim3(b0 + b1), dim3(256), 0, s, jobs));
  ILSM_CUDA(launch_pdl(grid_alloc_kernel, dim3(b0 + b1), dim3(256), 0, s, jobs));
  ILSM_CUDA(launch_pdl(grid_scatter_kernel, dim3(b0 + b1), dim3(256), 0, s, jobs));
  count_launches(3);
  return ILSM_OK;
}

int Map::build_dev(const float* d_src, int n_pts, int stride_bytes, float cell_size) {
  if (in_line) {
    cudaStream_t cs = ctx->stream;
    if (pending) ILSM_CUDA(cudaStreamWaitEvent(cs, ready, 0));
    pending = false;
    BuildJobs jobs = {};
    int rc = prepare_build(d_src, n_pts, stride_bytes, cell_size, cs, &jobs.j[0]);
    if (rc) return rc;
    if ((rc = launch_build(jobs, 1, cs))) return rc;
    return check_launch("map_build");
  }
  cudaStream_t s = stream;
  // order this (re)build after everything already enqueued on the context stream (previous users of the map,
  // producers of d_src), then run it on the map's own stream
  ILSM_CUDA(cudaEventRecord(ctx_done, ctx->stream));
  ILSM_CUDA(cudaStreamWaitEvent(s, ctx_done, 0));
  if (pending) ILSM_CUDA(cudaStreamWaitEvent(s, ready, 0));  // the previous build may have run on a partner map's stream (pair build)
  BuildJobs jobs = {};
  int rc = prepare_build(d_src, n_pts, stride_bytes, cell_size, s, &jobs.j[0]);
  if (rc) return rc;
  if ((rc = launch_build(jobs, 1, s))) return rc;
  ILSM_CUDA(cudaEventRecord(ready, s));
  pending = true;
  return check_launch("map_build");
}

// The two search structures of a frame (kdtreeCornerFromMap / kdtreeSurfFromMap, laserMapping.cpp:631-634) in ONE set of
// three launches on map a's stream.
int build_pair_dev(Map* a, const float* d_a, int na, Map* b, const float* d_b, int nb, int stride_bytes, float cell_size) {
  if (!a || !b || a == b || a->ctx != b->ctx) return fail(ILSM_ERR_INVALID_ARG, "map_build_pair: two maps of one context expected");
  Ctx* ctx = a->ctx;
  const bool in_line = a->in_line && b->in_line;
  cudaStream_t s = in_line ? ctx->stream : a->stream;
  if (in_line) {
    if (a->pending) ILSM_CUDA(cudaStreamWaitEvent(s, a->ready, 0));  // (a build made before the maps were set in line)
    if (b->pending) ILSM_CUDA(cudaStreamWaitEvent(s, b->ready, 0));
    a->pending = b->pending = false;
  } else {
    ILSM_CUDA(cudaEventRecord(a->ctx_done, ctx->stream));
    ILSM_CUDA(cudaStreamWaitEvent(s, a->ctx_done, 0));
    if (a->pending) ILSM_CUDA(cudaStreamWaitEvent(s, a->ready, 0));  // earlier builds may have run on another stream
    if (b->pending) ILSM_CUDA(cudaStreamWaitEvent(s, b->ready, 0));
  }
  BuildJobs jobs = {};
  int rc;
  if ((rc = a->prepare_build(d_a, na, stride_bytes, cell_size, s, &jobs.j[0])) || (rc = b->prepare_build(d_b, nb, stride_bytes, cell_size, s, &jobs.j[1])))
    return rc;
  if ((rc = launch_build(jobs, 2, s))) return rc;
  if (!in_line) {
    ILSM_CUDA(cudaEventRecord(a->ready, s));
    ILSM_CUDA(cudaEventRecord(b->ready, s));
    a->pending = b->pending = true;
  }
  return check_launch("map_build_pair");
}

GridView Map::view() const {
  GridView g;
  g.cells = cells.p + (size_t)cur * table_cap;
  g.sorted = sorted.p;
  g.orig = orig.p;
  g.bbox = bbox.p + 8 * cur;
  g.mask = table_size - 1;
  g.log2_size = log2_size;
  g.cell = cell;
  g.inv_cell = inv_cell;
  g.n = n;
  return g;
}

template <int K>
static int launch_knn(const GridView& g, const float* d_q, int nq, int stride_f, int k, float max_d2, int32_t* d_idx,
                       float* d_d2, cudaStream_t s, int sm_count) {
  // one warp per query; at most ~16 resident warps per SM, further queries are taken grid-stride
  long long blocks = ((long long)nq + 3) / 4, cap = (long long)sm_count * 4 * 4;
  if (blocks > cap) blocks = cap;
  ILSM_CUDA(launch_pdl(knn_kernel<K>, dim3((unsigned)blocks), dim3(128), 0, s, g, d_q, nq, stride_f, k, max_d2, d_idx, d_d2));
  return ILSM_OK;
}

int Map::knn_dev(const float* d_q, int nq, int stride_bytes, int k, float max_dist, int32_t* d_idx, float* d_d2) {
  if (nq < 0 || k < 1 || k > 8 || !valid_stride(stride_bytes))
    return fail(ILSM_ERR_INVALID_ARG, "knn: bad nq/k/stride");
  if (table_size == 0) return fail(ILSM_ERR_STATE, "knn: map not built");
  if (nq == 0) return ILSM_OK;
  // throughput regime: bin the queries by voxel and serve each group with one warp (knn_binned.cu); small query sets are
  // latency-bound and keep one warp per query
  if (nq >= ctx->knn_binned_min && n > 0) return knn_binned_dev(ctx, this, d_q, nq, stride_bytes, k, max_dist, d_idx, d_d2);
  GridView g = view();
  float max_d2 = max_dist > 0.f ? max_dist * max_dist : 0.f;
  cudaStream_t s = ctx->stream;
  {
    int rc = wait_ready(s);
    if (rc) return rc;
  }
  int stride_f = stride_bytes / 4;
  int rc;
  if (k == 1)
    rc = launch_knn<1>(g, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, s, ctx->sm_count);
  else if (k <= 5)
    rc = launch_knn<5>(g, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, s, ctx->sm_count);
  else
    rc = launch_knn<8>(g, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, s, ctx->sm_count);
  if (rc) return rc;
  count_launches(1);
  return check_launch("knn");
}

}  // namespace ilsm
