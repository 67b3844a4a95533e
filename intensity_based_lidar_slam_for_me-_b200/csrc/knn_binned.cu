// knn_binned.cu -- K1 in the throughput regime (a whole frame of queries against a large map): query-cooperative exact
// k-NN with shared-memory staged candidates.
//
// The per-query kernel (map_grid.cu: one warp per query) re-probes the voxel hash and re-reads the 27 neighbour voxels
// for every query and pays a 5-step binary search per candidate: 1161 warp instructions per query at N = 2 M,
// Q = 65 536 (ncu), instruction-bound.  A LiDAR frame's queries are spatially coherent -- tens of returns fall into the
// same 1 m voxel -- so here the queries are binned by voxel first (the same counting structure the map build uses,
// run over the query cloud), and one warp serves up to 32 queries of one voxel:
//   * the 3x3x3 (then shell by shell) neighbour voxels are probed ONCE per group,
//   * their points are staged ONCE into a shared-memory tile (coalesced loads, next tile prefetched while the
//     current one is scanned),
//   * every lane scans the tile for its own query with broadcast shared-memory reads and keeps its K best in registers.
// Groups with fewer than 32 queries split the candidate tile between 32 / pow2(count) lanes per query ("slices") and
// merge the slices' lists afterwards (REDUX arg-min for wide splits, a shuffle butterfly for narrow ones), so that a
// lone far-range query still uses the whole warp.  Termination is the per-query exact bound of knn_search, evaluated
// per lane; the group expands ring by ring until every query of it is done.
// Results are identical to the per-query kernel (same distance arithmetic, same (d2, index) total order).
#include "ilsm_host.hpp"

namespace ilsm {

constexpr int kGroupDefault = 8;  // queries per group (runtime parameter `gsz`, a power of two <= 32): every query's candidate scan is split over >= 4 lanes (32 / kGroup slices), which keeps
                          // one warp's serial work short -- with 32-query groups the kernel's duration was the heaviest group's scan
                          // (ncu: 18.8 % of the warps active on average)

struct QWork {  // one group: <= kGroup queries of one voxel
  int cx, cy, cz;
  uint32_t pack;  // (first query in the sorted query array) << 5 | (count - 1)
};

// occupied query voxels -> work items (chunks of <= 32 queries); voxels with many queries are written out by the
// whole warp
__global__ void qbin_work_kernel(const GridCell* __restrict__ cells, const uint32_t* __restrict__ occ, const uint32_t* __restrict__ counters,
                                 int occ_slot, QWork* __restrict__ work, uint32_t* __restrict__ n_work, uint32_t kGroup) {
  pdl_entry();
  const uint32_t n_occ = counters[occ_slot];
  const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31;
  uint32_t start = 0, cnt = 0;
  int cx = 0, cy = 0, cz = 0;
  if (li < n_occ) {
    const uint4 e = *reinterpret_cast<const uint4*>(cells + occ[li]);
    const u64 key = ((u64)e.y << 32) | e.x;
    cx = (int)((key >> 42) & 0x1FFFFF) - kCoordOff, cy = (int)((key >> 21) & 0x1FFFFF) - kCoordOff, cz = (int)(key & 0x1FFFFF) - kCoordOff;
    start = e.z, cnt = e.w;
  }
  const uint32_t nch = (cnt + kGroup - 1) / kGroup;
  // warp-aggregated reservation of work slots
  uint32_t inc = nch;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= (unsigned)off) inc += v;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
  uint32_t base = 0;
  if (lane == 31 && total) base = atomicAdd(n_work, total);
  base = __shfl_sync(0xffffffffu, base, 31) + inc - nch;
  if (nch == 1) {
    QWork w{cx, cy, cz, (start << 5) | (cnt - 1)};
    work[base] = w;
  }
  // voxels with several chunks: medium ones are written out by their warp, huge ones (thousands of queries in one voxel:
  // the no-return rays) are handed to the whole block through shared memory
  __shared__ uint32_t s_big[8][4];
  __shared__ int s_bigc[8][3];
  __shared__ int s_nbig;
  if (threadIdx.x == 0) s_nbig = 0;
  __syncthreads();
  const bool huge = nch > 64;
  if (huge) {
    const int k = atomicAdd(&s_nbig, 1);
    if (k < 8) s_big[k][0] = base, s_big[k][1] = cnt, s_big[k][2] = start, s_bigc[k][0] = cx, s_bigc[k][1] = cy, s_bigc[k][2] = cz;
  }
  unsigned big = __ballot_sync(0xffffffffu, nch > 1 && !huge);
  while (big) {
    const int src = __ffs(big) - 1;
    big &= big - 1;
    const uint32_t b = __shfl_sync(0xffffffffu, base, src), c = __shfl_sync(0xffffffffu, cnt, src), s = __shfl_sync(0xffffffffu, start, src);
    const int x = __shfl_sync(0xffffffffu, cx, src), y = __shfl_sync(0xffffffffu, cy, src), z = __shfl_sync(0xffffffffu, cz, src);
    const uint32_t n = (c + kGroup - 1) / kGroup;
    for (uint32_t k = lane; k < n; k += 32) {
      const uint32_t left = c - kGroup * k;
      QWork w{x, y, z, ((s + kGroup * k) << 5) | ((left < kGroup ? left : kGroup) - 1)};
      work[b + k] = w;
    }
  }
  __syncthreads();
  const int nbig = s_nbig < 8 ? s_nbig : 8;
  for (int h = 0; h < nbig; ++h) {
    const uint32_t b = s_big[h][0], c = s_big[h][1], s = s_big[h][2];
    const uint32_t n = (c + kGroup - 1) / kGroup;
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
      const uint32_t left = c - kGroup * k;
      QWork w{s_bigc[h][0], s_bigc[h][1], s_bigc[h][2], ((s + kGroup * k) << 5) | ((left < kGroup ? left : kGroup) - 1)};
      work[b + k] = w;
    }
  }
  if (huge && s_nbig > 8) {  // more than 8 huge voxels in one block (not seen in practice): their own thread writes them
    bool mine_listed = false;
    for (int h = 0; h < 8; ++h) mine_listed = mine_listed || (s_big[h][0] == base);
    if (!mine_listed)
      for (uint32_t k = 0; k < nch; ++k) {
        const uint32_t left = cnt - kGroup * k;
        QWork w{cx, cy, cz, ((start + kGroup * k) << 5) | ((left < kGroup ? left : kGroup) - 1)};
        work[base + k] = w;
      }
  }
}

// merge of the slices' lists of one query: K rounds of a 64-bit arg-min over the lanes named by `mask` (the lanes that
// hold slices of the same query), two 32-bit REDUX each
template <int K>
__device__ __forceinline__ void group_merge_redux(CandList<K, false>& best, unsigned mask, u64 (&res)[K]) {
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const uint32_t hi = (uint32_t)(best.key[0] >> 32), lo = (uint32_t)best.key[0];
    const uint32_t mhi = redux_min_u32(mask, hi);
    const uint32_t mlo = redux_min_u32(mask, hi == mhi ? lo : 0xFFFFFFFFu);
    const u64 m = ((u64)mhi << 32) | mlo;
    res[k] = m;
    if (best.key[0] == m && m != kSentinel) best.pop_front();
  }
}

template <int K>
__global__ void __launch_bounds__(128)
    knn_binned_kernel(GridView g, const float4* __restrict__ qsorted, const QWork* __restrict__ work, const uint32_t* __restrict__ n_work_p,
                      int k_out, float max_d2, int32_t* __restrict__ idx, float* __restrict__ d2) {
  pdl_entry();
  __shared__ WarpScratch scratch[4];
  __shared__ float4 tiles[4][32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch& ws = scratch[warp];
  float4* tile = tiles[warp];
  int bb[6];
  load_bbox(g, bb);
  const uint32_t n_work = *n_work_p;
  const uint32_t nwarps = gridDim.x * 4;
#pragma unroll 1
  for (uint32_t wi = blockIdx.x * 4 + warp; wi < n_work; wi += nwarps) {
    const QWork w = work[wi];
    const int cx = w.cx, cy = w.cy, cz = w.cz;
    const uint32_t q0 = w.pack >> 5, cnt_raw = (w.pack & 31u) + 1u;
    // A group whose queries are all the same point (the no-return rays of a LiDAR frame all map to the sensor origin:
    // half of an OS0-64 frame) is ONE query: it is searched once, split over the whole warp, and the result is written
    // to every member -- instead of 32 lanes scanning the same candidates for the same answer.
    bool same_pt = false;
    if (cnt_raw > 1) {
      const float4 mine = __ldg(qsorted + q0 + (lane < cnt_raw ? lane : 0u));
      const float4 first = __ldg(qsorted + q0);
      same_pt = __all_sync(0xffffffffu, mine.x == first.x && mine.y == first.y && mine.z == first.z);
    }
    const uint32_t cnt = same_pt ? 1u : cnt_raw;
    // lanes = (query, slice): nqp = pow2 >= cnt queries side by side, S = 32 / nqp slices of the candidate tile each
    const uint32_t nqp = cnt <= 1 ? 1u : 1u << (32 - __clz(cnt - 1));
    const uint32_t S = 32u / nqp;
    const uint32_t my_q = lane & (nqp - 1u), slice = lane / nqp;
    const bool valid = my_q < cnt;
    const float4 qv = __ldg(qsorted + q0 + (valid ? my_q : 0u));
    const float qx = qv.x, qy = qv.y, qz = qv.z;
    const float ux = __fmul_rn(qx, g.inv_cell), uy = __fmul_rn(qy, g.inv_cell), uz = __fmul_rn(qz, g.inv_cell);
    const float fx = ux - (float)cx, fy = uy - (float)cy, fz = uz - (float)cz;
    const float fmin_ = fminf(fminf(fminf(fx, 1.f - fx), fminf(fy, 1.f - fy)), fminf(fz, 1.f - fz));
    const float umax = fmaxf(fmaxf(fabsf(ux), fabsf(uy)), fabsf(uz));
    // lanes that hold slices of the same query (for the REDUX merge): every nqp-th lane from my_q
    const unsigned gmask = (nqp == 1 ? 0xffffffffu : nqp == 2 ? 0x55555555u : nqp == 4 ? 0x11111111u : 0u) << my_q;

    CandList<K, false> best;
    best.clear();
    const float kInf = __int_as_float(0x7f800000);
    float ext = kInf;    // K-th distance of the merged list of the previous rings (exact upper bound for the final K-th)
    float worst = kInf;  // pruning threshold of the scan: min(ext, K-th distance of this lane's own list)
    bool done = !valid;
    int r = 1;
#pragma unroll 1
    for (;;) {
      const bool brute = r > kMaxRing;
      const int side = 2 * r + 1, total = brute ? 1 : side * side * side;
#pragma unroll 1
      for (int base = 0; base < total; base += 32) {
        const int t = base + (int)lane;
        uint32_t start = 0, c = 0;
        if (brute) {
          if (lane == 0) c = (uint32_t)g.n;
        } else if (t < total) {
          int dz = t / (side * side), rem = t - dz * side * side;
          int dy = rem / side, dx = rem - dy * side;
          dx -= r, dy -= r, dz -= r;
          const bool interior = r > 1 && abs(dx) < r && abs(dy) < r && abs(dz) < r;  // visited by earlier passes
          const int vx = cx + dx, vy = cy + dy, vz = cz + dz;
          if (!interior && vx >= bb[0] && vx <= bb[3] && vy >= bb[1] && vy <= bb[4] && vz >= bb[2] && vz <= bb[5])
            c = probe_voxel(g, pack_voxel(vx, vy, vz), start);
        }
        uint32_t inc = c;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const uint32_t v = __shfl_up_sync(0xffffffffu, inc, off);
          if (lane >= (unsigned)off) inc += v;
        }
        const uint32_t ncand = __shfl_sync(0xffffffffu, inc, 31);
        ws.start[lane] = start;
        ws.prefix[lane + 1] = inc;
        if (lane == 0) ws.prefix[0] = 0;
        __syncwarp();
        // candidate k of this round -> its point (the binary search runs once per candidate, not once per query)
        auto fetch = [&](uint32_t k) -> float4 {
          if (k >= ncand) return make_float4(0.f, 0.f, 0.f, 0.f);
          int cc = 0;
#pragma unroll
          for (int step = 16; step > 0; step >>= 1)
            if (ws.prefix[cc + step] <= k) cc += step;
          return __ldg(g.sorted + ws.start[cc] + (k - ws.prefix[cc]));
        };
        float4 nxt = fetch(lane);
#pragma unroll 1
        for (uint32_t t0 = 0; t0 < ncand; t0 += 32) {
          tile[lane] = nxt;
          __syncwarp();
          nxt = fetch(t0 + 32 + lane);  // in flight while the tile is scanned
          const uint32_t m = ncand - t0 < 32u ? ncand - t0 : 32u;
          if (!done) {
#pragma unroll 4
            for (uint32_t j = slice; j < m; j += S) {
              const float4 p = tile[j];
              const float d = dist2_rn(qx, qy, qz, p.x, p.y, p.z);
              if (d <= worst) {  // ties go through: insert() decides them by index
                best.insert(pack_cand(d, __float_as_uint(p.w)), 0.f, 0.f, 0.f);
                worst = best.key[K - 1] == kSentinel ? ext : fminf(ext, cand_d2(best.key[K - 1]));
              }
            }
          }
          __syncwarp();
        }
      }
      // merge the slices of every query; afterwards slice 0 carries the list, the others restart empty but keep the
      // merged K-th distance as their pruning threshold
      if (S > 1) {
        if (S >= 8) {
          u64 res[K];
          group_merge_redux<K>(best, gmask, res);
#pragma unroll
          for (int k = 0; k < K; ++k) best.key[k] = res[k];
        } else {
          // few slices (2 or 4): K rounds of "minimum of the slices' heads" by xor shuffles over the slice bits; the lane
          // that owns the minimum pops it (keys are unique)
          u64 res[K];
#pragma unroll
          for (int k = 0; k < K; ++k) {
            u64 m = best.key[0];
            for (uint32_t bit = nqp; bit < 32u; bit <<= 1) {
              const u64 o = __shfl_xor_sync(0xffffffffu, m, bit);
              m = o < m ? o : m;
            }
            res[k] = m;
            if (best.key[0] == m && m != kSentinel) best.pop_front();
          }
#pragma unroll
          for (int k = 0; k < K; ++k) best.key[k] = res[k];
        }
      }
      ext = best.key[K - 1] == kSentinel ? kInf : cand_d2(best.key[K - 1]);  // (S == 1: the lane's own list is the merged one)
      worst = ext;
      if (brute) break;
      // per-query exact termination (see knn_search): the K-th distance is provably below anything unvisited, or the
      // visited block contains the ball max_d2, or it covers the occupied bounding box
      const float margin = (umax + (float)r + 2.f) * 2.4e-7f;
      const float bound = ((float)r + fmin_ - margin) * g.cell;
      const float b2 = bound > 0.f ? bound * bound * 0.999999f : 0.f;
      const bool have = best.key[K - 1] != kSentinel;
      done = done || (have && cand_d2(best.key[K - 1]) < b2) || (max_d2 > 0.f && b2 >= max_d2) ||
             (cx - r <= bb[0] && cx + r >= bb[3] && cy - r <= bb[1] && cy + r >= bb[4] && cz - r <= bb[2] && cz + r >= bb[5]);
      if (__all_sync(0xffffffffu, done)) break;
      ++r;
      if (r > kMaxRing) {  // brute force revisits everything: the queries still open restart from scratch
        if (!done) best.clear(), ext = kInf, worst = kInf;
      } else if (S > 1 && slice != 0) {
        best.clear();  // slice 0 carries the merged list forward
      }
    }
    if (same_pt) {
      // after the merge every lane holds the list (S = 32 -> REDUX merge leaves it in all lanes): lane l writes member l
      if (lane < cnt_raw) {
        const size_t o = (size_t)__float_as_uint(__ldg(qsorted + q0 + lane).w) * k_out;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          if (k < k_out) {
            const bool have = best.key[k] != kSentinel;
            idx[o + k] = have ? cand_idx(best.key[k]) : -1;
            d2[o + k] = have ? cand_d2(best.key[k]) : __int_as_float(0x7f800000);
          }
        }
      }
    } else if (valid && slice == 0) {
      const size_t o = (size_t)__float_as_uint(qv.w) * k_out;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (k < k_out) {
          const bool have = best.key[k] != kSentinel;
          idx[o + k] = have ? cand_idx(best.key[k]) : -1;
          d2[o + k] = have ? cand_d2(best.key[k]) : __int_as_float(0x7f800000);
        }
      }
    }
    __syncwarp();
  }
}

// queries the binning skipped (non-finite or outside the addressable voxel range): the per-query search, which
// falls back to an exact brute-force sweep for them.  Normally there are none and the kernel returns at once.
template <int K>
__global__ void __launch_bounds__(128)
    knn_outlier_kernel(GridView g, const float* __restrict__ q, int nq, int stride_f, const uint32_t* __restrict__ slot_of,
                       const uint32_t* __restrict__ counters, int k_out, float max_d2, int32_t* __restrict__ idx, float* __restrict__ d2) {
  pdl_entry();
  if (counters[2] == 0) return;
  __shared__ WarpScratch scratch[4];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int bb[6];
  load_bbox(g, bb);
  for (int gid = blockIdx.x * 4 + warp; gid < nq; gid += gridDim.x * 4) {
    if (slot_of[gid] != 0xFFFFFFFFu) continue;
    const float* qp = q + (size_t)gid * stride_f;
    KnnResult<K, false> res;
    knn_search<K, false>(g, bb, __ldg(qp), __ldg(qp + 1), __ldg(qp + 2), max_d2, lane, scratch[warp], res);
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (k < k_out) {
          const bool have = res.key[k] != kSentinel;
          idx[(size_t)gid * k_out + k] = have ? cand_idx(res.key[k]) : -1;
          d2[(size_t)gid * k_out + k] = have ? cand_d2(res.key[k]) : __int_as_float(0x7f800000);
        }
      }
    }
  }
}

// upper bound of the number of groups: every occupied voxel contributes ceil(count / kGroup) <= count / kGroup + 1
static inline size_t qwork_items(int nq) { return (size_t)2 * nq + 64; }

template <int K>
static int launch_binned(Ctx* ctx, Map* m, Map* qb, const float* d_q, int nq, int stride_f, int k, float max_d2, int32_t* d_idx,
                         float* d_d2, int occ_slot) {
  cudaStream_t s = ctx->stream;
  const GridView g = m->view();
  QWork* work = reinterpret_cast<QWork*>(ctx->qwork.p);
  uint32_t* n_work = reinterpret_cast<uint32_t*>(ctx->qwork.p + (size_t)4 * qwork_items(nq));
  ILSM_CUDA(cudaMemsetAsync(n_work, 0, sizeof(uint32_t), s));
  ILSM_CUDA(launch_pdl(qbin_work_kernel, dim3((nq + 255) / 256), dim3(256), 0, s, qb->cur_cells(), qb->cur_occ(),
                       qb->cur_counters(), occ_slot, work, n_work, (uint32_t)ctx->knn_group));
  // one warp per group; grid = a few resident waves, further groups are taken grid-stride
  long long blocks = ((long long)nq + 3) / 4, cap = (long long)ctx->sm_count * 16;
  if (blocks > cap) blocks = cap;
  ILSM_CUDA(launch_pdl(knn_binned_kernel<K>, dim3((unsigned)blocks), dim3(128), 0, s, g, (const float4*)qb->sorted.p, (const QWork*)work,
                       (const uint32_t*)n_work, k, max_d2, d_idx, d_d2));
  ILSM_CUDA(launch_pdl(knn_outlier_kernel<K>, dim3(ctx->sm_count), dim3(128), 0, s, g, d_q, nq, stride_f, (const uint32_t*)qb->slot_of.p,
                       qb->cur_counters(), k, max_d2, d_idx, d_d2));
  count_launches(3);
  return ILSM_OK;
}

// Exact k-NN of a large query set: bin the queries by voxel (the map's own cell size), then one warp per group.
int knn_binned_dev(Ctx* ctx, Map* m, const float* d_q, int nq, int stride_bytes, int k, float max_dist, int32_t* d_idx, float* d_d2) {
  int rc;
  if (!ctx->qbin) {  // installed only once it is complete: a failed init leaves the context without one
    std::unique_ptr<Map> qb(new (std::nothrow) Map());
    if (!qb) return fail(ILSM_ERR_OUT_OF_MEMORY, "host allocation failed");
    if ((rc = qb->init(ctx))) return rc;
    ctx->qbin = std::move(qb);
  }
  Map* qb = ctx->qbin.get();
  if ((rc = ctx->qwork.reserve((size_t)4 * qwork_items(nq) + 16))) return rc;  // QWork = 4 ints; the counter sits behind the list
  // the query cloud through the map build's count / alloc / scatter: queries grouped by voxel, original index in .w
  const int occ_slot = 4;  // occupied-voxel count of the build's own counter set
  if ((rc = qb->build_dev(d_q, nq, stride_bytes, m->cell))) return rc;
  if ((rc = m->wait_ready(ctx->stream)) || (rc = qb->wait_ready(ctx->stream))) return rc;
  const float max_d2 = max_dist > 0.f ? max_dist * max_dist : 0.f;
  const int stride_f = stride_bytes / 4;
  if (k == 1) rc = launch_binned<1>(ctx, m, qb, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, occ_slot);
  else if (k <= 5) rc = launch_binned<5>(ctx, m, qb, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, occ_slot);
  else rc = launch_binned<8>(ctx, m, qb, d_q, nq, stride_f, k, max_d2, d_idx, d_d2, occ_slot);
  if (rc) return rc;
  return check_launch("knn_binned");
}

}  // namespace ilsm
