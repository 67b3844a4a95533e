// ikdmap.cu -- incremental map maintenance with the ikd-Tree down-sampling policy (KD_TREE::Add_Points with
// downsample_on = true, ikd_Tree.cpp:570-640) and the point export (flatten, ikd_Tree.cpp).
//
// The reference inserts points one at a time: the box of edge `ds` around the new point is searched, the point of
// {box contents, new point} nearest to the box centre survives (strict `<`: the new point wins ties against what
// is already there, a later new point wins ties against an earlier one), the box is emptied and the survivor
// re-added.  Processed as a batch this is a per-voxel arg-min, so the whole Add_Points call becomes:
//   vox_new   : hash the new points by voxel, atomicMin of (d2 bits, ~sequence)            (best new point)
//   vox_old   : every existing point looks its voxel up; touched voxels: atomicMin of (d2 bits, index)
//   decide    : survivors = existing points of untouched voxels, best-old of a voxel when strictly nearer than
//               best-new, best-new otherwise
//   scan + compact (stable: survivors in their old order, then the winning new points in batch order)
//   rebuild of the search structure (map_grid.cu)
// No rebalancing, lazy deletion, rebuild thread or operation log is needed: the voxel hash has no shape to balance.
#include "ilsm_host.hpp"

namespace ilsm {

struct VoxSlot {
  u64 key;
  u64 best_new;  // (d2 bits << 32) | ~seq
  u64 best_old;  // (d2 bits << 32) | index
};

__global__ void vox_clear_kernel(VoxSlot* t, uint32_t size) {
  pdl_entry();
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < size) t[i].key = kEmptyKey, t[i].best_new = ~0ull, t[i].best_old = ~0ull;
}

// Box of voxel index k along one axis exactly as Add_Points builds it from a point with floor(x/ds) == k:
// min = k*ds, max = min + ds, mid = min + (max - min)/2.0 (float, float, double->float).
__device__ __forceinline__ void vox_box(int k, float ds, float& mn, float& mx, float& mid) {
  mn = __fmul_rn((float)k, ds);
  mx = __fadd_rn(mn, ds);
  mid = (float)((double)mn + (double)__fsub_rn(mx, mn) / 2.0);
}
__device__ __forceinline__ int vox_index(float x, float ds) { return __float2int_rd(floorf(__fdiv_rn(x, ds))); }

// voxel index of an EXISTING point under the reference's explicit box test (min <= x && max > x,
// ikd_Tree.cpp:1607-1637); the neighbours are tried when the coordinate sits within an ulp of a face.
__device__ __forceinline__ bool vox_member_axis(float x, float ds, int& k) {
  const int k0 = vox_index(x, ds);
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int kk = k0 + (t == 0 ? 0 : (t == 1 ? -1 : 1));
    float mn, mx, mid;
    vox_box(kk, ds, mn, mx, mid);
    if (mn <= x && mx > x) {
      k = kk;
      return true;
    }
  }
  return false;
}

__device__ __forceinline__ float centre_dist(float x, float y, float z, int kx, int ky, int kz, float ds) {
  float mn, mx, cx, cy, cz;
  vox_box(kx, ds, mn, mx, cx);
  vox_box(ky, ds, mn, mx, cy);
  vox_box(kz, ds, mn, mx, cz);
  return dist2_rn(x, y, z, cx, cy, cz);  // calc_dist(point, mid_point), ikd_Tree.cpp:2224-2230
}

__device__ __forceinline__ uint32_t vox_hash(u64 key, int log2_size) { return hash_voxel(key, log2_size); }

__global__ void vox_new_kernel(const float* __restrict__ src, int n, int stride_f, float ds, VoxSlot* table, uint32_t mask,
                               int log2_size, uint32_t* __restrict__ slot_of, float4* __restrict__ packed) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = src + (size_t)i * stride_f;
  const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
  packed[i] = make_float4(x, y, z, stride_f >= 4 ? __ldg(p + (stride_f >= 8 ? 4 : 3)) : 0.f);
  if (!(isfinite(x) && isfinite(y) && isfinite(z)) || fabsf(x / ds) >= (float)kCoordLim || fabsf(y / ds) >= (float)kCoordLim ||
      fabsf(z / ds) >= (float)kCoordLim) {
    slot_of[i] = 0xFFFFFFFFu;
    return;
  }
  const int kx = vox_index(x, ds), ky = vox_index(y, ds), kz = vox_index(z, ds);
  const u64 key = pack_voxel(kx, ky, kz);
  uint32_t slot = vox_hash(key, log2_size);
  for (;;) {
    const u64 prev = atomicCAS(&table[slot].key, kEmptyKey, key);
    if (prev == kEmptyKey || prev == key) break;
    slot = (slot + 1) & mask;
  }
  slot_of[i] = slot;
  const float d = centre_dist(x, y, z, kx, ky, kz, ds);
  atomicMin(&table[slot].best_new, ((u64)__float_as_uint(d) << 32) | (uint32_t)(~(uint32_t)i));
}

__global__ void vox_old_kernel(const float4* __restrict__ pts, int n, float ds, VoxSlot* table, uint32_t mask, int log2_size,
                               uint32_t* __restrict__ slot_of) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  int kx, ky, kz;
  uint32_t found = 0xFFFFFFFFu;
  if (vox_member_axis(p.x, ds, kx) && vox_member_axis(p.y, ds, ky) && vox_member_axis(p.z, ds, kz)) {
    const u64 key = pack_voxel(kx, ky, kz);
    uint32_t slot = vox_hash(key, log2_size);
    for (;;) {
      const u64 k = table[slot].key;
      if (k == key) {
        found = slot;
        break;
      }
      if (k == kEmptyKey) break;
      slot = (slot + 1) & mask;
    }
    if (found != 0xFFFFFFFFu) {
      const float d = centre_dist(p.x, p.y, p.z, kx, ky, kz, ds);
      atomicMin(&table[found].best_old, ((u64)__float_as_uint(d) << 32) | (uint32_t)i);
    }
  }
  slot_of[i] = found;  // 0xFFFFFFFF: voxel not touched by this batch
}

// keep flags: [0, n_old) existing points, [n_old, n_old + n_new) new points
__global__ void vox_decide_kernel(const VoxSlot* __restrict__ table, const uint32_t* __restrict__ slot_old, int n_old,
                                  const uint32_t* __restrict__ slot_new, int n_new, uint32_t* __restrict__ keep) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_old + n_new) return;
  uint32_t k = 0;
  if (i < n_old) {
    const uint32_t s = slot_old[i];
    if (s == 0xFFFFFFFFu) {
      k = 1;
    } else {
      const VoxSlot v = table[s];
      // an existing point stays only when it is the best existing one AND strictly nearer than the best new one
      k = ((uint32_t)v.best_old == (uint32_t)i) && ((v.best_old >> 32) < (v.best_new >> 32)) ? 1u : 0u;
    }
  } else {
    const int j = i - n_old;
    const uint32_t s = slot_new[j];
    if (s != 0xFFFFFFFFu) {
      const VoxSlot v = table[s];
      const bool best = (uint32_t)v.best_new == (uint32_t)(~(uint32_t)j);
      const bool old_wins = v.best_old != ~0ull && (v.best_old >> 32) < (v.best_new >> 32);
      k = best && !old_wins ? 1u : 0u;
    }
  }
  keep[i] = k;
}

// ---------------------------------------------------------------------------------------------------
// exclusive scan of 0/1 flags (up to 4 Mi elements): block sums -> one block scans them -> apply
// ---------------------------------------------------------------------------------------------------
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock) scan_block_kernel(const uint32_t* __restrict__ in, int n, uint32_t* __restrict__ out,
                                                                uint32_t* __restrict__ block_sums) {
  pdl_entry();
  __shared__ uint32_t wsum[32];
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  const uint32_t v = i < n ? in[i] : 0u;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= off) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = wsum[lane], winc = w;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, winc, off);
      if (lane >= off) winc += t;
    }
    wsum[lane] = winc - w;
    if (lane == 31) block_sums[blockIdx.x] = winc;
  }
  __syncthreads();
  if (i < n) out[i] = wsum[warp] + inc - v;
}
__global__ void __launch_bounds__(1024) scan_sums_kernel(uint32_t* sums, int nb, uint32_t* total) {
  pdl_entry();
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < nb; base += 1024) {
    const int i = base + threadIdx.x;
    const uint32_t v = i < nb ? sums[i] : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
      if (lane >= off) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = wsum[lane], winc = w;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, winc, off);
        if (lane >= off) winc += t;
      }
      wsum[lane] = winc - w;
    }
    __syncthreads();
    const uint32_t c = carry;
    if (i < nb) sums[i] = c + wsum[warp] + inc - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = c + wsum[warp] + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}
__global__ void compact_points_kernel(const float4* __restrict__ old_pts, int n_old, const float4* __restrict__ new_pts,
                                      int n_new, const uint32_t* __restrict__ keep, const uint32_t* __restrict__ pos,
                                      const uint32_t* __restrict__ block_off, float4* __restrict__ out) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_old + n_new || !keep[i]) return;
  const uint32_t o = pos[i] + block_off[i / kScanBlock];
  out[o] = i < n_old ? old_pts[i] : new_pts[i - n_old];
}

// Add_Points(points, downsample_on): policy 1 = nearest-to-centre per `ds` voxel, 0 = plain append
int Map::insert_dev(const float* d_src, int n_new, int stride_bytes, int policy, float ds) {
  if (n_new < 0 || !valid_stride(stride_bytes)) return fail(ILSM_ERR_INVALID_ARG, "map_insert: bad n/stride");
  if (policy == 1 && !(ds > 0.f)) return fail(ILSM_ERR_INVALID_ARG, "map_insert: downsample size must be positive");
  if (n_new == 0) return ILSM_OK;
  const int n_old = n;
  const long long tot = (long long)n_old + n_new;
  if (tot > (long long)kScanBlock * 4096) return fail(ILSM_ERR_INVALID_ARG, "map_insert: more than 4 Mi points");
  cudaStream_t s = stream;
  ILSM_CUDA(cudaEventRecord(ctx_done, ctx->stream));
  ILSM_CUDA(cudaStreamWaitEvent(s, ctx_done, 0));
  int rc;
  int log2 = 10;
  while ((1u << log2) < 2u * (uint32_t)n_new) ++log2;
  const uint32_t tsize = 1u << log2;
  const int nb = (int)((tot + kScanBlock - 1) / kScanBlock);
  if ((rc = vox_table.reserve((size_t)tsize * 3)) || (rc = ins_new.reserve(n_new + 1)) ||
      (rc = ins_slot_new.reserve(n_new + 1)) || (rc = ins_slot_old.reserve(n_old + 1)) || (rc = ins_keep.reserve(tot + 1)) ||
      (rc = ins_pos.reserve(tot + 1)) || (rc = ins_bsum.reserve(nb + 2)) || (rc = ins_out.reserve(tot + 1)))
    return rc;
  VoxSlot* table = reinterpret_cast<VoxSlot*>(vox_table.p);
  const int T = 256;
  if (policy == 1) {
    ILSM_CUDA(launch_pdl(vox_clear_kernel, dim3((tsize + T - 1) / T), dim3(T), 0, s, table, tsize));
    ILSM_CUDA(launch_pdl(vox_new_kernel, dim3((n_new + T - 1) / T), dim3(T), 0, s, d_src, n_new, stride_bytes / 4, ds, table, tsize - 1, log2, ins_slot_new.p, ins_new.p));
    if (n_old > 0)
      ILSM_CUDA(launch_pdl(vox_old_kernel, dim3((n_old + T - 1) / T), dim3(T), 0, s, orig.p, n_old, ds, table, tsize - 1, log2, ins_slot_old.p));
    ILSM_CUDA(launch_pdl(vox_decide_kernel, dim3(((int)tot + T - 1) / T), dim3(T), 0, s, table, ins_slot_old.p, n_old, ins_slot_new.p, n_new, ins_keep.p));
    ILSM_CUDA(launch_pdl(scan_block_kernel, dim3(nb), dim3(kScanBlock), 0, s, ins_keep.p, (int)tot, ins_pos.p, ins_bsum.p));
    ILSM_CUDA(launch_pdl(scan_sums_kernel, dim3(1), dim3(1024), 0, s, ins_bsum.p, nb, ins_bsum.p + nb));
    ILSM_CUDA(launch_pdl(compact_points_kernel, dim3(((int)tot + T - 1) / T), dim3(T), 0, s, orig.p, n_old, ins_new.p, n_new, ins_keep.p, ins_pos.p, ins_bsum.p, ins_out.p));
    count_launches(n_old > 0 ? 7 : 6);
    // the survivor count decides the grid of the rebuild: one small D2H read (the reference's Add_Points is
    // synchronous too and returns the number of points it added)
    uint32_t h_total = 0;
    ILSM_CUDA(cudaMemcpyAsync(&h_total, ins_bsum.p + nb, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ILSM_CUDA(cudaStreamSynchronize(s));
    return build_dev(reinterpret_cast<const float*>(ins_out.p), (int)h_total, 16, cell);
  }
  // plain append (downsample_on = false)
  ILSM_CUDA(cudaMemcpyAsync(ins_out.p, orig.p, (size_t)n_old * 16, cudaMemcpyDeviceToDevice, s));
  ILSM_CUDA(launch_pdl(vox_clear_kernel, dim3((tsize + T - 1) / T), dim3(T), 0, s, table, tsize));
  ILSM_CUDA(launch_pdl(vox_new_kernel, dim3((n_new + T - 1) / T), dim3(T), 0, s, d_src, n_new, stride_bytes / 4, 1.0f, table, tsize - 1, log2, ins_slot_new.p, ins_out.p + n_old));
  count_launches(2);
  return build_dev(reinterpret_cast<const float*>(ins_out.p), (int)tot, 16, cell);
}

}  // namespace ilsm
