// scancontext.cu -- K5: ScanContext descriptor (makeScancontext) and loop-closure candidate scoring over a
// (sharded) keyframe database with local top-k.
//
// Replaces SCManager::makeScancontext (Scancontext.cpp:160-204), makeSectorkeyFromScancontext (:222-235),
// fastAlignUsingVkey (:104-124), distDirectSC (:79-101), distanceBtnScanContext (:126-157) and the candidate loop
// of detectLoopClosureID (:299-312), scored over EVERY database entry instead of the 10 ring-key candidates (a
// superset of the reference's search; each rank of a sharded run keeps its local top-k, the ranks exchange
// k x 16 B with one all-gather and merge identically).
//
// Descriptor values are floats in the reference (SCPointType is float, widened into a MatrixXd), so the database
// is stored as float32 [20][60] row-major = 4800 B per keyframe without loss; all arithmetic is fp64 like Eigen's.
// The kernel is HBM-bound for one query (4800 B per candidate, ~12 kFLOP fp64); no tensor cores: the 7-shift
// column-cosine search after sector-key alignment is not a dense contraction at batch size 1.
#include <utility>

#include "ilsm_host.hpp"

namespace ilsm {

constexpr int kNR = 20, kNS = 60, kDesc = kNR * kNS;

struct ScQuery {  // prepared once per query, read by every scoring block
  double desc[kDesc];
  double norm[kNS];
  double key[kNS];
};

// ---------------------------------------------------------------------------------------------------
// makeScancontext: max (z + 2.0) per polar bin, empty bins -> 0
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float atan_rf(float v) { return (float)atan((double)v); }
__device__ __forceinline__ float xy2theta_dev(float x, float y) {
  const double k = 180.0 / 3.14159265358979323846;
  if (x >= 0 && y >= 0) return (float)(k * (double)atan_rf(__fdiv_rn(y, x)));
  if (x < 0 && y >= 0) return (float)(180.0 - (k * (double)atan_rf(__fdiv_rn(y, -x))));
  if (x < 0 && y < 0) return (float)(180.0 + (k * (double)atan_rf(__fdiv_rn(y, x))));
  return (float)(360.0 - (k * (double)atan_rf(__fdiv_rn(-y, x))));
}

__device__ __forceinline__ int float_order(float f) {  // monotone float -> int map for atomicMax
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float order_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF); }

__global__ void sc_make_clear_kernel(int* bins) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kDesc) bins[i] = float_order(-1000.0f);
}
__global__ void sc_make_kernel(const float* __restrict__ pts, int n, int stride_f, int* bins) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = pts + (size_t)i * stride_f;
  const float x = __ldg(p), y = __ldg(p + 1);
  const float z = (float)((double)__ldg(p + 2) + 2.0);  // LIDAR_HEIGHT, Scancontext.h:77
  const float range = __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
  const float angle = xy2theta_dev(x, y);
  if ((double)range > 80.0) return;
  int ring = __double2int_ru(((double)range / 80.0) * 20.0);
  int sector = __double2int_ru(((double)angle / 360.0) * 60.0);
  ring = max(min(kNR, ring), 1);
  sector = max(min(kNS, sector), 1);
  atomicMax(&bins[(ring - 1) * kNS + (sector - 1)], float_order(z));
}
__global__ void sc_make_finish_kernel(const int* bins, float* desc) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kDesc) {
    const float v = order_float(bins[i]);
    desc[i] = v == -1000.0f ? 0.f : v;
  }
}

// ---------------------------------------------------------------------------------------------------
// scoring
// ---------------------------------------------------------------------------------------------------
__global__ void sc_query_prep_kernel(const float* __restrict__ qdesc, ScQuery* q) {
  pdl_entry();
  qdesc += (size_t)blockIdx.x * kDesc;  // one block per query of a batch
  q += blockIdx.x;
  const int c = threadIdx.x;
  for (int i = threadIdx.x; i < kDesc; i += blockDim.x) q->desc[i] = (double)qdesc[i];
  if (c < kNS) {
    double s = 0, n2 = 0;
    for (int r = 0; r < kNR; ++r) {
      const double v = (double)qdesc[r * kNS + c];
      s += v;
      n2 += v * v;
    }
    q->key[c] = s / kNR;
    const double nrm = sqrt(n2);
    q->norm[c] = nrm != 0.0 ? 1.0 / nrm : 0.0;  // inverse column norm; 0 marks an empty column
  }
}

constexpr int kScWarps = 8;
constexpr int kTopKMax = 16;

// shared-memory layout of the scoring kernel (dynamic): the query once per block, one candidate per warp.
// Candidates are staged as the floats they are stored as and widened at use (exact), the query as doubles.
struct ScWarpSmem {
  float cd[kDesc];      // candidate descriptor as stored (widened on use: exact); half the bytes of a double copy, so three
                        // blocks (24 warps) fit an SM instead of two
  double ck2[2 * kNS];  // candidate sector key, stored twice: circshift index c - s + 60 needs no wrap
  double cin[kNS];      // inverse column norms (0 = empty column)
  u64 tk_d[kTopKMax];   // this warp's running top-k: distance bits, id, shift (ascending (d, id))
  int tk_id[kTopKMax];
  int tk_sh[kTopKMax];
};
struct ScBlockSmem {
  double qd[kDesc];
  double qin[kNS], qk[kNS];
  ScWarpSmem w[kScWarps];
};

__device__ __forceinline__ bool sc_key_less(u64 da, int ia, u64 db, int ib) { return da < db || (da == db && ia < ib); }
// Distances travel through the top-k machinery as 64-bit keys whose unsigned order is the order of the doubles --
// INCLUDING negative ones: 1 - mean(cos) of a descriptor against itself can come out as -2e-16, and raw IEEE bits would
// sort that last.  +inf maps below the all-ones "nothing" key.
__device__ __forceinline__ u64 dkey(double d) {
  const u64 b = (u64)__double_as_longlong(d);
  return b ^ ((b >> 63) ? ~0ull : 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(u64 k) {
  return __longlong_as_double((long long)(k ^ ((k >> 63) ? 0x8000000000000000ull : ~0ull)));
}

// One warp per candidate keyframe, grid-stride; every warp keeps its k best (distance, id) in shared memory, the
// block merges its warps' lists at the end and writes k entries, a small second kernel merges the blocks' lists.
//   fastAlignUsingVkey  (Scancontext.cpp:104-124): argmin_s || qk - circshift(ck, s) ||, first minimum wins
//   distDirectSC        (:79-101)                : 1 - mean over columns with both norms != 0 of cos(col_q, col_c)
//   distanceBtnScanContext (:126-157)            : the 7 shifts around the aligned one, ascending, first minimum wins
// kList: score only the entries named by cand_keys[0, n) (low word = database index; ~0 = none) and write each one's
// (distance, shift) to list_dist / list_shift in list order -- the candidate loop of detectLoopClosureID
// (Scancontext.cpp:299-312) over the ring-key candidates -- instead of keeping a top-k over the whole database.
// kMode 2 (indirect): the entries come from a per-query list as well (cand_keys[0, *n_ptr), built by the tensor-core
// prefilter, scancontext_tc.cu) but the block keeps a top-k like the full scan.  blockIdx.y = query of the batch: the
// query record, the list (list_stride entries apart) and the per-block outputs are offset by it.
template <int kMode>
__global__ void __launch_bounds__(kScWarps * 32, 3)
    sc_score_kernel(const float* __restrict__ db, int n, const ScQuery* __restrict__ q, int k, u64* __restrict__ part_d,
                    int* __restrict__ part_id, int* __restrict__ part_sh, const u64* __restrict__ cand_keys,
                    double* __restrict__ list_dist, int* __restrict__ list_shift, const int* __restrict__ n_ptr, int list_stride) {
  pdl_entry();
  constexpr bool kList = kMode == 1;
  if (kMode == 2) {
    const int y = blockIdx.y;
    q += y;
    cand_keys += (size_t)y * list_stride;
    n = min(n_ptr[y], list_stride);
    part_d += (size_t)y * gridDim.x * k, part_id += (size_t)y * gridDim.x * k, part_sh += (size_t)y * gridDim.x * k;
  }
  extern __shared__ __align__(16) unsigned char sc_smem_raw[];
  ScBlockSmem& sm = *reinterpret_cast<ScBlockSmem*>(sc_smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ScWarpSmem& w = sm.w[warp];
  for (int i = threadIdx.x; i < kDesc; i += blockDim.x) sm.qd[i] = q->desc[i];
  if (threadIdx.x < kNS) sm.qin[threadIdx.x] = q->norm[threadIdx.x], sm.qk[threadIdx.x] = q->key[threadIdx.x];
  if (lane < kTopKMax) w.tk_d[lane] = ~0ull, w.tk_id[lane] = INT_MAX, w.tk_sh[lane] = 0;
  __syncthreads();
  const int nwarps = gridDim.x * kScWarps;
  for (int item = blockIdx.x * kScWarps + warp; item < n; item += nwarps) {
    int cand = item;
    if (kMode == 2) cand = (int)(uint32_t)cand_keys[item];
    if (kList) {
      const u64 ck = cand_keys[item];
      if (ck == ~0ull) {  // fewer database entries than candidates asked for
        if (lane == 0) list_dist[item] = __longlong_as_double(0x7ff0000000000000ll), list_shift[item] = 0;
        continue;
      }
      cand = (int)(uint32_t)ck;
    }
    // stage the candidate: 4800 B of coalesced 128-bit loads, kept as float
    const float4* src = reinterpret_cast<const float4*>(db + (size_t)cand * kDesc);
    for (int i = lane; i < kDesc / 4; i += 32) reinterpret_cast<float4*>(w.cd)[i] = __ldg(src + i);
    __syncwarp();
    // sector key (column means) and inverse column norms of the candidate
    for (int c = lane; c < kNS; c += 32) {
      double s = 0, n2 = 0;
      const float* col = w.cd + c;
#pragma unroll
      for (int r = 0; r < kNR; ++r) {
        const double v = (double)col[r * kNS];
        s += v;
        n2 = fma(v, v, n2);  // v is a widened float: v * v is exact in double, so the fused form rounds identically
      }
      const double key = s / kNR;
      w.ck2[c] = key, w.ck2[c + kNS] = key;
      w.cin[c] = n2 != 0.0 ? frsqrt(n2) : 0.0;
    }
    __syncwarp();
    // fastAlignUsingVkey: lane -> shifts s = lane and lane + 32, each a sequential sum over the 60 columns; the two
    // sums are independent dependency chains and share the query-key load
    double best = 10000000;
    int arg = 0;
    {
      const int s1 = lane + 32 < kNS ? lane + 32 : lane;  // lanes 28..31 repeat their first shift (result unused)
      const double* ckp0 = w.ck2 + (kNS - lane);          // ckp[c] = ck[(c - s) mod 60]
      const double* ckp1 = w.ck2 + (kNS - s1);
      double ss0 = 0, ss1 = 0;
#pragma unroll 10
      for (int c = 0; c < kNS; ++c) {
        const double qv = sm.qk[c];
        const double d0 = qv - ckp0[c], d1 = qv - ckp1[c];
        ss0 += d0 * d0;
        ss1 += d1 * d1;
      }
      const double n0 = sqrt(ss0), n1 = sqrt(ss1);
      if (n0 < best) best = n0, arg = lane;  // ascending s within the lane, first minimum wins
      if (lane + 32 < kNS && n1 < best) best = n1, arg = lane + 32;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, off);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, off);
      if (ob < best || (ob == best && oa < arg)) best = ob, arg = oa;
    }
    // the 7 shifts around the aligned one in ascending order: a run arg-3 .. arg+3 that may wrap once
    int shifts[7];
    {
      const int lo = arg - 3, hi = arg + 3;
      // wrapped members (lo + t < 0 -> +60, lo + t > 59 -> -60) sort before / after the unwrapped ones
      const int n_hi_wrap = hi > kNS - 1 ? hi - (kNS - 1) : 0;  // values 0 .. n_hi_wrap-1 come first
      const int n_lo_wrap = lo < 0 ? -lo : 0;                   // values 60+lo .. 59 come last
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        int v;
        if (t < n_hi_wrap) v = t;                                    // wrapped high end
        else if (t >= 7 - n_lo_wrap) v = kNS + lo + (t - (7 - n_lo_wrap));  // wrapped low end
        else v = lo + n_lo_wrap + (t - n_hi_wrap);                   // the unwrapped run, ascending
        shifts[t] = v;
      }
    }
    double sum[7];
    int eff[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) sum[t] = 0.0, eff[t] = 0;
    for (int j = lane; j < kNS; j += 32) {
      const double iq = sm.qin[j];
      int jb[7];
      double dot[7];
      const float* ccol[7];
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        int b = j - shifts[t];
        jb[t] = b + (b < 0 ? kNS : 0);
        ccol[t] = w.cd + jb[t];
        dot[t] = 0.0;
      }
      const double* qcol = sm.qd + j;
#pragma unroll
      for (int r = 0; r < kNR; ++r) {  // fully unrolled: immediate shared-memory offsets, 1 + 7 loads and 7 DFMA per row
        const double qv = qcol[r * kNS];
#pragma unroll
        for (int t = 0; t < 7; ++t) dot[t] = fma(qv, (double)ccol[t][r * kNS], dot[t]);  // products of widened floats are exact
      }
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        const double ic = w.cin[jb[t]];
        if (iq != 0.0 && ic != 0.0) {
          sum[t] += dot[t] * (iq * ic);
          eff[t] += 1;
        }
      }
    }
    // warp totals: the 7 effective-column counts (each <= 60) travel packed in one 64-bit word
    u64 effp = 0;
#pragma unroll
    for (int t = 0; t < 7; ++t) effp |= (u64)eff[t] << (8 * t);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      effp += __shfl_xor_sync(0xffffffffu, effp, off);
#pragma unroll
      for (int t = 0; t < 7; ++t) sum[t] += __shfl_xor_sync(0xffffffffu, sum[t], off);
    }
    // lane t < 7 turns shift t's totals into a distance (one division per lane instead of seven per warp), then the
    // first minimum in ascending shift order wins: arg-min on (distance, t)
    double myd = __longlong_as_double(0x7ff0000000000000ll);
    int mysh = 0, myt = 99;
    {
      // select this lane's shift with predicated moves, then ONE division per lane: seven `if (lane == t)` bodies would
      // be seven serialised division sequences (~210 instructions per candidate)
      double s_t = 0.0;
      int sh_t = 0;
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        s_t = lane == t ? sum[t] : s_t;
        sh_t = lane == t ? shifts[t] : sh_t;
      }
      const int ek = lane < 7 ? (int)((effp >> (8 * lane)) & 0xFF) : 0;
      if (lane < 7) {
        if (ek > 0) myd = 1.0 - s_t / (double)ek;
        mysh = sh_t, myt = lane;
      }
    }
    const bool cand_ok = lane < 7 && myd < 10000000.0;  // min_sc_dist starts at 10000000 (strict <)
    if (!cand_ok) myd = 10000000.0, mysh = 0, myt = 99;
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, myd, off);
      const int os = __shfl_xor_sync(0xffffffffu, mysh, off);
      const int ot = __shfl_xor_sync(0xffffffffu, myt, off);
      if (od < myd || (od == myd && ot < myt)) myd = od, mysh = os, myt = ot;
    }
    const double bd = __shfl_sync(0xffffffffu, myd, 0);
    const int bs = __shfl_sync(0xffffffffu, mysh, 0);
    if (kList) {
      // distanceBtnScanContext's result as it is (10000000 when no shift had an effective column: never < min_dist)
      if (lane == 0) list_dist[item] = bd, list_shift[item] = bs;
    } else if (lane == 0) {  // insertion into this warp's sorted top-k
      const u64 kd = dkey(bd);
      if (sc_key_less(kd, cand, w.tk_d[k - 1], w.tk_id[k - 1])) {
        int pos = k - 1;
        while (pos > 0 && sc_key_less(kd, cand, w.tk_d[pos - 1], w.tk_id[pos - 1])) {
          w.tk_d[pos] = w.tk_d[pos - 1], w.tk_id[pos] = w.tk_id[pos - 1], w.tk_sh[pos] = w.tk_sh[pos - 1];
          --pos;
        }
        w.tk_d[pos] = kd, w.tk_id[pos] = cand, w.tk_sh[pos] = bs;
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (kList) return;
  if (threadIdx.x == 0) {  // k-way merge of the warps' lists (heads only): k x kScWarps comparisons
    int head[kScWarps];
#pragma unroll
    for (int i = 0; i < kScWarps; ++i) head[i] = 0;
    for (int j = 0; j < k; ++j) {
      int bw = 0;
#pragma unroll
      for (int i = 1; i < kScWarps; ++i) {
        const ScWarpSmem &a = sm.w[i], &b = sm.w[bw];
        if (sc_key_less(a.tk_d[head[i]], a.tk_id[head[i]], b.tk_d[head[bw]], b.tk_id[head[bw]])) bw = i;
      }
      const ScWarpSmem& b = sm.w[bw];
      const size_t o = (size_t)blockIdx.x * k + j;
      part_d[o] = b.tk_d[head[bw]], part_id[o] = b.tk_id[head[bw]], part_sh[o] = b.tk_sh[head[bw]];
      // exhausted lists present (~0, INT_MAX) sentinels: k <= kTopKMax keeps head within the array
      if (head[bw] < kTopKMax - 1) head[bw]++;
      else sm.w[bw].tk_d[kTopKMax - 1] = ~0ull, sm.w[bw].tk_id[kTopKMax - 1] = INT_MAX;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// ring keys and the reference's candidate selection (Scancontext.cpp:206-220, 270-295)
// ---------------------------------------------------------------------------------------------------
// makeRingkeyFromScancontext + eig2stdvec: row means in double, stored as float (polarcontext_invkeys_mat_).
__global__ void sc_ringkey_kernel(const float* __restrict__ db, int first, int count, float* __restrict__ keys) {
  pdl_entry();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * kNR) return;
  const int e = first + t / kNR, r = t % kNR;
  const float* row = db + (size_t)e * kDesc + r * kNS;
  double s = 0;
  for (int c = 0; c < kNS; ++c) s += (double)row[c];
  keys[(size_t)e * kNR + r] = (float)(s / kNS);
}

// nanoflann L2_Adaptor<float>::evalMetric over 20 dimensions (the metric of KDTreeVectorOfVectorsAdaptor,
// include/nanoflann.hpp): groups of four, result += ((d0*d0 + d1*d1) + d2*d2) + d3*d3, float, no FMA.
__device__ __forceinline__ float ringkey_l2(const float* q, const float4* key5) {
  float result = 0.f;
#pragma unroll
  for (int g = 0; g < kNR / 4; ++g) {
    const float4 b = __ldg(key5 + g);
    const float d0 = __fsub_rn(q[4 * g], b.x), d1 = __fsub_rn(q[4 * g + 1], b.y), d2 = __fsub_rn(q[4 * g + 2], b.z),
                d3 = __fsub_rn(q[4 * g + 3], b.w);
    result = __fadd_rn(result, __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)), __fmul_rn(d3, d3)));
  }
  return result;
}

// block-wide k smallest of one u64 per thread (unique keys; ~0 = none), written in ascending order
__device__ __forceinline__ void block_k_smallest(u64 mine, int k, u64* __restrict__ out) {
  __shared__ u64 s_w[32];
  __shared__ u64 s_win;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int round = 0; round < k; ++round) {
    u64 m = mine;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const u64 o = __shfl_xor_sync(0xffffffffu, m, off);
      m = o < m ? o : m;
    }
    if (lane == 0) s_w[warp] = m;
    __syncthreads();
    if (warp == 0) {
      u64 w = lane < nw ? s_w[lane] : ~0ull;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const u64 o = __shfl_xor_sync(0xffffffffu, w, off);
        w = o < w ? o : w;
      }
      if (lane == 0) s_win = w, out[round] = w;
    }
    __syncthreads();
    if (mine == s_win) mine = ~0ull;
    __syncthreads();
  }
}

// stage 1: every thread one database ring key -> (float distance bits, index) -> the block's k smallest
__global__ void __launch_bounds__(1024)
    sc_ringkey_select_kernel(const float* __restrict__ keys, int n, const float* __restrict__ qdesc, int k, u64* __restrict__ part) {
  pdl_entry();
  __shared__ float qk[kNR];
  if (threadIdx.x < kNR) {  // the query's own ring key, the same arithmetic as sc_ringkey_kernel
    const float* row = qdesc + threadIdx.x * kNS;
    double s = 0;
    for (int c = 0; c < kNS; ++c) s += (double)row[c];
    qk[threadIdx.x] = (float)(s / kNS);
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  u64 mine = ~0ull;
  if (i < n) mine = ((u64)__float_as_uint(ringkey_l2(qk, reinterpret_cast<const float4*>(keys + (size_t)i * kNR))) << 32) | (uint32_t)i;
  block_k_smallest(mine, k, part + (size_t)blockIdx.x * k);
}

// stage 2: the k smallest of the blocks' lists (m entries), ascending (distance, index) = nanoflann's result order
__global__ void __launch_bounds__(1024) sc_ringkey_final_kernel(const u64* __restrict__ part, int m, int k, u64* __restrict__ out) {
  pdl_entry();
  // a thread's strided slice is reduced to its smallest entry above the previous winner, round by round
  __shared__ u64 s_last;
  if (threadIdx.x == 0) s_last = 0;
  __syncthreads();
  for (int round = 0; round < k; ++round) {
    const u64 last = s_last;
    u64 mine = ~0ull;
    for (int e = threadIdx.x; e < m; e += blockDim.x) {
      const u64 v = part[e];
      if ((round == 0 || v > last) && v < mine) mine = v;
    }
    __syncthreads();
    block_k_smallest(mine, 1, out + round);
    if (threadIdx.x == 0) s_last = out[round];
    __syncthreads();
  }
}

// candidate list -> ids and float key distances for the caller
__global__ void sc_list_unpack_kernel(const u64* __restrict__ sel, int k, int* __restrict__ id, float* __restrict__ key_d2) {
  pdl_entry();
  const int i = threadIdx.x;
  if (i >= k) return;
  const u64 v = sel[i];
  id[i] = v == ~0ull ? -1 : (int)(uint32_t)v;
  key_d2[i] = v == ~0ull ? __int_as_float(0x7f800000) : __uint_as_float((uint32_t)(v >> 32));
}

// Final merge of the blocks' lists (n = blocks * k entries, a few thousand): every thread holds up to kFinalPer
// entries, k rounds of a block-wide arg-min on (distance bits, id).
constexpr int kFinalThreads = 1024, kFinalPer = 8;
__global__ void __launch_bounds__(kFinalThreads)
    sc_topk_final_kernel(const u64* __restrict__ part_d, const int* __restrict__ part_id, const int* __restrict__ part_sh, int n,
                         int id_offset, int k, double* __restrict__ o_dist, int* __restrict__ o_id, int* __restrict__ o_shift,
                         unsigned char* __restrict__ o_packed) {
  pdl_entry();
  if (o_packed) {  // batched: block b merges query b's n entries into record b of the packed output (16 k bytes each)
    part_d += (size_t)blockIdx.x * n, part_id += (size_t)blockIdx.x * n, part_sh += (size_t)blockIdx.x * n;
    unsigned char* rec = o_packed + (size_t)blockIdx.x * 16 * k;
    o_dist = reinterpret_cast<double*>(rec), o_id = reinterpret_cast<int*>(rec + (size_t)8 * k), o_shift = reinterpret_cast<int*>(rec + (size_t)12 * k);
  }
  __shared__ u64 s_d[32];
  __shared__ int s_id[32], s_sh[32];
  __shared__ int s_win;
  u64 d[kFinalPer];
  int id[kFinalPer], sh[kFinalPer];
#pragma unroll
  for (int e = 0; e < kFinalPer; ++e) {
    const int i = threadIdx.x + e * kFinalThreads;
    const bool in = i < n;
    d[e] = in ? part_d[i] : ~0ull;
    id[e] = in ? part_id[i] : INT_MAX;
    sh[e] = in ? part_sh[i] : 0;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int round = 0; round < k; ++round) {
    u64 md = ~0ull;
    int mi = INT_MAX, ms = 0;
#pragma unroll
    for (int e = 0; e < kFinalPer; ++e)
      if (sc_key_less(d[e], id[e], md, mi)) md = d[e], mi = id[e], ms = sh[e];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const u64 od = __shfl_xor_sync(0xffffffffu, md, off);
      const int oi = __shfl_xor_sync(0xffffffffu, mi, off);
      const int os = __shfl_xor_sync(0xffffffffu, ms, off);
      if (sc_key_less(od, oi, md, mi)) md = od, mi = oi, ms = os;
    }
    if (lane == 0) s_d[warp] = md, s_id[warp] = mi, s_sh[warp] = ms;
    __syncthreads();
    if (warp == 0) {
      u64 wd = s_d[lane];
      int wi = s_id[lane], wsft = s_sh[lane];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const u64 od = __shfl_xor_sync(0xffffffffu, wd, off);
        const int oi = __shfl_xor_sync(0xffffffffu, wi, off);
        const int os = __shfl_xor_sync(0xffffffffu, wsft, off);
        if (sc_key_less(od, oi, wd, wi)) wd = od, wi = oi, wsft = os;
      }
      if (lane == 0) {
        s_win = wi;
        const bool have = wi != INT_MAX;
        o_dist[round] = have ? dkey_inv(wd) : __longlong_as_double(0x7ff0000000000000ll);
        o_id[round] = have ? wi + id_offset : -1;
        o_shift[round] = have ? wsft : 0;
      }
    }
    __syncthreads();
    const int win = s_win;
    if (win != INT_MAX) {
#pragma unroll
      for (int e = 0; e < kFinalPer; ++e)
        if (id[e] == win) d[e] = ~0ull, id[e] = INT_MAX;
    }
    __syncthreads();
  }
}

// Merge of gathered per-shard top-k lists on the device (what every rank runs after the all-gather).  Packed layout
// per shard: k x f64 distance | k x i32 id | k x i32 shift (16 k bytes).  One warp; round j picks the smallest
// (distance, id) strictly above round j-1's winner (ids are unique across shards), so the result is the same
// ascending (distance, id) order as ilsm_sc_merge_topk on the host.
// Batched form: block b merges query b; shard r's record of query b sits at packed + r * shard_stride + b * 16 k (the
// layout an all-gather of per-rank [B][16 k] buffers produces), the merged record goes to out + b * 16 k.
__global__ void sc_merge_kernel(const unsigned char* __restrict__ packed, int shards, int k, unsigned char* __restrict__ out,
                                size_t shard_stride) {
  pdl_entry();
  const int lane = threadIdx.x;
  const size_t rec = (size_t)16 * k;
  packed += (size_t)blockIdx.x * rec;
  out += (size_t)blockIdx.x * rec;
  u64 last_d = 0;
  int last_id = -1;
  bool first = true;
  double* o_dist = reinterpret_cast<double*>(out);
  int* o_id = reinterpret_cast<int*>(out + (size_t)8 * k);
  int* o_shift = reinterpret_cast<int*>(out + (size_t)12 * k);
  for (int j = 0; j < k; ++j) {
    u64 bd = ~0ull;
    int bid = INT_MAX, bsh = 0;
    for (int e = lane; e < shards * k; e += 32) {
      const unsigned char* base = packed + (size_t)(e / k) * shard_stride;
      const int i = e % k;
      const int id = reinterpret_cast<const int*>(base + (size_t)8 * k)[i];
      if (id < 0) continue;
      const u64 d = dkey(reinterpret_cast<const double*>(base)[i]);
      const bool above = first || d > last_d || (d == last_d && id > last_id);
      if (above && (d < bd || (d == bd && id < bid))) bd = d, bid = id, bsh = reinterpret_cast<const int*>(base + (size_t)12 * k)[i];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const u64 od = __shfl_xor_sync(0xffffffffu, bd, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bid, off);
      const int os = __shfl_xor_sync(0xffffffffu, bsh, off);
      if (od < bd || (od == bd && oi < bid)) bd = od, bid = oi, bsh = os;
    }
    const bool have = bid != INT_MAX;
    if (lane == 0) {
      o_dist[j] = have ? dkey_inv(bd) : __longlong_as_double(0x7ff0000000000000ll);
      o_id[j] = have ? bid : -1;
      o_shift[j] = have ? bsh : 0;
    }
    if (have) last_d = bd, last_id = bid, first = false;
    else last_d = ~0ull, last_id = INT_MAX, first = false;
  }
}

int sc_merge_dev(Ctx* ctx, const void* d_packed, int shards, int k, void* d_out, int batch, size_t shard_stride) {
  if (shard_stride == 0) shard_stride = (size_t)16 * k;
  ILSM_CUDA(launch_pdl(sc_merge_kernel, dim3(batch), dim3(32), 0, ctx->stream, reinterpret_cast<const unsigned char*>(d_packed), shards, k,
                       reinterpret_cast<unsigned char*>(d_out), shard_stride));
  count_launches(1);
  return check_launch("sc_merge");
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
ScDb::ScDb() = default;
ScDb::~ScDb() = default;

int ScDb::append_dev(const float* d_desc, int n_add, bool from_host) {
  if (n_add <= 0) return ILSM_OK;
  const size_t need = (size_t)(count + n_add) * kDesc;
  if (need > db.cap) {  // grow and keep the contents
    DevBuf<float> bigger;
    int rc = bigger.reserve(need * 2);
    if (rc) return rc;
    if (count > 0)
      ILSM_CUDA(cudaMemcpyAsync(bigger.p, db.p, (size_t)count * kDesc * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    ILSM_CUDA(cudaStreamSynchronize(ctx->stream));
    db = std::move(bigger);
  }
  ILSM_CUDA(cudaMemcpyAsync(db.p + (size_t)count * kDesc, d_desc, (size_t)n_add * kDesc * sizeof(float),
                            from_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
  // polarcontext_invkeys_mat_.push_back(ring key as floats)  Scancontext.cpp:243,249
  const size_t need_k = (size_t)(count + n_add) * kNR;
  if (need_k > ringkey.cap) {
    DevBuf<float> bigger;
    int rc = bigger.reserve(need_k * 2);
    if (rc) return rc;
    if (count > 0)
      ILSM_CUDA(cudaMemcpyAsync(bigger.p, ringkey.p, (size_t)count * kNR * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    ILSM_CUDA(cudaStreamSynchronize(ctx->stream));
    ringkey = std::move(bigger);
  }
  ILSM_CUDA(launch_pdl(sc_ringkey_kernel, dim3((n_add * kNR + 255) / 256), dim3(256), 0, ctx->stream, (const float*)db.p, count, n_add,
                       ringkey.p));
  count_launches(1);
  count += n_add;
  return check_launch("sc_add");
}

int ScDb::make_dev(const float* d_pts, int n, int stride_bytes, float* d_desc) {
  int rc;
  if ((rc = bins.reserve(kDesc))) return rc;
  cudaStream_t s = ctx->stream;
  ILSM_CUDA(launch_pdl(sc_make_clear_kernel, dim3((kDesc + 255) / 256), dim3(256), 0, s, bins.p));
  if (n > 0) ILSM_CUDA(launch_pdl(sc_make_kernel, dim3((n + 255) / 256), dim3(256), 0, s, d_pts, n, stride_bytes / 4, bins.p));
  ILSM_CUDA(launch_pdl(sc_make_finish_kernel, dim3((kDesc + 255) / 256), dim3(256), 0, s, bins.p, d_desc));
  count_launches(n > 0 ? 3 : 2);
  return check_launch("sc_make");
}

int ScDb::query_dev(const float* d_qdesc, int n_search, int id_offset, int k, double* d_dist, int* d_id, int* d_shift) {
  n_search = searched(n_search);
  if (k < 1 || k > kTopKMax) return fail(ILSM_ERR_INVALID_ARG, "sc_query: k must be in [1,16]");
  if (n_search < 0 || n_search > count) return fail(ILSM_ERR_INVALID_ARG, "sc_query: n_search exceeds the database");
  // two resident blocks of 8 warps per SM; fewer blocks when the shard is small.  The final merge holds at most
  // kFinalThreads * kFinalPer entries.
  long long blocks = ((long long)n_search + kScWarps - 1) / kScWarps, cap = (long long)ctx->sm_count * 3;  // three resident blocks per SM
  if (blocks > cap) blocks = cap;
  if (blocks * k > (long long)kFinalThreads * kFinalPer) blocks = (long long)kFinalThreads * kFinalPer / k;
  if (blocks < 1) blocks = 1;
  int rc;
  if ((rc = query.reserve(1)) || (rc = part_d.reserve((size_t)blocks * kTopKMax)) ||
      (rc = part_id.reserve((size_t)blocks * kTopKMax)) || (rc = part_sh.reserve((size_t)blocks * kTopKMax)))
    return rc;
  cudaStream_t s = ctx->stream;
  ILSM_CUDA(cudaFuncSetAttribute(sc_score_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScBlockSmem)));
  ILSM_CUDA(launch_pdl(sc_query_prep_kernel, dim3(1), dim3(64), 0, s, d_qdesc, query.p));
  ILSM_CUDA(launch_pdl(sc_score_kernel<0>, dim3((unsigned)blocks), dim3(kScWarps * 32), sizeof(ScBlockSmem), s, (const float*)db.p, n_search,
                       (const ScQuery*)query.p, k, part_d.p, part_id.p, part_sh.p, (const u64*)nullptr, (double*)nullptr, (int*)nullptr,
                       (const int*)nullptr, 0));
  ILSM_CUDA(launch_pdl(sc_topk_final_kernel, dim3(1), dim3(kFinalThreads), 0, s, part_d.p, part_id.p, part_sh.p, (int)(blocks * k), id_offset, k, d_dist, d_id, d_shift,
                       (unsigned char*)nullptr));
  count_launches(3);
  return check_launch("sc_query");
}

// B queries against the shard, one after the other on the stream (the scoring kernel already fills the GPU for one
// query); record b of d_packed receives query b's top-k in the packed layout (k x f64 | k x i32 | k x i32).
// Exact scoring of per-query candidate lists (built by the prefilter): B queries, lists list_cap entries apart, lengths
// on the device; writes B packed top-k records.
int sc_score_lists_dev(ScDb* d, const float* d_qdesc, int B, int k, const u64* d_lists, const int* d_list_n, int list_cap, int id_offset,
                       int n_search, unsigned char* d_packed) {
  Ctx* ctx = d->ctx;
  // lists hold tens to a few thousand entries (mostly pairs whose alignment the prefilter could not decide)
  const int blocks = 48;
  int rc;
  if ((rc = d->query.reserve(B)) || (rc = d->part_d.reserve((size_t)B * blocks * kTopKMax)) || (rc = d->part_id.reserve((size_t)B * blocks * kTopKMax)) ||
      (rc = d->part_sh.reserve((size_t)B * blocks * kTopKMax)))
    return rc;
  cudaStream_t s = ctx->stream;
  ILSM_CUDA(cudaFuncSetAttribute(sc_score_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScBlockSmem)));
  ILSM_CUDA(launch_pdl(sc_query_prep_kernel, dim3(B), dim3(64), 0, s, d_qdesc, d->query.p));
  ILSM_CUDA(launch_pdl(sc_score_kernel<2>, dim3(blocks, B), dim3(kScWarps * 32), sizeof(ScBlockSmem), s, (const float*)d->db.p, 0,
                       (const ScQuery*)d->query.p, k, d->part_d.p, d->part_id.p, d->part_sh.p, d_lists, (double*)nullptr, (int*)nullptr, d_list_n,
                       list_cap));
  ILSM_CUDA(launch_pdl(sc_topk_final_kernel, dim3(B), dim3(kFinalThreads), 0, s, (const u64*)d->part_d.p, (const int*)d->part_id.p,
                       (const int*)d->part_sh.p, blocks * k, id_offset, k, (double*)nullptr, (int*)nullptr, (int*)nullptr, d_packed));
  count_launches(3);
  return check_launch("sc_score_lists");
}

int ScDb::query_batch_dev(const float* d_qdesc, int B, int n_search, int id_offset, int k, unsigned char* d_packed) {
  n_search = searched(n_search);
  // large shards: approximate scoring of every pair on the tensor cores, exact rescoring of the few that can matter
  if (n_search >= tc_min) return query_batch_tc_dev(d_qdesc, B, n_search, id_offset, k, d_packed, nullptr);
  for (int b = 0; b < B; ++b) {
    unsigned char* base = d_packed + (size_t)b * 16 * k;
    int rc = query_dev(d_qdesc + (size_t)b * kDesc, n_search, id_offset, k, reinterpret_cast<double*>(base),
                       reinterpret_cast<int*>(base + (size_t)8 * k), reinterpret_cast<int*>(base + (size_t)12 * k));
    if (rc) return rc;
  }
  return ILSM_OK;
}

// detectLoopClosureID's two steps (Scancontext.cpp:283-312) over entries [0, n_search): the num_cand nearest ring keys
// (float L2 as nanoflann evaluates it, ties by lower index), then distanceBtnScanContext for exactly those, in that
// order.  Outputs (device): ids, float key distances, distances, shifts -- num_cand entries each, id -1 when the
// database holds fewer entries.
int ScDb::candidates_dev(const float* d_qdesc, int n_search, int num_cand, int* d_id, float* d_key_d2, double* d_dist, int* d_shift) {
  n_search = searched(n_search);
  if (num_cand < 1 || num_cand > kTopKMax) return fail(ILSM_ERR_INVALID_ARG, "sc_candidates: num_candidates must be in [1,16]");
  if (n_search < 0 || n_search > count) return fail(ILSM_ERR_INVALID_ARG, "sc_candidates: n_search exceeds the database");
  const int blocks = n_search > 0 ? (n_search + 1023) / 1024 : 1;
  int rc;
  if ((rc = query.reserve(1)) || (rc = rk_part.reserve((size_t)blocks * kTopKMax + kTopKMax))) return rc;
  u64* sel = rk_part.p + (size_t)blocks * kTopKMax;
  cudaStream_t s = ctx->stream;
  ILSM_CUDA(launch_pdl(sc_ringkey_select_kernel, dim3(blocks), dim3(1024), 0, s, (const float*)ringkey.p, n_search, d_qdesc, num_cand, rk_part.p));
  ILSM_CUDA(launch_pdl(sc_ringkey_final_kernel, dim3(1), dim3(1024), 0, s, (const u64*)rk_part.p, blocks * num_cand, num_cand, sel));
  ILSM_CUDA(launch_pdl(sc_list_unpack_kernel, dim3(1), dim3(32), 0, s, (const u64*)sel, num_cand, d_id, d_key_d2));
  ILSM_CUDA(cudaFuncSetAttribute(sc_score_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScBlockSmem)));
  ILSM_CUDA(launch_pdl(sc_query_prep_kernel, dim3(1), dim3(64), 0, s, d_qdesc, query.p));
  ILSM_CUDA(launch_pdl(sc_score_kernel<1>, dim3((num_cand + kScWarps - 1) / kScWarps), dim3(kScWarps * 32), sizeof(ScBlockSmem), s,
                       (const float*)db.p, num_cand, (const ScQuery*)query.p, num_cand, (u64*)nullptr, (int*)nullptr, (int*)nullptr, (const u64*)sel,
                       d_dist, d_shift, (const int*)nullptr, 0));
  count_launches(5);
  return check_launch("sc_candidates");
}

}  // namespace ilsm
