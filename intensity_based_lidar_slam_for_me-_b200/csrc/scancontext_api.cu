// scancontext_api.cu -- the ScanContext entry points beyond the single-query brute-force scorer:
//   ilsm_sc_query_candidates     detectLoopClosureID's own two steps (ring-key 10-NN, then only those scored)
//   ilsm_sc_query_topk_batch     B queries per call
//   ilsm_sc_init_nccl[_rank]     the database as one shard of R, NCCL communicator behind the C ABI
//   ilsm_sc_query_topk_sharded   score the local shard -> ONE ncclAllGather of the packed per-rank top-k records for
//                                the whole batch -> identical deterministic merge on every rank; nothing visits the
//                                host between the scoring kernels, the all-gather and the merge
// NCCL is resolved at run time (dlopen of the libnccl.so.2 already in the process -- torch's bundled copy under
// Python -- else the system one): libilsm_cuda.so has no link-time NCCL dependency, and a host that never shards
// never loads it.
#include <dlfcn.h>
#include <nccl.h>  // types only; every function is looked up with dlsym
#include <string.h>

#include "ilsm_host.hpp"

namespace ilsm {
int sc_merge_dev(Ctx* ctx, const void* d_packed, int shards, int k, void* d_out, int batch, size_t shard_stride);

namespace {
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  bool ok = false;
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

int nccl_load() {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.ok) return ILSM_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names)
    if ((h = dlopen(n, RTLD_NOW | RTLD_NOLOAD))) break;  // the copy already in the process (torch's bundled NCCL)
  for (const char* n : names) {
    if (h) break;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
  }
  if (!h) return fail(ILSM_ERR_STATE, "sc_init_nccl: libnccl.so.2 not found (dlopen)");
  g_nccl.lib = h;
#define ILSM_NCCL_SYM(field, name)                                                    \
  *reinterpret_cast<void**>(&g_nccl.field) = dlsym(h, name);                          \
  if (!g_nccl.field) return fail(ILSM_ERR_STATE, "sc_init_nccl: symbol " name " missing in libnccl")
  ILSM_NCCL_SYM(GetUniqueId, "ncclGetUniqueId");
  ILSM_NCCL_SYM(CommInitRank, "ncclCommInitRank");
  ILSM_NCCL_SYM(CommDestroy, "ncclCommDestroy");
  ILSM_NCCL_SYM(AllGather, "ncclAllGather");
  ILSM_NCCL_SYM(GetErrorString, "ncclGetErrorString");
  ILSM_NCCL_SYM(GetVersion, "ncclGetVersion");
#undef ILSM_NCCL_SYM
  g_nccl.ok = true;
  return ILSM_OK;
}

int nccl_fail(ncclResult_t r, const char* where) {
  char msg[256];
  snprintf(msg, sizeof(msg), "%s: NCCL error %d (%s)", where, (int)r, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  return fail(ILSM_ERR_CUDA, msg);
}
}  // namespace

void sc_nccl_release(ScDb& d) {
  if (d.nccl_comm && d.nccl_owned && g_nccl.ok) g_nccl.CommDestroy(reinterpret_cast<ncclComm_t>(d.nccl_comm));
  d.nccl_comm = nullptr, d.nccl_owned = false, d.nccl_ranks = 1, d.nccl_rank = 0;
}
}  // namespace ilsm

using namespace ilsm;

extern "C" {

ILSM_API int ilsm_sc_query_candidates(ilsm_sc* sc, const float* desc_20x60, int n_search, int num_candidates, int32_t* cand_id,
                                      float* cand_key_d2, double* cand_dist, int32_t* cand_shift) {
  if (!sc || !desc_20x60 || !cand_id || !cand_dist || !cand_shift) return fail(ILSM_ERR_INVALID_ARG, "sc_candidates: null argument");
  if (num_candidates < 1 || num_candidates > 16) return fail(ILSM_ERR_INVALID_ARG, "sc_candidates: num_candidates must be in [1,16]");
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = d.count;
  const int k = num_candidates;
  int rc;
  if ((rc = d.stage.reserve(1200 + 8)) || (rc = d.cand_out.reserve(24 * 16 + 64)) || (rc = c.pinned.reserve(4096))) return rc;
  // device layout: k x f64 distances | k x i32 ids | k x i32 shifts | k x f32 key distances
  unsigned char* o = d.cand_out.p;
  double* o_dist = reinterpret_cast<double*>(o);
  int* o_id = reinterpret_cast<int*>(o + 8 * 16);
  int* o_sh = reinterpret_cast<int*>(o + 12 * 16);
  float* o_kd = reinterpret_cast<float*>(o + 16 * 16);
  ILSM_CUDA(cudaMemcpyAsync(d.stage.p, desc_20x60, 1200 * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  if ((rc = d.candidates_dev(d.stage.p, n_search, k, o_id, o_kd, o_dist, o_sh))) return rc;
  unsigned char* pin = c.pinned.p;
  ILSM_CUDA(cudaMemcpyAsync(pin, o, 20 * 16, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  memcpy(cand_dist, pin, (size_t)k * 8);
  memcpy(cand_id, pin + 8 * 16, (size_t)k * 4);
  memcpy(cand_shift, pin + 12 * 16, (size_t)k * 4);
  if (cand_key_d2) memcpy(cand_key_d2, pin + 16 * 16, (size_t)k * 4);
  return ILSM_OK;
}

static int batch_args_ok(const ilsm_sc* sc, const void* desc, int n_queries, int k, const void* a, const void* b, const void* c3,
                         const char* who) {
  if (!sc || !desc || !a || !b || !c3) return fail(ILSM_ERR_INVALID_ARG, who);
  if (n_queries < 1 || n_queries > 4096 || k < 1 || k > 16) return fail(ILSM_ERR_INVALID_ARG, who);
  return ILSM_OK;
}

// packed device records [B][16 k] -> the caller's three host arrays ([B][k] each)
static int unpack_to_host(Ctx& c, const unsigned char* d_packed, int B, int k, double* dist, int32_t* id, int32_t* shift) {
  const size_t bytes = (size_t)B * 16 * k;
  int rc;
  if ((rc = c.pinned.reserve(bytes + 64))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(c.pinned.p, d_packed, bytes, cudaMemcpyDeviceToHost, c.stream));
  ILSM_CUDA(cudaStreamSynchronize(c.stream));
  for (int b = 0; b < B; ++b) {
    const unsigned char* r = c.pinned.p + (size_t)b * 16 * k;
    memcpy(dist + (size_t)b * k, r, (size_t)8 * k);
    memcpy(id + (size_t)b * k, r + (size_t)8 * k, (size_t)4 * k);
    memcpy(shift + (size_t)b * k, r + (size_t)12 * k, (size_t)4 * k);
  }
  return ILSM_OK;
}

ILSM_API int ilsm_sc_query_topk_batch(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                      double* dist, int32_t* id, int32_t* shift) {
  int rc = batch_args_ok(sc, desc_20x60, n_queries, k, dist, id, shift, "sc_query_batch: bad argument");
  if (rc) return rc;
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = d.count;
  if ((rc = d.qbatch.reserve((size_t)n_queries * 1200 + 8)) || (rc = d.pk_out.reserve((size_t)n_queries * 16 * k + 64))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(d.qbatch.p, desc_20x60, (size_t)n_queries * 1200 * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  if ((rc = d.query_batch_dev(d.qbatch.p, n_queries, n_search, id_offset, k, d.pk_out.p))) return rc;
  return unpack_to_host(c, d.pk_out.p, n_queries, k, dist, id, shift);
}

ILSM_API int ilsm_sc_query_topk_batch_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                          void* d_packed) {
  if (!sc || !d_desc_20x60 || !d_packed || n_queries < 1 || k < 1 || k > 16) return fail(ILSM_ERR_INVALID_ARG, "sc_query_batch_dev: bad argument");
  Ctx& c = *sc->d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = sc->d.count;
  return sc->d.query_batch_dev(d_desc_20x60, n_queries, n_search, id_offset, k, reinterpret_cast<unsigned char*>(d_packed));
}

// Testing aid: the tensor-core prefilter alone.  approx[q * n_search + c] = approximate distance (-1: pair flagged for
// exact rescoring), aligned_shift likewise (the sector-key alignment it used).  n_queries <= 8.
ILSM_API int ilsm_sc_prefilter_debug(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, float* approx,
                                     uint8_t* aligned_shift) {
  if (!sc || !desc_20x60 || !approx || !aligned_shift || n_queries < 1 || n_queries > 8) return fail(ILSM_ERR_INVALID_ARG, "sc_prefilter_debug: bad argument");
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = d.count;
  if (n_search < 1 || n_search > d.count) return fail(ILSM_ERR_INVALID_ARG, "sc_prefilter_debug: bad n_search");
  int rc;
  DevBuf<unsigned char> sh;
  if ((rc = d.qbatch.reserve((size_t)n_queries * 1200 + 8)) || (rc = d.pk_out.reserve((size_t)n_queries * 16 * 10 + 64)) ||
      (rc = sh.reserve((size_t)8 * n_search + 16)))
    return rc;
  ILSM_CUDA(cudaMemcpyAsync(d.qbatch.p, desc_20x60, (size_t)n_queries * 1200 * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  rc = d.query_batch_tc_dev(d.qbatch.p, n_queries, n_search, 0, 10, d.pk_out.p, sh.p);
  if (!rc) {
    ILSM_CUDA(cudaMemcpyAsync(approx, d.pf_dist.p, (size_t)n_queries * n_search * sizeof(float), cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaMemcpyAsync(aligned_shift, sh.p, (size_t)n_queries * n_search, cudaMemcpyDeviceToHost, c.stream));
    ILSM_CUDA(cudaStreamSynchronize(c.stream));
  }
  return rc;
}

// ------------------------------------------------------------------------------------------- sharded database (NCCL)
ILSM_API int ilsm_sc_nccl_unique_id(char id_out[128]) {
  if (!id_out) return fail(ILSM_ERR_INVALID_ARG, "sc_nccl_unique_id: null argument");
  int rc = nccl_load();
  if (rc) return rc;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) return nccl_fail(r, "ncclGetUniqueId");
  memcpy(id_out, &id, 128);
  return ILSM_OK;
}

ILSM_API int ilsm_sc_init_nccl_rank(ilsm_sc* sc, const char id[128], int n_ranks, int rank) {
  if (!sc || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(ILSM_ERR_INVALID_ARG, "sc_init_nccl_rank: bad argument");
  int rc = nccl_load();
  if (rc) return rc;
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  sc_nccl_release(d);
  ncclUniqueId uid;
  memcpy(&uid, id, 128);
  ncclComm_t comm = nullptr;
  ncclResult_t r = g_nccl.CommInitRank(&comm, n_ranks, uid, rank);
  if (r != ncclSuccess) return nccl_fail(r, "ncclCommInitRank");
  d.nccl_comm = comm, d.nccl_owned = true, d.nccl_ranks = n_ranks, d.nccl_rank = rank;
  return ILSM_OK;
}

ILSM_API int ilsm_sc_init_nccl(ilsm_sc* sc, void* nccl_comm, int n_ranks, int rank) {
  if (!sc || !nccl_comm || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(ILSM_ERR_INVALID_ARG, "sc_init_nccl: bad argument");
  int rc = nccl_load();
  if (rc) return rc;
  ScDb& d = sc->d;
  std::lock_guard<std::mutex> lk(d.ctx->mu);
  sc_nccl_release(d);
  d.nccl_comm = nccl_comm, d.nccl_owned = false, d.nccl_ranks = n_ranks, d.nccl_rank = rank;
  return ILSM_OK;
}

ILSM_API int ilsm_sc_nccl_version(int* version) {
  if (!version) return fail(ILSM_ERR_INVALID_ARG, "sc_nccl_version: null argument");
  int rc = nccl_load();
  if (rc) return rc;
  ncclResult_t r = g_nccl.GetVersion(version);
  return r == ncclSuccess ? ILSM_OK : nccl_fail(r, "ncclGetVersion");
}

// enqueue: local scoring -> all-gather -> merge, all on the context stream; the merged records land in d.pk_out
static int sharded_enqueue(ScDb& d, const float* d_q, int B, int n_search, int id_offset, int k) {
  Ctx& c = *d.ctx;
  const size_t rec = (size_t)16 * k, local = (size_t)B * rec;
  const int R = d.nccl_ranks;
  int rc;
  if ((rc = d.pk_local.reserve(local + 64)) || (rc = d.pk_all.reserve(local * R + 64)) || (rc = d.pk_out.reserve(local + 64))) return rc;
  if ((rc = d.query_batch_dev(d_q, B, n_search, id_offset, k, d.pk_local.p))) return rc;
  if (R > 1) {
    if (!d.nccl_comm) return fail(ILSM_ERR_STATE, "sc_query_sharded: no communicator (ilsm_sc_init_nccl)");
    ncclResult_t r = g_nccl.AllGather(d.pk_local.p, d.pk_all.p, local, ncclChar, reinterpret_cast<ncclComm_t>(d.nccl_comm), c.stream);
    if (r != ncclSuccess) return nccl_fail(r, "ncclAllGather");
    return sc_merge_dev(&c, d.pk_all.p, R, k, d.pk_out.p, B, local);
  }
  return sc_merge_dev(&c, d.pk_local.p, 1, k, d.pk_out.p, B, local);
}

ILSM_API int ilsm_sc_query_topk_sharded(ilsm_sc* sc, const float* desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                        double* dist, int32_t* id, int32_t* shift) {
  int rc = batch_args_ok(sc, desc_20x60, n_queries, k, dist, id, shift, "sc_query_sharded: bad argument");
  if (rc) return rc;
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = d.count;
  if ((rc = d.qbatch.reserve((size_t)n_queries * 1200 + 8))) return rc;
  ILSM_CUDA(cudaMemcpyAsync(d.qbatch.p, desc_20x60, (size_t)n_queries * 1200 * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  if ((rc = sharded_enqueue(d, d.qbatch.p, n_queries, n_search, id_offset, k))) return rc;
  return unpack_to_host(c, d.pk_out.p, n_queries, k, dist, id, shift);
}

ILSM_API int ilsm_sc_query_topk_sharded_dev(ilsm_sc* sc, const float* d_desc_20x60, int n_queries, int n_search, int id_offset, int k,
                                            void* d_packed_out) {
  if (!sc || !d_desc_20x60 || !d_packed_out || n_queries < 1 || k < 1 || k > 16)
    return fail(ILSM_ERR_INVALID_ARG, "sc_query_sharded_dev: bad argument");
  ScDb& d = sc->d;
  Ctx& c = *d.ctx;
  std::lock_guard<std::mutex> lk(c.mu);
  ILSM_CUDA(cudaSetDevice(c.device));
  if (n_search < 0) n_search = d.count;
  int rc = sharded_enqueue(d, d_desc_20x60, n_queries, n_search, id_offset, k);
  if (rc) return rc;
  ILSM_CUDA(cudaMemcpyAsync(d_packed_out, d.pk_out.p, (size_t)n_queries * 16 * k, cudaMemcpyDeviceToDevice, c.stream));
  return ILSM_OK;
}

}  // extern "C"
