// sip_comm.cu -- multi-GPU layer of the C ABI (SURVEY 8e; include/sipnet_gpu.h "multi-GPU").
//
// Members are independent, so `run` needs no communication: every rank (one rank = one GPU) integrates its share.
// NCCL appears only in the final gather:
//   * log-likelihoods: one all-gather of a double per member, rank-major;
//   * ensemble summaries of a site whose members are spread over ranks: the lockstep select of sip_gsum.cu --
//     per level an all-reduce of 8 KB of histogram per row, plus small all-gathers -- instead of moving the
//     members' values (1 MB per row and rank at 131072 members).
// Two ways to form the team, same code below:
//   * one process per GPU (torchrun, MPI, ...): sipnet_gpu_comm_init_rank() with an id made by rank 0 and
//     broadcast by the caller's launcher;
//   * one process, one host thread, all GPUs: sipnet_gpu_multi_* (ncclCommInitAll, grouped calls).
// The host sides of the ensemble adjustment Kalman filter (kernels: sip_assim.cu), of the particle filter
// (sip_resample.cu) and of its parameter move (sip_jitter.cu) live here too: a single handle runs them as a team of
// one, which needs no exchange.
// NCCL is bound at run time (dlopen of libnccl.so.2): single-GPU use never loads it, and a process that already
// carries an NCCL (e.g. PyTorch's) shares that copy.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <numeric>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "sip_assim.cuh"
#include "sip_gsum.cuh"
#include "sip_handle.h"
#include "sip_jitter.cuh"
#include "sip_resample.cuh"

using namespace sip;

namespace {

struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

const NcclApi *nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api.lib ? &api : nullptr;
  tried = true;
  const char *names[] = {getenv("SIPNET_GPU_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void *lib = nullptr;
  for (const char *n : names) {
    if (!n || !*n) continue;
    lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (lib) break;
  }
  if (!lib) return nullptr;
#define SIP_BIND(field, sym)                                              \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(lib, sym));      \
  if (!api.field) return nullptr;
  SIP_BIND(GetUniqueId, "ncclGetUniqueId")
  SIP_BIND(CommInitRank, "ncclCommInitRank")
  SIP_BIND(CommInitAll, "ncclCommInitAll")
  SIP_BIND(CommDestroy, "ncclCommDestroy")
  SIP_BIND(AllReduce, "ncclAllReduce")
  SIP_BIND(AllGather, "ncclAllGather")
  SIP_BIND(Send, "ncclSend")
  SIP_BIND(Recv, "ncclRecv")
  SIP_BIND(GroupStart, "ncclGroupStart")
  SIP_BIND(GroupEnd, "ncclGroupEnd")
  SIP_BIND(GetErrorString, "ncclGetErrorString")
#undef SIP_BIND
  api.lib = lib;
  return &api;
}

#define CUDA_OK(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "%s failed: %s", #expr, cudaGetErrorString(e__));      \
  } while (0)
#define NCCL_OK(expr)                                                                              \
  do {                                                                                             \
    ncclResult_t r__ = (expr);                                                                     \
    if (r__ != ncclSuccess)                                                                        \
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "%s failed: %s", #expr, nccl_api()->GetErrorString(r__)); \
  } while (0)

// `p` holds at least `need` elements (at least one), reallocated after `stream` has finished with the old buffer
template <class T>
int grow(T *&p, size_t &cap, size_t need, cudaStream_t stream) {
  if (need <= cap && p) return 0;
  CUDA_OK(cudaStreamSynchronize(stream));
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  CUDA_OK(cudaMalloc((void **)&p, std::max<size_t>(need, 1) * sizeof(T)));
  cap = std::max<size_t>(need, 1);
  return 0;
}

// count a launch on `h` and map its error
int launched(sipnet_gpu_handle *h, cudaError_t e, const char *what) {
  h->launches++;
  return e == cudaSuccess ? 0 : fail(SIPNET_GPU_ERR_NO_DEVICE, "%s launch failed: %s", what, cudaGetErrorString(e));
}

// one local rank of the team: a handle, its communicator and its scratch for the cross-rank summaries
struct Local {
  sipnet_gpu_handle *h = nullptr;
  ncclComm_t comm = nullptr;
  int rank = 0;
  // scratch, sized for `rowsCap` rows
  int64_t rowsCap = 0;
  gs::GsStat *statAll = nullptr;
  double *q2All = nullptr;
  uint32_t *hist = nullptr;
  gs::GsRow *state = nullptr;
  gs::GsTie *tieAll = nullptr;
  uint64_t *emitAll = nullptr;
  int32_t *flags = nullptr;
  double *list = nullptr;  // candidate lists (only where they are worth their memory, see ensure_scratch)
  int32_t *listN = nullptr;
  // [nranks][bytes per rank] of one all-gather at a time: argument hashes, the filters' per-site partials, member words
  unsigned char *xchg = nullptr;
  size_t xchgCap = 0;
};

}  // namespace

struct sipnet_gpu_comm {
  int nranks = 1;
  bool loopback = false;                 // every rank on one device: the collectives are device copies, not NCCL
  std::vector<Local> local;              // the ranks this process drives (1 with one process per GPU)
  std::vector<int64_t> memberCounts;     // [nranks]
  int lastLevels = 0;
};

namespace {

// all scratch of `l`: the rank keeps its handle, communicator and rank
void free_local(Local &l) {
  if (l.h) cudaSetDevice(l.h->device);
  void *ptrs[] = {l.statAll, l.q2All, l.hist, l.state, l.tieAll, l.emitAll, l.flags, l.list, l.listN, l.xchg};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  l = Local{l.h, l.comm, l.rank};
}

// one handle alone: a team of one rank, which needs no exchange
sipnet_gpu_comm team_of_one(sipnet_gpu_handle *h) {
  sipnet_gpu_comm one;
  one.local.resize(1);
  one.local[0].h = h;
  one.memberCounts.assign(1, h->nmembers);
  return one;
}

// collectives over the team; with one rank they are no-ops (local data already sits at index `rank` = 0)
struct Group {
  const sipnet_gpu_comm *c;
  bool grouped;
  explicit Group(const sipnet_gpu_comm *cc) : c(cc), grouped(cc->nranks > 1 && cc->local.size() > 1) {}
  int begin() const {
    if (grouped) NCCL_OK(nccl_api()->GroupStart());
    return 0;
  }
  int end() const {
    if (grouped) NCCL_OK(nccl_api()->GroupEnd());
    return 0;
  }
};

// f(i, local rank i) on every local rank, with its device current; stops at the first non-zero return
template <class F>
int each_rank(sipnet_gpu_comm *c, F f) {
  for (size_t i = 0; i < c->local.size(); ++i) {
    CUDA_OK(cudaSetDevice(c->local[i].h->device));
    if (int rc = f(i, c->local[i])) return rc;
  }
  return 0;
}

// the local streams, all finished (the loopback collectives copy between the ranks' buffers on one device)
int sync_all(sipnet_gpu_comm *c) {
  return each_rank(c, [](size_t, Local &l) {
    CUDA_OK(cudaStreamSynchronize(l.h->stream));
    return 0;
  });
}

int all_gather_bytes(sipnet_gpu_comm *c, size_t bytesPerRank, void *(*buf)(Local &)) {
  if (c->nranks == 1) return 0;
  if (c->loopback) {
    if (int rc = sync_all(c)) return rc;
    for (Local &to : c->local)
      for (Local &from : c->local)
        if (&to != &from) {
          const size_t off = (size_t)from.rank * bytesPerRank;
          CUDA_OK(cudaMemcpyAsync(static_cast<char *>(buf(to)) + off, static_cast<char *>(buf(from)) + off, bytesPerRank,
                                  cudaMemcpyDeviceToDevice, to.h->stream));
        }
    return sync_all(c);
  }
  const Group g(c);
  if (int rc = g.begin()) return rc;
  if (int rc = each_rank(c, [&](size_t, Local &l) {
        char *base = static_cast<char *>(buf(l));
        NCCL_OK(nccl_api()->AllGather(base + (size_t)l.rank * bytesPerRank, base, bytesPerRank, ncclUint8, l.comm,
                                      l.h->stream));
        return 0;
      }))
    return rc;
  return g.end();
}

int all_reduce_hist(sipnet_gpu_comm *c, size_t words) {
  if (c->nranks == 1) return 0;
  if (c->loopback) {  // sum into rank 0's buffer, then copy the sum back to every other rank
    if (int rc = sync_all(c)) return rc;
    Local &l0 = c->local[0];
    CUDA_OK(cudaSetDevice(l0.h->device));
    for (size_t i = 1; i < c->local.size(); ++i) CUDA_OK(gs::launch_add_u32(l0.hist, c->local[i].hist, words, l0.h->stream));
    for (size_t i = 1; i < c->local.size(); ++i)
      CUDA_OK(cudaMemcpyAsync(c->local[i].hist, l0.hist, words * sizeof(uint32_t), cudaMemcpyDeviceToDevice, l0.h->stream));
    return sync_all(c);
  }
  const Group g(c);
  if (int rc = g.begin()) return rc;
  if (int rc = each_rank(c, [&](size_t, Local &l) {
        NCCL_OK(nccl_api()->AllReduce(l.hist, l.hist, words, ncclUint32, ncclSum, l.comm, l.h->stream));
        return 0;
      }))
    return rc;
  return g.end();
}

// Candidate lists are kept when the rank's members per site are at least 4 x kGsListCap: then a list costs at most a
// quarter of the memory of the summary columns themselves and saves the later scans most of a row.  Whether a rank
// keeps lists is its own choice (each rank scans its own list or row); what it compacts is decided from global counts.
int ensure_scratch(sipnet_gpu_comm *c, Local &l, int64_t rows, bool lists) {
  if (rows <= l.rowsCap && (!lists || l.list)) return 0;
  const int R = c->nranks;
  sipnet_gpu_handle *h = l.h;
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  free_local(l);
  CUDA_OK(cudaMalloc((void **)&l.statAll, (size_t)R * rows * sizeof(gs::GsStat)));
  CUDA_OK(cudaMalloc((void **)&l.q2All, (size_t)R * rows * sizeof(double)));
  CUDA_OK(cudaMalloc((void **)&l.hist, (size_t)rows * gs::kGsHistWords * sizeof(uint32_t)));
  CUDA_OK(cudaMalloc((void **)&l.state, (size_t)rows * sizeof(gs::GsRow)));
  CUDA_OK(cudaMalloc((void **)&l.tieAll, (size_t)R * rows * gs::kGsMaxStat * sizeof(gs::GsTie)));
  CUDA_OK(cudaMalloc((void **)&l.emitAll, (size_t)R * rows * gs::kGsMaxStat * gs::kGsEmit * sizeof(uint64_t)));
  CUDA_OK(cudaMalloc((void **)&l.flags, 16));
  if (lists) {
    CUDA_OK(cudaMalloc((void **)&l.list, (size_t)rows * gs::kGsListCap * sizeof(double)));
    CUDA_OK(cudaMalloc((void **)&l.listN, (size_t)rows * sizeof(int32_t)));
  }
  l.rowsCap = rows;
  return 0;
}

// The summaries of the last run range over the WHOLE team, into every local handle's mean / var / quant buffers.
int team_summaries(sipnet_gpu_comm *c) {
  Local &l0 = c->local[0];
  sipnet_gpu_handle *h0 = l0.h;
  const int64_t n = h0->lastEnd - h0->lastBegin;
  if (n <= 0) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no run range to summarise");
  const int ncols = (int)h0->summaryCols.size();
  if (ncols <= 0 || ncols > gs::kGsMaxCols)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "cross-rank summaries take 1..%d summary columns", gs::kGsMaxCols);
  if (!h0->mean && !h0->quant) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no summary output was requested at init");
  const int nqTotal = h0->quant ? (int)h0->quantiles.size() : 0;
  const int64_t rows = (int64_t)h0->nsites * ncols * n;
  for (Local &l : c->local) {
    sipnet_gpu_handle *h = l.h;
    if (h->lastEnd - h->lastBegin != n || h->nsites != h0->nsites || (int)h->summaryCols.size() != ncols)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the ranks of a team must hold the same sites, columns and run range");
    const bool lists = nqTotal > 0 && h->ld >= 4 * (int64_t)gs::kGsListCap * h->nsites;
    if (int rc = ensure_scratch(c, l, rows, lists)) return rc;
  }
  std::vector<gs::GsArgs> args(c->local.size());
  for (size_t i = 0; i < c->local.size(); ++i) {
    Local &l = c->local[i];
    sipnet_gpu_handle *h = l.h;
    gs::GsArgs &a = args[i];
    memset(&a, 0, sizeof a);
    a.out = h->out;
    a.ld = h->ld;
    a.nsteps = n;
    a.sites = h->sites;
    a.nsites = (int32_t)h->nsites;
    a.ncols = ncols;
    for (int k = 0; k < ncols; ++k) a.colSlot[k] = h->colSlot[h->summaryCols[(size_t)k]];
    a.nranks = c->nranks;
    a.rank = l.rank;
    a.wantMoments = h->mean != nullptr;
    a.statAll = l.statAll;
    a.q2All = l.q2All;
    a.hist = l.hist;
    a.state = l.state;
    a.tieAll = l.tieAll;
    a.emitAll = l.emitAll;
    a.flags = l.flags;
    a.list = l.list;
    a.listN = l.listN;
    a.mean = h->mean;
    a.var = h->var;
    a.quant = h->quant;
    a.nqTotal = nqTotal;
  }
  c->lastLevels = 0;
  // the select takes the probabilities ascending (sip_gsum.cu resolve_level); results go to the caller's order
  std::vector<int> order((size_t)nqTotal);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [h0](int i, int j) { return h0->quantiles[(size_t)i] < h0->quantiles[(size_t)j]; });
  // quantiles in groups of kGsMaxQ; the moments ride with the first group
  for (int q0 = 0; q0 < std::max(nqTotal, 1); q0 += gs::kGsMaxQ) {
    const int nq = std::min(gs::kGsMaxQ, nqTotal - q0);
    if (int rc = each_rank(c, [&](size_t i, Local &l) {
          gs::GsArgs &a = args[i];
          a.nq = std::max(nq, 0);
          for (int k = 0; k < a.nq; ++k) {
            a.qOut[k] = order[(size_t)(q0 + k)];
            a.probs[k] = l.h->quantiles[(size_t)a.qOut[k]];
          }
          a.wantMoments = (l.h->mean != nullptr && q0 == 0) ? 1 : 0;
          return launched(l.h, gs::launch_pass0(a, l.h->stream), "summary");
        }))
      return rc;
    if (int rc = all_gather_bytes(c, (size_t)rows * sizeof(gs::GsStat), [](Local &l) -> void * { return l.statAll; })) return rc;
    if (args[0].nq > 0)
      if (int rc = all_reduce_hist(c, (size_t)rows * gs::kGsHistWords)) return rc;
    for (int level = 1; level <= gs::kGsLevels; ++level) {
      if (int rc = each_rank(c, [&](size_t i, Local &l) {
            CUDA_OK(cudaMemsetAsync(l.flags, 0, 16, l.h->stream));
            return launched(l.h, gs::launch_level(args[i], level, l.h->stream), "summary");
          }))
        return rc;
      // the flag is a function of exchanged data only: every rank reads the same value
      int32_t flag = 0;
      {
        Local &l = c->local[0];
        CUDA_OK(cudaSetDevice(l.h->device));
        CUDA_OK(cudaMemcpyAsync(&flag, l.flags, sizeof flag, cudaMemcpyDeviceToHost, l.h->stream));
        CUDA_OK(cudaStreamSynchronize(l.h->stream));
      }
      if (level == 1 && args[0].wantMoments)
        if (int rc = all_gather_bytes(c, (size_t)rows * sizeof(double), [](Local &l) -> void * { return l.q2All; })) return rc;
      if (!flag) break;
      c->lastLevels = std::max(c->lastLevels, level);
      if (int rc = all_reduce_hist(c, (size_t)rows * gs::kGsHistWords)) return rc;
      if (int rc = all_gather_bytes(c, (size_t)rows * gs::kGsMaxStat * sizeof(gs::GsTie), [](Local &l) -> void * { return l.tieAll; }))
        return rc;
    }
    if (args[0].nq > 0) {
      if (int rc = each_rank(c, [&](size_t i, Local &l) {
            return launched(l.h, gs::launch_emit(args[i], l.h->stream), "summary");
          }))
        return rc;
      if (int rc = all_gather_bytes(c, (size_t)rows * gs::kGsMaxStat * gs::kGsEmit * sizeof(uint64_t),
                                    [](Local &l) -> void * { return l.emitAll; }))
        return rc;
    }
    if (int rc = each_rank(c, [&](size_t i, Local &l) {
          return launched(l.h, gs::launch_finish(args[i], l.h->stream), "summary");
        }))
      return rc;
  }
  for (Local &l : c->local) l.h->summariesValid = true;
  return 0;
}

}  // namespace

// ---- C ABI: one process per GPU ---------------------------------------------------------------------------------
extern "C" int sipnet_gpu_comm_unique_id(void *id) {
  if (!id) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL id");
  const NcclApi *api = nccl_api();
  if (!api) return fail(SIPNET_GPU_ERR_NO_DEVICE, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror());
  ncclUniqueId uid;
  NCCL_OK(api->GetUniqueId(&uid));
  static_assert(sizeof(uid) == SIPNET_GPU_COMM_ID_BYTES, "id size");
  memcpy(id, &uid, sizeof uid);
  return 0;
}

// mine[i] of every local rank i, all-gathered through xchg: every rank's word, rank-major, on the host
static int gather_words(sipnet_gpu_comm *c, const std::vector<uint64_t> &mine, std::vector<uint64_t> &all) {
  if (int rc = each_rank(c, [&](size_t i, Local &l) {
        if (int rc = grow(l.xchg, l.xchgCap, (size_t)c->nranks * sizeof(uint64_t), l.h->stream)) return rc;
        CUDA_OK(cudaMemcpyAsync(l.xchg + l.rank * sizeof(uint64_t), &mine[i], sizeof(uint64_t), cudaMemcpyHostToDevice,
                                l.h->stream));
        CUDA_OK(cudaStreamSynchronize(l.h->stream));
        return 0;
      }))
    return rc;
  if (int rc = all_gather_bytes(c, sizeof(uint64_t), [](Local &l) -> void * { return l.xchg; })) return rc;
  all.resize((size_t)c->nranks);
  Local &l0 = c->local[0];
  CUDA_OK(cudaSetDevice(l0.h->device));
  CUDA_OK(cudaMemcpyAsync(all.data(), l0.xchg, all.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, l0.h->stream));
  CUDA_OK(cudaStreamSynchronize(l0.h->stream));
  return 0;
}

static int finish_comm(sipnet_gpu_comm *c) {
  // member counts of all ranks (for the log-likelihood gather's layout); no exchange when this process drives them all
  c->memberCounts.assign((size_t)c->nranks, 0);
  if ((int)c->local.size() == c->nranks) {
    for (const Local &l : c->local) c->memberCounts[(size_t)l.rank] = l.h->nmembers;
    return 0;
  }
  std::vector<uint64_t> mine, all;
  for (const Local &l : c->local) mine.push_back((uint64_t)l.h->nmembers);
  if (int rc = gather_words(c, mine, all)) return rc;
  for (int q = 0; q < c->nranks; ++q) c->memberCounts[(size_t)q] = (int64_t)all[(size_t)q];
  return 0;
}

extern "C" int sipnet_gpu_comm_init_rank(sipnet_gpu_handle *h, int32_t nranks, int32_t rank, const void *id,
                                         sipnet_gpu_comm **out) {
  if (out) *out = nullptr;
  if (!h || !out) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or comm pointer");
  if (nranks < 1 || rank < 0 || rank >= nranks) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "bad rank %d of %d", rank, nranks);
  sipnet_gpu_comm *c = new sipnet_gpu_comm();
  c->nranks = nranks;
  c->local.resize(1);
  c->local[0].h = h;
  c->local[0].rank = rank;
  if (nranks > 1) {
    if (!id) {
      delete c;
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL id");
    }
    const NcclApi *api = nccl_api();
    if (!api) {
      delete c;
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror());
    }
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof uid);
    cudaSetDevice(h->device);
    ncclResult_t r = api->CommInitRank(&c->local[0].comm, nranks, uid, rank);
    if (r != ncclSuccess) {
      delete c;
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "ncclCommInitRank failed: %s", api->GetErrorString(r));
    }
  }
  if (int rc = finish_comm(c)) {
    sipnet_gpu_comm_destroy(c);
    return rc;
  }
  *out = c;
  return 0;
}

extern "C" void sipnet_gpu_comm_destroy(sipnet_gpu_comm *c) {
  if (!c) return;
  for (Local &l : c->local) {
    if (l.h) {
      cudaSetDevice(l.h->device);
      cudaStreamSynchronize(l.h->stream);
    }
    free_local(l);
    if (l.comm) nccl_api()->CommDestroy(l.comm);
  }
  delete c;
}

extern "C" int32_t sipnet_gpu_comm_nranks(const sipnet_gpu_comm *c) { return c ? c->nranks : 0; }

extern "C" int sipnet_gpu_comm_summaries(sipnet_gpu_comm *c) {
  if (!c) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm");
  return team_summaries(c);
}

extern "C" int32_t sipnet_gpu_comm_last_levels(const sipnet_gpu_comm *c) { return c ? c->lastLevels : 0; }

// one 8-byte word per member of the team (`src` of every handle: log-likelihoods, ancestors), rank-major, into each
// local rank's gather buffer, and to `dst` on the host when given
static int team_member_words(sipnet_gpu_comm *c, void *dst, size_t bytes, const void *(*src)(const sipnet_gpu_handle *),
                             const char *what) {
  int64_t total = 0, width = 0;
  for (int64_t m : c->memberCounts) {
    total += m;
    width = std::max(width, m);
  }
  if (dst && bytes != (size_t)total * sizeof(double))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "%s gather: buffer is %zu bytes, expected %zu", what, bytes,
                (size_t)total * sizeof(double));
  if (int rc = each_rank(c, [&](size_t, Local &l) {
        sipnet_gpu_handle *h = l.h;
        const void *from = src(h);
        if (!from) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "%s output was not requested at init", what);
        if (int rc = grow(l.xchg, l.xchgCap, (size_t)c->nranks * width * sizeof(double), h->stream)) return rc;
        CUDA_OK(cudaMemcpyAsync(l.xchg + (size_t)l.rank * width * sizeof(double), from, (size_t)h->nmembers * sizeof(double),
                                cudaMemcpyDeviceToDevice, h->stream));
        return 0;
      }))
    return rc;
  if (int rc = all_gather_bytes(c, (size_t)width * sizeof(double), [](Local &l) -> void * { return l.xchg; })) return rc;
  if (dst) {
    Local &l = c->local[0];
    CUDA_OK(cudaSetDevice(l.h->device));
    int64_t off = 0;
    for (int q = 0; q < c->nranks; ++q) {
      CUDA_OK(cudaMemcpyAsync(static_cast<double *>(dst) + off, l.xchg + (size_t)q * width * sizeof(double),
                              (size_t)c->memberCounts[(size_t)q] * sizeof(double), cudaMemcpyDeviceToHost, l.h->stream));
      off += c->memberCounts[(size_t)q];
    }
    CUDA_OK(cudaStreamSynchronize(l.h->stream));
  }
  // every local stream has finished its part before the caller reuses the handles
  return sync_all(c);
}

extern "C" int sipnet_gpu_comm_gather_loglik(sipnet_gpu_comm *c, double *dst, size_t bytes) {
  if (!c || !dst) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm or destination");
  return team_member_words(c, dst, bytes, [](const sipnet_gpu_handle *h) -> const void * { return h->loglik; },
                           "log-likelihood");
}

extern "C" int sipnet_gpu_comm_member_counts(const sipnet_gpu_comm *c, int64_t *counts) {
  if (!c || !counts) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL argument");
  for (int q = 0; q < c->nranks; ++q) counts[q] = c->memberCounts[(size_t)q];
  return 0;
}

// ---- C ABI: one process, all GPUs ---------------------------------------------------------------------------------
// The configuration is the single-GPU one; members are partitioned like this:
//   * at least as many sites as devices: whole sites per device (forcing is not replicated), contiguous site ranges;
//   * fewer sites than devices: every device gets every site and an even, contiguous share of each site's members;
//     the summaries of such split sites go through the team select above.
struct sipnet_gpu_multi {
  sipnet_gpu_comm *comm = nullptr;
  std::vector<sipnet_gpu_handle *> handles;
  bool split = false;  // sites are split over devices (else whole sites per device)
  int64_t nmembers = 0, nsites = 0, nsummary = 0, nquant = 0;
  uint32_t outputs = 0;
  // per device: its site range, and its members as runs of consecutive members, `count` members from local index
  // `local0` and configuration index `global0` on (whole sites: one run; split sites: one run per site)
  struct Run {
    int64_t local0, global0, count;
  };
  struct Part {
    int64_t site0 = 0, site1 = 0;
    std::vector<Run> runs;
  };
  std::vector<Part> parts;
};

extern "C" void sipnet_gpu_multi_destroy(sipnet_gpu_multi *m) {
  if (!m) return;
  sipnet_gpu_comm_destroy(m->comm);  // first: it synchronises the handles' streams
  for (sipnet_gpu_handle *h : m->handles) sipnet_gpu_destroy(h);
  delete m;
}

extern "C" int sipnet_gpu_multi_init(const sipnet_gpu_config *cfg, int32_t ndevices, const int32_t *devices,
                                     sipnet_gpu_multi **out) {
  if (out) *out = nullptr;
  if (!cfg || !out) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL config or handle pointer");
  int visible = 0;
  if (cudaGetDeviceCount(&visible) != cudaSuccess || visible <= 0)
    return fail(SIPNET_GPU_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
  std::vector<int> devs;
  if (ndevices <= 0) {
    for (int d = 0; d < visible; ++d) devs.push_back(d);
  } else {
    for (int i = 0; i < ndevices; ++i) devs.push_back(devices ? devices[i] : i);
  }
  // one device named several times: a loopback team, every rank on that device (a test seam for the team select)
  bool loopback = false;
  {
    std::vector<int> u(devs);
    std::sort(u.begin(), u.end());
    if (std::unique(u.begin(), u.end()) != u.end()) {
      if (u.front() != u.back())
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "a device list names distinct devices once each, or one device repeatedly");
      loopback = true;
    }
  }
  for (int d : devs)
    if (d < 0 || d >= visible) return fail(SIPNET_GPU_ERR_NO_DEVICE, "device %d not present", d);
  if (cfg->nsites <= 0 || !cfg->sites || cfg->nmembers <= 0 || !cfg->params)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no sites / members");
  if (cfg->stream) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "a caller stream cannot be shared by several devices");
  // never more devices than members
  while ((int64_t)devs.size() > cfg->nmembers) devs.pop_back();
  int D = (int)devs.size();

  sipnet_gpu_multi *m = new sipnet_gpu_multi();
  m->nmembers = cfg->nmembers;
  m->nsites = cfg->nsites;
  m->nsummary = cfg->n_summary_cols;
  m->nquant = cfg->n_quantiles;
  m->outputs = cfg->outputs;
  m->split = cfg->nsites < D;
  std::vector<int32_t> memberSite((size_t)cfg->nmembers, 0);
  if (cfg->member_site)
    for (int64_t i = 0; i < cfg->nmembers; ++i) memberSite[(size_t)i] = cfg->member_site[i];
  // first member and count of every site (validated again by sipnet_gpu_init)
  std::vector<int64_t> siteM0((size_t)cfg->nsites, 0), siteCnt((size_t)cfg->nsites, 0);
  for (int64_t i = 0; i < cfg->nmembers; ++i) {
    const int32_t s = memberSite[(size_t)i];
    if (s < 0 || s >= cfg->nsites || (i > 0 && s < memberSite[(size_t)i - 1])) {
      delete m;
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "member_site must be non-decreasing and in range");
    }
    if (siteCnt[(size_t)s]++ == 0) siteM0[(size_t)s] = i;
  }

  // the same mean-NPP ring capacity on every device (sipnet_gpu_init sizes it from the shortest step it sees)
  int32_t ringSlots = cfg->ring_slots;
  if (ringSlots == 0) {
    double minLen = 1e300;
    for (int64_t s = 0; s < cfg->nsites; ++s)
      for (int64_t t = 0; t < cfg->sites[s].nsteps && cfg->sites[s].length; ++t)
        if (cfg->sites[s].length[t] > 0) minLen = std::min(minLen, cfg->sites[s].length[t]);
    const double bound = std::floor(kMeanNppDays / minLen) + 3.0;
    ringSlots = (int32_t)std::min<double>(kRingMax, std::max(2.0, bound));
  }

  // the partition over D devices; a device that would get no member is left out, so the team may be smaller than D
  std::vector<std::vector<int64_t>> picks;  // per kept device: its global member indices, ascending
  std::vector<int> keptDevs;
  for (int d = 0; d < D; ++d) {
    sipnet_gpu_multi::Part p;
    std::vector<int64_t> pick;
    if (!m->split) {
      p.site0 = (cfg->nsites * d) / D;
      p.site1 = (cfg->nsites * (d + 1)) / D;
      for (int64_t i = 0; i < cfg->nmembers; ++i)
        if (memberSite[(size_t)i] >= p.site0 && memberSite[(size_t)i] < p.site1) pick.push_back(i);
      if (!pick.empty()) p.runs.push_back({0, pick.front(), (int64_t)pick.size()});  // member_site is non-decreasing
    } else {
      p.site0 = 0;
      p.site1 = cfg->nsites;
      for (int64_t s = 0; s < cfg->nsites; ++s) {
        const int64_t lo = (siteCnt[(size_t)s] * d) / D, hi = (siteCnt[(size_t)s] * (d + 1)) / D;
        p.runs.push_back({(int64_t)pick.size(), siteM0[(size_t)s] + lo, hi - lo});
        for (int64_t i = lo; i < hi; ++i) pick.push_back(siteM0[(size_t)s] + i);
      }
    }
    if (pick.empty()) continue;
    m->parts.push_back(p);
    picks.push_back(std::move(pick));
    keptDevs.push_back(devs[(size_t)d]);
  }
  devs = keptDevs;
  D = (int)devs.size();
  // whole sites: the site ranges of the devices left out hold no member; the kept devices take them over (each one
  // up to the next kept device's first site), so the summaries still cover every site in order
  if (!m->split)
    for (int d = 0; d < D; ++d) {
      m->parts[(size_t)d].site0 = d == 0 ? 0 : m->parts[(size_t)d - 1].site1;
      m->parts[(size_t)d].site1 = d + 1 < D ? m->parts[(size_t)d + 1].site0 : cfg->nsites;
    }

  for (int d = 0; d < D; ++d) {
    const sipnet_gpu_multi::Part &p = m->parts[(size_t)d];
    const std::vector<int64_t> &pick = picks[(size_t)d];
    sipnet_gpu_config sub = *cfg;
    sub.device = devs[(size_t)d];
    sub.ring_slots = ringSlots;
    std::vector<int32_t> subSite;
    std::vector<double> subParams;
    sub.nsites = p.site1 - p.site0;
    sub.sites = cfg->sites + p.site0;
    for (int64_t i : pick) subSite.push_back(memberSite[(size_t)i] - (int32_t)p.site0);
    const int64_t nm = (int64_t)pick.size();
    subParams.resize((size_t)SIPNET_GPU_NPARAMS * (size_t)nm);
    for (int k = 0; k < SIPNET_GPU_NPARAMS; ++k)
      for (int64_t j = 0; j < nm; ++j)
        subParams[(size_t)k * (size_t)nm + (size_t)j] = cfg->params[(size_t)k * (size_t)cfg->params_ld + (size_t)pick[(size_t)j]];
    sub.nmembers = nm;
    sub.member_site = subSite.data();
    sub.params = subParams.data();
    sub.params_ld = nm;
    sipnet_gpu_handle *h = nullptr;
    const int rc = sipnet_gpu_init(&sub, &h);
    if (rc) {
      sipnet_gpu_multi_destroy(m);
      return rc;
    }
    m->handles.push_back(h);
  }

  // the team: needed when sites are split (summaries) or log-likelihoods are gathered through NCCL; one device
  // needs none
  sipnet_gpu_comm *c = new sipnet_gpu_comm();
  c->nranks = D;
  c->local.resize((size_t)D);
  for (int d = 0; d < D; ++d) {
    c->local[(size_t)d].h = m->handles[(size_t)d];
    c->local[(size_t)d].rank = d;
  }
  m->comm = c;
  c->loopback = loopback && D > 1;
  if (D > 1 && !c->loopback) {
    const NcclApi *api = nccl_api();
    if (!api) {
      sipnet_gpu_multi_destroy(m);
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror());
    }
    std::vector<ncclComm_t> comms((size_t)D, nullptr);
    ncclResult_t r = api->CommInitAll(comms.data(), D, devs.data());
    if (r != ncclSuccess) {
      sipnet_gpu_multi_destroy(m);
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "ncclCommInitAll failed: %s", api->GetErrorString(r));
    }
    for (int d = 0; d < D; ++d) c->local[(size_t)d].comm = comms[(size_t)d];
  }
  if (int rc = finish_comm(c)) {
    sipnet_gpu_multi_destroy(m);
    return rc;
  }
  *out = m;
  return 0;
}

extern "C" int32_t sipnet_gpu_multi_ndevices(const sipnet_gpu_multi *m) { return m ? (int32_t)m->handles.size() : 0; }
extern "C" sipnet_gpu_handle *sipnet_gpu_multi_handle(sipnet_gpu_multi *m, int32_t i) {
  return (m && i >= 0 && i < (int32_t)m->handles.size()) ? m->handles[(size_t)i] : nullptr;
}

extern "C" int sipnet_gpu_multi_run(sipnet_gpu_multi *m, int64_t step_begin, int64_t step_end) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  for (sipnet_gpu_handle *h : m->handles) {  // asynchronous launches: all devices run side by side
    // a device whose sites are all shorter than the range runs what it has
    const int64_t e = std::min<int64_t>(step_end, h->maxSteps);
    const int64_t b = std::min<int64_t>(step_begin, e);
    if (int rc = sipnet_gpu_run(h, b, e)) return rc;
  }
  return 0;
}

extern "C" int sipnet_gpu_multi_reset(sipnet_gpu_multi *m) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  for (sipnet_gpu_handle *h : m->handles)
    if (int rc = sipnet_gpu_reset(h)) return rc;
  return 0;
}

extern "C" int sipnet_gpu_multi_sync(sipnet_gpu_multi *m) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  for (sipnet_gpu_handle *h : m->handles)
    if (int rc = sipnet_gpu_sync(h)) return rc;
  return 0;
}

// steps of the last run range over all devices (a device whose sites are shorter ran fewer)
static int64_t multi_range_steps(const sipnet_gpu_multi *m) {
  int64_t n = 0;
  for (const sipnet_gpu_handle *h : m->handles) n = std::max(n, h->lastEnd - h->lastBegin);
  return n;
}

// per-member outputs: `rows` rows of M elements of `elem` bytes; per-step outputs have rows = columns x steps
static bool member_output_shape(const sipnet_gpu_multi *m, int what, size_t *cols, bool *perStep, size_t *elem) {
  const sipnet_gpu_handle *h0 = m->handles[0];
  *perStep = false;
  *elem = 8;
  switch (what) {
    case SIPNET_GPU_GATHER_FULL: *cols = SIPNET_GPU_NOUT; *perStep = true; return (h0->outputs & SIPNET_GPU_OUT_FULL) != 0;
    case SIPNET_GPU_GATHER_DEBUG: *cols = SIPNET_GPU_NDEBUG; *perStep = true; return h0->dbg != nullptr;
    case SIPNET_GPU_GATHER_BALANCE: *cols = SIPNET_GPU_NBALANCE; *perStep = true; return h0->dbg != nullptr;
    case SIPNET_GPU_GATHER_LOGLIK:
    case SIPNET_GPU_GATHER_LOGLIK_N: *cols = 1; return h0->loglik != nullptr;
    case SIPNET_GPU_GATHER_STATUS: *cols = 1; *elem = 4; return true;
    case SIPNET_GPU_GATHER_STATE: *cols = SIPNET_GPU_NSTATE; return true;
    case SIPNET_GPU_GATHER_PARAMS: *cols = SIPNET_GPU_NPARAMS; return true;
    case SIPNET_GPU_GATHER_RING_VALUES:
    case SIPNET_GPU_GATHER_RING_WEIGHTS: *cols = (size_t)h0->ringCap; return true;
    case SIPNET_GPU_GATHER_EVENT_COUNTS: *cols = 1; *elem = 4; return h0->recCount != nullptr;
    case SIPNET_GPU_GATHER_EVENT_RECORDS:
      *cols = 1;
      *elem = (size_t)h0->maxRecs * sizeof(sipnet_gpu_event_record);
      return h0->recs != nullptr;
    default: return false;
  }
}

extern "C" size_t sipnet_gpu_multi_gather_bytes(const sipnet_gpu_multi *m, int what) {
  if (!m || m->handles.empty()) return 0;
  const sipnet_gpu_handle *h0 = m->handles[0];
  const size_t n = (size_t)multi_range_steps(m);
  const size_t ns = h0->summaryCols.size();
  switch (what) {
    case SIPNET_GPU_GATHER_MEAN:
    case SIPNET_GPU_GATHER_VARIANCE: return h0->mean ? (size_t)m->nsites * ns * n * 8 : 0;
    case SIPNET_GPU_GATHER_QUANTILES: return h0->quant ? (size_t)m->nsites * ns * h0->quantiles.size() * n * 8 : 0;
    default: break;
  }
  size_t cols = 0, elem = 8;
  bool perStep = false;
  if (!member_output_shape(m, what, &cols, &perStep, &elem)) return 0;
  return cols * (perStep ? n : 1) * (size_t)m->nmembers * elem;
}

extern "C" int sipnet_gpu_multi_gather(sipnet_gpu_multi *m, int what, void *dst, size_t bytes) {
  if (!m || !dst) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or destination");
  const size_t need = sipnet_gpu_multi_gather_bytes(m, what);
  if (need == 0) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "gather(%d): output was not requested at init or nothing has run", what);
  if (bytes != need) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "gather(%d): buffer is %zu bytes, expected %zu", what, bytes, need);
  const size_t D = m->handles.size();
  const size_t n = (size_t)multi_range_steps(m);
  const bool summary = what == SIPNET_GPU_GATHER_MEAN || what == SIPNET_GPU_GATHER_VARIANCE || what == SIPNET_GPU_GATHER_QUANTILES;
  if (summary) {
    if (m->split) {  // every device ends with the team's result: take device 0's
      if (!m->handles[0]->summariesValid)
        if (int rc = team_summaries(m->comm)) return rc;
      return sipnet_gpu_gather(m->handles[0], what, dst, bytes);
    }
    // whole sites per device: local summaries; rows [site][col]([q])[n], a shorter device's rows are NaN-padded
    const sipnet_gpu_handle *h0 = m->handles[0];
    const size_t per = h0->summaryCols.size() * (what == SIPNET_GPU_GATHER_QUANTILES ? h0->quantiles.size() : 1);
    double *out = static_cast<double *>(dst);
    std::vector<double> tmp;
    for (size_t d = 0; d < D; ++d) {
      sipnet_gpu_handle *h = m->handles[d];
      const size_t nd = (size_t)(h->lastEnd - h->lastBegin);
      const size_t rowsD = (size_t)h->nsites * per;
      if (nd == n) {
        if (int rc = sipnet_gpu_gather(h, what, out, rowsD * n * 8)) return rc;
      } else {
        for (size_t i = 0; i < rowsD * n; ++i) out[i] = __builtin_nan("");
        if (nd > 0) {
          tmp.resize(rowsD * nd);
          if (int rc = sipnet_gpu_gather(h, what, tmp.data(), rowsD * nd * 8)) return rc;
          for (size_t r = 0; r < rowsD; ++r) memcpy(out + r * n, tmp.data() + r * nd, nd * 8);
        }
      }
      out += rowsD * n;
    }
    return 0;
  }
  size_t cols = 0, elem = 8;
  bool perStep = false;
  member_output_shape(m, what, &cols, &perStep, &elem);
  const size_t M = (size_t)m->nmembers;
  const size_t steps = perStep ? n : 1;
  std::vector<char> tmp;
  for (size_t d = 0; d < D; ++d) {
    sipnet_gpu_handle *h = m->handles[d];
    const size_t nm = (size_t)h->nmembers;
    const size_t nd = perStep ? (size_t)(h->lastEnd - h->lastBegin) : 1;
    if (nd > 0) {
      tmp.resize(cols * nd * nm * elem);
      if (int rc = sipnet_gpu_gather(h, what, tmp.data(), tmp.size())) return rc;
    }
    for (const sipnet_gpu_multi::Run &r : m->parts[d].runs)
      for (size_t c = 0; c < cols; ++c)
        for (size_t t = 0; t < steps; ++t) {
          char *to = static_cast<char *>(dst) + ((c * steps + t) * M + (size_t)r.global0) * elem;
          if (t < nd) {
            memcpy(to, tmp.data() + ((c * nd + t) * nm + (size_t)r.local0) * elem, (size_t)r.count * elem);
          } else {  // steps this device's (shorter) sites never ran: NaN, as on one GPU
            memset(to, 0xFF, (size_t)r.count * elem);
          }
        }
  }
  return 0;
}

// ---- the ensemble filters: one run over a team, from a handle, a comm or a multi-GPU handle -----------------------
namespace {

// One site pass on every local rank: launch(i, l) queues the members and site launches; a team then all-gathers the
// [nsites][rec] per-site partials (doubles) in xchg, and combine(i, l) sums them in rank order on every rank.  A team
// of one makes no exchange and no host round trip.
template <class Launch, class Combine>
int site_pass(sipnet_gpu_comm *c, size_t rec, Launch launch, Combine combine) {
  if (int rc = each_rank(c, launch)) return rc;
  if (c->nranks == 1) return 0;
  const size_t bytes = (size_t)c->local[0].h->nsites * rec * sizeof(double);
  if (int rc = all_gather_bytes(c, bytes, [](Local &l) -> void * { return l.xchg; })) return rc;
  return each_rank(c, combine);
}

// A filter through the multi-GPU interface: split sites, run(m->comm, 0) over every device; whole sites, run(its team
// of one, d) for each device d.  Device d's per-site arrays start at site m->parts[d].site0 (0 when sites are split).
template <class F>
int multi_run(sipnet_gpu_multi *m, F run) {
  if (m->split) return run(m->comm, 0);
  for (size_t d = 0; d < m->handles.size(); ++d) {
    sipnet_gpu_comm one = team_of_one(m->handles[d]);
    if (int rc = run(&one, d)) return rc;
  }
  return 0;
}

// sites [site0, ...) of an array of `per` elements per site; NULL stays NULL
template <class T>
T *from_site(T *p, int64_t site0, size_t per) {
  return p ? p + (size_t)site0 * per : nullptr;
}

// a configuration-order array [rows][M] as every device's [rows][its members] copy; at[d] is device d's
struct Copies {
  std::vector<std::vector<double>> v;
  std::vector<const double *> at;
};

Copies device_copies(const sipnet_gpu_multi *m, const double *a, size_t rows) {
  Copies c;
  const size_t M = (size_t)m->nmembers;
  for (size_t d = 0; d < m->handles.size(); ++d) {
    const size_t nm = (size_t)m->handles[d]->nmembers;
    c.v.emplace_back(rows * nm);
    for (size_t j = 0; j < rows; ++j)
      for (const sipnet_gpu_multi::Run &r : m->parts[d].runs)
        memcpy(c.v[d].data() + j * nm + r.local0, a + j * M + r.global0, (size_t)r.count * sizeof(double));
  }
  for (const std::vector<double> &v : c.v) c.at.push_back(v.data());
  return c;
}

// the configuration index of each of device d's members
std::vector<int64_t> config_index(const sipnet_gpu_multi *m, size_t d) {
  std::vector<int64_t> g((size_t)m->handles[d]->nmembers);
  for (const sipnet_gpu_multi::Run &r : m->parts[d].runs)
    std::iota(g.begin() + r.local0, g.begin() + r.local0 + r.count, r.global0);
  return g;
}

}  // namespace

// ---- sequential data assimilation: the ensemble adjustment Kalman filter (sip_assim.cuh) --------------------------
namespace {

// the spec against `nsites` sites: 0, or SIPNET_GPU_ERR_BAD_ARGUMENT with the reason
int check_obs(const sipnet_gpu_obs_spec *o, int64_t nsites) {
  if (!o || !o->rows || !o->op || !o->value || !o->variance)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL observation spec or array");
  if (o->n_rows < 1 || o->n_obs < 1) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "n_rows and n_obs must be at least 1");
  if (o->n_rows > as::kMaxRows) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "at most %d rows", as::kMaxRows);
  bool seen[as::kMaxRows] = {};
  for (int j = 0; j < o->n_rows; ++j) {
    const int32_t r = o->rows[j];
    if (r < SIPNET_S_plantWoodC || r > SIPNET_S_plantStorageN)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "state row %d is not a pool the analysis adjusts (0..11)", r);
    if (seen[r]) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "state row %d listed twice", r);
    seen[r] = true;
  }
  for (int k = 0; k < o->n_obs; ++k) {
    bool nonzero = false;
    for (int j = 0; j < o->n_rows; ++j) {
      const double v = o->op[(size_t)k * o->n_rows + j];
      if (!std::isfinite(v)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "op[%d][%d] is not finite", k, j);
      nonzero = nonzero || v != 0.0;
    }
    if (!nonzero) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "op row %d is all zero", k);
  }
  for (size_t i = 0; i < (size_t)nsites * (size_t)o->n_obs; ++i) {
    const double v = o->value[i], r = o->variance[i];
    if (std::isinf(v)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "observation value %zu is infinite", i);
    if (std::isfinite(v) && !(std::isfinite(r) && r > 0.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "observation %zu needs a finite variance > 0", i);
  }
  return 0;
}

// FNV-1a of a collective's arguments, for team_agree: never 0, which stands for invalid arguments
struct ArgHash {
  uint64_t h = 0xcbf29ce484222325ull;
  ArgHash &add(const void *p, size_t n) {
    const unsigned char *b = static_cast<const unsigned char *>(p);
    for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 0x100000001b3ull;
    return *this;
  }
  uint64_t value() const { return h == 0 ? 1 : h; }
};

uint64_t spec_hash(const sipnet_gpu_obs_spec *o, int64_t nsites) {
  const size_t nv = (size_t)nsites * (size_t)o->n_obs;
  return ArgHash()
      .add(&o->n_rows, sizeof o->n_rows)
      .add(o->rows, (size_t)o->n_rows * sizeof(int32_t))
      .add(&o->n_obs, sizeof o->n_obs)
      .add(o->op, (size_t)o->n_obs * o->n_rows * sizeof(double))
      .add(o->value, nv * sizeof(double))
      .add(o->variance, nv * sizeof(double))
      .value();
}

// the inflation arguments against `nsites` sites: 0, or SIPNET_GPU_ERR_BAD_ARGUMENT with the reason
int check_inflation(const sipnet_gpu_inflation_spec *f, int64_t nsites) {
  if (!f || !f->lambda) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL inflation spec or lambda");
  if (!(std::isfinite(f->lambda_min) && std::isfinite(f->lambda_max) && f->lambda_min > 0.0 &&
        f->lambda_min <= f->lambda_max))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "lambda bounds must be finite with 0 < lambda_min <= lambda_max");
  if (!(std::isfinite(f->sd_min) && f->sd_min >= 0.0))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "sd_min must be finite and >= 0");
  for (int64_t s = 0; s < nsites; ++s) {
    const double l = f->lambda[s];
    if (!std::isnan(l) && !(std::isfinite(l) && l > 0.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "lambda[%lld] = %g is neither NaN nor finite and > 0", (long long)s, l);
    if (!f->lambda_sd) continue;
    const double sd = f->lambda_sd[s];
    if (!(std::isfinite(sd) && sd >= 0.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "lambda_sd[%lld] = %g is not finite and >= 0", (long long)s, sd);
    if (sd > 0.0 && sd < f->sd_min)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "lambda_sd[%lld] = %g is below sd_min", (long long)s, sd);
    if (sd > 0.0 && std::isfinite(l) && (l < f->lambda_min || l > f->lambda_max))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "lambda[%lld] = %g is adaptive but outside the bounds", (long long)s, l);
  }
  return 0;
}

// the inflation arguments of sites [site0, ...): the multi-GPU partition's slice
sipnet_gpu_inflation_spec inflation_slice(const sipnet_gpu_inflation_spec *f, int64_t site0) {
  sipnet_gpu_inflation_spec g = *f;
  g.lambda += site0;
  g.lambda_sd = from_site(g.lambda_sd, site0, 1);
  return g;
}

// Queue the analysis on every local rank of `c`: value / variance (and infl, NULL = no inflation) hold the handles'
// sites (all ranks hold the same sites).  A team of one needs no exchange and no host round trip; a larger team
// all-gathers each pass's per-site partial sums and sums them in rank order on every rank.
int run_assimilation(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *o, const double *value, const double *variance,
                     const sipnet_gpu_inflation_spec *infl) {
  const int R = c->nranks, nobs = o->n_obs, nr = o->n_rows;
  const int64_t S = c->local[0].h->nsites;
  std::vector<as::Args> args(c->local.size());
  std::vector<double> f0;  // {λ0, λ, σ} per site
  bool inflate = false;    // some site may be inflated: run the moment pass
  if (infl) {
    f0.resize((size_t)S * 3);
    for (int64_t s = 0; s < S; ++s) {
      const double l = infl->lambda[s];
      f0[3 * s] = f0[3 * s + 1] = l;
      f0[3 * s + 2] = infl->lambda_sd ? infl->lambda_sd[s] : 0.0;
      inflate = inflate || (std::isfinite(l) && l != 1.0);
    }
  }
  for (size_t i = 0; i < c->local.size(); ++i) {
    Local &l = c->local[i];
    sipnet_gpu_handle *h = l.h;
    if (h->nsites != S) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the ranks of a team must hold the same sites");
    CUDA_OK(cudaSetDevice(h->device));
    if (int rc = as::ensure_scratch(h, nobs)) return rc;
    if (infl)
      if (int rc = as::ensure_inflation(h)) return rc;
    if (R > 1)
      if (int rc = grow(l.xchg, l.xchgCap, (size_t)R * h->nsites * as::kRec * sizeof(double), h->stream)) return rc;
    const size_t nv = (size_t)h->nsites * nobs;
    CUDA_OK(cudaMemcpyAsync(h->asObs, value, nv * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->asObs + nv, variance, nv * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemsetAsync(h->asCoef, 0, (size_t)h->nsites * as::kRec * sizeof(double), h->stream));
    if (infl) CUDA_OK(cudaMemcpyAsync(h->asInfl, f0.data(), f0.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    as::Args &a = args[i];
    memset(&a, 0, sizeof a);
    a.state = h->state;
    a.status = h->status;
    a.ld = h->ld;
    a.sites = h->sites;
    a.nsites = (int32_t)h->nsites;
    a.nchunks = (int32_t)h->nchunks;
    a.chunk = h->chunk;
    a.siteChunks = h->siteChunks;
    a.nrows = nr;
    a.nobs = nobs;
    a.nranks = R;
    a.rank = l.rank;
    for (int j = 0; j < nr; ++j) a.rows[j] = o->rows[j];
    a.part = h->asPart;
    a.mom = h->asMom;
    a.coef = h->asCoef;
    a.value = h->asObs;
    a.variance = h->asObs + nv;
    a.diag = h->asDiag;
    a.rankRec = reinterpret_cast<double *>(l.xchg);
    if (infl) {
      a.infl = h->asInfl;
      a.lamMin = infl->lambda_min;
      a.lamMax = infl->lambda_max;
      a.sdMin = infl->sd_min;
    }
  }
  // one members pass and its site reduction on every rank; a team then exchanges and combines the site partials
  auto run_pass = [&](int pass, bool apply, bool inflatePass) {
    const char *what = "assimilation";
    return site_pass(
        c, as::kRec,
        [&](size_t i, Local &l) {
          if (int rc = launched(l.h, as::launch_members(args[i], pass, apply, false, inflatePass, l.h->stream), what))
            return rc;
          return launched(l.h, as::launch_site_reduce(args[i], pass, l.h->stream), what);
        },
        [&](size_t i, Local &l) { return launched(l.h, as::launch_site_combine(args[i], pass, l.h->stream), what); });
  };
  if (inflate)  // the means the inflation centres on
    if (int rc = run_pass(as::kInflPass, false, false)) return rc;
  for (int k = 0; k < nobs; ++k) {
    for (as::Args &a : args) {
      a.k = k;
      for (int j = 0; j < nr; ++j) {
        a.opCur[j] = o->op[(size_t)k * nr + j];
        a.opPrev[j] = k > 0 ? o->op[(size_t)(k - 1) * nr + j] : 0.0;
      }
    }
    // pass 1 of observation k first applies observation k - 1, or (k = 0) the inflation
    if (int rc = run_pass(1, k > 0, k == 0 && inflate)) return rc;
    if (int rc = run_pass(2, false, false)) return rc;
  }
  return each_rank(c, [&](size_t i, Local &l) {  // the last observation's update and the floor
    as::Args &a = args[i];
    for (int j = 0; j < nr; ++j) a.opPrev[j] = o->op[(size_t)(nobs - 1) * nr + j];
    return launched(l.h, as::launch_members(a, 0, true, true, false, l.h->stream), "assimilation");
  });
}

// wait for the analysis of `h`; diag (may be NULL) gets its [nsites][nobs][4] diagnostics, infl (may be NULL) the
// updated lambda / lambda_sd of its sites
int finish_assimilation(sipnet_gpu_handle *h, double *diag, int nobs, const sipnet_gpu_inflation_spec *infl) {
  CUDA_OK(cudaSetDevice(h->device));
  if (diag)
    CUDA_OK(cudaMemcpyAsync(diag, h->asDiag, (size_t)h->nsites * nobs * 4 * sizeof(double), cudaMemcpyDeviceToHost,
                            h->stream));
  std::vector<double> f(infl ? (size_t)h->nsites * 3 : 0);
  if (infl) CUDA_OK(cudaMemcpyAsync(f.data(), h->asInfl, f.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  for (int64_t s = 0; infl && s < h->nsites; ++s) {
    infl->lambda[s] = f[3 * s + 1];
    if (infl->lambda_sd) infl->lambda_sd[s] = f[3 * s + 2];
  }
  return 0;
}

// sipnet_gpu_assimilate(), with the inflation unless infl is NULL (the same for the comm and multi variants below)
int assimilate_handle(sipnet_gpu_handle *h, const sipnet_gpu_obs_spec *obs, sipnet_gpu_inflation_spec *infl,
                      double *diag) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_obs(obs, h->nsites)) return rc;
  if (infl)
    if (int rc = check_inflation(infl, h->nsites)) return rc;
  sipnet_gpu_comm one = team_of_one(h);
  if (int rc = run_assimilation(&one, obs, obs->value, obs->variance, infl)) return rc;
  return finish_assimilation(h, diag, obs->n_obs, infl);
}

}  // namespace

extern "C" int sipnet_gpu_assimilate(sipnet_gpu_handle *h, const sipnet_gpu_obs_spec *obs, double *diag) {
  return assimilate_handle(h, obs, nullptr, diag);
}

extern "C" int sipnet_gpu_assimilate_inflated(sipnet_gpu_handle *h, const sipnet_gpu_obs_spec *obs,
                                              sipnet_gpu_inflation_spec *infl, double *diag) {
  if (!infl) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL inflation spec");
  return assimilate_handle(h, obs, infl, diag);
}

// Collective: every rank sees every rank's argument hash (`mine`; 0 = this rank's arguments are invalid, with the
// reason in the last error) before any rank returns, so a bad or differing argument fails on all of them.
static int team_agree(sipnet_gpu_comm *c, int bad, uint64_t mine, const char *what) {
  if (c->nranks == 1) return bad;
  const std::string why = bad ? sipnet_gpu_last_error() : "";
  std::vector<uint64_t> all;
  if (int rc = gather_words(c, std::vector<uint64_t>(c->local.size(), mine), all)) return rc;
  for (uint64_t v : all)
    if (v == 0 || v != all[0]) {
      if (bad) return fail(bad, "%s", why.c_str());
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the ranks of the team passed different or invalid %s", what);
    }
  return bad;
}

namespace {

// the spec's hash, extended by the inflation arguments (infl NULL: spec_hash)
uint64_t assim_hash(const sipnet_gpu_obs_spec *o, const sipnet_gpu_inflation_spec *f, int64_t nsites) {
  const uint64_t h0 = spec_hash(o, nsites);
  if (!f) return h0;
  const uint8_t hasSd = f->lambda_sd != nullptr;
  ArgHash h;
  h.add(&h0, sizeof h0).add(f->lambda, (size_t)nsites * sizeof(double)).add(&hasSd, 1);
  if (hasSd) h.add(f->lambda_sd, (size_t)nsites * sizeof(double));
  return h.add(&f->lambda_min, sizeof(double)).add(&f->lambda_max, sizeof(double)).add(&f->sd_min, sizeof(double))
      .value();
}

int assimilate_comm(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *obs, sipnet_gpu_inflation_spec *infl,
                    double *diag) {
  if (!c) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm");
  const int64_t S = c->local[0].h->nsites;
  int bad = check_obs(obs, S);
  if (!bad && infl) bad = check_inflation(infl, S);
  if (int rc = team_agree(c, bad, bad ? 0 : assim_hash(obs, infl, S), "observation specs")) return rc;
  if (int rc = run_assimilation(c, obs, obs->value, obs->variance, infl)) return rc;
  return finish_assimilation(c->local[0].h, diag, obs->n_obs, infl);
}

int assimilate_multi(sipnet_gpu_multi *m, const sipnet_gpu_obs_spec *obs, sipnet_gpu_inflation_spec *infl,
                     double *diag) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_obs(obs, m->nsites)) return rc;
  if (infl)
    if (int rc = check_inflation(infl, m->nsites)) return rc;
  const int nobs = obs->n_obs;
  std::vector<sipnet_gpu_inflation_spec> slice(m->handles.size());
  if (int rc = multi_run(m, [&](sipnet_gpu_comm *c, size_t d) {  // whole sites: all devices side by side
        const int64_t s0 = m->parts[d].site0;
        if (infl) slice[d] = inflation_slice(infl, s0);
        return run_assimilation(c, obs, obs->value + s0 * nobs, obs->variance + s0 * nobs, infl ? &slice[d] : nullptr);
      }))
    return rc;
  // split sites: every device ends with the same diagnostics and inflation, take device 0's
  for (size_t d = 0; d < m->handles.size(); ++d) {
    const bool out = d == 0 || !m->split;
    if (int rc = finish_assimilation(m->handles[d], out ? from_site(diag, m->parts[d].site0, (size_t)nobs * 4) : nullptr,
                                     nobs, out && infl ? &slice[d] : nullptr))
      return rc;
  }
  return 0;
}

}  // namespace

extern "C" int sipnet_gpu_comm_assimilate(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *obs, double *diag) {
  return assimilate_comm(c, obs, nullptr, diag);
}

extern "C" int sipnet_gpu_comm_assimilate_inflated(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *obs,
                                                   sipnet_gpu_inflation_spec *infl, double *diag) {
  if (!infl) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL inflation spec");
  return assimilate_comm(c, obs, infl, diag);
}

extern "C" int sipnet_gpu_multi_assimilate(sipnet_gpu_multi *m, const sipnet_gpu_obs_spec *obs, double *diag) {
  return assimilate_multi(m, obs, nullptr, diag);
}

extern "C" int sipnet_gpu_multi_assimilate_inflated(sipnet_gpu_multi *m, const sipnet_gpu_obs_spec *obs,
                                                    sipnet_gpu_inflation_spec *infl, double *diag) {
  if (!infl) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL inflation spec");
  return assimilate_multi(m, obs, infl, diag);
}

// ---- the particle filter: per-site systematic resampling (sip_resample.cuh) ---------------------------------------
namespace {

typedef unsigned __int128 u128;

int check_resample(const sipnet_gpu_handle *h, const double *u, int64_t nsites, double essFraction, const double *logw) {
  if (!u) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL u");
  if (std::isnan(essFraction) || essFraction < 0.0)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "ess_fraction must be >= 0 (INFINITY: always resample)");
  for (int64_t s = 0; s < nsites; ++s)
    if (!std::isnan(u[s]) && !(u[s] >= 0.0 && u[s] < 1.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "u[%lld] = %g is neither NaN nor in [0, 1)", (long long)s, u[s]);
  if (!logw && !h->loglik)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no log_weights, and the handle keeps no log-likelihood (SIPNET_GPU_OUT_LOGLIK)");
  return 0;
}

uint64_t resample_hash(const sipnet_gpu_handle *h, const double *u, double essFraction) {
  const int64_t S = h->nsites, words = rs::record_words(h);
  return ArgHash()
      .add(&S, sizeof S)
      .add(&words, sizeof words)
      .add(&essFraction, sizeof essFraction)
      .add(u, (size_t)S * sizeof(double))
      .value();
}

// K(C): the first slot k with t_k >= C, i.e. clamp(ceil((ceil(C n 2^32 / T) - U) / 2^32), 0, n)
int64_t first_slot(uint64_t C, uint64_t T, uint64_t U, int64_t n) {
  const u128 a = ((((u128)C * (uint64_t)n) << 32) + T - 1) / T;
  if (a <= U) return 0;
  const u128 k = (a - U + 0xffffffffu) >> 32;
  return k < (u128)n ? (int64_t)k : n;
}

// every rank's per-site record of the last site pass, rank-major, on the host
int site_records(sipnet_gpu_comm *c, std::vector<uint64_t> &out) {
  const size_t S = (size_t)c->local[0].h->nsites;
  if (int rc = all_gather_bytes(c, S * rs::kRec * sizeof(uint64_t), [](Local &l) -> void * { return l.h->rsSite; }))
    return rc;
  Local &l0 = c->local[0];
  out.resize((size_t)c->nranks * S * rs::kRec);
  CUDA_OK(cudaSetDevice(l0.h->device));
  CUDA_OK(cudaMemcpyAsync(out.data(), l0.h->rsSite, out.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, l0.h->stream));
  CUDA_OK(cudaStreamSynchronize(l0.h->stream));
  return 0;
}

// this rank's part of the copy: segment sizes (records) and where they sit (doubles)
struct CopyPlan {
  std::vector<int64_t> tab;
  std::vector<int64_t> sendCnt, sendBase, recvCnt, recvBase;
};

// the resampler's arguments for the members of `h` and their records (the rest zero)
void member_args(const sipnet_gpu_handle *h, rs::Args &a) {
  memset(&a, 0, sizeof a);
  a.status = h->status;
  a.sites = h->sites;
  a.memberSite = h->memberSite;
  a.nmembers = h->nmembers;
  a.ld = h->ld;
  a.nsites = (int32_t)h->nsites;
  a.nchunks = (int32_t)h->nchunks;
  a.chunk = h->chunk;
  a.siteChunks = h->siteChunks;
  a.params = h->params;
  a.state = h->state;
  a.ringV = h->ringV;
  a.ringW = h->ringW;
  a.loglik = h->loglik;
  a.loglikN = h->loglikN;
  a.counters = h->counters;
  a.recs = h->recs;
  a.recCount = h->recCount;
  a.ringCap = h->ringCap;
  a.maxRecs = h->maxRecs;
  a.words = rs::record_words(h);
}

// Resample every local rank of `c` (all ranks hold the same sites): logw[i] is local rank i's host log-weights or
// NULL (its log-likelihood).  diag (may be NULL) gets [nsites][4]; ancAll the team's ancestors, rank-major.
int run_resample(sipnet_gpu_comm *c, const double *u, double essFraction, const double *const *logw, double *diag,
                 std::vector<int64_t> &ancAll) {
  const int R = c->nranks;
  const int64_t S = c->local[0].h->nsites;
  const int words = rs::record_words(c->local[0].h);
  const size_t L = c->local.size();
  std::vector<rs::Args> args(L);
  std::vector<int64_t> rankBase((size_t)R + 1, 0);
  for (int q = 0; q < R; ++q) rankBase[(size_t)q + 1] = rankBase[(size_t)q] + c->memberCounts[(size_t)q];
  for (size_t i = 0; i < L; ++i) {
    Local &l = c->local[i];
    sipnet_gpu_handle *h = l.h;
    if (h->nsites != S || rs::record_words(h) != words)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the ranks of a team must hold the same sites and outputs");
    CUDA_OK(cudaSetDevice(h->device));
    if (int rc = rs::ensure_scratch(h)) return rc;
    if (int rc = grow(h->rsSite, h->rsSiteCap, (size_t)R * S * rs::kRec, h->stream)) return rc;
    if (logw[i])
      CUDA_OK(cudaMemcpyAsync(h->rsLogw, logw[i], (size_t)h->nmembers * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    rs::Args &a = args[i];
    member_args(h, a);
    a.logw = logw[i] ? h->rsLogw : h->loglik;
    a.nranks = R;
    a.rank = l.rank;
    a.idBase = rankBase[(size_t)l.rank];
    a.part = h->rsPart;
    a.w = h->rsW;
    a.c = h->rsC;
    a.siteRec = h->rsSite;
    a.lmax = h->rsLmax;
    a.anc = h->rsAnc;
    if (int rc = launched(h, rs::launch_weights(a, 0, h->stream), "resampling")) return rc;
    if (int rc = launched(h, rs::launch_site(a, 0, h->stream), "resampling")) return rc;
  }
  // pass a over the ranks: participants, members and the largest log-weight of every site
  std::vector<uint64_t> recA, recB;
  if (int rc = site_records(c, recA)) return rc;
  std::vector<double> lmax((size_t)S, -INFINITY);
  std::vector<int64_t> N((size_t)S, 0), n((size_t)S, 0);
  for (int r = 0; r < R; ++r)
    for (int64_t s = 0; s < S; ++s) {
      const uint64_t *p = &recA[((size_t)r * S + s) * rs::kRec];
      if (p[3]) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "a log-weight of site %lld is +inf", (long long)s);
      N[(size_t)s] += (int64_t)p[0];
      n[(size_t)s] += (int64_t)p[2];
      double v;
      memcpy(&v, &p[1], sizeof v);
      if (p[0]) lmax[(size_t)s] = std::max(lmax[(size_t)s], v);
    }
  for (int64_t s = 0; s < S; ++s)
    if (n[(size_t)s] > rs::kMaxSiteMembers)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "site %lld has %lld members; resampling takes at most 2^23 per site",
                  (long long)s, (long long)n[(size_t)s]);
  if (int rc = each_rank(c, [&](size_t i, Local &l) {
        sipnet_gpu_handle *h = l.h;
        CUDA_OK(cudaMemcpyAsync(h->rsLmax, lmax.data(), (size_t)S * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        if (int rc = launched(h, rs::launch_weights(args[i], 1, h->stream), "resampling")) return rc;
        return launched(h, rs::launch_site(args[i], 1, h->stream), "resampling");
      }))
    return rc;
  // pass b over the ranks: ESS, the decision and the slot ranges of every site (integer sums: any order, same bits)
  if (int rc = site_records(c, recB)) return rc;
  const size_t R1 = (size_t)R + 1;
  std::vector<int64_t> flag((size_t)S, 0), U((size_t)S, 0), T((size_t)S, 0), slot0((size_t)S * R1, 0), mem0((size_t)S * R1, 0);
  std::vector<uint64_t> toff((size_t)S * R1, 0);
  std::vector<double> dg((size_t)S * 4, 0.0);
  for (int64_t s = 0; s < S; ++s) {
    u128 f1 = 0, f2 = 0;
    for (int r = 0; r < R; ++r) {
      const uint64_t *p = &recB[((size_t)r * S + s) * rs::kRec];
      f1 += (u128)p[1] << 64 | p[0];
      f2 += (u128)p[3] << 64 | p[2];
      toff[(size_t)s * R1 + r + 1] = toff[(size_t)s * R1 + r] + p[4];
      mem0[(size_t)s * R1 + r + 1] = mem0[(size_t)s * R1 + r] + (int64_t)recA[((size_t)r * S + s) * rs::kRec + 2];
    }
    double *d = &dg[(size_t)s * 4];
    d[0] = (double)N[(size_t)s];
    d[1] = d[2] = __builtin_nan("");
    if (N[(size_t)s] == 0) continue;
    const double s1 = std::ldexp((double)f1, -rs::kFixBits), s2 = std::ldexp((double)f2, -rs::kFixBits);
    d[1] = s1 * s1 / s2;
    d[2] = lmax[(size_t)s] + std::log(s1 / (double)N[(size_t)s]);
    if (std::isnan(u[s]) || !(d[1] < essFraction * (double)n[(size_t)s])) continue;
    flag[(size_t)s] = 1;
    U[(size_t)s] = (int64_t)(uint64_t)std::ldexp(u[s], 32);
    T[(size_t)s] = (int64_t)toff[(size_t)s * R1 + R];
    for (size_t p = 0; p <= (size_t)R; ++p)
      slot0[(size_t)s * R1 + p] = first_slot(toff[(size_t)s * R1 + p], (uint64_t)T[(size_t)s], (uint64_t)U[(size_t)s], n[(size_t)s]);
  }
  // records travelling from rank p to rank q for site s
  auto count = [&](int p, int q, int64_t s) {
    const int64_t *a = &slot0[(size_t)s * R1], *b = &mem0[(size_t)s * R1];
    return std::max<int64_t>(0, std::min(a[p + 1], b[q + 1]) - std::max(a[p], b[q]));
  };
  std::vector<CopyPlan> plan(L);
  for (size_t i = 0; i < L; ++i) {
    Local &l = c->local[i];
    sipnet_gpu_handle *h = l.h;
    const int r = l.rank;
    CopyPlan &P = plan[i];
    P.sendCnt.assign((size_t)R, 0);
    P.recvCnt.assign((size_t)R, 0);
    P.sendBase.assign((size_t)R, 0);
    P.recvBase.assign((size_t)R, 0);
    std::vector<int64_t> sendPos((size_t)S * R), recvPos((size_t)S * R), outPre((size_t)S + 1, 0), rtoff((size_t)S);
    for (int64_t s = 0; s < S; ++s) {
      for (int q = 0; q < R; ++q) {
        sendPos[(size_t)s * R + q] = P.sendCnt[(size_t)q];
        P.sendCnt[(size_t)q] += count(r, q, s);
        recvPos[(size_t)s * R + q] = P.recvCnt[(size_t)q];
        P.recvCnt[(size_t)q] += count(q, r, s);
      }
      outPre[(size_t)s + 1] = outPre[(size_t)s] + slot0[(size_t)s * R1 + r + 1] - slot0[(size_t)s * R1 + r];
      rtoff[(size_t)s] = (int64_t)toff[(size_t)s * R1 + r];
    }
    size_t sendWords = 0, recvWords = 0;
    for (int q = 0; q < R; ++q) {
      P.sendBase[(size_t)q] = (int64_t)sendWords;
      sendWords += (size_t)P.sendCnt[(size_t)q] * words;
      if (q == r) continue;
      P.recvBase[(size_t)q] = (int64_t)recvWords;
      recvWords += (size_t)P.recvCnt[(size_t)q] * words;
    }
    CUDA_OK(cudaSetDevice(h->device));
    if (int rc = grow(h->rsSend, h->rsSendCap, sendWords, h->stream)) return rc;
    if (int rc = grow(h->rsRecv, h->rsRecvCap, recvWords, h->stream)) return rc;
    std::vector<int64_t> src((size_t)R);
    for (int p = 0; p < R; ++p)
      src[(size_t)p] = reinterpret_cast<int64_t>(p == r ? h->rsSend + P.sendBase[(size_t)r] : h->rsRecv + P.recvBase[(size_t)p]);
    std::vector<int64_t> &tab = P.tab;
    std::vector<size_t> at;
    for (const std::vector<int64_t> *v : {&flag, &U, &T, &n, &rtoff, &slot0, &mem0, &sendPos, &recvPos, &outPre, &P.sendBase,
                                          &P.sendCnt, &P.recvCnt, &src}) {
      at.push_back(tab.size());
      tab.insert(tab.end(), v->begin(), v->end());
    }
    if (int rc = grow(h->rsTab, h->rsTabCap, tab.size(), h->stream)) return rc;
    CUDA_OK(cudaMemcpyAsync(h->rsTab, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    rs::Args &a = args[i];
    const int64_t *t = h->rsTab;
    a.flag = t + at[0];
    a.U = t + at[1];
    a.T = t + at[2];
    a.n = t + at[3];
    a.toff = t + at[4];
    a.slot0 = t + at[5];
    a.mem0 = t + at[6];
    a.sendPos = t + at[7];
    a.recvPos = t + at[8];
    a.outPre = t + at[9];
    a.sendBase = t + at[10];
    a.sendCnt = t + at[11];
    a.recvCnt = t + at[12];
    a.src = reinterpret_cast<double *const *>(t + at[13]);
    a.sendBuf = h->rsSend;
    a.nOut = outPre[(size_t)S];
    if (int rc = launched(h, rs::launch_prefix(a, h->stream), "resampling")) return rc;
    if (int rc = launched(h, rs::launch_pack(a, h->stream), "resampling")) return rc;
  }
  // the segments between ranks
  if (R > 1 && c->loopback) {
    if (int rc = sync_all(c)) return rc;
    for (size_t i = 0; i < L; ++i)
      for (size_t j = 0; j < L; ++j) {
        const int p = c->local[j].rank, q = c->local[i].rank;
        const int64_t cnt = plan[i].recvCnt[(size_t)p];
        if (p == q || cnt == 0) continue;
        CUDA_OK(cudaMemcpyAsync(c->local[i].h->rsRecv + plan[i].recvBase[(size_t)p],
                                c->local[j].h->rsSend + plan[j].sendBase[(size_t)q], (size_t)cnt * words * sizeof(double),
                                cudaMemcpyDeviceToDevice, c->local[i].h->stream));
      }
    if (int rc = sync_all(c)) return rc;
  } else if (R > 1) {  // send and receive of one pair must sit in one group
    NCCL_OK(nccl_api()->GroupStart());
    for (size_t i = 0; i < L; ++i) {
      Local &l = c->local[i];
      CUDA_OK(cudaSetDevice(l.h->device));
      for (int q = 0; q < R; ++q) {
        if (q == l.rank) continue;
        if (const int64_t cnt = plan[i].sendCnt[(size_t)q])
          NCCL_OK(nccl_api()->Send(l.h->rsSend + plan[i].sendBase[(size_t)q], (size_t)cnt * words * sizeof(double), ncclUint8,
                                   q, l.comm, l.h->stream));
        if (const int64_t cnt = plan[i].recvCnt[(size_t)q])
          NCCL_OK(nccl_api()->Recv(l.h->rsRecv + plan[i].recvBase[(size_t)q], (size_t)cnt * words * sizeof(double), ncclUint8,
                                   q, l.comm, l.h->stream));
      }
    }
    NCCL_OK(nccl_api()->GroupEnd());
  }
  if (int rc = each_rank(c, [&](size_t i, Local &l) {
        return launched(l.h, rs::launch_unpack(args[i], l.h->stream), "resampling");
      }))
    return rc;
  // the ancestors of the whole team, and the distinct ancestors of every resampled site
  ancAll.assign((size_t)rankBase[(size_t)R], -1);
  if (R == 1) {
    sipnet_gpu_handle *h = c->local[0].h;
    CUDA_OK(cudaMemcpyAsync(ancAll.data(), h->rsAnc, ancAll.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(cudaStreamSynchronize(h->stream));
  } else if (int rc = team_member_words(c, ancAll.data(), ancAll.size() * sizeof(int64_t),
                                        [](const sipnet_gpu_handle *h) -> const void * { return h->rsAnc; }, "ancestor")) {
    return rc;
  }
  std::vector<int64_t> last((size_t)S, -1);
  for (int r = 0; r < R; ++r) {
    const int64_t *a = ancAll.data() + rankBase[(size_t)r];
    for (int64_t s = 0; s < S; ++s) {  // a rank's members are in site order
      const int64_t cnt = (int64_t)recA[((size_t)r * S + s) * rs::kRec + 2];
      for (int64_t k = 0; k < cnt; ++k, ++a)
        if (*a >= 0 && *a != last[(size_t)s]) {
          dg[(size_t)s * 4 + 3] += 1.0;
          last[(size_t)s] = *a;
        }
    }
  }
  if (diag) memcpy(diag, dg.data(), dg.size() * sizeof(double));
  return 0;
}

}  // namespace

extern "C" int sipnet_gpu_resample(sipnet_gpu_handle *h, const double *u, double ess_fraction, const double *log_weights,
                                   int64_t *ancestors, double *diag) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_resample(h, u, h->nsites, ess_fraction, log_weights)) return rc;
  sipnet_gpu_comm one = team_of_one(h);
  std::vector<int64_t> anc;
  if (int rc = run_resample(&one, u, ess_fraction, &log_weights, diag, anc)) return rc;
  if (ancestors) memcpy(ancestors, anc.data(), anc.size() * sizeof(int64_t));
  return 0;
}

extern "C" int sipnet_gpu_comm_resample(sipnet_gpu_comm *c, const double *u, double ess_fraction, const double *log_weights,
                                        int64_t *ancestors, double *diag) {
  if (!c) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm");
  sipnet_gpu_handle *h = c->local[0].h;
  const int64_t S = h->nsites;
  const int bad = check_resample(h, u, S, ess_fraction, log_weights);
  if (int rc = team_agree(c, bad, bad ? 0 : resample_hash(h, u, ess_fraction), "resampling arguments")) return rc;
  std::vector<int64_t> anc;
  if (int rc = run_resample(c, u, ess_fraction, &log_weights, diag, anc)) return rc;
  if (ancestors) memcpy(ancestors, anc.data(), anc.size() * sizeof(int64_t));
  return 0;
}

extern "C" int sipnet_gpu_multi_resample(sipnet_gpu_multi *m, const double *u, double ess_fraction, const double *log_weights,
                                         int64_t *ancestors, double *diag) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_resample(m->handles[0], u, m->nsites, ess_fraction, log_weights)) return rc;
  const size_t D = m->handles.size();
  // the log-weights per device, checked here: a device must not resample before another one rejects the call
  std::vector<double> all;
  if (!log_weights) {
    all.resize((size_t)m->nmembers);
    if (int rc = sipnet_gpu_multi_gather(m, SIPNET_GPU_GATHER_LOGLIK, all.data(), all.size() * sizeof(double))) return rc;
    log_weights = all.data();
  }
  for (int64_t i = 0; i < m->nmembers; ++i)
    if (log_weights[i] == INFINITY) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "log_weights[%lld] is +inf", (long long)i);
  std::vector<int64_t> siteN((size_t)m->nsites, 0);
  for (size_t d = 0; d < D; ++d)
    for (size_t s = 0; s < m->handles[d]->hostSites.size(); ++s)
      siteN[(size_t)m->parts[d].site0 + s] += m->handles[d]->hostSites[s].memberCount;
  for (int64_t s = 0; s < m->nsites; ++s)
    if (siteN[(size_t)s] > rs::kMaxSiteMembers)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "site %lld has %lld members; resampling takes at most 2^23 per site",
                  (long long)s, (long long)siteN[(size_t)s]);
  const Copies lw = device_copies(m, log_weights, 1);
  std::vector<std::vector<int64_t>> glob;
  for (size_t d = 0; d < D; ++d) glob.push_back(config_index(m, d));
  return multi_run(m, [&](sipnet_gpu_comm *c, size_t d) {
    const int64_t s0 = m->parts[d].site0;
    std::vector<int64_t> anc;
    if (int rc = run_resample(c, u + s0, ess_fraction, lw.at.data() + d, from_site(diag, s0, 4), anc)) return rc;
    if (ancestors) {  // rank-major -> configuration order
      std::vector<int64_t> base(1, 0);
      for (int64_t n : c->memberCounts) base.push_back(base.back() + n);
      for (size_t i = 0; i < c->local.size(); ++i)
        for (size_t j = 0; j < glob[d + i].size(); ++j) {
          const int64_t v = anc[(size_t)base[i] + j];
          int64_t g = -1;
          if (v >= 0) {
            const size_t q = (size_t)(std::upper_bound(base.begin(), base.end(), v) - base.begin()) - 1;
            g = glob[d + q][(size_t)(v - base[q])];
          }
          ancestors[glob[d + i][j]] = g;
        }
    }
    return 0;
  });
}

// ---- parameter rejuvenation: the Liu-West move (sip_jitter.cuh) ---------------------------------------------------
namespace {

bool derived_row(int32_t r) { return r == SIPNET_P_psnTMax || r == SIPNET_P_coarseRootAllocation; }

// the moved rows of a spec (both moves): 0, or SIPNET_GPU_ERR_BAD_ARGUMENT with the reason
int check_rows(int32_t nRows, const int32_t *rows, const int32_t *transform, const double *lower, const double *upper) {
  if (nRows < 1 || nRows > jt::kMaxRows) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "n_rows must be 1..%d", jt::kMaxRows);
  bool seen[SIPNET_GPU_NPARAMS] = {};
  for (int j = 0; j < nRows; ++j) {
    const int32_t r = rows[j], tf = transform[j];
    if (r < 0 || r >= SIPNET_GPU_NPARAMS) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "parameter row %d out of range", r);
    if (derived_row(r)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "parameter row %d is derived by setupModel()", r);
    if (seen[r]) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "parameter row %d listed twice", r);
    seen[r] = true;
    if (tf != SIPNET_GPU_TF_IDENTITY && tf != SIPNET_GPU_TF_LOG && tf != SIPNET_GPU_TF_LOGIT)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "unknown transform %d of row %d", tf, r);
    if (tf == SIPNET_GPU_TF_LOGIT) {
      if (!lower || !upper) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "LOGIT row %d without lower / upper", r);
      const double lo = lower[j], hi = upper[j];
      if (!std::isfinite(lo) || !std::isfinite(hi) || !(lo < hi))
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "LOGIT bounds of row %d must be finite with lower < upper", r);
    }
  }
  return 0;
}

int check_normals(const double *z, int32_t nRows, int64_t nmembers) {
  for (size_t i = 0; i < (size_t)nRows * (size_t)nmembers; ++i)
    if (!std::isfinite(z[i])) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "z[%zu] is not finite", i);
  return 0;
}

// the spec against `nsites` sites and `nmembers` members (z): 0, or SIPNET_GPU_ERR_BAD_ARGUMENT with the reason
int check_jitter(const sipnet_gpu_jitter_spec *sp, int64_t nsites, int64_t nmembers) {
  if (!sp || !sp->rows || !sp->transform || !sp->shrink || !sp->z)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL jitter spec or array");
  if (int rc = check_rows(sp->n_rows, sp->rows, sp->transform, sp->lower, sp->upper)) return rc;
  for (int64_t s = 0; s < nsites; ++s) {
    const double a = sp->shrink[s];
    if (!std::isnan(a) && !(a > 0.0 && a < 1.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "shrink[%lld] = %g is neither NaN nor in (0, 1)", (long long)s, a);
  }
  return check_normals(sp->z, sp->n_rows, nmembers);
}

uint64_t jitter_hash(const sipnet_gpu_jitter_spec *sp, int64_t nsites) {
  ArgHash h;
  h.add(&nsites, sizeof nsites)
      .add(&sp->n_rows, sizeof sp->n_rows)
      .add(sp->rows, (size_t)sp->n_rows * sizeof(int32_t))
      .add(sp->transform, (size_t)sp->n_rows * sizeof(int32_t));
  for (int j = 0; j < sp->n_rows; ++j)
    if (sp->transform[j] == SIPNET_GPU_TF_LOGIT) h.add(&sp->lower[j], sizeof(double)).add(&sp->upper[j], sizeof(double));
  return h.add(sp->shrink, (size_t)nsites * sizeof(double)).value();
}

// The arguments of the move's kernels on local rank `l` (scratch made, rows checked): the handle, the rows, the
// chunk records and a team's exchange buffer (grown here); the caller sets the per-site move arguments.
int jitter_args(sipnet_gpu_comm *c, Local &l, int32_t n, const int32_t *rows, const int32_t *transform,
                const double *lower, const double *upper, jt::Args &a) {
  sipnet_gpu_handle *h = l.h;
  const int R = c->nranks;
  const int64_t S = h->nsites;
  if (S != c->local[0].h->nsites) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the ranks of a team must hold the same sites");
  CUDA_OK(cudaSetDevice(h->device));
  if (int rc = jt::ensure_scratch(h)) return rc;
  if (R > 1)
    if (int rc = grow(l.xchg, l.xchgCap, (size_t)R * S * jt::kRec * sizeof(double), h->stream)) return rc;
  memset(&a, 0, sizeof a);
  a.params = h->params;
  a.status = h->status;
  a.ld = h->ld;
  a.nmembers = h->nmembers;
  a.sites = h->sites;
  a.nsites = (int32_t)S;
  a.nchunks = (int32_t)h->nchunks;
  a.chunk = h->chunk;
  a.siteChunks = h->siteChunks;
  a.nrows = n;
  a.nranks = R;
  a.rank = l.rank;
  for (int j = 0; j < n; ++j) {
    a.rows[j] = rows[j];
    a.transform[j] = transform[j];
    a.lower[j] = transform[j] == SIPNET_GPU_TF_LOGIT ? lower[j] : 0.0;
    a.upper[j] = transform[j] == SIPNET_GPU_TF_LOGIT ? upper[j] : 0.0;
  }
  a.z = h->jtZ;
  a.part = h->jtPart;
  a.mom = h->jtMom;
  a.coef = h->jtCoef;
  a.diag = h->jtDiag;
  a.rankRec = reinterpret_cast<double *>(l.xchg);
  return 0;
}

// One pass of the move on every local rank: members(pass) (unless the chunk records are already written), site(pass),
// and for a team the exchange of the per-site partials and combine(pass).
int jitter_pass(sipnet_gpu_comm *c, std::vector<jt::Args> &args, int pass, bool members, const char *what) {
  return site_pass(
      c, jt::kRec,
      [&](size_t i, Local &l) {
        if (members)
          if (int rc = launched(l.h, jt::launch_members(args[i], pass, l.h->stream), what)) return rc;
        return launched(l.h, jt::launch_site(args[i], pass, l.h->stream), what);
      },
      [&](size_t i, Local &l) { return launched(l.h, jt::launch_combine(args[i], pass, l.h->stream), what); });
}

// local rank 0's diagnostics into diag (may be NULL), and every local stream finished
int jitter_diag(sipnet_gpu_comm *c, double *diag) {
  if (diag) {
    sipnet_gpu_handle *h = c->local[0].h;
    CUDA_OK(cudaSetDevice(h->device));
    CUDA_OK(cudaMemcpyAsync(diag, h->jtDiag, (size_t)h->nsites * 4 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  }
  return sync_all(c);
}

// Move every local rank of `c` (all ranks hold the same sites): shrink holds the handles' sites, z[i] local rank i's
// members.  A team of one needs no exchange and no host round trip; a larger team all-gathers the per-site partial
// sums of the two moment passes and of the counts, and sums them in rank order on every rank.  diag (may be NULL)
// gets local rank 0's [nsites][4].
int run_rejuvenate(sipnet_gpu_comm *c, const sipnet_gpu_jitter_spec *sp, const double *shrink, const double *const *z,
                   double *diag) {
  const int n = sp->n_rows;
  std::vector<jt::Args> args(c->local.size());
  for (size_t i = 0; i < c->local.size(); ++i) {
    sipnet_gpu_handle *h = c->local[i].h;
    if (int rc = jitter_args(c, c->local[i], n, sp->rows, sp->transform, sp->lower, sp->upper, args[i])) return rc;
    CUDA_OK(cudaMemcpyAsync(h->jtShrink, shrink, (size_t)h->nsites * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->jtZ, z[i], (size_t)n * h->nmembers * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    args[i].shrink = h->jtShrink;
  }
  for (int pass = 1; pass <= 3; ++pass)
    if (int rc = jitter_pass(c, args, pass, true, "rejuvenation")) return rc;
  return jitter_diag(c, diag);
}

}  // namespace

extern "C" int sipnet_gpu_rejuvenate(sipnet_gpu_handle *h, const sipnet_gpu_jitter_spec *spec, double *diag) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_jitter(spec, h->nsites, h->nmembers)) return rc;
  sipnet_gpu_comm one = team_of_one(h);
  return run_rejuvenate(&one, spec, spec->shrink, &spec->z, diag);
}

extern "C" int sipnet_gpu_comm_rejuvenate(sipnet_gpu_comm *c, const sipnet_gpu_jitter_spec *spec, double *diag) {
  if (!c) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm");
  sipnet_gpu_handle *h = c->local[0].h;
  const int64_t S = h->nsites;
  const int bad = check_jitter(spec, S, h->nmembers);
  if (int rc = team_agree(c, bad, bad ? 0 : jitter_hash(spec, S), "rejuvenation specs")) return rc;
  return run_rejuvenate(c, spec, spec->shrink, &spec->z, diag);
}

extern "C" int sipnet_gpu_multi_rejuvenate(sipnet_gpu_multi *m, const sipnet_gpu_jitter_spec *spec, double *diag) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_jitter(spec, m->nsites, m->nmembers)) return rc;
  const Copies z = device_copies(m, spec->z, (size_t)spec->n_rows);
  return multi_run(m, [&](sipnet_gpu_comm *c, size_t d) {
    const int64_t s0 = m->parts[d].site0;
    return run_rejuvenate(c, spec, spec->shrink + s0, z.at.data() + d, from_site(diag, s0, 4));
  });
}

// ---- parameter calibration: the Metropolis-Hastings move (sip_jitter.cuh proposes, sip_resample.cuh decides) ------
namespace {

// the spec against `nsites` sites, `nmembers` members, the next step and whether the handles keep a log-likelihood
int check_mh(const sipnet_gpu_mh_spec *sp, int64_t nsites, int64_t nmembers, int64_t step, bool hasLoglik) {
  if (!sp || !sp->rows || !sp->transform || !sp->prior || !sp->prior_a || !sp->prior_b || !sp->scale || !sp->tempering ||
      !sp->current_loglik || !sp->z || !sp->log_u)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL Metropolis-Hastings spec or array");
  if (int rc = check_rows(sp->n_rows, sp->rows, sp->transform, sp->lower, sp->upper)) return rc;
  for (int j = 0; j < sp->n_rows; ++j) {
    const double a = sp->prior_a[j], b = sp->prior_b[j];
    if (sp->prior[j] == SIPNET_GPU_PRIOR_FLAT) {
      if (std::isnan(a) || std::isnan(b) || !(a < b))
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "FLAT prior of row %d needs prior_a < prior_b", sp->rows[j]);
      if (sp->transform[j] == SIPNET_GPU_TF_LOGIT && !(a >= sp->lower[j] && b <= sp->upper[j]))
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "FLAT prior of LOGIT row %d must lie inside [lower, upper]", sp->rows[j]);
    } else if (sp->prior[j] == SIPNET_GPU_PRIOR_NORMAL) {
      if (!std::isfinite(a) || !std::isfinite(b) || !(b > 0.0))
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NORMAL prior of row %d needs a finite mean and a finite sd > 0",
                    sp->rows[j]);
    } else {
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "unknown prior %d of row %d", sp->prior[j], sp->rows[j]);
    }
  }
  for (int64_t s = 0; s < nsites; ++s) {
    const double h = sp->scale[s], t = sp->tempering[s];
    if (!std::isnan(h) && !(std::isfinite(h) && h > 0.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "scale[%lld] = %g is neither NaN nor finite > 0", (long long)s, h);
    if (!(t >= 0.0 && t <= 1.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "tempering[%lld] = %g is not in [0, 1]", (long long)s, t);
    if (!std::isnan(h) && t > 0.0 && !hasLoglik)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "tempering[%lld] > 0 on a handle without SIPNET_GPU_OUT_LOGLIK", (long long)s);
  }
  if (int rc = check_normals(sp->z, sp->n_rows, nmembers)) return rc;
  for (int64_t i = 0; i < nmembers; ++i)
    if (!(sp->log_u[i] <= 0.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "log_u[%lld] = %g is not <= 0", (long long)i, sp->log_u[i]);
  if (step < 1) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "the window [0, s) is empty: run at least one step first");
  return 0;
}

// everything the ranks of a team must agree on (all but the per-member arrays)
uint64_t mh_hash(const sipnet_gpu_mh_spec *sp, int64_t nsites, int64_t step, bool hasLoglik) {
  const size_t n = (size_t)sp->n_rows;
  const uint8_t ll = hasLoglik;
  ArgHash h;
  h.add(&nsites, sizeof nsites).add(&step, sizeof step).add(&ll, 1).add(&sp->n_rows, sizeof sp->n_rows)
      .add(sp->rows, n * sizeof(int32_t)).add(sp->transform, n * sizeof(int32_t)).add(sp->prior, n * sizeof(int32_t))
      .add(sp->prior_a, n * sizeof(double)).add(sp->prior_b, n * sizeof(double));
  for (size_t j = 0; j < n; ++j)
    if (sp->transform[j] == SIPNET_GPU_TF_LOGIT) h.add(&sp->lower[j], sizeof(double)).add(&sp->upper[j], sizeof(double));
  return h.add(sp->scale, (size_t)nsites * sizeof(double)).add(sp->tempering, (size_t)nsites * sizeof(double)).value();
}

// reset() and run(0, s) of one handle, in pieces its output buffers hold
int rerun_window(sipnet_gpu_handle *h, int64_t s) {
  if (int rc = sipnet_gpu_reset(h)) return rc;
  const int64_t piece = (h->out || h->dbg) && h->outCap > 0 ? h->outCap : s;
  for (int64_t b = 0; b < s; b += piece)
    if (int rc = sipnet_gpu_run(h, b, std::min(s, b + piece))) return rc;
  return 0;
}

// Move every local rank of `c` (all ranks hold the same sites): scale and tau hold the handles' sites, curL[i], z[i]
// and logU[i] local rank i's members.  The sequence: the two moment passes (a team exchanges their partials), the
// snapshot, the proposal, reset and run of every local handle over its window (no exchange), the accept pass, and the
// site pass of the counts (a team exchanges them).  diag (may be NULL) gets local rank 0's [nsites][4].
int run_mh(sipnet_gpu_comm *c, const sipnet_gpu_mh_spec *sp, const double *scale, const double *tau,
           const double *const *curL, const double *const *z, const double *const *logU, double *diag) {
  const int n = sp->n_rows;
  const int64_t S = c->local[0].h->nsites;
  const size_t L = c->local.size();
  if (std::all_of(scale, scale + S, [](double v) { return std::isnan(v); })) {  // no site moves: nothing to launch
    if (diag)
      for (int64_t s = 0; s < S; ++s) {
        double *d = diag + s * 4;
        d[0] = __builtin_nan("");
        d[1] = -1.0;
        d[2] = d[3] = 0.0;
      }
    return 0;
  }
  std::vector<jt::Args> args(L);
  std::vector<rs::Args> acc(L);
  std::vector<int64_t> window(L);
  for (size_t i = 0; i < L; ++i) {
    sipnet_gpu_handle *h = c->local[i].h;
    if (int rc = jitter_args(c, c->local[i], n, sp->rows, sp->transform, sp->lower, sp->upper, args[i])) return rc;
    if (int rc = rs::ensure_mh_scratch(h)) return rc;
    const size_t M = (size_t)h->nmembers;
    CUDA_OK(cudaMemcpyAsync(h->mhScale, scale, (size_t)S * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->mhTau, tau, (size_t)S * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->jtZ, z[i], (size_t)n * M * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->mhCurL, curL[i], M * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->mhLogU, logU[i], M * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    jt::Args &a = args[i];
    a.scale = h->mhScale;
    a.curLoglik = h->mhCurL;
    for (int j = 0; j < n; ++j) {
      a.prior[j] = sp->prior[j];
      a.priorA[j] = sp->prior_a[j];
      a.priorB[j] = sp->prior_b[j];
    }
    a.valid = h->mhValid;
    a.dlp = h->mhDlp;
    rs::Args &r = acc[i];
    member_args(h, r);
    r.snap = h->mhSnap;
    r.valid = h->mhValid;
    r.dlp = h->mhDlp;
    r.curLoglik = h->mhCurL;
    r.logU = h->mhLogU;
    r.tau = h->mhTau;
    r.count = h->jtPart;
    r.countStride = jt::kRec;
    window[i] = h->stepsDone;
  }
  for (int pass = 1; pass <= 2; ++pass)
    if (int rc = jitter_pass(c, args, pass, true, "Metropolis-Hastings")) return rc;
  if (int rc = each_rank(c, [&](size_t i, Local &l) {
        if (int rc = launched(l.h, rs::launch_snapshot(acc[i], l.h->stream), "Metropolis-Hastings")) return rc;
        return launched(l.h, jt::launch_members(args[i], 3, l.h->stream), "Metropolis-Hastings");
      }))
    return rc;
  // asynchronous: the devices run side by side
  if (int rc = each_rank(c, [&](size_t i, Local &l) { return rerun_window(l.h, window[i]); })) return rc;
  if (int rc = each_rank(c, [&](size_t i, Local &l) {
        sipnet_gpu_handle *h = l.h;
        if (int rc = launched(h, rs::launch_accept(acc[i], h->stream), "Metropolis-Hastings")) return rc;
        h->lastBegin = h->lastEnd = window[i];  // no run range: its outputs are the proposals' (or are gone)
        h->summariesValid = false;
        return 0;
      }))
    return rc;
  if (int rc = jitter_pass(c, args, 3, false, "Metropolis-Hastings")) return rc;
  return jitter_diag(c, diag);
}

}  // namespace

extern "C" int sipnet_gpu_mh_move(sipnet_gpu_handle *h, const sipnet_gpu_mh_spec *spec, double *diag) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (int rc = check_mh(spec, h->nsites, h->nmembers, h->stepsDone, h->loglik != nullptr)) return rc;
  sipnet_gpu_comm one = team_of_one(h);
  return run_mh(&one, spec, spec->scale, spec->tempering, &spec->current_loglik, &spec->z, &spec->log_u, diag);
}

extern "C" int sipnet_gpu_comm_mh_move(sipnet_gpu_comm *c, const sipnet_gpu_mh_spec *spec, double *diag) {
  if (!c) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL comm");
  sipnet_gpu_handle *h = c->local[0].h;
  const int64_t S = h->nsites;
  const bool ll = h->loglik != nullptr;
  const int bad = check_mh(spec, S, h->nmembers, h->stepsDone, ll);
  if (int rc = team_agree(c, bad, bad ? 0 : mh_hash(spec, S, h->stepsDone, ll), "Metropolis-Hastings specs")) return rc;
  return run_mh(c, spec, spec->scale, spec->tempering, &spec->current_loglik, &spec->z, &spec->log_u, diag);
}

extern "C" int sipnet_gpu_multi_mh_move(sipnet_gpu_multi *m, const sipnet_gpu_mh_spec *spec, double *diag) {
  if (!m) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  int64_t step = 0;
  for (const sipnet_gpu_handle *h : m->handles) step = std::max(step, h->stepsDone);
  if (int rc = check_mh(spec, m->nsites, m->nmembers, step, m->handles[0]->loglik != nullptr)) return rc;
  const Copies z = device_copies(m, spec->z, (size_t)spec->n_rows), cl = device_copies(m, spec->current_loglik, 1),
               lu = device_copies(m, spec->log_u, 1);
  return multi_run(m, [&](sipnet_gpu_comm *c, size_t d) {
    const int64_t s0 = m->parts[d].site0;
    return run_mh(c, spec, spec->scale + s0, spec->tempering + s0, cl.at.data() + d, z.at.data() + d, lu.at.data() + d,
                  from_site(diag, s0, 4));
  });
}
