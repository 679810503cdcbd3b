// sip_handle.h -- the handle behind the C ABI (private to the library: sipnet_gpu.cu, sip_comm.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "sip_types.cuh"

struct sipnet_gpu_handle {
  int device = 0;
  uint32_t flags = 0;
  uint32_t outputs = 0;
  int math = 0;
  int64_t nmembers = 0, ld = 0, nsites = 0, maxSteps = 0, maxSiteMembers = 0;
  int64_t outCap = 0;      // steps of output kept per run
  int64_t stepsDone = 0;   // next step to run
  int64_t lastBegin = 0, lastEnd = 0;
  int blockThreads = 128, nblocks = 0, ringCap = 0;
  int ncols = 0;  // column slots in `out`
  int8_t colSlot[SIPNET_GPU_NOUT];
  std::vector<int32_t> summaryCols;
  std::vector<double> quantiles;
  int maxRecs = 0;
  double sigma = 1.0;
  bool sitesDiffer = false;
  bool anyObs = false;

  cudaStream_t stream = nullptr;
  bool ownStream = false;
  cudaEvent_t evStart = nullptr, evStop = nullptr, evT0 = nullptr, evT1 = nullptr;
  cudaStream_t copyStream = nullptr;
  cudaEvent_t evRunDone[2] = {nullptr, nullptr}, evCopyDone[2] = {nullptr, nullptr};
  int64_t launches = 0;

  // device memory
  double *params = nullptr, *state = nullptr, *ringV = nullptr, *ringW = nullptr;
  uint32_t *status = nullptr;
  uint32_t *counters = nullptr;  // [SIPNET_GPU_NCOUNTERS][ld], with the debug dump only
  int32_t *memberSite = nullptr;
  sip::BlockDesc *blocks = nullptr;
  sip::SiteDev *sites = nullptr;
  std::vector<void *> siteAllocs;
  double *out = nullptr, *dbg = nullptr, *loglik = nullptr, *loglikN = nullptr;
  sipnet_gpu_event_record *recs = nullptr;
  int32_t *recCount = nullptr;
  double *mean = nullptr, *var = nullptr, *quant = nullptr;
  bool staticSched = false;
  unsigned char *sched = nullptr;  // work counter (8 B, padded to 16) + per-block progress words (dynamic scheduling)
  // segment-start copies for the replay of members flagged by the optimistic kernel (MATH_FAST only)
  double *stateBk = nullptr, *ringVBk = nullptr, *ringWBk = nullptr, *loglikBk = nullptr, *loglikNBk = nullptr;
  uint32_t *statusBk = nullptr;
  int32_t *recCountBk = nullptr;
  bool summariesValid = false;
  std::vector<sip::SiteDev> hostSites;
  bool mixedBlocks = false;          // some block holds members of two sites
  sip::StepConsts kc = {};           // launch-lifetime constants of the step (device-evaluated at init)
  // the chunk tables of the ensemble filters (sip::ensure_chunks), made by the first filter call
  int64_t nchunks = 0;
  int2 *chunk = nullptr, *siteChunks = nullptr;
  // ensemble adjustment Kalman filter scratch (sip_assim.cu), made by the first assimilation
  int asObsCap = 0;
  double *asPart = nullptr, *asMom = nullptr, *asCoef = nullptr, *asObs = nullptr, *asDiag = nullptr;
  double *asInfl = nullptr;  // [nsites][3] {λ0, λ, σ} of the prior inflation, made by the first inflated call
  // particle filter scratch (sip_resample.cu), made by the first resampling; the tables and the record buffers grow
  uint64_t *rsW = nullptr, *rsC = nullptr, *rsSite = nullptr, *rsPart = nullptr;
  double *rsLogw = nullptr, *rsLmax = nullptr, *rsSend = nullptr, *rsRecv = nullptr;
  int64_t *rsAnc = nullptr, *rsTab = nullptr;
  size_t rsSiteCap = 0, rsTabCap = 0, rsSendCap = 0, rsRecvCap = 0;  // elements
  // parameter move scratch (sip_jitter.cu), made by the first rejuvenation
  double *jtPart = nullptr, *jtMom = nullptr, *jtCoef = nullptr, *jtDiag = nullptr, *jtShrink = nullptr, *jtZ = nullptr;
};

namespace sip {
// error plumbing shared by the translation units of the library (sipnet_gpu.cu)
int fail(int code, const char *fmt, ...);
// queue the local row summaries of the last run range (sipnet_gpu.cu)
int ensure_summaries(sipnet_gpu_handle *h);

// The ensemble filters (sip_assim.cu, sip_resample.cu, sip_jitter.cu) reduce over chunks of kChunk consecutive
// SITE-LOCAL member indices, so their sums depend on a site's members and not on the handle's block layout.
constexpr int kChunk = 128;
// members no filter counts or changes
constexpr uint32_t kExcluded = SIPNET_GPU_ST_BAD_ALLOCATION | SIPNET_GPU_ST_NONFINITE;
// the handle's chunk tables, made once (sipnet_gpu.cu): chunk[nchunks] = (site, first site-local member),
// siteChunks[nsites] = (first chunk, chunk count), sites in order and a site's chunks in member order
int ensure_chunks(sipnet_gpu_handle *h);
}  // namespace sip
