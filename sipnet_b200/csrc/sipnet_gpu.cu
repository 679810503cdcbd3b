// sipnet_gpu.cu -- implementation of the C ABI in include/sipnet_gpu.h.
//
// Host-side responsibilities (everything that is state-independent is decided
// here, once, so the device loop carries no control plane):
//   * validate the configuration the way the reference would fail at run time
//     (processEvents(): non-positive step length -> 3, event without climate
//     record -> 5, unknown irrigation method / event type -> 4; frontend.c:217:
//     first event before first climate record -> 5)
//   * bind every events.in row to the climate step on which the reference's
//     gEvent pointer walk (events.c:471-481) would fire it
//   * size the mean-NPP ring from the site's step lengths
//   * build the block -> (site, member range) table
//   * own all device memory, the stream and the timing events
// There is no CPU compute path: without a CUDA device init() fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "sip_handle.h"
#include "sip_libm.cuh"
#include "sip_types.cuh"

namespace sip {
namespace k1 {
// mode: 0 = exact (validation), 1 = fast (optimistic), 2 = replay of flagged members
cudaError_t launch_run(const RunArgs &a, int nblocks, int blockThreads, bool debug, int mode, cudaStream_t stream);
cudaError_t launch_derive(double *params, int64_t ld, int64_t nmembers, uint32_t *status, cudaStream_t stream);
cudaError_t launch_consts(StepConsts *out, cudaStream_t stream);
cudaError_t launch_init_state(const double *params, int64_t ld, int64_t nmembers, const int32_t *memberSite,
                              const SiteDev *sites, uint32_t flags, double *state, double *ringV, double *ringW,
                              uint32_t *status, double *loglik, double *loglikN, int32_t *recCount,
                              cudaStream_t stream);
}  // namespace k1
cudaError_t launch_row_summary(const double *cols, int64_t ld, int64_t nsteps, const SiteDev *sites, int64_t nsites,
                               int64_t maxMembers, const double *probs, int nq, double *mean, double *var,
                               int64_t momStride, double *quant, int64_t qStride, cudaStream_t stream);
cudaError_t measure_fp64_peak(int device, double *tflops);
cudaError_t eval_libm(int device, int op, const double *x, const double *y, double *out, int64_t n);
}  // namespace sip

using namespace sip;

static thread_local std::string g_err;
int sip::fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CUDA_OK(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(SIPNET_GPU_ERR_NO_DEVICE, "%s failed: %s", #expr, cudaGetErrorString(e__));      \
  } while (0)

static uint32_t flag_mask(const sipnet_gpu_flags &f) {
  uint32_t m = 0;
  if (f.events) m |= F_EVENTS;
  if (f.gdd) m |= F_GDD;
  if (f.growthResp) m |= F_GROWTH_RESP;
  if (f.leafWater) m |= F_LEAF_WATER;
  if (f.litterPool) m |= F_LITTER_POOL;
  if (f.snow) m |= F_SNOW;
  if (f.soilPhenol) m |= F_SOIL_PHENOL;
  if (f.waterHResp) m |= F_WATER_HRESP;
  if (f.nitrogenCycle) m |= F_NITROGEN;
  if (f.anaerobic) m |= F_ANAEROBIC;
  if (f.flooding) m |= F_FLOODING;
  if (f.carbonSaturation) m |= F_CSAT;
  return m;
}

template <class T>
static cudaError_t dalloc(T **p, size_t count) {
  return cudaMalloc((void **)p, std::max<size_t>(count, 1) * sizeof(T));
}

// Build one site's ClimRec stream with events bound to steps, into recs[0 .. nsteps) and evs[0 .. nevents).
// Returns 0 or a reference exit code with its message in `err` (called from worker threads: no global state).
static int site_fail(std::string &err, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  err = buf;
  return code;
}

static int64_t site_event_count(const sipnet_gpu_site &s, bool eventsOn) {
  return (eventsOn && s.events != nullptr) ? s.nevents : 0;  // initEvents(), events.c:427-433
}

static int build_site(const sipnet_gpu_site &s, bool eventsOn, ClimRec *recs, EventDev *evs, double &minLen,
                      int64_t siteIndex, std::string &err) {
  if (s.nsteps <= 0) return site_fail(err, SIPNET_GPU_ERR_INPUT_FILE, "site %lld: no climate data", (long long)siteIndex);
  const void *need[] = {s.year, s.day, s.time, s.length, s.tair, s.tsoil, s.par, s.precip,
                        s.vpd,  s.vpdSoil, s.vPress, s.wspd, s.gdd};
  for (const void *p : need)
    if (p == nullptr) return site_fail(err, SIPNET_GPU_ERR_BAD_ARGUMENT, "site %lld: NULL climate array", (long long)siteIndex);
  const int64_t nev = site_event_count(s, eventsOn);
  if (nev > 0) {  // frontend.c:217-222 / isFirstEventBefore(), events.c:437-447
    const sipnet_gpu_event &e0 = s.events[0];
    const bool before = (e0.year != s.year[0]) ? (e0.year < s.year[0]) : (e0.day < s.day[0]);
    if (before)
      return site_fail(err, SIPNET_GPU_ERR_INPUT_FILE, "site %lld: first event occurs before the start of the climate file",
                       (long long)siteIndex);
  }
  int64_t e = 0;
  double prevLen = -1.0, prevDecay = 0.0, prevInv = 0.0;  // step lengths repeat: their functions are reused
  for (int64_t t = 0; t < s.nsteps; ++t) {
    ClimRec &c = recs[(size_t)t];
    c.length = s.length[t];
    c.tair = s.tair[t];
    c.tsoil = s.tsoil[t];
    c.par = s.par[t];
    c.precip = s.precip[t];
    c.vpd = s.vpd[t];
    c.vpdSoil = s.vpdSoil[t];
    c.vPress = s.vPress[t];
    c.wspd = s.wspd[t];
    c.gdd = s.gdd[t];
    c.year = s.year[t];
    c.day = s.day[t];
    c.dayFrac = (double)c.day + s.time[t] / 24.0;
    if (!(c.length > 0))  // events.c:460-465
      return site_fail(err, SIPNET_GPU_ERR_BAD_PARAMETER_VALUE,
                       "site %lld: climate length (%f) on year %d day %d is non-positive", (long long)siteIndex, c.length,
                       c.year, c.day);
    minLen = std::min(minLen, c.length);
    if (c.length != prevLen) {
      prevLen = c.length;
      prevDecay = std::exp(-c.length * (1 / 30.0));  // events.c:816, events.h:58
      int ex = 0;
      const double mant = std::frexp(c.length, &ex);  // power of two <=> mantissa 0.5: then x / length == x * (1 / length)
      prevInv = (mant == 0.5 && ex > -500 && ex < 500) ? 1.0 / c.length : 0.0;
    }
    c.tillDecay = prevDecay;
    c.invLenPow2 = prevInv;
    {
      const libm::LogHL l = libm::pow_log(c.vpd);  // host evaluation of the same operations
      c.logVpdHi = l.hi;
      c.logVpdLo = l.lo;
    }
    c.tair10 = c.tair / 10.0;
    c.tsoil10 = c.tsoil / 10.0;
    c.precipRate = c.precip / c.length;
    c.sublK = ((1.3 * 1005.) / 66. * (1. / 2835000.) * 1000. * 1000. * (1. / 10000) * 86400.0) * (0.6 - c.vPress);
    c.evapK = ((1.3 * 1005.) / 66. * (1. / 2501000.) * 1000. * 1000. * (1. / 10000) * 86400.0) * c.vpdSoil;
    c.evBegin = (int32_t)e;
    while (e < nev && s.events[e].year <= c.year && s.events[e].day <= c.day) {  // events.c:471
      const sipnet_gpu_event &ev = s.events[e];
      if (ev.year < c.year || ev.day < c.day)  // events.c:476-481
        return site_fail(err, SIPNET_GPU_ERR_INPUT_FILE,
                         "site %lld: agronomic event for year %d day %d has no corresponding climate record",
                         (long long)siteIndex, ev.year, ev.day);
      if (ev.type < SIPNET_EV_FERTILIZATION || ev.type > SIPNET_EV_PLANTDEATH)  // events.c:735-737
        return site_fail(err, SIPNET_GPU_ERR_UNKNOWN_EVENT, "site %lld: unknown event type %d", (long long)siteIndex, ev.type);
      if (ev.type == SIPNET_EV_IRRIGATION && ev.method != 0 && ev.method != 1)  // events.c:498-501
        return site_fail(err, SIPNET_GPU_ERR_UNKNOWN_EVENT, "site %lld: unknown irrigation method type: %d",
                         (long long)siteIndex, ev.method);
      EventDev &d = evs[(size_t)e];
      for (int k = 0; k < 4; ++k) d.p[k] = ev.p[k];
      d.type = ev.type;
      d.method = ev.method;
      d.pad0 = d.pad1 = 0;
      ++e;
    }
    c.evEnd = (int32_t)e;
  }
  // events past the last climate record never fire (the reference's pointer walk ends with the climate list);
  // their slots keep a harmless filler
  for (; e < nev; ++e) {
    EventDev &d = evs[(size_t)e];
    for (int k = 0; k < 4; ++k) d.p[k] = 0.0;
    d.type = SIPNET_EV_PLANTDEATH;
    d.method = d.pad0 = d.pad1 = 0;
  }
  return 0;
}

// All sites of a launch -> three device arenas (forcing records, events, observations), prepared by the host cores
// in parallel and uploaded batch by batch from two pinned staging buffers, so the upload of one batch overlaps
// the preparation of the next.  Sites are independent; the first failing site IN ORDER decides the error, as a
// sequential pass would.  (10 000 ten-year sites: 12.9 GB of records; ~4 s on one thread with one allocation per
// site before, a few hundred ms now.)
static int upload_sites(sipnet_gpu_handle *h, const sipnet_gpu_config *cfg, double &minLenOut) {
  const int64_t S = cfg->nsites;
  const bool eventsOn = cfg->flags.events != 0;
  const bool wantObs = (cfg->outputs & SIPNET_GPU_OUT_LOGLIK) != 0;
  std::vector<int64_t> recOff((size_t)S + 1, 0), evOff((size_t)S + 1, 0), obsOff((size_t)S + 1, 0);
  for (int64_t s = 0; s < S; ++s) {
    const sipnet_gpu_site &st = cfg->sites[s];
    if (st.nsteps <= 0) return fail(SIPNET_GPU_ERR_INPUT_FILE, "site %lld: no climate data", (long long)s);
    recOff[(size_t)s + 1] = recOff[(size_t)s] + st.nsteps;
    evOff[(size_t)s + 1] = evOff[(size_t)s] + site_event_count(st, eventsOn);
    obsOff[(size_t)s + 1] = obsOff[(size_t)s] + ((wantObs && st.nee_obs) ? st.nsteps : 0);
  }
  const bool trace = getenv("SIPNET_GPU_TRACE_INIT") != nullptr;  // phase times of the site upload on stderr
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double tTrace0 = now();
  double tBuild = 0.0;
  ClimRec *dRec = nullptr;
  EventDev *dEv = nullptr;
  double *dObs = nullptr;
  CUDA_OK(dalloc(&dRec, (size_t)recOff[(size_t)S]));
  h->siteAllocs.push_back(dRec);
  CUDA_OK(dalloc(&dEv, (size_t)evOff[(size_t)S]));
  h->siteAllocs.push_back(dEv);
  CUDA_OK(dalloc(&dObs, (size_t)obsOff[(size_t)S]));
  h->siteAllocs.push_back(dObs);

  // batches of whole sites, about kBatchBytes of records each
  const size_t kBatchBytes = (size_t)64 << 20;  // pinning the two staging buffers is part of init: keep them small
  std::vector<int64_t> batchBegin{0};
  {
    size_t acc = 0;
    for (int64_t s = 0; s < S; ++s) {
      const size_t b = (size_t)cfg->sites[s].nsteps * sizeof(ClimRec) +
                       (size_t)(evOff[(size_t)s + 1] - evOff[(size_t)s]) * sizeof(EventDev);
      if (acc > 0 && acc + b > kBatchBytes) {
        batchBegin.push_back(s);
        acc = 0;
      }
      acc += b;
    }
    batchBegin.push_back(S);
  }
  size_t stageBytes = 0;
  for (size_t b = 0; b + 1 < batchBegin.size(); ++b) {
    const int64_t s0 = batchBegin[b], s1 = batchBegin[b + 1];
    stageBytes = std::max(stageBytes, (size_t)(recOff[(size_t)s1] - recOff[(size_t)s0]) * sizeof(ClimRec) +
                                          (size_t)(evOff[(size_t)s1] - evOff[(size_t)s0]) * sizeof(EventDev));
  }
  unsigned char *stage[2] = {nullptr, nullptr};
  cudaEvent_t copied[2] = {nullptr, nullptr};
  const int nbuf = batchBegin.size() > 2 ? 2 : 1;
  int rc = 0;
  std::vector<int> siteRc((size_t)S, 0);
  std::vector<std::string> siteErr((size_t)S);
  std::vector<double> siteMin((size_t)S, 1e300);
  unsigned nthreads = std::thread::hardware_concurrency();
  if (const char *e = getenv("SIPNET_GPU_INIT_THREADS")) nthreads = (unsigned)std::max(1, atoi(e));
  nthreads = std::max(1u, std::min(nthreads, 64u));
  for (int i = 0; i < nbuf && rc == 0; ++i) {
    if (cudaHostAlloc((void **)&stage[i], std::max<size_t>(stageBytes, 16), cudaHostAllocDefault) != cudaSuccess ||
        cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming) != cudaSuccess)
      rc = fail(SIPNET_GPU_ERR_NO_DEVICE, "pinned staging allocation of %zu bytes failed", stageBytes);
  }
  const double tPinned = now();
  for (size_t b = 0; rc == 0 && b + 1 < batchBegin.size(); ++b) {
    const int64_t s0 = batchBegin[b], s1 = batchBegin[b + 1];
    const int buf = (int)(b % (size_t)nbuf);
    if (b >= (size_t)nbuf && cudaEventSynchronize(copied[buf]) != cudaSuccess) {  // this buffer's previous upload is done
      rc = fail(SIPNET_GPU_ERR_NO_DEVICE, "site upload failed");
      break;
    }
    ClimRec *recs = reinterpret_cast<ClimRec *>(stage[buf]);
    const size_t nrec = (size_t)(recOff[(size_t)s1] - recOff[(size_t)s0]);
    EventDev *evs = reinterpret_cast<EventDev *>(stage[buf] + nrec * sizeof(ClimRec));
    const size_t nev = (size_t)(evOff[(size_t)s1] - evOff[(size_t)s0]);
    std::atomic<int64_t> next{s0};
    auto work = [&]() {
      for (;;) {
        const int64_t s = next.fetch_add(1);
        if (s >= s1) break;
        siteRc[(size_t)s] = build_site(cfg->sites[s], eventsOn, recs + (recOff[(size_t)s] - recOff[(size_t)s0]),
                                       evs + (evOff[(size_t)s] - evOff[(size_t)s0]), siteMin[(size_t)s], s, siteErr[(size_t)s]);
      }
    };
    const unsigned nt = (unsigned)std::min<int64_t>(nthreads, s1 - s0);
    std::vector<std::thread> pool;
    const double tb0 = now();
    for (unsigned i = 1; i < nt; ++i) pool.emplace_back(work);
    work();
    for (std::thread &t : pool) t.join();
    tBuild += now() - tb0;
    for (int64_t s = s0; s < s1 && rc == 0; ++s)
      if (siteRc[(size_t)s]) rc = fail(siteRc[(size_t)s], "%s", siteErr[(size_t)s].c_str());
    if (rc) break;
    cudaError_t e = cudaMemcpyAsync(dRec + recOff[(size_t)s0], recs, nrec * sizeof(ClimRec), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess && nev > 0)
      e = cudaMemcpyAsync(dEv + evOff[(size_t)s0], evs, nev * sizeof(EventDev), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaEventRecord(copied[buf], h->stream);
    if (e != cudaSuccess) rc = fail(SIPNET_GPU_ERR_NO_DEVICE, "site upload failed: %s", cudaGetErrorString(e));
  }
  if (rc == 0 && cudaStreamSynchronize(h->stream) != cudaSuccess) rc = fail(SIPNET_GPU_ERR_NO_DEVICE, "site upload failed");
  const double tDone = now();
  for (int i = 0; i < 2; ++i) {
    if (copied[i]) cudaEventDestroy(copied[i]);
    if (stage[i]) cudaFreeHost(stage[i]);
  }
  if (trace)
    fprintf(stderr, "[sipnet_gpu] sites: %lld, records %.2f GB, %u threads, %zu batches: alloc+pin %.3f s, build %.3f s, "
                    "build+upload %.3f s, unpin %.3f s\n",
            (long long)S, (double)recOff[(size_t)S] * sizeof(ClimRec) / 1e9, nthreads, batchBegin.size() - 1, tPinned - tTrace0,
            tBuild, tDone - tPinned, now() - tDone);
  if (rc) return rc;
  // observations go up straight from the caller's arrays
  int64_t firstLen = cfg->sites[0].nsteps;
  minLenOut = 1e300;
  for (int64_t s = 0; s < S; ++s) {
    const sipnet_gpu_site &st = cfg->sites[s];
    SiteDev &sd = h->hostSites[(size_t)s];
    sd.nsteps = st.nsteps;
    sd.member0 = 0;
    sd.memberCount = 0;
    sd.clim = dRec + recOff[(size_t)s];
    sd.events = dEv + evOff[(size_t)s];
    sd.neeObs = nullptr;
    if (wantObs && st.nee_obs) {
      CUDA_OK(cudaMemcpyAsync(dObs + obsOff[(size_t)s], st.nee_obs, (size_t)st.nsteps * sizeof(double), cudaMemcpyHostToDevice,
                              h->stream));
      sd.neeObs = dObs + obsOff[(size_t)s];
      h->anyObs = true;
    }
    h->maxSteps = std::max(h->maxSteps, sd.nsteps);
    if (sd.nsteps != firstLen) h->sitesDiffer = true;
    minLenOut = std::min(minLenOut, siteMin[(size_t)s]);
  }
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return 0;
}

static void free_handle(sipnet_gpu_handle *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  void *ptrs[] = {h->params, h->state, h->ringV, h->ringW, h->status, h->memberSite, h->blocks, h->sites, h->out,
                  h->dbg,    h->counters, h->loglik, h->loglikN, h->recs, h->recCount, h->mean, h->var, h->quant,
                  h->stateBk, h->ringVBk, h->ringWBk, h->loglikBk, h->loglikNBk, h->statusBk,
                  h->recCountBk, h->sched, h->chunk, h->siteChunks, h->asPart, h->asMom, h->asCoef,
                  h->asObs, h->asDiag, h->asInfl, h->rsW, h->rsC, h->rsSite, h->rsPart, h->rsLogw, h->rsLmax, h->rsSend, h->rsRecv,
                  h->rsAnc, h->rsTab, h->jtPart, h->jtMom, h->jtCoef, h->jtDiag, h->jtShrink, h->jtZ,
                  h->mhSnap, h->mhDlp, h->mhCurL, h->mhLogU, h->mhScale, h->mhTau, h->mhValid};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  for (void *p : h->siteAllocs)
    if (p) cudaFree(p);
  if (h->evStart) cudaEventDestroy(h->evStart);
  if (h->evStop) cudaEventDestroy(h->evStop);
  if (h->evT0) cudaEventDestroy(h->evT0);
  if (h->evT1) cudaEventDestroy(h->evT1);
  for (int i = 0; i < 2; ++i) {
    if (h->evRunDone[i]) cudaEventDestroy(h->evRunDone[i]);
    if (h->evCopyDone[i]) cudaEventDestroy(h->evCopyDone[i]);
  }
  if (h->copyStream) cudaStreamDestroy(h->copyStream);
  if (h->ownStream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

static int run_init_state(sipnet_gpu_handle *h) {
  // rings start zeroed so that never-written slots read the same after a reset as after init
  CUDA_OK(cudaMemsetAsync(h->ringV, 0, (size_t)h->ringCap * h->ld * sizeof(double), h->stream));
  CUDA_OK(cudaMemsetAsync(h->ringW, 0, (size_t)h->ringCap * h->ld * sizeof(double), h->stream));
  if (h->counters) CUDA_OK(cudaMemsetAsync(h->counters, 0, (size_t)SIPNET_GPU_NCOUNTERS * h->ld * sizeof(uint32_t), h->stream));
  cudaError_t e = k1::launch_init_state(h->params, h->ld, h->nmembers, h->memberSite, h->sites, h->flags, h->state,
                                        h->ringV, h->ringW, h->status, h->loglik, h->loglikN, h->recCount, h->stream);
  h->launches++;
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "init_state launch failed: %s", cudaGetErrorString(e));
  h->stepsDone = 0;
  h->lastBegin = h->lastEnd = 0;
  h->summariesValid = false;
  return 0;
}

static int derive_params(sipnet_gpu_handle *h);

extern "C" int sipnet_gpu_init(const sipnet_gpu_config *cfg, sipnet_gpu_handle **out) {
  if (out) *out = nullptr;
  if (!cfg || !out) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL config or handle pointer");
  if (cfg->abi_version != SIPNET_GPU_ABI_VERSION)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "ABI version mismatch: caller %d, library %d", cfg->abi_version,
                SIPNET_GPU_ABI_VERSION);
  if (cfg->nsites <= 0 || !cfg->sites) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no sites");
  if (cfg->nmembers <= 0 || !cfg->params) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no members / params");
  if (cfg->params_ld < cfg->nmembers) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "params_ld < nmembers");
  if (cfg->math != SIPNET_GPU_MATH_VALIDATION && cfg->math != SIPNET_GPU_MATH_FAST && cfg->math != SIPNET_GPU_MATH_THROUGHPUT)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "unknown math mode %d", cfg->math);
  if (cfg->block_threads != 0 && cfg->block_threads != 32 && cfg->block_threads != 128)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "block_threads must be 0, 32 or 128");
  if (cfg->ring_slots != 0 && (cfg->ring_slots < 2 || cfg->ring_slots > SIPNET_GPU_RING_SLOTS_REFERENCE))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "ring_slots must be 0 or in [2, %d]", SIPNET_GPU_RING_SLOTS_REFERENCE);
  if ((cfg->outputs & SIPNET_GPU_OUT_LOGLIK) && !(cfg->nee_sigma > 0))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "nee_sigma must be > 0");
  if ((cfg->outputs & (SIPNET_GPU_OUT_MOMENTS | SIPNET_GPU_OUT_QUANTILES)) &&
      (cfg->n_summary_cols <= 0 || !cfg->summary_cols))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "summary outputs need summary_cols");
  if ((cfg->outputs & SIPNET_GPU_OUT_QUANTILES) && (cfg->n_quantiles <= 0 || !cfg->quantiles))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "quantile output needs quantiles");
  for (int i = 0; i < cfg->n_summary_cols; ++i)
    if (cfg->summary_cols[i] < 0 || cfg->summary_cols[i] >= SIPNET_GPU_NOUT)
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "summary column %d out of range", cfg->summary_cols[i]);
  for (int i = 0; i < cfg->n_quantiles; ++i)
    if (!(cfg->quantiles[i] >= 0.0 && cfg->quantiles[i] <= 1.0))
      return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "quantile probability out of [0,1]");

  // member -> site map: non-decreasing
  std::vector<int32_t> memberSite((size_t)cfg->nmembers, 0);
  if (cfg->member_site) {
    for (int64_t m = 0; m < cfg->nmembers; ++m) {
      const int32_t s = cfg->member_site[m];
      if (s < 0 || s >= cfg->nsites) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "member_site[%lld] out of range", (long long)m);
      if (m > 0 && s < cfg->member_site[m - 1])
        return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "member_site must be non-decreasing");
      memberSite[(size_t)m] = s;
    }
  }

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(SIPNET_GPU_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(SIPNET_GPU_ERR_NO_DEVICE, "device %d not present", cfg->device);
  CUDA_OK(cudaSetDevice(cfg->device));

  sipnet_gpu_handle *h = new sipnet_gpu_handle();
  h->device = cfg->device;
  h->flags = flag_mask(cfg->flags);
  h->outputs = cfg->outputs;
  h->math = cfg->math;
  h->nmembers = cfg->nmembers;
  h->ld = (cfg->nmembers + 15) / 16 * 16;
  h->nsites = cfg->nsites;
  h->sigma = cfg->nee_sigma > 0 ? cfg->nee_sigma : 1.0;
  h->maxRecs = (cfg->outputs & SIPNET_GPU_OUT_EVENTS) ? std::max(cfg->max_event_records, 0) : 0;
  h->summaryCols.assign(cfg->summary_cols, cfg->summary_cols + std::max(cfg->n_summary_cols, 0));
  h->quantiles.assign(cfg->quantiles, cfg->quantiles + std::max(cfg->n_quantiles, 0));

#define INIT_CUDA(expr)                                                                                  \
  do {                                                                                                   \
    cudaError_t e__ = (expr);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      int rc__ = fail(SIPNET_GPU_ERR_NO_DEVICE, "%s failed: %s", #expr, cudaGetErrorString(e__));        \
      free_handle(h);                                                                                    \
      return rc__;                                                                                       \
    }                                                                                                    \
  } while (0)

  if (cfg->stream) {
    h->stream = (cudaStream_t)cfg->stream;
  } else {
    INIT_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->ownStream = true;
  }
  INIT_CUDA(cudaEventCreate(&h->evStart));
  INIT_CUDA(cudaEventCreate(&h->evStop));
  INIT_CUDA(cudaEventCreate(&h->evT0));
  INIT_CUDA(cudaEventCreate(&h->evT1));

  // ---- sites ----
  h->hostSites.resize((size_t)cfg->nsites);
  double minLen = 1e300;
  {
    const int rc = upload_sites(h, cfg, minLen);
    if (rc) {
      free_handle(h);
      return rc;
    }
  }
  // ring capacity: occupancy <= 1 partially evicted entry + floor(5/minLen) whole entries (+ slack), capped like
  // the reference (MEAN_NPP_MAX_ENTRIES, sipnet.c:40) so the overflow condition is the reference's.
  {
    double bound = std::floor(kMeanNppDays / minLen) + 3.0;
    h->ringCap = (int)std::min<double>(kRingMax, std::max(2.0, bound));
    // an explicit slot count is honoured as given: fewer slots than `bound` can overflow (status bit) where the
    // reference would not, the reference's own count reproduces its ring layout slot for slot
    if (cfg->ring_slots != 0) h->ringCap = cfg->ring_slots;
  }
  if ((uint64_t)h->ringCap * (uint64_t)h->ld >= (1ull << 32)) {  // the kernel forms ring offsets as 32-bit products
    free_handle(h);
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "%lld members x %d ring slots exceed the 2^32 ring entries one handle addresses",
                (long long)cfg->nmembers, h->ringCap);
  }

  // ---- members, blocks ----
  {
    int64_t m = 0;
    while (m < cfg->nmembers) {
      const int32_t s = memberSite[(size_t)m];
      int64_t m1 = m;
      while (m1 < cfg->nmembers && memberSite[(size_t)m1] == s) ++m1;
      h->hostSites[(size_t)s].member0 = (int32_t)m;
      h->hostSites[(size_t)s].memberCount = (int32_t)(m1 - m);
      m = m1;
    }
  }
  for (const SiteDev &sd : h->hostSites) h->maxSiteMembers = std::max<int64_t>(h->maxSiteMembers, sd.memberCount);
  auto count_blocks = [&](int bt) {
    int64_t n = 0;
    for (const SiteDev &sd : h->hostSites) n += (sd.memberCount + bt - 1) / bt;
    return n;
  };
  if (cfg->block_threads) {
    h->blockThreads = cfg->block_threads;
  } else {
    int smCount = 148;
    cudaDeviceGetAttribute(&smCount, cudaDevAttrMultiProcessorCount, cfg->device);
    h->blockThreads = 32;
    for (int bt : {128}) {  // largest block that still gives every SM >= 2 blocks
      if (count_blocks(bt) >= 2 * (int64_t)smCount) {
        h->blockThreads = bt;
        break;
      }
    }
  }
  std::vector<BlockDesc> blocks;
  {
    const int32_t B = h->blockThreads;
    const bool mix = B == 128 && getenv("SIPNET_GPU_NO_MIXED_BLOCKS") == nullptr;  // (A/B switch for measurements)
    std::vector<int64_t> live;  // sites that have members, in member order
    for (int64_t s = 0; s < cfg->nsites; ++s)
      if (h->hostSites[(size_t)s].memberCount > 0) live.push_back(s);
    int32_t taken = 0;  // members of the current site already placed in the previous (mixed) block
    for (size_t i = 0; i < live.size(); ++i) {
      const SiteDev &sd = h->hostSites[(size_t)live[i]];
      int32_t off = taken;
      taken = 0;
      for (; off < sd.memberCount; off += B) {
        BlockDesc bd{};
        bd.site = bd.site1 = (int32_t)live[i];
        bd.member0 = sd.member0 + off;
        bd.count = bd.count0 = std::min(B, sd.memberCount - off);
        if (mix && bd.count < B && i + 1 < live.size()) {  // the site's tail shares its block with the next site's head
          const SiteDev &nx = h->hostSites[(size_t)live[i + 1]];
          if (nx.member0 == bd.member0 + bd.count) {
            taken = std::min(B - bd.count, nx.memberCount);
            bd.site1 = (int32_t)live[i + 1];
            bd.count += taken;
            h->mixedBlocks = true;
          }
        }
        blocks.push_back(bd);
      }
    }
  }
  h->nblocks = (int)blocks.size();

  INIT_CUDA(dalloc(&h->sites, h->hostSites.size()));
  INIT_CUDA(cudaMemcpy(h->sites, h->hostSites.data(), h->hostSites.size() * sizeof(SiteDev), cudaMemcpyHostToDevice));
  INIT_CUDA(dalloc(&h->blocks, blocks.size()));
  INIT_CUDA(cudaMemcpy(h->blocks, blocks.data(), blocks.size() * sizeof(BlockDesc), cudaMemcpyHostToDevice));
  INIT_CUDA(dalloc(&h->memberSite, memberSite.size()));
  INIT_CUDA(cudaMemcpy(h->memberSite, memberSite.data(), memberSite.size() * sizeof(int32_t), cudaMemcpyHostToDevice));

  // ---- parameters: upload raw rows, derive in place ----
  INIT_CUDA(dalloc(&h->params, (size_t)kNParamDev * h->ld));
  INIT_CUDA(cudaMemsetAsync(h->params, 0, (size_t)kNParamDev * h->ld * sizeof(double), h->stream));
  INIT_CUDA(cudaMemcpy2DAsync(h->params, h->ld * sizeof(double), cfg->params, cfg->params_ld * sizeof(double),
                              cfg->nmembers * sizeof(double), SIPNET_GPU_NPARAMS, cudaMemcpyHostToDevice, h->stream));
  INIT_CUDA(dalloc(&h->status, (size_t)h->ld));
  INIT_CUDA(cudaMemsetAsync(h->status, 0, (size_t)h->ld * sizeof(uint32_t), h->stream));
  INIT_CUDA(dalloc(&h->state, (size_t)SIPNET_GPU_NSTATE * h->ld));
  INIT_CUDA(cudaMemsetAsync(h->state, 0, (size_t)SIPNET_GPU_NSTATE * h->ld * sizeof(double), h->stream));
  INIT_CUDA(dalloc(&h->ringV, (size_t)h->ringCap * h->ld));
  INIT_CUDA(dalloc(&h->ringW, (size_t)h->ringCap * h->ld));
  INIT_CUDA(cudaMemsetAsync(h->ringV, 0, (size_t)h->ringCap * h->ld * sizeof(double), h->stream));
  INIT_CUDA(cudaMemsetAsync(h->ringW, 0, (size_t)h->ringCap * h->ld * sizeof(double), h->stream));

  // ---- outputs ----
  h->outCap = cfg->out_steps_capacity > 0 ? std::min(cfg->out_steps_capacity, h->maxSteps) : h->maxSteps;
  for (int c = 0; c < SIPNET_GPU_NOUT; ++c) h->colSlot[c] = -1;
  if (cfg->outputs & SIPNET_GPU_OUT_FULL) {
    for (int c = 0; c < SIPNET_GPU_NOUT; ++c) h->colSlot[c] = (int8_t)c;
    h->ncols = SIPNET_GPU_NOUT;
  } else if (cfg->outputs & (SIPNET_GPU_OUT_MOMENTS | SIPNET_GPU_OUT_QUANTILES)) {
    for (int32_t c : h->summaryCols)
      if (h->colSlot[c] < 0) h->colSlot[c] = (int8_t)h->ncols++;
  }
  if (h->ncols > 0) INIT_CUDA(dalloc(&h->out, (size_t)h->ncols * h->outCap * h->ld));
  if (cfg->outputs & SIPNET_GPU_OUT_DEBUG) INIT_CUDA(dalloc(&h->dbg, (size_t)(SIPNET_GPU_NDEBUG + SIPNET_GPU_NBALANCE) * h->outCap * h->ld));
  if (cfg->outputs & SIPNET_GPU_OUT_DEBUG) INIT_CUDA(dalloc(&h->counters, (size_t)SIPNET_GPU_NCOUNTERS * h->ld));
  if (cfg->outputs & SIPNET_GPU_OUT_LOGLIK) {
    INIT_CUDA(dalloc(&h->loglik, (size_t)h->ld));
    INIT_CUDA(dalloc(&h->loglikN, (size_t)h->ld));
  }
  if (cfg->outputs & SIPNET_GPU_OUT_EVENTS) {
    INIT_CUDA(dalloc(&h->recCount, (size_t)h->ld));
    if (h->maxRecs > 0) INIT_CUDA(dalloc(&h->recs, (size_t)h->nmembers * h->maxRecs));
  }
  if (h->math != SIPNET_GPU_MATH_VALIDATION) {
    INIT_CUDA(dalloc(&h->stateBk, (size_t)SIPNET_GPU_NSTATE * h->ld));
    INIT_CUDA(dalloc(&h->ringVBk, (size_t)h->ringCap * h->ld));
    INIT_CUDA(dalloc(&h->ringWBk, (size_t)h->ringCap * h->ld));
    INIT_CUDA(dalloc(&h->statusBk, (size_t)h->ld));
    if (h->loglik) {
      INIT_CUDA(dalloc(&h->loglikBk, (size_t)h->ld));
      INIT_CUDA(dalloc(&h->loglikNBk, (size_t)h->ld));
    }
    if (h->recCount) INIT_CUDA(dalloc(&h->recCountBk, (size_t)h->ld));
  }
  const size_t nsum = (size_t)h->nsites * h->summaryCols.size() * h->outCap;
  if (cfg->outputs & SIPNET_GPU_OUT_MOMENTS) {
    INIT_CUDA(dalloc(&h->mean, nsum));
    INIT_CUDA(dalloc(&h->var, nsum));
  }
  if (cfg->outputs & SIPNET_GPU_OUT_QUANTILES) {
    INIT_CUDA(dalloc(&h->quant, nsum * h->quantiles.size()));
  }

  {  // dynamic scheduling words: counter + one progress word per block descriptor
    void *p = nullptr;
    INIT_CUDA(cudaMalloc(&p, 16 + (size_t)h->nblocks * sizeof(unsigned int)));
    h->sched = (unsigned char *)p;
    const char *env = getenv("SIPNET_GPU_STATIC_SCHED");  // A/B switch for measurements: one CTA per block, whole range
    h->staticSched = env && env[0] == '1';
  }

  {  // launch-lifetime constants, evaluated by the device
    StepConsts *dkc = nullptr;
    INIT_CUDA(dalloc(&dkc, 1));
    cudaError_t e = k1::launch_consts(dkc, h->stream);
    h->launches++;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h->kc, dkc, sizeof h->kc, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(dkc);
    INIT_CUDA(e);
  }

  // ---- setupModel() on the device ----
  {
    int rc = derive_params(h);
    if (rc) {
      free_handle(h);
      return rc;
    }
  }
  {
    int rc = run_init_state(h);
    if (rc) {
      free_handle(h);
      return rc;
    }
  }
  INIT_CUDA(cudaStreamSynchronize(h->stream));
#undef INIT_CUDA
  *out = h;
  return SIPNET_GPU_OK;
}

static int derive_params(sipnet_gpu_handle *h) {
  cudaError_t e = k1::launch_derive(h->params, h->ld, h->nmembers, h->status, h->stream);
  h->launches++;
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "derive launch failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int sipnet_gpu_set_params(sipnet_gpu_handle *h, const double *params, int64_t params_ld) {
  if (!h || !params) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or params");
  if (params_ld < h->nmembers) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "params_ld < nmembers");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaMemcpy2DAsync(h->params, h->ld * sizeof(double), params, params_ld * sizeof(double),
                            h->nmembers * sizeof(double), SIPNET_GPU_NPARAMS, cudaMemcpyHostToDevice, h->stream));
  int rc = derive_params(h);
  if (rc) return rc;
  return run_init_state(h);
}

extern "C" int sipnet_gpu_timer_start(sipnet_gpu_handle *h) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaEventRecord(h->evT0, h->stream));
  return 0;
}

extern "C" int sipnet_gpu_timer_stop_ms(sipnet_gpu_handle *h, float *ms) {
  if (!h || !ms) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL argument");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaEventRecord(h->evT1, h->stream));
  CUDA_OK(cudaEventSynchronize(h->evT1));
  CUDA_OK(cudaEventElapsedTime(ms, h->evT0, h->evT1));
  return 0;
}

extern "C" int sipnet_gpu_reset(sipnet_gpu_handle *h) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  CUDA_OK(cudaSetDevice(h->device));
  return run_init_state(h);
}

extern "C" int32_t sipnet_gpu_ring_slots(const sipnet_gpu_handle *h) { return h ? h->ringCap : 0; }

extern "C" int sipnet_gpu_set_state(sipnet_gpu_handle *h, const double *state, int64_t state_ld, const double *ring_values,
                                    const double *ring_weights, int64_t ring_ld, int64_t next_step) {
  if (!h || !state) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or state");
  if (state_ld < h->nmembers) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "state_ld < nmembers");
  if ((ring_values == nullptr) != (ring_weights == nullptr))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "ring values and weights go together");
  if (ring_values && ring_ld < h->nmembers) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "ring_ld < nmembers");
  if (next_step < 0 || next_step > h->maxSteps) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "next_step out of range");
  // ring cursors index the device ring: reject what restartLoadCheckpoint() rejects (restart.c:976-981)
  for (int64_t m = 0; m < h->nmembers; ++m) {
    const double a = state[(size_t)SIPNET_S_meanStart * (size_t)state_ld + (size_t)m];
    const double b = state[(size_t)SIPNET_S_meanLast * (size_t)state_ld + (size_t)m];
    if (!(a >= 0 && a < h->ringCap && b >= 0 && b < h->ringCap))
      return fail(SIPNET_GPU_ERR_BAD_RESTART, "mean-tracker cursor out of range for member %lld", (long long)m);
  }
  CUDA_OK(cudaSetDevice(h->device));
  const size_t w = (size_t)h->nmembers * sizeof(double);
  CUDA_OK(cudaMemcpy2DAsync(h->state, (size_t)h->ld * sizeof(double), state, (size_t)state_ld * sizeof(double), w,
                            SIPNET_GPU_NSTATE, cudaMemcpyHostToDevice, h->stream));
  if (ring_values) {
    CUDA_OK(cudaMemcpy2DAsync(h->ringV, (size_t)h->ld * sizeof(double), ring_values, (size_t)ring_ld * sizeof(double), w,
                              (size_t)h->ringCap, cudaMemcpyHostToDevice, h->stream));
    CUDA_OK(cudaMemcpy2DAsync(h->ringW, (size_t)h->ld * sizeof(double), ring_weights, (size_t)ring_ld * sizeof(double), w,
                              (size_t)h->ringCap, cudaMemcpyHostToDevice, h->stream));
  }
  CUDA_OK(cudaStreamSynchronize(h->stream));
  h->stepsDone = next_step;
  h->lastBegin = h->lastEnd = next_step;
  h->summariesValid = false;
  return 0;
}

// one contiguous segment; `outbuf` = where the column outputs of this segment go (h->out or one of its halves)
static int run_segment(sipnet_gpu_handle *h, int64_t step_begin, int64_t step_end, double *outbuf, int64_t outCapSteps) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  if (step_begin != h->stepsDone)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "step_begin %lld is not the next step (%lld): segments must be contiguous",
                (long long)step_begin, (long long)h->stepsDone);
  if (step_end < step_begin || step_end > h->maxSteps)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "bad step range [%lld, %lld) for %lld steps", (long long)step_begin,
                (long long)step_end, (long long)h->maxSteps);
  const bool keeps = (h->out != nullptr) || (h->dbg != nullptr);
  if (keeps && step_end - step_begin > outCapSteps)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "run range of %lld steps exceeds out_steps_capacity %lld",
                (long long)(step_end - step_begin), (long long)outCapSteps);
  CUDA_OK(cudaSetDevice(h->device));
  h->lastBegin = step_begin;
  h->lastEnd = step_end;
  h->summariesValid = false;
  if (step_end == step_begin) return SIPNET_GPU_OK;

  RunArgs a;
  memset(&a, 0, sizeof a);
  a.ld = h->ld;
  a.nmembers = h->nmembers;
  a.params = h->params;
  a.state = h->state;
  a.ringV = h->ringV;
  a.ringW = h->ringW;
  a.status = h->status;
  a.counters = h->counters;
  a.blocks = h->blocks;
  a.sites = h->sites;
  a.stepBegin = step_begin;
  a.stepEnd = step_end;
  a.out = outbuf;
  a.outSteps = step_end - step_begin;
  a.dbg = h->dbg;
  a.loglik = h->loglik;
  a.loglikN = h->loglikN;
  a.recs = h->recs;
  a.recCount = h->recCount;
  a.maxRecs = h->maxRecs;
  a.ringCap = h->ringCap;
  a.flags = h->flags;
  a.kc = h->kc;
  a.mixedBlocks = h->mixedBlocks ? 1 : 0;
  a.invSigma = 1.0 / h->sigma;
  a.logNorm = -std::log(h->sigma) - 0.5 * std::log(2.0 * M_PI);
  memcpy(a.colSlot, h->colSlot, sizeof a.colSlot);
  for (int c = 0; c < SIPNET_GPU_NOUT; ++c)
    if (h->colSlot[c] >= 0) {
      a.slotCol[h->colSlot[c]] = (int8_t)c;
      a.nOutCols = std::max<int32_t>(a.nOutCols, h->colSlot[c] + 1);
    }
  a.neeOff = a.gppOff = -1;
  a.nSlowCols = 0;
  for (int c = 0; c < SIPNET_GPU_NOUT; ++c) {
    if (h->colSlot[c] < 0) continue;
    const int64_t off = (int64_t)h->colSlot[c] * a.outSteps * h->ld * (int64_t)sizeof(double);
    if (c == SIPNET_O_nee) {
      a.neeOff = off;
    } else if (c == SIPNET_O_gpp) {
      a.gppOff = off;
    } else {
      a.slowCol[a.nSlowCols] = (int8_t)c;
      a.slowOff[a.nSlowCols++] = off;
    }
  a.onlyNeeGpp = (a.out != nullptr && a.neeOff >= 0 && a.gppOff >= 0 && a.nSlowCols == 0) ? 1 : 0;
  }

  if (h->sitesDiffer) {  // steps past a shorter site's end are never written: make them NaN
    if (outbuf) CUDA_OK(cudaMemsetAsync(outbuf, 0xFF, (size_t)h->ncols * a.outSteps * h->ld * sizeof(double), h->stream));
    if (h->dbg)
      CUDA_OK(cudaMemsetAsync(h->dbg, 0xFF, (size_t)(SIPNET_GPU_NDEBUG + SIPNET_GPU_NBALANCE) * a.outSteps * h->ld * sizeof(double),
                              h->stream));
  }
  const bool debug = h->dbg != nullptr;
  const bool optimistic = (h->math != SIPNET_GPU_MATH_VALIDATION) && !debug;
  if (optimistic) {  // keep the segment's start state so flagged members can be replayed exactly
    const size_t ldB = (size_t)h->ld * sizeof(double);
    CUDA_OK(cudaMemcpyAsync(h->stateBk, h->state, SIPNET_GPU_NSTATE * ldB, cudaMemcpyDeviceToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->ringVBk, h->ringV, h->ringCap * ldB, cudaMemcpyDeviceToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->ringWBk, h->ringW, h->ringCap * ldB, cudaMemcpyDeviceToDevice, h->stream));
    CUDA_OK(cudaMemcpyAsync(h->statusBk, h->status, (size_t)h->ld * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
    if (h->loglik) {
      CUDA_OK(cudaMemcpyAsync(h->loglikBk, h->loglik, ldB, cudaMemcpyDeviceToDevice, h->stream));
      CUDA_OK(cudaMemcpyAsync(h->loglikNBk, h->loglikN, ldB, cudaMemcpyDeviceToDevice, h->stream));
    }
    if (h->recCount)
      CUDA_OK(cudaMemcpyAsync(h->recCountBk, h->recCount, (size_t)h->ld * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
    a.stateBackup = h->stateBk;
    a.ringVBackup = h->ringVBk;
    a.ringWBackup = h->ringWBk;
    a.statusBackup = h->statusBk;
    a.loglikBackup = h->loglikBk;
    a.loglikNBackup = h->loglikNBk;
    a.recCountBackup = h->recCountBk;
  }
  if (!h->staticSched) {
    CUDA_OK(cudaMemsetAsync(h->sched, 0, 16 + (size_t)h->nblocks * sizeof(unsigned int), h->stream));
    a.workCounter = reinterpret_cast<unsigned long long *>(h->sched);
    a.progress = reinterpret_cast<unsigned int *>(h->sched + 16);
  }
  CUDA_OK(cudaEventRecord(h->evStart, h->stream));
  const int mode = !optimistic ? 0 : (h->math == SIPNET_GPU_MATH_THROUGHPUT ? 3 : 1);
  cudaError_t e = k1::launch_run(a, h->nblocks, h->blockThreads, debug, mode, h->stream);
  h->launches++;
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "run launch failed: %s", cudaGetErrorString(e));
  CUDA_OK(cudaEventRecord(h->evStop, h->stream));
  if (optimistic) {  // members outside the optimistic guards (normally none) are re-run by the general kernel
    e = k1::launch_run(a, h->nblocks, h->blockThreads, false, 2, h->stream);
    h->launches++;
    if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "replay launch failed: %s", cudaGetErrorString(e));
  }
  h->stepsDone = step_end;
  return SIPNET_GPU_OK;
}

extern "C" int sipnet_gpu_run(sipnet_gpu_handle *h, int64_t step_begin, int64_t step_end) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  return run_segment(h, step_begin, step_end, h->out, h->outCap);
}

extern "C" int sipnet_gpu_run_to_host(sipnet_gpu_handle *h, int64_t step_begin, int64_t step_end, double *dst,
                                      size_t bytes, int64_t chunk_steps) {
  if (!h || !dst) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or destination");
  if (!(h->outputs & SIPNET_GPU_OUT_FULL)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "run_to_host needs SIPNET_GPU_OUT_FULL");
  if (h->dbg) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "run_to_host is not available with the debug dump");
  const int64_t total = step_end - step_begin;
  if (total <= 0) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "empty step range");
  const size_t M = (size_t)h->nmembers;
  if (bytes != (size_t)SIPNET_GPU_NOUT * (size_t)total * M * sizeof(double))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "run_to_host: buffer is %zu bytes, expected %zu", bytes,
                (size_t)SIPNET_GPU_NOUT * (size_t)total * M * sizeof(double));
  const int64_t half = h->outCap / 2;
  if (half < 1) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "out_steps_capacity must be at least 2 for run_to_host");
  int64_t tc = chunk_steps > 0 ? chunk_steps : 512;
  if (tc > half) tc = half;
  CUDA_OK(cudaSetDevice(h->device));
  if (!h->copyStream) {
    CUDA_OK(cudaStreamCreateWithFlags(&h->copyStream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CUDA_OK(cudaEventCreateWithFlags(&h->evRunDone[i], cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&h->evCopyDone[i], cudaEventDisableTiming));
    }
  }
  double *bufs[2] = {h->out, h->out + (size_t)h->ncols * (size_t)half * (size_t)h->ld};
  int64_t k = 0;
  for (int64_t t0 = step_begin; t0 < step_end; t0 += tc, ++k) {
    const int64_t t1 = t0 + tc < step_end ? t0 + tc : step_end;
    const int64_t n = t1 - t0;
    const int b = (int)(k & 1);
    if (k >= 2) CUDA_OK(cudaStreamWaitEvent(h->stream, h->evCopyDone[b], 0));  // this half has been drained
    int rc = run_segment(h, t0, t1, bufs[b], half);
    if (rc) return rc;
    CUDA_OK(cudaEventRecord(h->evRunDone[b], h->stream));
    CUDA_OK(cudaStreamWaitEvent(h->copyStream, h->evRunDone[b], 0));
    {  // all 32 columns of the segment in ONE 3-D copy: device [col][n][ld] -> host [col][total][M] at step t0
      cudaMemcpy3DParms p3;
      memset(&p3, 0, sizeof p3);
      p3.srcPtr = make_cudaPitchedPtr(bufs[b], (size_t)h->ld * sizeof(double), M * sizeof(double), (size_t)n);
      p3.dstPtr = make_cudaPitchedPtr(dst, M * sizeof(double), M * sizeof(double), (size_t)total);
      p3.dstPos = make_cudaPos(0, (size_t)(t0 - step_begin), 0);
      p3.extent = make_cudaExtent(M * sizeof(double), (size_t)n, SIPNET_GPU_NOUT);
      p3.kind = cudaMemcpyDeviceToHost;
      CUDA_OK(cudaMemcpy3DAsync(&p3, h->copyStream));
    }
    CUDA_OK(cudaEventRecord(h->evCopyDone[b], h->copyStream));
  }
  // join: later work on the handle's stream (and the stopwatch) sees the copies as done
  CUDA_OK(cudaStreamWaitEvent(h->stream, h->evCopyDone[(k - 1) & 1], 0));
  if (k >= 2) CUDA_OK(cudaStreamWaitEvent(h->stream, h->evCopyDone[k & 1], 0));
  CUDA_OK(cudaStreamSynchronize(h->copyStream));
  h->lastBegin = step_end;  // the device buffer no longer holds one contiguous range: gather(FULL) is not valid
  h->lastEnd = step_end;
  return SIPNET_GPU_OK;
}

int sip::ensure_summaries(sipnet_gpu_handle *h) {
  if (h->summariesValid) return 0;
  const int64_t n = h->lastEnd - h->lastBegin;
  if (n <= 0) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "no run range to summarise");
  // summary columns occupy `out` slots; with OUT_FULL the slot of column c is c itself.
  // Device layout = the ABI's: mean/var [site][col][n], quantiles [site][col][q][n].
  const int ns = (int)h->summaryCols.size();
  const int64_t nq = (int64_t)h->quantiles.size();
  for (int i = 0; i < ns; ++i) {
    const int slot = h->colSlot[h->summaryCols[(size_t)i]];
    const double *cols = h->out + (size_t)slot * n * h->ld;
    cudaError_t e = launch_row_summary(cols, h->ld, n, h->sites, h->nsites, h->maxSiteMembers, h->quantiles.data(),
                                       h->quant ? (int)nq : 0, h->mean ? h->mean + (size_t)i * n : nullptr,
                                       h->var ? h->var + (size_t)i * n : nullptr, (int64_t)ns * n,
                                       h->quant ? h->quant + (size_t)i * nq * n : nullptr, (int64_t)ns * nq * n, h->stream);
    h->launches++;
    if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "summary launch failed: %s", cudaGetErrorString(e));
  }
  h->summariesValid = true;
  return 0;
}

int sip::ensure_chunks(sipnet_gpu_handle *h) {
  if (h->chunk) return 0;
  const size_t S = (size_t)h->nsites;
  std::vector<int2> chunk, siteChunks(S);
  for (size_t s = 0; s < S; ++s) {
    const int32_t cnt = h->hostSites[s].memberCount;
    siteChunks[s] = make_int2((int)chunk.size(), (cnt + kChunk - 1) / kChunk);
    for (int32_t i = 0; i < cnt; i += kChunk) chunk.push_back(make_int2((int)s, i));
  }
  cudaError_t e = cudaMalloc((void **)&h->chunk, std::max<size_t>(chunk.size(), 1) * sizeof(int2));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->siteChunks, S * sizeof(int2));
  if (e == cudaSuccess && !chunk.empty())
    e = cudaMemcpy(h->chunk, chunk.data(), chunk.size() * sizeof(int2), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->siteChunks, siteChunks.data(), S * sizeof(int2), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "chunk tables: %s", cudaGetErrorString(e));
  h->nchunks = (int64_t)chunk.size();
  return 0;
}

extern "C" size_t sipnet_gpu_gather_bytes(const sipnet_gpu_handle *h, int what) {
  if (!h) return 0;
  const size_t n = (size_t)(h->lastEnd - h->lastBegin);
  const size_t M = (size_t)h->nmembers;
  const size_t ns = h->summaryCols.size();
  switch (what) {
    case SIPNET_GPU_GATHER_FULL: return (h->outputs & SIPNET_GPU_OUT_FULL) ? SIPNET_GPU_NOUT * n * M * 8 : 0;
    case SIPNET_GPU_GATHER_DEBUG: return h->dbg ? (size_t)SIPNET_GPU_NDEBUG * n * M * 8 : 0;
    case SIPNET_GPU_GATHER_BALANCE: return h->dbg ? (size_t)SIPNET_GPU_NBALANCE * n * M * 8 : 0;
    case SIPNET_GPU_GATHER_LOGLIK:
    case SIPNET_GPU_GATHER_LOGLIK_N: return h->loglik ? M * 8 : 0;
    case SIPNET_GPU_GATHER_STATUS: return M * 4;
    case SIPNET_GPU_GATHER_COUNTERS: return h->counters ? (size_t)SIPNET_GPU_NCOUNTERS * M * 4 : 0;
    case SIPNET_GPU_GATHER_STATE: return (size_t)SIPNET_GPU_NSTATE * M * 8;
    case SIPNET_GPU_GATHER_RING_VALUES:
    case SIPNET_GPU_GATHER_RING_WEIGHTS: return (size_t)h->ringCap * M * 8;
    case SIPNET_GPU_GATHER_MEAN:
    case SIPNET_GPU_GATHER_VARIANCE: return h->mean ? (size_t)h->nsites * ns * n * 8 : 0;
    case SIPNET_GPU_GATHER_QUANTILES: return h->quant ? (size_t)h->nsites * ns * h->quantiles.size() * n * 8 : 0;
    case SIPNET_GPU_GATHER_EVENT_COUNTS: return h->recCount ? M * 4 : 0;
    case SIPNET_GPU_GATHER_EVENT_RECORDS: return h->recs ? M * (size_t)h->maxRecs * sizeof(sipnet_gpu_event_record) : 0;
    case SIPNET_GPU_GATHER_PARAMS: return (size_t)SIPNET_GPU_NPARAMS * M * 8;
    default: return 0;
  }
}

// rows x nmembers doubles out of a [rows][ld] device array
static int copy_rows(sipnet_gpu_handle *h, void *dst, const void *src, size_t rows, size_t elem) {
  CUDA_OK(cudaMemcpy2DAsync(dst, (size_t)h->nmembers * elem, src, (size_t)h->ld * elem, (size_t)h->nmembers * elem, rows,
                            cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return 0;
}

extern "C" int sipnet_gpu_gather(sipnet_gpu_handle *h, int what, void *dst, size_t bytes) {
  if (!h || !dst) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle or destination");
  const size_t need = sipnet_gpu_gather_bytes(h, what);
  if (need == 0) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "gather(%d): output was not requested at init or nothing has run", what);
  if (bytes != need)
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "gather(%d): buffer is %zu bytes, expected %zu", what, bytes, need);
  CUDA_OK(cudaSetDevice(h->device));
  const size_t n = (size_t)(h->lastEnd - h->lastBegin);
  switch (what) {
    case SIPNET_GPU_GATHER_FULL: return copy_rows(h, dst, h->out, SIPNET_GPU_NOUT * n, 8);
    case SIPNET_GPU_GATHER_DEBUG: return copy_rows(h, dst, h->dbg, (size_t)SIPNET_GPU_NDEBUG * n, 8);
    case SIPNET_GPU_GATHER_BALANCE:
      return copy_rows(h, dst, h->dbg + (size_t)SIPNET_GPU_NDEBUG * n * (size_t)h->ld, (size_t)SIPNET_GPU_NBALANCE * n, 8);
    case SIPNET_GPU_GATHER_LOGLIK: return copy_rows(h, dst, h->loglik, 1, 8);
    case SIPNET_GPU_GATHER_LOGLIK_N: return copy_rows(h, dst, h->loglikN, 1, 8);
    case SIPNET_GPU_GATHER_STATUS: return copy_rows(h, dst, h->status, 1, 4);
    case SIPNET_GPU_GATHER_COUNTERS: return copy_rows(h, dst, h->counters, SIPNET_GPU_NCOUNTERS, 4);
    case SIPNET_GPU_GATHER_STATE: return copy_rows(h, dst, h->state, SIPNET_GPU_NSTATE, 8);
    case SIPNET_GPU_GATHER_PARAMS: return copy_rows(h, dst, h->params, SIPNET_GPU_NPARAMS, 8);
    case SIPNET_GPU_GATHER_RING_VALUES: return copy_rows(h, dst, h->ringV, (size_t)h->ringCap, 8);
    case SIPNET_GPU_GATHER_RING_WEIGHTS: return copy_rows(h, dst, h->ringW, (size_t)h->ringCap, 8);
    case SIPNET_GPU_GATHER_EVENT_COUNTS: return copy_rows(h, dst, h->recCount, 1, 4);
    case SIPNET_GPU_GATHER_EVENT_RECORDS:
      CUDA_OK(cudaMemcpyAsync(dst, h->recs, need, cudaMemcpyDeviceToHost, h->stream));
      CUDA_OK(cudaStreamSynchronize(h->stream));
      return 0;
    case SIPNET_GPU_GATHER_MEAN:
    case SIPNET_GPU_GATHER_VARIANCE:
    case SIPNET_GPU_GATHER_QUANTILES: {
      int rc = ensure_summaries(h);
      if (rc) return rc;
      const double *src = what == SIPNET_GPU_GATHER_MEAN ? h->mean : what == SIPNET_GPU_GATHER_VARIANCE ? h->var : h->quant;
      CUDA_OK(cudaMemcpyAsync(dst, src, need, cudaMemcpyDeviceToHost, h->stream));
      CUDA_OK(cudaStreamSynchronize(h->stream));
      return 0;
    }
    default: return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "unknown gather selector %d", what);
  }
}

extern "C" int sipnet_gpu_sync(sipnet_gpu_handle *h) {
  if (!h) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL handle");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return 0;
}

extern "C" void sipnet_gpu_destroy(sipnet_gpu_handle *h) { free_handle(h); }

extern "C" int sipnet_gpu_last_run_ms(sipnet_gpu_handle *h, float *ms) {
  if (!h || !ms) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL argument");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaEventSynchronize(h->evStop));
  CUDA_OK(cudaEventElapsedTime(ms, h->evStart, h->evStop));
  return 0;
}

extern "C" int64_t sipnet_gpu_launch_count(const sipnet_gpu_handle *h) { return h ? h->launches : 0; }

extern "C" void *sipnet_gpu_device_ptr(sipnet_gpu_handle *h, int what) {
  if (!h) return nullptr;
  switch (what) {
    case SIPNET_GPU_GATHER_FULL: return h->out;
    case SIPNET_GPU_GATHER_DEBUG: return h->dbg;
    case SIPNET_GPU_GATHER_LOGLIK: return h->loglik;
    case SIPNET_GPU_GATHER_LOGLIK_N: return h->loglikN;
    case SIPNET_GPU_GATHER_STATUS: return h->status;
    case SIPNET_GPU_GATHER_COUNTERS: return h->counters;
    case SIPNET_GPU_GATHER_STATE: return h->state;
    case SIPNET_GPU_GATHER_MEAN: return ensure_summaries(h) ? nullptr : h->mean;
    case SIPNET_GPU_GATHER_VARIANCE: return ensure_summaries(h) ? nullptr : h->var;
    case SIPNET_GPU_GATHER_QUANTILES: return ensure_summaries(h) ? nullptr : h->quant;
    default: return nullptr;
  }
}

extern "C" void *sipnet_gpu_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}
extern "C" void sipnet_gpu_host_free(void *p) {
  if (p) cudaFreeHost(p);
}
extern "C" const char *sipnet_gpu_last_error(void) { return g_err.c_str(); }
extern "C" int sipnet_gpu_abi_version(void) { return SIPNET_GPU_ABI_VERSION; }

extern "C" int sipnet_gpu_measure_fp64_peak(int device, double *tflops) {
  if (!tflops) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "NULL argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
    return fail(SIPNET_GPU_ERR_NO_DEVICE, "device %d not present", device);
  CUDA_OK(measure_fp64_peak(device, tflops));
  return 0;
}

extern "C" int sipnet_gpu_eval_libm(int device, int op, const double *x, const double *y, double *out, int64_t n) {
  if (!x || !out || n <= 0 || op < 0 || op > 8 || (op != 0 && op != 2 && op != 8 && !y))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "bad eval_libm arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
    return fail(SIPNET_GPU_ERR_NO_DEVICE, "device %d not present", device);
  CUDA_OK(eval_libm(device, op, x, y, out, n));
  return 0;
}

extern "C" int sipnet_gpu_rows_summary(int device, const double *d_rows, int64_t nrows, int64_t ncols, int64_t ld,
                                       const double *probs, int32_t nq, double *d_mean, double *d_var, double *d_quant,
                                       void *stream) {
  if (!d_rows || nrows <= 0 || ncols <= 0 || ld < ncols || nq < 0 || (nq > 0 && (!probs || !d_quant)))
    return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "bad rows_summary arguments");
  if ((d_mean == nullptr) != (d_var == nullptr)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "mean and var go together");
  for (int i = 0; i < nq; ++i)
    if (!(probs[i] >= 0.0 && probs[i] <= 1.0)) return fail(SIPNET_GPU_ERR_BAD_ARGUMENT, "quantile probability out of [0,1]");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
    return fail(SIPNET_GPU_ERR_NO_DEVICE, "device %d not present", device);
  CUDA_OK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  // row span and probabilities travel as kernel parameters: no device scratch, nothing that synchronises
  CUDA_OK(launch_row_summary(d_rows, ld, nrows, nullptr, 1, ncols, probs, nq, d_mean, d_var, nrows, d_quant,
                             (int64_t)nq * nrows, st));
  if (st == nullptr) CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}
