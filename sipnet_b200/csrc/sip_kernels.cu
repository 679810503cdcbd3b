// sip_kernels.cu -- setup kernels (setupModel() on the device) and the dispatcher of the fused step kernel K1.
//
// K1 itself (run_item / run_kernel) is a template in sip_run.cuh, instantiated in sip_run_exact.cu and
// sip_run_fast_*.cu.  Everything is compiled with -fmad=false: the model arithmetic keeps the reference's
// operation order, and exp/pow/division are explicit operation sequences (sip_libm.cuh, sip_num.cuh), so every
// kernel is bit-identical to the reference binary.
#include <cuda_runtime.h>

#include "sip_derive.cuh"
#include "sip_step.cuh"

namespace sip {
namespace k1 {

// ---- setup kernels: setupModel(), sipnet.c:1858-1951 ----------------------------------------
// (1) parameter derivation, in place on the uploaded raw rows: the unit changes, then the rows that depend on other
// rows (sip_derive.cuh, shared with the parameter move of sip_jitter.cu)
__global__ void derive_params_kernel(double *params, int64_t ld, int64_t nmembers, uint32_t *status) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= nmembers) return;
  auto P = [&](int k) -> double & { return params[(int64_t)k * ld + m]; };
  P(SIPNET_P_baseVegResp) /= 365.0;  // :1873-1877
  P(SIPNET_P_litterBreakdownRate) /= 365.0;
  P(SIPNET_P_baseSoilResp) /= 365.0;
  P(SIPNET_P_woodTurnoverRate) /= 365.0;
  P(SIPNET_P_leafTurnoverRate) /= 365.0;
  P(SIPNET_P_fineRootTurnoverRate) /= 365.0;  // :1898-1902
  P(SIPNET_P_coarseRootTurnoverRate) /= 365.0;
  P(SIPNET_P_baseCoarseRootResp) /= 365.0;
  P(SIPNET_P_baseFineRootResp) /= 365.0;
  status[m] = derive_dependent(P) ? SIPNET_GPU_ST_BAD_ALLOCATION : 0u;
}

// (2) initial pools / trackers (also used by reset())
__global__ void init_state_kernel(const double *params, int64_t ld, int64_t nmembers, const int32_t *memberSite,
                                  const SiteDev *sites, uint32_t flags, double *state, double *ringV, double *ringW,
                                  uint32_t *status, double *loglik, double *loglikN, int32_t *recCount) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= nmembers) return;
  auto P = [&](int k) -> double { return params[(int64_t)k * ld + m]; };
  auto S = [&](int k) -> double & { return state[(int64_t)k * ld + m]; };
  const RuntimeFlags fl(flags);
  for (int k = 0; k < SIPNET_GPU_NSTATE; ++k) S(k) = 0.0;
  S(SIPNET_S_plantWoodC) = (1 - P(SIPNET_P_coarseRootFrac) - P(SIPNET_P_fineRootFrac)) * P(SIPNET_P_plantWoodInit);
  S(SIPNET_S_plantCAccountingDelta) = 0.0;
  S(SIPNET_S_plantLeafC) = P(SIPNET_P_laiInit) * P(SIPNET_P_leafCSpWt);
  S(SIPNET_S_litterC) = fl.on(F_LITTER_POOL) ? P(SIPNET_P_litterInit) : 0.0;
  S(SIPNET_S_soilC) = P(SIPNET_P_soilInit);
  S(SIPNET_S_coarseRootC) = P(SIPNET_P_coarseRootFrac) * P(SIPNET_P_plantWoodInit);
  S(SIPNET_S_fineRootC) = P(SIPNET_P_fineRootFrac) * P(SIPNET_P_plantWoodInit);
  double water = P(SIPNET_P_soilWFracInit) * P(SIPNET_P_soilWHC);
  if (water < 0) water = 0;
  S(SIPNET_S_soilWater) = water;
  S(SIPNET_S_snow) = P(SIPNET_P_snowInit);
  if (fl.on(F_NITROGEN)) {
    S(SIPNET_S_minN) = P(SIPNET_P_minNInit);
    S(SIPNET_S_soilOrgN) = P(SIPNET_P_soilOrgNInit);
    S(SIPNET_S_litterN) = P(SIPNET_P_litterOrgNInit);
    S(SIPNET_S_plantStorageN) = P(SIPNET_P_plantStorageNInit);
  }
  // initTrackers, :1406-1413
  S(SIPNET_S_soilWetnessFrac) = water / P(SIPNET_P_soilWHC);
  S(SIPNET_S_trackersLastYear) = -1.0;
  // initPhenologyTrackers, :1501-1527, against the site's FIRST climate record
  const SiteDev site = sites[memberSite[m]];
  int didGrowth = 0, didFall = 0, year0 = 0;
  if (site.nsteps > 0) {
    const ClimRec c = site.clim[0];
    year0 = c.year;
    if (fl.on(F_GDD)) {
      didGrowth = c.gdd >= P(SIPNET_P_gddLeafOn);  // trackers.lastYear == -1, so no carry-over term
    } else if (fl.on(F_SOIL_PHENOL)) {
      didGrowth = c.tsoil >= P(SIPNET_P_soilTempLeafOn);
    } else if (P(SIPNET_P_leafOnDay) > 0) {
      didGrowth = c.dayFrac >= P(SIPNET_P_leafOnDay);
    }
    if (P(SIPNET_P_leafOffDay) > 0) didFall = c.dayFrac >= P(SIPNET_P_leafOffDay);
    if (didFall && !didGrowth) didGrowth = 1;
  }
  S(SIPNET_S_didLeafGrowth) = didGrowth;
  S(SIPNET_S_didLeafFall) = didFall;
  S(SIPNET_S_phenLastYear) = year0;
  // resetMeanTracker(meanNPP, 0), :1948
  ringV[m] = 0.0;
  ringW[m] = kMeanNppDays;
  S(SIPNET_S_meanSum) = 0.0 * kMeanNppDays;
  status[m] &= SIPNET_GPU_ST_BAD_ALLOCATION;  // keep the static verdict, clear run-time bits
  if (loglik != nullptr) loglik[m] = 0.0;
  if (loglikN != nullptr) loglikN[m] = 0.0;
  if (recCount != nullptr) recCount[m] = 0;
}

// (3) launch-lifetime constants (StepConsts): the division seeds of the literal divisors come from the device's own
// reciprocal approximation, so they are evaluated here, once per handle
__global__ void consts_kernel(StepConsts *out) {
  const FastNum fn;
  const libm::LogHL l2 = libm::pow_log(2.0);  // pow(2, y), sipnet.c:551
  out->log2Hi = l2.hi;
  out->log2Lo = l2.lo;
  out->seed10 = fn.seed(10.0);
  out->seed5 = fn.seed(kMeanNppDays);
  out->seed18 = fn.seed(3.0 * 6);
  out->seed24 = fn.seed(24.0);
}

// ---- host-side launchers (C++ linkage inside the library) -------------------------------------
constexpr uint32_t kMaskDefault = F_EVENTS | F_GDD | F_SNOW | F_WATER_HRESP;                       // context.c:35-46
constexpr uint32_t kMaskCropN = kMaskDefault | F_LITTER_POOL | F_ANAEROBIC | F_NITROGEN;          // russell_2 / C2-C5

// K1 instantiations live in sip_run_exact.cu / sip_run_fast_*.cu
cudaError_t launch_exact(const RunArgs &a, int nblocks, int blockThreads, bool debug, int mode, cudaStream_t stream);
cudaError_t launch_fast_default_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_fast_default_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_fast_cropn_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_fast_cropn_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_fast_generic_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_fast_generic_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);

cudaError_t launch_thr_default_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_thr_default_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_thr_cropn_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_thr_cropn_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_thr_generic_32(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);
cudaError_t launch_thr_generic_128(const RunArgs &a, int nblocks, bool full, cudaStream_t stream);

// mode: 0 = exact (validation), 1 = fast (optimistic), 2 = replay of flagged members (exact), 3 = throughput policy
cudaError_t launch_run(const RunArgs &a, int nblocks, int blockThreads, bool debug, int mode, cudaStream_t stream) {
  if (blockThreads != 32 && blockThreads != 128) return cudaErrorInvalidValue;
  if ((mode != 1 && mode != 3) || debug) return launch_exact(a, nblocks, blockThreads, debug, mode, stream);
  const uint32_t arith = a.flags & ~(uint32_t)F_SNOW;  // ctx.snow has no arithmetic effect (SURVEY 8a trap 6)
  bool full = a.out != nullptr;
  for (int c = 0; c < SIPNET_GPU_NOUT; ++c) full = full && a.colSlot[c] == c;
  using Launcher = cudaError_t (*)(const RunArgs &, int, bool, cudaStream_t);
  // [numerics: optimistic, throughput][flag policy: default, crop-N, generic][block: 32, 128]
  // (256-member blocks, one per SM, were measured: 3-4 % slower than two 128-member blocks)
  static const Launcher table[2][3][2] = {
      {{launch_fast_default_32, launch_fast_default_128},
       {launch_fast_cropn_32, launch_fast_cropn_128},
       {launch_fast_generic_32, launch_fast_generic_128}},
      {{launch_thr_default_32, launch_thr_default_128},
       {launch_thr_cropn_32, launch_thr_cropn_128},
       {launch_thr_generic_32, launch_thr_generic_128}}};
  const int policy = arith == (kMaskDefault & ~(uint32_t)F_SNOW) ? 0 : (arith == (kMaskCropN & ~(uint32_t)F_SNOW) ? 1 : 2);
  const int block = blockThreads == 32 ? 0 : 1;
  return table[mode == 3 ? 1 : 0][policy][block](a, nblocks, full, stream);
}

cudaError_t launch_derive(double *params, int64_t ld, int64_t nmembers, uint32_t *status, cudaStream_t stream) {
  const int threads = 128;
  const int blocks = (int)((nmembers + threads - 1) / threads);
  derive_params_kernel<<<blocks, threads, 0, stream>>>(params, ld, nmembers, status);
  return cudaGetLastError();
}

cudaError_t launch_consts(StepConsts *out, cudaStream_t stream) {
  consts_kernel<<<1, 1, 0, stream>>>(out);
  return cudaGetLastError();
}

cudaError_t launch_init_state(const double *params, int64_t ld, int64_t nmembers, const int32_t *memberSite,
                              const SiteDev *sites, uint32_t flags, double *state, double *ringV, double *ringW,
                              uint32_t *status, double *loglik, double *loglikN, int32_t *recCount,
                              cudaStream_t stream) {
  const int threads = 128;
  const int blocks = (int)((nmembers + threads - 1) / threads);
  init_state_kernel<<<blocks, threads, 0, stream>>>(params, ld, nmembers, memberSite, sites, flags, state, ringV,
                                                    ringW, status, loglik, loglikN, recCount);
  return cudaGetLastError();
}

}  // namespace k1
}  // namespace sip
