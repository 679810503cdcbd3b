// sip_derive.cuh -- the rows setupModel() derives from other parameter rows (sipnet.c:1858-1951), as one device
// function shared by the setup kernel (sip_kernels.cu) and the parameter move (sip_jitter.cu), so both give the same
// bits.  It reads no row that setupModel() rescales (the nine rates / 365), so it may run before or after them.
#pragma once
#include "sip_math.cuh"
#include "sip_num.cuh"
#include "sip_types.cuh"

namespace sip {

// ensureAllocation, sipnet.c:1111-1123: true when the allocation fractions are not a valid split
__device__ __forceinline__ bool allocation_fails(double leaf, double wood, double fineRoot, double coarseRoot) {
  return (leaf >= 1.0) || (wood >= 1.0) || (fineRoot >= 1.0) || (coarseRoot < 0);
}

// coarseRootAllocation, psnTMax, the fAnoxia / anaerobicDecompRate clamps and the internal rows kPsnTRangeSqSlot ..
// kOneMinusFracLitResp of one member; `P(k)` is a reference to row k.  Returns the allocation verdict.
template <class Row>
__device__ __forceinline__ bool derive_dependent(Row P) {
  P(SIPNET_P_coarseRootAllocation) =
      1 - P(SIPNET_P_leafAllocation) - P(SIPNET_P_woodAllocation) - P(SIPNET_P_fineRootAllocation);
  const bool bad = allocation_fails(P(SIPNET_P_leafAllocation), P(SIPNET_P_woodAllocation),
                                    P(SIPNET_P_fineRootAllocation), P(SIPNET_P_coarseRootAllocation));
  P(SIPNET_P_psnTMax) = P(SIPNET_P_psnTOpt) + (P(SIPNET_P_psnTOpt) - P(SIPNET_P_psnTMin));  // :1880-1881
  if (P(SIPNET_P_fAnoxia) <= 0.0) {  // :1905-1909
    P(SIPNET_P_fAnoxia) = kTiny;
  } else if (P(SIPNET_P_fAnoxia) >= 1.0) {
    P(SIPNET_P_fAnoxia) = 1.0 - kTiny;
  }
  if (P(SIPNET_P_anaerobicDecompRate) <= 0.0) {  // :1912-1916
    P(SIPNET_P_anaerobicDecompRate) = kTiny;
  } else if (P(SIPNET_P_anaerobicDecompRate) > 1.0) {
    P(SIPNET_P_anaerobicDecompRate) = 1.0;
  }
  // member constant of potPsn(): pow((psnTMax - psnTMin) / 2.0, 2), sipnet.c:622
  P(kPsnTRangeSqSlot) = sip_pow((P(SIPNET_P_psnTMax) - P(SIPNET_P_psnTMin)) / 2.0, 2.0);
  // division seeds of the member-constant divisors and member-constant sub-expressions (sip_num.cuh)
  {
    const FastNum fn;
    P(kOneMinusFa) = 1 - P(SIPNET_P_fAnoxia);
    P(kTwoWhc) = 2.0 * P(SIPNET_P_soilWHC);
    P(kOneMinusFracLitResp) = 1.0 - P(SIPNET_P_fracLitterRespired);
    P(kRespPerGram) = P(SIPNET_P_baseFolRespFrac) * P(SIPNET_P_aMax);
    P(kGrossAMax) = P(SIPNET_P_aMax) * P(SIPNET_P_aMaxFrac) + P(kRespPerGram);
    P(kConvBase) = 12.0 * (1.0 / 1000000000.0) * (P(SIPNET_P_leafCSpWt) / P(SIPNET_P_cFracLeaf));
    P(kSeedLeafCSpWt) = fn.seed(P(SIPNET_P_leafCSpWt));
    P(kSeedPsnTRangeSq) = fn.seed(P(kPsnTRangeSqSlot));
    P(kSeedHalfSatPar) = fn.seed(P(SIPNET_P_halfSatPar));
    P(kSeedWhc) = fn.seed(P(SIPNET_P_soilWHC));
    P(kSeedTwoWhc) = fn.seed(P(kTwoWhc));
    P(kSeedLeafCN) = fn.seed(P(SIPNET_P_leafCN));
    P(kSeedWoodCN) = fn.seed(P(SIPNET_P_woodCN));
    P(kSeedFineRootCN) = fn.seed(P(SIPNET_P_fineRootCN));
    P(kSeedFAnoxia) = fn.seed(P(SIPNET_P_fAnoxia));
    P(kSeedOneMinusFa) = fn.seed(P(kOneMinusFa));
    P(kSeedCSat) = fn.seed(P(SIPNET_P_soilCSaturation));
  }
  // log_inline() of the member-constant pow() bases
  const int bases[4] = {SIPNET_P_vegRespQ10, SIPNET_P_coarseRootQ10, SIPNET_P_fineRootQ10, SIPNET_P_soilRespQ10};
  const int slots[4] = {kLogVegQ10, kLogCoarseQ10, kLogFineQ10, kLogSoilQ10};
  for (int i = 0; i < 4; ++i) {
    const libm::LogHL l = libm::pow_log(P(bases[i]));
    P(slots[i]) = l.hi;
    P(slots[i] + 1) = l.lo;
  }
  return bad;
}

}  // namespace sip
