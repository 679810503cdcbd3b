// sip_assim.cuh -- the serial ensemble adjustment Kalman filter (EAKF; Anderson 2001/2003) on a handle's carried
// pools: launchers and scratch of sip_assim.cu.  The host driver (one handle, or a team that exchanges per-site
// partial sums) is in sip_comm.cu.
//
// Per observation k the device runs
//   members(pass 1)  partial sums N, Σy, Σx_j of every chunk (fused with the update of observation k-1)
//   site_reduce(1)   chunk partials -> per site; one rank: the means ȳ, x̄_j (a team: its partial, then exchange +
//                    site_combine(1), which sums the ranks' partials in rank order)
//   members(pass 2)  Σ(y-ȳ)², Σ(x_j-x̄_j)(y-ȳ) of every chunk
//   site_reduce(2)   -> per site coefficients ȳ_a - ȳ, α - 1, S_jy / S_yy and the diagnostics (team: + combine)
// and after the last observation members(apply + floor).  With prior inflation at some site, the call first runs
//   members(pass 3)  partial sums N, Σx_j of every chunk
//   site_reduce(3)   -> per site x̄_j and sqrt(λ0), or "not inflated" (team: + combine)
// and observation 0's members(pass 1) inflates before it sums.  The adaptive update of λ, σ runs in finish(2).
//
// Reduction order: a chunk is kChunk consecutive SITE-LOCAL member indices; inside a chunk each lane sums its members
// in index order and the 32 lane sums meet in a fixed xor tree; a site sums its chunks in the same way.  Nothing
// depends on the handle's block layout, and there are no floating-point atomics: the same members of a site give the
// same bits in any handle.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "sip_handle.h"

namespace sip {
namespace as {

constexpr int kMaxRows = 12;   // the pools SIPNET_S_plantWoodC .. SIPNET_S_plantStorageN
constexpr int kRec = 16;       // doubles per chunk / site / rank record
constexpr int kInflPass = 3;   // the inflation's moment pass

// Record layouts (doubles):
//   pass-1 partial  [0] N  [1] Σy  [2+j] Σx_j          means  [0] N  [1] ȳ  [2+j] x̄_j
//   pass-3 partial  [0] N  [2+j] Σx_j                 inflation (in `mom` until pass 1 of observation 0 replaces it)
//                                                     [0] 1: inflate, 0: not  [1] sqrt(λ0)  [2+j] x̄_j
//   pass-2 partial  [0] S_yy  [1+j] S_jy
//   coefficients    [0] flags (bit 0: this observation applies, bit 1: some observation of the call applied)
//                   [1] ȳ_a - ȳ  [2] α - 1  [3] ȳ  [4+j] S_jy / S_yy
struct Args {
  double *state;
  uint32_t *status;
  int64_t ld;
  const SiteDev *sites;
  int32_t nsites;
  int32_t nchunks;
  const int2 *chunk;       // [nchunks]: (site, first site-local member)
  const int2 *siteChunks;  // [nsites]: (first chunk, chunk count)
  int32_t nrows, nobs, k;  // k: the observation of this launch
  int32_t nranks, rank;
  int32_t rows[kMaxRows];
  double opPrev[kMaxRows];  // operator of observation k - 1 (the update applied by a pass)
  double opCur[kMaxRows];   // operator of observation k
  double *part;             // [nchunks][kRec]
  double *mom;              // [nsites][kRec] means of observation k
  double *coef;             // [nsites][kRec]
  const double *value;      // [nsites][nobs]
  const double *variance;   // [nsites][nobs]
  double *diag;             // [nsites][nobs][4]
  double *rankRec;          // [nranks][nsites][kRec] (teams only)
  double *infl;             // [nsites][3] {λ0, λ, σ} of the inflation, or NULL (sipnet_gpu_assimilate)
  double lamMin, lamMax, sdMin;
};

// the handle's chunk tables and per-call buffers (made once; the observation buffers grow with nobs)
int ensure_scratch(sipnet_gpu_handle *h, int nobs);
// the per-site {λ0, λ, σ} buffer of the inflation (made once)
int ensure_inflation(sipnet_gpu_handle *h);
// pass 0 / 1 / 2 / kInflPass; `apply`: first add the update of observation k - 1; `floor`: then the final floor;
// `inflate` (pass 1 of observation 0): first the prior inflation
cudaError_t launch_members(const Args &a, int pass, bool apply, bool floor, bool inflate, cudaStream_t stream);
// chunks -> site; one rank finishes the pass, a team writes its partial to rankRec[rank]
cudaError_t launch_site_reduce(const Args &a, int pass, cudaStream_t stream);
// team: the ranks' partials, summed in rank order, finish the pass on every rank
cudaError_t launch_site_combine(const Args &a, int pass, cudaStream_t stream);

}  // namespace as
}  // namespace sip
