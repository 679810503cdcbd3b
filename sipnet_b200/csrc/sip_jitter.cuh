// sip_jitter.cuh -- the Liu & West (2001) kernel-shrinkage move of the parameter rows, per site, after a resample:
// launchers and scratch of sip_jitter.cu.  The host driver (one handle, or a team that exchanges per-site partial
// sums) is in sip_comm.cu; the definition is in include/sipnet_gpu.h (sipnet_gpu_rejuvenate).
//
// One call runs
//   members(1)      per chunk: N and the sums of phi_j (phi = the transformed rows)
//   site(1)         chunks -> per site; one rank: N and the means (a team: its partial, then exchange + combine(1),
//                   which sums the ranks' partials in rank order)
//   members(2)      per chunk: the centred cross sums sum (phi_j - mean_j)(phi_l - mean_l), l <= j
//   site(2)         -> per site: V, its semidefinite Cholesky factor L and the move's coefficients (team: + combine)
//   members(3)      propose, invert, re-derive (sip_derive.cuh), accept or keep; moved / kept per chunk
//   site(3)         -> per site diagnostics {N, rank, moved, kept} (team: + combine)
// Six launches on one GPU, whatever the number of sites.
// The Metropolis-Hastings move (Args::scale set) runs the same passes with a = 1, h = scale and its own participants;
// members(3) also records each member's verdict, and site(3) runs after the accept pass of sip_resample.cu, whose
// per-chunk counts {invalid, accepted} it turns into diag (sip_comm.cu run_mh).
//
// Reduction order: the handle's 128-member chunks of site-local indices (sipnet_gpu_handle::chunk).  Inside a chunk,
// a lane sums one quantity over the chunk's members in index order; a site sums its chunks in chunk order; a team
// sums the ranks' partials in rank order.  No floating-point atomics: the same members of a site give the same bits
// in any handle.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "sip_handle.h"

namespace sip {
namespace jt {

constexpr int kMaxRows = 16;
constexpr int kTri = kMaxRows * (kMaxRows + 1) / 2;  // lower triangle of V (l <= j), row-major
constexpr int kSum0 = 1 + kMaxRows;                  // first cross sum in a record
constexpr int kRec = kSum0 + kTri;                   // doubles per chunk / site / rank record: N, sums of phi, cross sums

// Coefficient record of a site (doubles): [0] 1 = the site moves  [1] a  [2] rank
//   [3 + j] (1 - a) mean_j  [3 + kMaxRows + tri(j, m)] h L_jm
constexpr int kCoef = 3 + kMaxRows + kTri;

__host__ __device__ constexpr int tri(int j, int l) { return j * (j + 1) / 2 + l; }

struct Args {
  double *params;
  uint32_t *status;
  int64_t ld;
  int64_t nmembers;
  const SiteDev *sites;
  int32_t nsites;
  int32_t nchunks;
  const int2 *chunk;       // [nchunks]: (site, first site-local member)
  const int2 *siteChunks;  // [nsites]: (first chunk, chunk count)
  int32_t nrows;
  int32_t nranks, rank;
  int32_t rows[kMaxRows];
  int32_t transform[kMaxRows];  // SIPNET_GPU_TF_*
  double lower[kMaxRows], upper[kMaxRows];
  const double *shrink;  // [nsites]
  const double *z;       // [nrows][nmembers]
  double *part;          // [nchunks][kRec]
  double *mom;           // [nsites][kRec]: N, means
  double *coef;          // [nsites][kCoef]
  double *diag;          // [nsites][4]
  double *rankRec;       // [nranks][nsites][kRec] (teams only)
  // The Metropolis-Hastings proposal (sipnet_gpu_mh_move) when scale != NULL: a = 1 and h = scale[s] per site (the
  // Liu-West move: a = shrink[s], h = sqrt(1 - a^2)); a participant also needs a finite current log-likelihood and
  // log prior; members(3) writes every member's verdict (kMh*) and, for a valid proposal, lp(phi') - lp(phi).
  const double *scale;      // [nsites]
  const double *curLoglik;  // [nmembers]
  int32_t prior[kMaxRows];  // SIPNET_GPU_PRIOR_*
  double priorA[kMaxRows], priorB[kMaxRows];
  int8_t *valid;            // [nmembers]
  double *dlp;              // [nmembers]
};

// the handle's chunk tables and scratch (made once, by the first call)
int ensure_scratch(sipnet_gpu_handle *h);
// pass 1 / 2 / 3
cudaError_t launch_members(const Args &a, int pass, cudaStream_t stream);
// chunks -> site; one rank finishes the pass, a team writes its partial to rankRec[rank]
cudaError_t launch_site(const Args &a, int pass, cudaStream_t stream);
// team: the ranks' partials, summed in rank order, finish the pass on every rank
cudaError_t launch_combine(const Args &a, int pass, cudaStream_t stream);

}  // namespace jt
}  // namespace sip
