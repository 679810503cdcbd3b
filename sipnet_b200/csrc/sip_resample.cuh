// sip_resample.cuh -- the per-site systematic particle filter (bootstrap filter; Gordon, Salmond & Smith 1993) on a
// handle's members: launchers and scratch of sip_resample.cu.  The host driver (one handle, or a team) is in
// sip_comm.cu; the definition is in include/sipnet_gpu.h (sipnet_gpu_resample).
//
// One call runs
//   weights_a    per chunk: participants N, max of l, a +inf flag
//   site_a       chunks -> this rank's per-site record;  (team: all-gather)  host: lmax of every site
//   weights_b    per chunk: w = exp(l - lmax), W = (uint64)(w 2^40) to scratch, sums of w and w^2 in 2^-100 fixed
//                point and of W
//   site_b       chunks -> this rank's per-site record, and the exclusive scan of the chunk totals of W;
//                (team: all-gather)  host: ESS, the decision, T, every rank's slot ranges and the record tables
//   prefix       per chunk: C_i = (W of the lower ranks) + (chunk offset) + warp exclusive scan of W
//   pack         one thread per outgoing slot: its ancestor (binary search on C), the ancestor's record into the
//                segment of the slot's destination rank;  (team: the segments travel, NCCL or device copies)
//   unpack       one thread per member: its slot's record from the segment of the source rank
// Seven launches, whatever the number of sites.  Every sum is an integer sum, so no order of reduction -- chunks,
// lanes, ranks -- changes a bit: a site gives the same ancestors and diagnostics in any partition.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "sip_handle.h"

namespace sip {
namespace rs {

constexpr int kRec = 6;             // uint64 words per (rank, site) record
constexpr int kFixBits = 100;     // w and w^2 are summed as floor(x 2^100)
constexpr int kWeightBits = 40;   // W = floor(w 2^40)
constexpr int64_t kMaxSiteMembers = int64_t(1) << 23;  // keeps T = sum W below 2^63

// Record layouts (uint64 words):
//   pass a  [0] participants N  [1] max l of the participants (double bits; -inf if none)  [2] members n
//           [3] some l is +inf
//   pass b  [0, 1] sum floor(w 2^100) (lo, hi)  [2, 3] sum floor(w^2 2^100) (lo, hi)  [4] sum W
// A member record (what a resampled slot receives) is `words` doubles: kNParamDev parameter rows, SIPNET_GPU_NSTATE
// state rows, ringCap values, ringCap weights, status | event count << 32, SIPNET_GPU_NCOUNTERS counters (two per
// word), maxRecs event records, and the ancestor's member index in the team's rank-major order.
struct Args {
  // the handle
  const double *logw;  // [ld] log-weights
  uint32_t *status;
  const SiteDev *sites;
  const int32_t *memberSite;
  int64_t nmembers, ld;
  int32_t nsites, nchunks;
  const int2 *chunk;       // [nchunks]: (site, first site-local member)
  const int2 *siteChunks;  // [nsites]: (first chunk, chunk count)
  double *params, *state, *ringV, *ringW, *loglik, *loglikN;
  uint32_t *counters;
  sipnet_gpu_event_record *recs;
  int32_t *recCount;
  int32_t ringCap, maxRecs, words;
  int32_t nranks, rank;
  int64_t idBase;  // rank-major index of this rank's first member
  // scratch
  uint64_t *part;     // [nchunks][kRec + 1]: the record, then [kRec] the chunk's exclusive prefix of W in its site
  uint64_t *w, *c;    // [ld]: W and C of every member
  uint64_t *siteRec;  // [nranks][nsites][kRec]: this rank writes its slot
  const double *lmax; // [nsites]
  int64_t *anc;       // [ld]: ancestor (rank-major index) of every member, -1 where its site was not resampled
  // tables of the copy (made on the host by sip_comm.cu run_resample)
  const int64_t *flag, *U, *T, *n, *toff;  // [nsites]: resampled?, U, T, n of the site, W of the lower ranks
  const int64_t *slot0;    // [nsites][nranks + 1]: first slot whose ancestor lives on rank p (p = nranks: n)
  const int64_t *mem0;     // [nsites][nranks + 1]: first slot held by rank q (q = nranks: n)
  const int64_t *sendPos;  // [nsites][nranks]: position of the site's first record in this rank's segment to q
  const int64_t *recvPos;  // [nsites][nranks]: position of the site's first record in p's segment to this rank
  const int64_t *outPre;   // [nsites + 1]: this rank's outgoing records before each site
  const int64_t *sendBase, *sendCnt, *recvCnt;  // [nranks]: segment to q at sendBuf + sendBase[q] (sendCnt[q] records);
                                                 // recvCnt[p] records come from p
  double *const *src;      // [nranks]: where the segment from p is read (this rank's own: in sendBuf)
  double *sendBuf;
  int64_t nOut;            // outgoing records
};

// the handle's chunk tables, chunk records and member scratch
int ensure_scratch(sipnet_gpu_handle *h);
// doubles of one member record
int record_words(const sipnet_gpu_handle *h);
cudaError_t launch_weights(const Args &a, int pass, cudaStream_t stream);  // pass 0 (a) or 1 (b)
cudaError_t launch_site(const Args &a, int pass, cudaStream_t stream);
cudaError_t launch_prefix(const Args &a, cudaStream_t stream);
cudaError_t launch_pack(const Args &a, cudaStream_t stream);
cudaError_t launch_unpack(const Args &a, cudaStream_t stream);

}  // namespace rs
}  // namespace sip
