// sip_gsum.cuh -- interface of the cross-rank ensemble summaries (sip_gsum.cu), driven by sip_comm.cu.
//
// A site's members may be spread over several ranks (one rank = one GPU).  Every rank holds the per-step output
// columns of ITS members; the summaries of the whole ensemble -- mean, population variance and exact quantiles
// (numpy "linear" rule) per (site, summary column, step) row -- are found WITHOUT moving the members' values:
//   * moments: per-rank (count, sum) and, against the global mean, per-rank sums of squared deviations are gathered
//     (a few bytes per row and rank) and added in rank order on every rank -- deterministic for a given partition;
//   * quantiles: a radix select on the order-preserving 64-bit keys of the values, all ranks in lockstep: per
//     level every rank histograms its members' next key bits (11, then 8 at a time) inside the bins that still
//     hold a wanted order statistic, the histograms are summed over the ranks (NCCL all-reduce) and every rank
//     resolves the same bin.  When a bin holds at most kGsEmit keys, the ranks emit those keys, gather them and
//     finish locally.  Traffic: 8 KB per row and level instead of the row itself (1 MB per rank at 131072 members).
// With one rank the exchange steps fall away and the same kernels give the local result.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "sip_types.cuh"

namespace sip {
namespace gs {

constexpr int kGsMaxQ = 4;              // quantiles per pass
constexpr int kGsMaxStat = 2 * kGsMaxQ; // order statistics: lo and lo + 1 of every quantile
constexpr int kGsEmit = 16;             // a bin with at most this many keys (over all ranks) is finished by gathering them
constexpr int kGsHistWords = 2048;      // per row and level: 2^11 bins (level 0) or kGsMaxStat slots x 2^8 bins
constexpr int kGsLevels = 8;            // key bits per level: 11, 8, 8, 8, 8, 8, 8, 5
constexpr int kGsMaxCols = 8;           // summary columns per pass
constexpr int kGsListCap = 4096;        // candidate list of a row (see GsArgs::list): at most this many keys, all ranks

struct GsStat {  // per row and rank, pass 0
  double count, sum;
  uint64_t rep;   // key of one finite member (valid when count > 0)
  uint64_t diff;  // OR of (key ^ rep) over the rank's finite members: 0 = they are all equal
};

struct GsTie {  // per row, histogram slot and rank, written by a level pass
  uint64_t rep;   // one key of the rank's members in the slot (kGsNoKey = none)
  uint64_t diff;  // OR of (key ^ rep) over them: 0 = they are all equal
};
constexpr uint64_t kGsNoKey = ~0ull;  // never the key of a finite value

struct GsRow {  // selection state of a row; identical on every rank after each exchange
  uint64_t prefix[kGsMaxStat];  // resolved leading key bits of each wanted order statistic (the key when bits == 64)
  uint64_t k[kGsMaxStat];       // its rank among the keys sharing the prefix
  uint32_t pop[kGsMaxStat];     // how many keys (all ranks) share the prefix
  uint8_t slotOf[kGsMaxStat];   // statistics with equal prefixes share a histogram slot (0xff = final)
  uint8_t rbits[kGsMaxStat];    // key bits resolved when the statistic became final (0 = not yet): its bin then held
                                // at most kGsEmit keys, or all 64 bits were resolved
  uint8_t nslots;
  uint8_t bits;                 // leading key bits resolved so far (same for every statistic of the row)
  uint8_t done;                 // 0 = needs another level, 1 = every statistic is resolved or ready to emit,
                                // 2 = constant row (value in prefix[0]), 3 = no finite member
  uint8_t listed;               // level whose pass copied this rank's candidates into GsArgs::list (0 = none)
  double n, mean;
};

struct GsArgs {
  // the run range's column buffer and its rows
  const double *out;
  int64_t ld, nsteps;
  const SiteDev *sites;
  int32_t nsites, ncols;
  int32_t colSlot[kGsMaxCols];  // slot of summary column i in `out`
  int32_t nq;
  double probs[kGsMaxQ];  // ascending (the caller sorts them; the slot assignment of resolve_level relies on it)
  int32_t qOut[kGsMaxQ];  // index of each probability's result among the column's nqTotal quantiles
  int32_t nranks, rank;
  int32_t wantMoments;
  // scratch (device).  *Local = this rank's contribution, *All = [nranks][...] after the gather (the same
  // allocation: local data sits at index `rank`)
  GsStat *statAll;
  double *q2All;
  uint32_t *hist;      // [rows][kGsHistWords], summed over ranks between the levels
  GsRow *state;        // [rows]
  GsTie *tieAll;       // [nranks][rows][kGsMaxStat]: are the keys of a slot all equal? (order statistics inside a
                       // large group of equal values -- exact zeros -- would otherwise need every key bit)
  uint64_t *emitAll;   // [nranks][rows][kGsMaxStat][kGsEmit]
  int32_t *flags;      // [0] = some row needs the next level
  // Candidate lists (nullptr: never compact).  A level pass whose filter -- the slots in play plus the bins of the
  // statistics waiting for the emit -- holds at most kGsListCap keys over ALL ranks copies this rank's finite members
  // inside it to list[row]; later levels and the emit scan that list instead of the row.  Later prefixes only extend
  // the filter's, so the list holds every key they look for; the global bound keeps every rank's share in the list.
  double *list;        // [rows][kGsListCap]
  int32_t *listN;      // [rows]: members in list[row]
  // results, in the handle's layout: mean/var [site][col][n], quant [site][col][q][n]
  double *mean, *var, *quant;
  int32_t nqTotal;  // quantiles per column (quant rows are [nqTotal] per column)
};

inline int64_t gs_rows(const GsArgs &a) { return (int64_t)a.nsites * a.ncols * a.nsteps; }

cudaError_t launch_pass0(const GsArgs &a, cudaStream_t stream);
cudaError_t launch_level(const GsArgs &a, int level, cudaStream_t stream);
cudaError_t launch_emit(const GsArgs &a, cudaStream_t stream);
cudaError_t launch_finish(const GsArgs &a, cudaStream_t stream);
// dst[i] += src[i] for i < n (the histogram sum of a team whose ranks share one device)
cudaError_t launch_add_u32(uint32_t *dst, const uint32_t *src, size_t n, cudaStream_t stream);

}  // namespace gs
}  // namespace sip
