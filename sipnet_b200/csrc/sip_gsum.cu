// sip_gsum.cu -- cross-rank ensemble summaries: kernels of the lockstep radix select (see sip_gsum.cuh).
//
// One CTA per (site, summary column, step) row; a row's local members are contiguous in the column buffer K1 wrote.
// Every kernel is a pure function of (local data, exchanged buffers), and the selection state it derives from the
// exchanged buffers is recomputed identically on every rank -- no rank ever waits for another inside a kernel.
// The reference has no ensemble code (SURVEY 8c): definitions as in sip_reduce.cu; tests compare with numpy.
#include "sip_gsum.cuh"

#include <algorithm>
#include <type_traits>

namespace sip {
namespace gs {

constexpr int kThreads = 512;
constexpr int kUnroll = 4;       // loads in flight per thread: emit and the 64-bit levels (more would spill)
// Levels 1-2 read whole rows at 2 blocks x 512 threads per SM, where 4 loads of 8 B in flight per thread are too
// few bytes in flight for HBM latency (level 1 on the C4 share: 4.9 -> 4.3 ms with 8; pass 0, at 3 blocks per SM,
// takes the same loop and stays at 3.0 ms).  Element i of a row is still handled by thread i % kThreads in
// ascending i for any unroll, so the per-thread sums -- and the moments -- are the same bits.
constexpr int kUnrollWide = 8;
constexpr uint64_t kSent = kGsNoKey;

__host__ __device__ constexpr int bits_after(int level) { return level < 7 ? 11 + 8 * level : 64; }
__host__ __device__ constexpr int shift_of(int level) { return 64 - bits_after(level); }
__host__ __device__ constexpr int bins_of(int level) { return level == 0 ? 2048 : (level < 7 ? 256 : 32); }

// order-preserving map double -> uint64 (ascending), as in sip_reduce.cu
__device__ __forceinline__ uint64_t key_of(double x) {
  const uint64_t b = (uint64_t)__double_as_longlong(x);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double val_of(uint64_t k) {
  const uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ bool finite_hi(double x) { return (((unsigned int)__double2hiint(x) >> 20) & 0x7ffu) != 0x7ffu; }

// histogram update for all 32 lanes (code < 0: nothing to count); the lanes agreeing with lane 0 add once.  One
// predicated atomic per lane: lane 0 and the lanes that differ from it do not take separate paths.
__device__ __forceinline__ void hist_add(unsigned int *hist, int code) {
  const int lead = __shfl_sync(0xffffffffu, code, 0);
  const unsigned same = __ballot_sync(0xffffffffu, code == lead);
  const bool first = (threadIdx.x & 31) == 0;
  if (code >= 0 && (first || code != lead)) atomicAdd(&hist[code], first ? (unsigned)__popc(same) : 1u);
}

__device__ __forceinline__ double block_sum(double v, double *sh) {  // fixed order
  const int tid = threadIdx.x;
  sh[tid] = v;
  __syncthreads();
  for (int s = kThreads / 2; s > 0; s >>= 1) {
    if (tid < s) sh[tid] += sh[tid + s];
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();
  return r;
}

struct RowRef {
  const double *p;
  int count;
  int64_t row;  // (site * ncols + col) * nsteps + t
};
__device__ __forceinline__ RowRef row_ref(const GsArgs &a) {
  const int64_t row = blockIdx.x;
  const int64_t t = row % a.nsteps;
  const int64_t sc = row / a.nsteps;
  const int ci = (int)(sc % a.ncols);
  const int site = (int)(sc / a.ncols);
  const SiteDev sd = a.sites[site];
  return RowRef{a.out + ((int64_t)a.colSlot[ci] * a.nsteps + t) * a.ld + sd.member0, sd.memberCount, row};
}

// ---- pass 0: finite count, sum, one representative key + OR of differences, level-0 histogram -----------------
__global__ void __launch_bounds__(kThreads, 2) gs_pass0_kernel(const GsArgs a) {
  __shared__ unsigned int hist[2048];
  __shared__ double red[kThreads];
  __shared__ int repTid;
  __shared__ unsigned long long repKey;
  __shared__ unsigned int diffLo, diffHi;
  const int tid = threadIdx.x;
  const RowRef r = row_ref(a);
  const bool wantHist = a.nq > 0;
  if (wantHist)
    for (int i = tid; i < 2048; i += kThreads) hist[i] = 0;
  if (tid == 0) {
    repTid = kThreads;
    diffLo = diffHi = 0;
  }
  __syncthreads();
  double s = 0.0, c = 0.0;
  uint64_t first = 0, diff = 0;
  bool have = false;
  for (int i0 = 0; i0 < r.count; i0 += kUnrollWide * kThreads) {
    double x[kUnrollWide];
#pragma unroll
    for (int u = 0; u < kUnrollWide; ++u) {
      const int i = i0 + u * kThreads + tid;
      x[u] = i < r.count ? r.p[i] : __longlong_as_double(0x7ff8000000000000ll);
    }
#pragma unroll
    for (int u = 0; u < kUnrollWide; ++u) {  // per thread the elements are accumulated in index order
      const bool fin = finite_hi(x[u]);
      int code = -1;
      if (fin) {
        s += x[u];
        c += 1.0;
        const uint64_t k = key_of(x[u]);
        if (!have) {
          first = k;
          have = true;
        }
        diff |= k ^ first;
        code = (int)(k >> 53);
      }
      if (wantHist) hist_add(hist, code);
    }
  }
  const double total = block_sum(s, red);
  const double n = block_sum(c, red);
  if (have) atomicMin(&repTid, tid);
  __syncthreads();
  if (tid == repTid) repKey = first;
  __syncthreads();
  if (have) {
    diff |= first ^ (uint64_t)repKey;
    if ((unsigned int)diff) atomicOr(&diffLo, (unsigned int)diff);
    if ((unsigned int)(diff >> 32)) atomicOr(&diffHi, (unsigned int)(diff >> 32));
  }
  __syncthreads();
  if (tid == 0) {
    GsStat st;
    st.count = n;
    st.sum = total;
    st.rep = n > 0 ? (uint64_t)repKey : 0;
    st.diff = ((uint64_t)diffHi << 32) | diffLo;
    a.statAll[(int64_t)a.rank * gridDim.x + r.row] = st;
  }
  if (wantHist) {
    unsigned int *g = a.hist + r.row * kGsHistWords;
    for (int i = tid; i < 2048; i += kThreads) g[i] = hist[i];
  }
}

// ---- selection state -----------------------------------------------------------------------------------------
// global stats of the row from the gathered per-rank stats, in rank order; initial state of the select
__device__ void init_state(const GsArgs &a, int64_t row, int64_t rows, GsRow &S) {
  double n = 0.0, sum = 0.0;
  bool constant = true, any = false;
  uint64_t rep = 0;
  for (int q = 0; q < a.nranks; ++q) {
    const GsStat st = a.statAll[(int64_t)q * rows + row];
    n += st.count;
    sum += st.sum;
    if (st.count > 0) {
      if (!any) {
        rep = st.rep;
        any = true;
      }
      if (st.diff != 0 || st.rep != rep) constant = false;
    }
  }
  S.n = n;
  S.mean = n > 0 ? sum / n : __longlong_as_double(0x7ff8000000000000ll);
  S.bits = 0;
  S.nslots = 1;
  S.listed = 0;
  for (int i = 0; i < kGsMaxStat; ++i) {
    S.prefix[i] = 0;
    S.k[i] = 0;
    S.pop[i] = 0;
    S.slotOf[i] = 0;
    S.rbits[i] = 0;
  }
  if (!(n > 0)) {
    S.done = 3;
  } else if (constant) {
    S.done = 2;
    S.prefix[0] = rep;
  } else {
    S.done = a.nq > 0 ? 0 : 1;
    for (int i = 0; i < a.nq; ++i) {
      const double pos = a.probs[i] * (n - 1.0);
      const double lo = floor(pos);
      const double fr = pos - lo;
      S.k[2 * i] = (uint64_t)lo;
      S.k[2 * i + 1] = (uint64_t)(fr > 0.0 ? lo + 1.0 : lo);
      S.pop[2 * i] = S.pop[2 * i + 1] = 0xffffffffu;
    }
  }
}

// resolve the histogram of `level` (summed over ranks) into the state: warp w handles statistic w.
// rbits[r] = key bits resolved when statistic r became final (pop <= kGsEmit, or all 64 bits).
__device__ void resolve_level(const GsArgs &a, GsRow &S, const unsigned int *hist, int level) {
  uint8_t *rbits = S.rbits;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nr = 2 * a.nq;
  if (warp < nr && rbits[warp] == 0) {
    const unsigned int *h = level == 0 ? hist : hist + (int)S.slotOf[warp] * 256;
    const int per = bins_of(level) / 32;
    unsigned long long mine = 0;
    for (int b = 0; b < per; ++b) mine += h[lane * per + b];
    unsigned long long incl = mine;
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    const unsigned long long k = S.k[warp];
    const unsigned owner = __ballot_sync(0xffffffffu, incl > k);
    const int who = __ffs(owner) - 1;  // first lane whose inclusive count exceeds k (exists: k < population)
    __syncwarp();  // every lane has read S.k[warp] before lane `who` overwrites it (the branch above is warp-uniform)
    if (lane == who) {
      unsigned long long acc = incl - mine;
      int bin = lane * per;
      for (; bin < lane * per + per - 1; ++bin) {
        const unsigned long long cnt = h[bin];
        if (acc + cnt > k) break;
        acc += cnt;
      }
      S.prefix[warp] |= (uint64_t)bin << shift_of(level);
      S.k[warp] = k - acc;
      S.pop[warp] = h[bin];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    S.bits = (uint8_t)bits_after(level);
    int ns = 0;
    bool done = true;
    for (int r = 0; r < nr; ++r) {
      if (rbits[r] == 0 && (S.pop[r] <= (uint32_t)kGsEmit || S.bits == 64)) rbits[r] = S.bits;
      if (rbits[r] != 0) {
        S.slotOf[r] = 0xff;
        continue;
      }
      done = false;
      // Precondition: the probabilities ascend, so a statistic's rank only steps back to a rank listed before it
      // (hi_i = lo_i + 1 > lo_{i+1} = lo_i).  An open statistic shares the slot of an earlier open one with the
      // same prefix, adjacent or not: two slots with one prefix would leave the first one's histogram empty.
      int e = 0;
      while (e < r && (rbits[e] != 0 || S.prefix[e] != S.prefix[r])) ++e;
      S.slotOf[r] = e < r ? S.slotOf[e] : (uint8_t)ns++;
    }
    S.nslots = (uint8_t)ns;
    S.done = done ? 1 : 0;
  }
  __syncthreads();
}


// ---- level l >= 1: resolve level l-1, then (rows still undecided) histogram the next key bits -------------------
template <bool HI32>
__global__ void __launch_bounds__(kThreads, 2) gs_level_kernel(const GsArgs a, const int level) {
  __shared__ unsigned int hist[kGsHistWords];
  __shared__ double red[kThreads];
  __shared__ GsRow S;
  __shared__ uint64_t slotTop[kGsMaxStat];
  __shared__ unsigned long long tieRep[kGsMaxStat];
  __shared__ unsigned int tieLo[kGsMaxStat], tieHi[kGsMaxStat];
  __shared__ uint64_t xTop[kGsMaxStat];  // the compacting pass: bins of the statistics waiting for the emit
  __shared__ int xSh[kGsMaxStat], nx;
  __shared__ unsigned int listFill;
  const int tid = threadIdx.x;
  const RowRef r = row_ref(a);
  const int64_t rows = gridDim.x;
  if (level == 1) {
    if (tid == 0) init_state(a, r.row, rows, S);
  } else {
    if (a.state[r.row].done != 0) return;  // decided at an earlier level (block-uniform)
    if (tid == 0) S = a.state[r.row];
  }
  __syncthreads();
  if (S.done == 0) {
    if (level >= 2 && tid < 2 * a.nq && S.rbits[tid] == 0) {
      // the previous pass looked at the keys of this statistic's slot on every rank: all equal => that key is it
      const int slot = S.slotOf[tid];
      bool any = false, same = true;
      uint64_t rep = 0;
      for (int q = 0; q < a.nranks; ++q) {
        const GsTie t = a.tieAll[((int64_t)q * rows + r.row) * kGsMaxStat + slot];
        if (t.rep == kGsNoKey) continue;
        if (!any) {
          rep = t.rep;
          any = true;
        }
        if (t.diff != 0 || t.rep != rep) same = false;
      }
      if (any && same) {
        S.prefix[tid] = rep;
        S.rbits[tid] = 64;
      }
    }
    const unsigned int *g = a.hist + r.row * kGsHistWords;
    for (int i = tid; i < kGsHistWords; i += kThreads) hist[i] = g[i];
    __syncthreads();
    resolve_level(a, S, hist, level - 1);
  }
  const bool pass = S.done == 0 && level < kGsLevels;
  const bool needSS = level == 1 && a.wantMoments && S.n > 0;
  if (tid == 0) {
    // compact when the filter -- every slot in play and every bin waiting for the emit, each counted once -- holds
    // at most kGsListCap keys over all ranks (the same decision on every rank: it reads exchanged data only)
    nx = 0;
    listFill = 0;
    if (pass && a.list && S.listed == 0) {
      uint64_t popSum = 0;
      for (int q = 0; q < 2 * a.nq; ++q) {
        bool first = true;
        if (S.rbits[q] == 0) {
          for (int e = 0; e < q; ++e) first = first && !(S.rbits[e] == 0 && S.slotOf[e] == S.slotOf[q]);
          if (first) popSum += S.pop[q];
        } else if (S.rbits[q] < 64) {
          const int shv = 64 - (int)S.rbits[q];
          for (int e = 0; e < nx; ++e) first = first && !(xSh[e] == shv && xTop[e] == S.prefix[q] >> shv);
          if (first) {
            popSum += S.pop[q];
            xTop[nx] = S.prefix[q] >> shv;
            xSh[nx++] = shv;
          }
        }
      }
      if (popSum <= (uint64_t)kGsListCap) S.listed = (uint8_t)level;
    }
    a.state[r.row] = S;
    if (pass) a.flags[0] = 1;
  }
  __syncthreads();  // S.listed
  if (!pass && !needSS) return;

  const int nslots = S.nslots;
  // a row compacted by an earlier level scans its list; the compacting pass (listed == level) reads the row
  const bool fromList = S.listed != 0 && S.listed < level;
  const bool listing = pass && S.listed == level;
  const double *src = fromList ? a.list + r.row * kGsListCap : r.p;
  const int count = fromList ? a.listN[r.row] : r.count;
  double *dstList = a.list + r.row * kGsListCap;
  if (pass) {
    for (int i = tid; i < nslots * 256; i += kThreads) hist[i] = 0;
    if (tid < 2 * a.nq && S.slotOf[tid] != 0xff) slotTop[S.slotOf[tid]] = S.prefix[tid] >> shift_of(level - 1);
    if (tid < kGsMaxStat) {
      tieRep[tid] = kGsNoKey;
      tieLo[tid] = tieHi[tid] = 0;
    }
  }
  __syncthreads();
  const int sh0 = shift_of(level - 1), sh1 = shift_of(level), bmask = bins_of(level) - 1;
  const double mu = S.mean;
  double q2 = 0.0;
  // the slots' resolved prefixes in registers (compared with every element); unused slots never match.  HI32 (levels
  // 1 and 2): the resolved bits AND the next 8 all sit in the key's high word -- 32-bit compares and shifts only.
  uint64_t top[kGsMaxStat];
  unsigned top32[kGsMaxStat];
#pragma unroll
  for (int s = 0; s < kGsMaxStat; ++s) {
    top[s] = (pass && s < nslots) ? slotTop[s] : kGsNoKey;
    top32[s] = (pass && s < nslots) ? (unsigned)slotTop[s] : 0xffffffffu;  // a prefix of <= 19 bits is never all ones
  }
  // "are the slot's keys all equal?" is only worth asking where a slot is still large after the first refinement:
  // a group of equal values (exact zeros) that holds a wanted order statistic
  unsigned trackMask = 0;
  if (pass && level >= 2)
    for (int r2 = 0; r2 < 2 * a.nq; ++r2)
      if (S.slotOf[r2] != 0xff && S.pop[r2] > 1024u) trackMask |= 1u << S.slotOf[r2];
  // The scan of the row, instantiated for the number of slots an element has to be matched against: most rows have one
  // or two bins in play, and eight compare + select pairs per element are most of what the later levels execute.
  const int nxs = nx;
  // LIST: the compacting pass (its own instantiation: the other passes keep the loop without the append)
  const auto scan = [&](auto nsTag, auto listTag) {
  constexpr int NS = decltype(nsTag)::value;
  constexpr bool LIST = decltype(listTag)::value;
  constexpr int UN = HI32 ? kUnrollWide : kUnroll;
  for (int i0 = 0; i0 < count; i0 += UN * kThreads) {
    double x[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int i = i0 + u * kThreads + tid;
      x[u] = i < count ? src[i] : __longlong_as_double(0x7ff8000000000000ll);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      int code = -1;
      bool keep = false;
      if (finite_hi(x[u])) {
        if (needSS) {
          const double d = x[u] - mu;
          q2 += d * d;
        }
        if (pass) {
          int slot = -1;
          int bin;
          if (HI32) {
            const unsigned hi = (unsigned)__double2hiint(x[u]);
            const unsigned khi = hi ^ ((unsigned)((int)hi >> 31) | 0x80000000u);  // high word of key_of(x)
            const unsigned t = khi >> (sh0 - 32);
#pragma unroll
            for (int s = 0; s < NS; ++s)
              if (top32[s] == t) slot = s;
            bin = (int)((khi >> (sh1 - 32)) & (unsigned)bmask);
          } else {
            const uint64_t k = key_of(x[u]);
            const uint64_t t = k >> sh0;
#pragma unroll
            for (int s = 0; s < NS; ++s)
              if (top[s] == t) slot = s;
            bin = (int)((k >> sh1) & (uint64_t)bmask);
          }
          if (LIST) {
            keep = slot >= 0;
            if (nxs > 0) {  // rare: a statistic already waits for the emit while others are open
              const uint64_t k = key_of(x[u]);
              for (int j = 0; j < nxs; ++j) keep = keep || (k >> xSh[j]) == xTop[j];
            }
          }
          if (slot >= 0) {
            code = slot * 256 + bin;
            if ((trackMask >> slot) & 1u) {  // one representative (first come) and the OR of the differences
              const uint64_t k = key_of(x[u]);
              unsigned long long rep = *(volatile unsigned long long *)&tieRep[slot];
              if (rep == kGsNoKey) {
                const unsigned long long old = atomicCAS(&tieRep[slot], (unsigned long long)kGsNoKey, (unsigned long long)k);
                rep = old == kGsNoKey ? k : old;
              }
              const uint64_t d = k ^ rep;
              if (d) {
                const unsigned int lo = (unsigned int)d, hi2 = (unsigned int)(d >> 32);
                if (lo & ~*(volatile unsigned int *)&tieLo[slot]) atomicOr(&tieLo[slot], lo);
                if (hi2 & ~*(volatile unsigned int *)&tieHi[slot]) atomicOr(&tieHi[slot], hi2);
              }
            }
          }
        }
      }
      // (warps in which no lane holds a candidate -- most of them from the second refinement on -- skip the update)
      if (!LIST) {
        if (pass && __any_sync(0xffffffffu, code >= 0)) hist_add(hist, code);
      } else {  // keep >= (code >= 0); one shared atomic per warp, and a warp's keys land side by side in the list
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m) {
          hist_add(hist, code);
          const int lane = tid & 31;
          unsigned base = 0;
          if (lane == 0) base = atomicAdd(&listFill, (unsigned)__popc(m));
          base = __shfl_sync(0xffffffffu, base, 0) + (unsigned)__popc(m & ((1u << lane) - 1u));
          if (keep && base < (unsigned)kGsListCap) dstList[base] = x[u];  // (the global bound keeps base below)
        }
      }
    }
  }
  };
  const auto slots = [&](auto listTag) {
    if (nslots <= 1) scan(std::integral_constant<int, 1>{}, listTag);
    else if (nslots <= 2) scan(std::integral_constant<int, 2>{}, listTag);
    else if (nslots <= 4) scan(std::integral_constant<int, 4>{}, listTag);
    else scan(std::integral_constant<int, kGsMaxStat>{}, listTag);
  };
  if (listing) slots(std::true_type{});
  else slots(std::false_type{});
  if (needSS) {
    const double ss = block_sum(q2, red);
    if (tid == 0) a.q2All[(int64_t)a.rank * rows + r.row] = ss;
  }
  if (pass) {
    __syncthreads();
    if (listing && tid == 0) a.listN[r.row] = (int)min(listFill, (unsigned)kGsListCap);
    unsigned int *g = a.hist + r.row * kGsHistWords;
    for (int i = tid; i < nslots * 256; i += kThreads) g[i] = hist[i];
    if (tid < kGsMaxStat) {
      GsTie t;  // a slot that was not watched reports "not all equal"
      const bool watched = (trackMask >> tid) & 1u;
      t.rep = watched ? tieRep[tid] : 0;
      t.diff = watched ? (((uint64_t)tieHi[tid] << 32) | tieLo[tid]) : ~0ull;
      a.tieAll[((int64_t)a.rank * rows + r.row) * kGsMaxStat + tid] = t;
    }
  }
}

// ---- emit: the local keys of every bin that is finished by gathering ------------------------------------------
__global__ void __launch_bounds__(kThreads, 2) gs_emit_kernel(const GsArgs a) {
  __shared__ GsRow S;
  __shared__ uint64_t top[kGsMaxStat];
  __shared__ int sh[kGsMaxStat];
  __shared__ int owner[kGsMaxStat];  // first statistic with the same (prefix, rbits): its emit slot is shared
  __shared__ unsigned int fill[kGsMaxStat];
  __shared__ int nemit;
  const int tid = threadIdx.x;
  const RowRef r = row_ref(a);
  const int64_t rows = gridDim.x;
  const GsRow *gx = a.state + r.row;
  uint64_t *dst = a.emitAll + ((int64_t)a.rank * rows + r.row) * (kGsMaxStat * kGsEmit);
  for (int i = tid; i < kGsMaxStat * kGsEmit; i += kThreads) dst[i] = kSent;
  if (gx->done != 1 || a.nq == 0) return;
  if (tid == 0) {
    S = *gx;
    int ne = 0;
    for (int s = 0; s < 2 * a.nq; ++s) {
      fill[s] = 0;
      owner[s] = -1;
      if (S.rbits[s] >= 64) continue;  // every bit resolved: the key is the prefix
      const int shv = 64 - (int)S.rbits[s];
      bool shared = false;
      for (int e = 0; e < s; ++e)
        if (owner[e] == e && S.rbits[e] == S.rbits[s] && (S.prefix[e] >> shv) == (S.prefix[s] >> shv)) {
          owner[s] = e;
          shared = true;
          break;
        }
      if (!shared) {
        owner[s] = s;
        ++ne;
      }
      top[s] = S.prefix[s] >> shv;
      sh[s] = shv;
    }
    nemit = ne;
  }
  __syncthreads();
  if (nemit == 0) return;
  const bool fromList = S.listed != 0;  // every emit bin lies inside the filter the list was cut with
  const double *src = fromList ? a.list + r.row * kGsListCap : r.p;
  const int count = fromList ? a.listN[r.row] : r.count;
  // the ACTIVE emit slots in registers, compacted (most rows have one to three): a key belongs to slot at[j] when
  // (key >> shv[j]) == tp[j].  When every slot was resolved within the key's high word (<= 32 bits: the usual case)
  // the test is a 32-bit shift and compare.  The scan is instantiated for the number of active slots.
  uint64_t tp[kGsMaxStat];
  unsigned tp32[kGsMaxStat];
  int shv[kGsMaxStat], at[kGsMaxStat];
  bool hi32 = true;
  {
    int j = 0;
#pragma unroll
    for (int s = 0; s < kGsMaxStat; ++s) {
      tp[s] = kGsNoKey;
      tp32[s] = 0xffffffffu;
      shv[s] = 32;
      at[s] = 0;
    }
#pragma unroll
    for (int s = 0; s < kGsMaxStat; ++s) {
      const bool on = s < 2 * a.nq && owner[s] == s;
      if (on) {
#pragma unroll
        for (int jj = 0; jj < kGsMaxStat; ++jj)
          if (jj == j) {
            tp[jj] = top[s];
            tp32[jj] = (unsigned)top[s];
            shv[jj] = sh[s];
            at[jj] = s;
          }
        if (sh[s] < 32) hi32 = false;
        ++j;
      }
    }
  }
  const auto scan = [&](auto neTag) {
    constexpr int NE = decltype(neTag)::value;
    for (int i0 = 0; i0 < count; i0 += kUnroll * kThreads) {
      double x[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const int i = i0 + u * kThreads + tid;
        x[u] = i < count ? src[i] : __longlong_as_double(0x7ff8000000000000ll);
      }
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        if (!finite_hi(x[u])) continue;
        if (hi32) {  // block-uniform
          const unsigned hi = (unsigned)__double2hiint(x[u]);
          const unsigned khi = hi ^ ((unsigned)((int)hi >> 31) | 0x80000000u);
          int hit = -1;
#pragma unroll
          for (int j = 0; j < NE; ++j)
            if ((khi >> (shv[j] - 32)) == tp32[j]) hit = at[j];  // emit slots hold disjoint key ranges
          if (hit >= 0) {
            const unsigned int pos = atomicAdd(&fill[hit], 1u);
            if (pos < (unsigned)kGsEmit) dst[hit * kGsEmit + pos] = key_of(x[u]);
          }
        } else {
          const uint64_t k = key_of(x[u]);
#pragma unroll
          for (int j = 0; j < NE; ++j) {
            if ((k >> shv[j]) == tp[j]) {
              const unsigned int pos = atomicAdd(&fill[at[j]], 1u);
              if (pos < (unsigned)kGsEmit) dst[at[j] * kGsEmit + pos] = k;
            }
          }
        }
      }
    }
  };
  if (nemit <= 1) scan(std::integral_constant<int, 1>{});
  else if (nemit <= 2) scan(std::integral_constant<int, 2>{});
  else if (nemit <= 4) scan(std::integral_constant<int, 4>{});
  else scan(std::integral_constant<int, kGsMaxStat>{});
}

// ---- finish: order statistics from the gathered keys, quantiles, moments ----------------------------------------
__global__ void gs_finish_kernel(const GsArgs a, const int64_t rows) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const GsRow *gx = a.state + row;
  const int64_t t = row % a.nsteps;
  const int64_t sc = row / a.nsteps;  // site * ncols + col
  const double nanv = __longlong_as_double(0x7ff8000000000000ll);
  const int done = gx->done;
  const int nr = 2 * a.nq;
  uint64_t key = 0;
  if (done == 1 && lane < nr) {
    const int s = lane;
    const int rb = gx->rbits[s];
    if (rb >= 64) {
      key = gx->prefix[s];
    } else {
      const int shv = 64 - rb;
      int e = s;  // emit slot = first statistic with the same (prefix, rbits)
      for (int j = 0; j < s; ++j)
        if (gx->rbits[j] == rb && (gx->prefix[j] >> shv) == (gx->prefix[s] >> shv)) {
          e = j;
          break;
        }
      uint64_t c[kGsEmit];
      int nc = 0;
      for (int q = 0; q < a.nranks; ++q) {  // at most kGsEmit keys over all ranks share the bin
        const uint64_t *src = a.emitAll + (((int64_t)q * rows + row) * kGsMaxStat + e) * kGsEmit;
        for (int i = 0; i < kGsEmit && nc < kGsEmit; ++i) {
          const uint64_t v = src[i];
          if (v == kSent) break;
          int p = nc++;
          while (p > 0 && c[p - 1] > v) {  // insertion into the ascending list
            c[p] = c[p - 1];
            --p;
          }
          c[p] = v;
        }
      }
      const uint64_t kk = gx->k[s];
      key = kk < (uint64_t)nc ? c[kk] : kSent;
    }
  }
  for (int i = 0; i < a.nq; ++i) {
    const uint64_t klo = __shfl_sync(0xffffffffu, key, 2 * i);
    const uint64_t khi = __shfl_sync(0xffffffffu, key, 2 * i + 1);
    if (lane != i) continue;
    double v = nanv;
    if (done == 2) {
      v = val_of(gx->prefix[0]);
    } else if (done == 1) {
      const double n = gx->n;
      const double pos = a.probs[i] * (n - 1.0);
      const double fr = pos - floor(pos);
      const double xlo = val_of(klo), xhi = val_of(khi);
      // numpy's _lerp: a + (b - a) t, evaluated from the b side when t >= 0.5
      v = (fr >= 0.5) ? xhi - (xhi - xlo) * (1.0 - fr) : xlo + (xhi - xlo) * fr;
    }
    a.quant[(sc * a.nqTotal + a.qOut[i]) * a.nsteps + t] = v;
  }
  if (a.wantMoments && lane == 0) {
    const double n = gx->n;
    double ss = 0.0;
    if (n > 0)
      for (int q = 0; q < a.nranks; ++q) ss += a.q2All[(int64_t)q * rows + row];
    a.mean[sc * a.nsteps + t] = gx->mean;
    a.var[sc * a.nsteps + t] = n > 0 ? ss / n : nanv;
  }
}

cudaError_t launch_pass0(const GsArgs &a, cudaStream_t stream) {
  gs_pass0_kernel<<<(unsigned)gs_rows(a), kThreads, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_level(const GsArgs &a, int level, cudaStream_t stream) {
  // levels 1 and 2 resolve key bits 11..26: shift_of(level) >= 32
  if (level <= 2) gs_level_kernel<true><<<(unsigned)gs_rows(a), kThreads, 0, stream>>>(a, level);
  else gs_level_kernel<false><<<(unsigned)gs_rows(a), kThreads, 0, stream>>>(a, level);
  return cudaGetLastError();
}
cudaError_t launch_emit(const GsArgs &a, cudaStream_t stream) {
  gs_emit_kernel<<<(unsigned)gs_rows(a), kThreads, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_finish(const GsArgs &a, cudaStream_t stream) {
  const int64_t rows = gs_rows(a);
  gs_finish_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, stream>>>(a, rows);
  return cudaGetLastError();
}

__global__ void add_u32_kernel(uint32_t *dst, const uint32_t *src, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] += src[i];
}
cudaError_t launch_add_u32(uint32_t *dst, const uint32_t *src, size_t n, cudaStream_t stream) {
  const size_t blocks = std::min<size_t>((n + 255) / 256, 4096);
  add_u32_kernel<<<(unsigned)std::max<size_t>(blocks, 1), 256, 0, stream>>>(dst, src, n);
  return cudaGetLastError();
}

}  // namespace gs
}  // namespace sip
