// sip_resample.cu -- kernels of the per-site systematic particle filter (see sip_resample.cuh for the sequence of
// launches).  Compiled with -fmad=false like the rest of the model path: the weights are the glibc-exact exp of
// sip_libm.cuh and every product below is rounded on its own, so the host reference can restate them bit for bit.
#include <cuda_runtime.h>

#include <algorithm>

#include "sip_math.cuh"
#include "sip_resample.cuh"

namespace sip {
namespace rs {
namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarps = 4;        // warps per CTA; one chunk or one site per warp
constexpr int kWordsPerY = 64;   // record words one pack / unpack thread copies
typedef unsigned __int128 u128;

__device__ __forceinline__ uint64_t shfl_xor(uint64_t v, int off) { return __shfl_xor_sync(kFull, v, off); }

// floor(x 2^kFixBits) for x in [0, 1]: exact (x 2^100 is a double with 53 significant bits, at most 2^100)
__device__ __forceinline__ u128 fixed(double x) {
  const double v = ldexp(x, kFixBits);
  if (!(v >= 1.0)) return 0;
  const uint64_t bits = (uint64_t)__double_as_longlong(v);
  const int e = (int)((bits >> 52) & 0x7ff) - 1075;
  const uint64_t m = (bits & ((uint64_t(1) << 52) - 1)) | (uint64_t(1) << 52);
  return e >= 0 ? (u128)m << e : (u128)(m >> -e);
}

__device__ __forceinline__ bool takes_part(uint32_t st, double l) { return (st & kExcluded) == 0 && isfinite(l); }

// one warp per chunk
template <int PASS>
__global__ void __launch_bounds__(kWarps * 32) weights_kernel(const Args a) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (c >= a.nchunks) return;  // warp-uniform
  const int2 ch = a.chunk[c];
  const int32_t member0 = a.sites[ch.x].member0, count = a.sites[ch.x].memberCount;
  const double lmax = PASS == 1 ? a.lmax[ch.x] : 0.0;
  uint64_t n = 0, inf = 0, T = 0;
  double mx = -INFINITY;
  u128 s1 = 0, s2 = 0;
  for (int i = 0; i < kChunk / 32; ++i) {
    const int idx = ch.y + lane + 32 * i;
    if (idx >= count) break;
    const int64_t m = (int64_t)member0 + idx;
    const double l = a.logw[m];
    const bool in = takes_part(a.status[m], l);
    if (PASS == 0) {
      inf |= (l == INFINITY) ? 1 : 0;
      if (in) {
        ++n;
        mx = fmax(mx, l);
      }
    } else {
      uint64_t W = 0;
      if (in) {
        const double w = sip_exp(l - lmax);
        W = (uint64_t)ldexp(w, kWeightBits);  // exact: a power-of-two scaling
        s1 += fixed(w);
        s2 += fixed(w * w);
      }
      a.w[m] = W;
      T += W;
    }
  }
  uint64_t *p = a.part + (size_t)c * (kRec + 1);
  if (PASS == 0) {
    for (int off = 16; off > 0; off >>= 1) {
      n += shfl_xor(n, off);
      inf |= shfl_xor(inf, off);
      mx = fmax(mx, __shfl_xor_sync(kFull, mx, off));
    }
    if (lane == 0) {
      p[0] = n;
      p[1] = (uint64_t)__double_as_longlong(mx);
      p[3] = inf;
    }
  } else {
    uint64_t v[5] = {(uint64_t)s1, (uint64_t)(s1 >> 64), (uint64_t)s2, (uint64_t)(s2 >> 64), T};
    for (int off = 16; off > 0; off >>= 1) {
      uint64_t o[5];
#pragma unroll
      for (int i = 0; i < 5; ++i) o[i] = shfl_xor(v[i], off);
      const u128 a1 = ((u128)v[1] << 64 | v[0]) + ((u128)o[1] << 64 | o[0]);
      const u128 a2 = ((u128)v[3] << 64 | v[2]) + ((u128)o[3] << 64 | o[2]);
      v[0] = (uint64_t)a1;
      v[1] = (uint64_t)(a1 >> 64);
      v[2] = (uint64_t)a2;
      v[3] = (uint64_t)(a2 >> 64);
      v[4] += o[4];
    }
    if (lane == 0)
#pragma unroll
      for (int i = 0; i < 5; ++i) p[i] = v[i];
  }
}

// One warp per site: its chunks -> this rank's site record; pass b also scans the chunk totals of W.
template <int PASS>
__global__ void __launch_bounds__(kWarps * 32) site_kernel(const Args a) {
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (s >= a.nsites) return;
  const int2 sc = a.siteChunks[s];
  uint64_t *r = a.siteRec + ((size_t)a.rank * a.nsites + s) * kRec;
  if (PASS == 0) {
    uint64_t n = 0, inf = 0;
    double mx = -INFINITY;
    for (int c = lane; c < sc.y; c += 32) {
      const uint64_t *p = a.part + (size_t)(sc.x + c) * (kRec + 1);
      n += p[0];
      mx = fmax(mx, __longlong_as_double((long long)p[1]));
      inf |= p[3];
    }
    for (int off = 16; off > 0; off >>= 1) {
      n += shfl_xor(n, off);
      inf |= shfl_xor(inf, off);
      mx = fmax(mx, __shfl_xor_sync(kFull, mx, off));
    }
    if (lane == 0) {
      r[0] = n;
      r[1] = (uint64_t)__double_as_longlong(mx);
      r[2] = (uint64_t)a.sites[s].memberCount;
      r[3] = inf;
    }
    return;
  }
  u128 s1 = 0, s2 = 0;
  uint64_t carry = 0;
  for (int c0 = 0; c0 < sc.y; c0 += 32) {
    const int c = c0 + lane;
    uint64_t t = 0;
    if (c < sc.y) {
      uint64_t *p = a.part + (size_t)(sc.x + c) * (kRec + 1);
      s1 += (u128)p[1] << 64 | p[0];
      s2 += (u128)p[3] << 64 | p[2];
      t = p[4];
    }
    uint64_t incl = t;  // inclusive scan of the 32 chunk totals
    for (int off = 1; off < 32; off <<= 1) {
      const uint64_t o = __shfl_up_sync(kFull, incl, off);
      if (lane >= off) incl += o;
    }
    if (c < sc.y) a.part[(size_t)(sc.x + c) * (kRec + 1) + kRec] = carry + incl - t;
    carry += __shfl_sync(kFull, incl, 31);
  }
  uint64_t v[4] = {(uint64_t)s1, (uint64_t)(s1 >> 64), (uint64_t)s2, (uint64_t)(s2 >> 64)};
  for (int off = 16; off > 0; off >>= 1) {
    uint64_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = shfl_xor(v[i], off);
    const u128 a1 = ((u128)v[1] << 64 | v[0]) + ((u128)o[1] << 64 | o[0]);
    const u128 a2 = ((u128)v[3] << 64 | v[2]) + ((u128)o[3] << 64 | o[2]);
    v[0] = (uint64_t)a1;
    v[1] = (uint64_t)(a1 >> 64);
    v[2] = (uint64_t)a2;
    v[3] = (uint64_t)(a2 >> 64);
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) r[i] = v[i];
    r[4] = carry;
  }
}

// one warp per chunk of a resampled site: C = toff + chunk offset + exclusive scan of W in member order
__global__ void __launch_bounds__(kWarps * 32) prefix_kernel(const Args a) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (c >= a.nchunks) return;
  const int2 ch = a.chunk[c];
  if (!a.flag[ch.x]) return;
  const int32_t member0 = a.sites[ch.x].member0, count = a.sites[ch.x].memberCount;
  uint64_t carry = (uint64_t)a.toff[ch.x] + a.part[(size_t)c * (kRec + 1) + kRec];
  for (int i = 0; i < kChunk / 32; ++i) {
    const int idx = ch.y + lane + 32 * i;
    const int64_t m = (int64_t)member0 + idx;
    const uint64_t W = idx < count ? a.w[m] : 0;
    uint64_t incl = W;
    for (int off = 1; off < 32; off <<= 1) {
      const uint64_t o = __shfl_up_sync(kFull, incl, off);
      if (lane >= off) incl += o;
    }
    if (idx < count) a.c[m] = carry + incl - W;
    carry += __shfl_sync(kFull, incl, 31);
  }
}

// word `k` of member j's record: read (LOAD) or write
template <bool LOAD>
__device__ __forceinline__ void record_word(const Args &a, int k, int64_t j, double &v) {
  auto io = [&](double *p) {
    if (LOAD) v = *p;
    else *p = v;
  };
  if (k < kNParamDev) return io(a.params + (int64_t)k * a.ld + j);
  k -= kNParamDev;
  if (k < SIPNET_GPU_NSTATE) return io(a.state + (int64_t)k * a.ld + j);
  k -= SIPNET_GPU_NSTATE;
  if (k < a.ringCap) return io(a.ringV + (int64_t)k * a.ld + j);
  k -= a.ringCap;
  if (k < a.ringCap) return io(a.ringW + (int64_t)k * a.ld + j);
  k -= a.ringCap;
  if (k == 0) {  // status (internal per-segment bits cleared) | event count << 32
    if (LOAD) {
      const uint64_t cnt = a.recCount ? (uint32_t)a.recCount[j] : 0u;
      v = __longlong_as_double((long long)((cnt << 32) | (a.status[j] & ~kStNeedsReplay)));
    } else {
      const uint64_t b = (uint64_t)__double_as_longlong(v);
      a.status[j] = (uint32_t)b;
      if (a.recCount) a.recCount[j] = (int32_t)(uint32_t)(b >> 32);
    }
    return;
  }
  k -= 1;
  if (k < (SIPNET_GPU_NCOUNTERS + 1) / 2) {
    if (!a.counters) {
      if (LOAD) v = 0.0;
      return;
    }
    uint32_t *c0 = a.counters + (int64_t)(2 * k) * a.ld + j;
    const bool two = 2 * k + 1 < SIPNET_GPU_NCOUNTERS;
    if (LOAD) {
      const uint64_t hi = two ? c0[a.ld] : 0u;
      v = __longlong_as_double((long long)(hi << 32 | *c0));
    } else {
      const uint64_t b = (uint64_t)__double_as_longlong(v);
      *c0 = (uint32_t)b;
      if (two) c0[a.ld] = (uint32_t)(b >> 32);
    }
    return;
  }
  k -= (SIPNET_GPU_NCOUNTERS + 1) / 2;
  constexpr int kRecWords = (int)(sizeof(sipnet_gpu_event_record) / sizeof(double));
  if (k < a.maxRecs * kRecWords) {
    if (a.recs) io(reinterpret_cast<double *>(a.recs + j * (int64_t)a.maxRecs) + k);
    else if (LOAD) v = 0.0;
    return;
  }
  // the last word (the ancestor's index) is handled by the callers
}

// one thread per outgoing slot (x) and group of record words (y)
__global__ void __launch_bounds__(128) pack_kernel(const Args a) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.nOut) return;
  const int R = a.nranks;
  int lo = 0, hi = a.nsites;  // the site: last s with outPre[s] <= g
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (a.outPre[mid] <= g) lo = mid;
    else hi = mid;
  }
  const int s = lo;
  const int64_t *slot0 = a.slot0 + (size_t)s * (R + 1), *mem0 = a.mem0 + (size_t)s * (R + 1);
  const int64_t k = slot0[a.rank] + (g - a.outPre[s]);
  int q = 0;  // the destination rank: the one that holds slot k
  while (q + 1 < R && mem0[q + 1] <= k) ++q;
  const int64_t pos = a.sendPos[(size_t)s * R + q] + (k - max(slot0[a.rank], mem0[q]));
  // t_k = floor((k 2^32 + U) T / (n 2^32)); its ancestor is the last local member with C <= t_k
  const u128 t = (((u128)k << 32) + (u128)a.U[s]) * (u128)(uint64_t)a.T[s] / ((u128)a.n[s] << 32);
  const int64_t b = a.sites[s].member0;
  int64_t jl = b, jh = b + a.sites[s].memberCount;
  while (jh - jl > 1) {
    const int64_t mid = (jl + jh) >> 1;
    if ((u128)a.c[mid] <= t) jl = mid;
    else jh = mid;
  }
  double *dst = a.sendBuf + a.sendBase[q] + pos;
  const int64_t cnt = a.sendCnt[q];
  const int k0 = blockIdx.y * kWordsPerY, k1 = min(k0 + kWordsPerY, a.words);
  for (int w = k0; w < k1; ++w) {
    double v;
    if (w == a.words - 1) v = __longlong_as_double((long long)(a.idBase + jl));
    else record_word<true>(a, w, jl, v);
    dst[(int64_t)w * cnt] = v;
  }
}

// one thread per member (x) and group of record words (y)
__global__ void __launch_bounds__(128) unpack_kernel(const Args a) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.nmembers) return;
  const int s = a.memberSite[m];
  if (!a.flag[s]) {
    if (blockIdx.y == 0) a.anc[m] = -1;
    return;
  }
  const int R = a.nranks;
  const int64_t *slot0 = a.slot0 + (size_t)s * (R + 1), *mem0 = a.mem0 + (size_t)s * (R + 1);
  const int64_t k = mem0[a.rank] + (m - a.sites[s].member0);
  int p = 0;  // the source rank: the one whose slot range holds k
  while (p + 1 < R && slot0[p + 1] <= k) ++p;
  const int64_t pos = a.recvPos[(size_t)s * R + p] + (k - max(slot0[p], mem0[a.rank]));
  const double *src = a.src[p] + pos;
  const int64_t cnt = a.recvCnt[p];
  const int k0 = blockIdx.y * kWordsPerY, k1 = min(k0 + kWordsPerY, a.words);
  for (int w = k0; w < k1; ++w) {
    double v = src[(int64_t)w * cnt];
    if (w == a.words - 1) a.anc[m] = (int64_t)__double_as_longlong(v);
    else record_word<false>(a, w, m, v);
  }
  if (blockIdx.y == 0 && a.loglik) {
    a.loglik[m] = 0.0;
    a.loglikN[m] = 0.0;
  }
}

unsigned blocks_for(int64_t units, int per) { return (unsigned)std::max<int64_t>((units + per - 1) / per, 1); }

}  // namespace

int record_words(const sipnet_gpu_handle *h) {
  return kNParamDev + SIPNET_GPU_NSTATE + 2 * h->ringCap + 1 + (SIPNET_GPU_NCOUNTERS + 1) / 2 +
         h->maxRecs * (int)(sizeof(sipnet_gpu_event_record) / sizeof(double)) + 1;
}

int ensure_scratch(sipnet_gpu_handle *h) {
  if (int rc = ensure_chunks(h)) return rc;
  if (h->rsW) return 0;
  const size_t ld = (size_t)h->ld, S = (size_t)h->nsites, nc = (size_t)std::max<int64_t>(h->nchunks, 1);
  cudaError_t e = cudaMalloc((void **)&h->rsW, ld * sizeof(uint64_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->rsPart, nc * (kRec + 1) * sizeof(uint64_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->rsC, ld * sizeof(uint64_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->rsLogw, ld * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->rsAnc, ld * sizeof(int64_t));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->rsLmax, S * sizeof(double));
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "resampling scratch: %s", cudaGetErrorString(e));
  return 0;
}

cudaError_t launch_weights(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nchunks, kWarps);
  if (pass == 0) weights_kernel<0><<<g, kWarps * 32, 0, stream>>>(a);
  else weights_kernel<1><<<g, kWarps * 32, 0, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_site(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nsites, kWarps);
  if (pass == 0) site_kernel<0><<<g, kWarps * 32, 0, stream>>>(a);
  else site_kernel<1><<<g, kWarps * 32, 0, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_prefix(const Args &a, cudaStream_t stream) {
  prefix_kernel<<<blocks_for(a.nchunks, kWarps), kWarps * 32, 0, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_pack(const Args &a, cudaStream_t stream) {
  const dim3 g(blocks_for(a.nOut, 128), (unsigned)((a.words + kWordsPerY - 1) / kWordsPerY));
  pack_kernel<<<g, 128, 0, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_unpack(const Args &a, cudaStream_t stream) {
  const dim3 g(blocks_for(a.nmembers, 128), (unsigned)((a.words + kWordsPerY - 1) / kWordsPerY));
  unpack_kernel<<<g, 128, 0, stream>>>(a);
  return cudaGetLastError();
}

}  // namespace rs
}  // namespace sip
