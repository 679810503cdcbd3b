// sip_jitter.cu -- kernels of the Liu-West parameter move and of the Metropolis-Hastings proposal (see sip_jitter.cuh for the sequence of launches and the
// reduction order).  Compiled with -fmad=false like the rest of the model path: every product and sum below is rounded
// on its own, and the re-derivation of the dependent rows is setupModel()'s own (sip_derive.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>

#include "sip_derive.cuh"
#include "sip_jitter.cuh"

namespace sip {
namespace jt {
namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarps = 2;       // warps per CTA of the members kernel, one chunk per warp
constexpr int kSiteThreads = 128;  // threads per site (site and combine kernels), one quantity per thread

__device__ __forceinline__ bool in_domain(double t, int tf, double lo, double hi) {
  if (!isfinite(t)) return false;
  if (tf == SIPNET_GPU_TF_LOG) return t > 0.0;
  if (tf == SIPNET_GPU_TF_LOGIT) return t > lo && t < hi;
  return true;
}

__device__ __forceinline__ double forward(double t, int tf, double lo, double hi) {
  if (tf == SIPNET_GPU_TF_LOG) return log(t);
  if (tf == SIPNET_GPU_TF_LOGIT) return log((t - lo) / (hi - t));
  return t;
}

__device__ __forceinline__ double inverse(double p, int tf, double lo, double hi) {
  if (tf == SIPNET_GPU_TF_LOG) return exp(p);
  if (tf == SIPNET_GPU_TF_LOGIT) return lo + (hi - lo) / (1.0 + exp(-p));
  return p;
}

// log density of row j's prior in phi at theta = t, phi = p, constants dropped (include/sipnet_gpu.h mh_move)
__device__ __forceinline__ double log_prior(const Args &a, int j, double t, double p) {
  if (a.prior[j] == SIPNET_GPU_PRIOR_NORMAL) {
    const double d = p - a.priorA[j];
    return -(d * d) / (2.0 * (a.priorB[j] * a.priorB[j]));
  }
  if (!(t >= a.priorA[j] && t <= a.priorB[j])) return -INFINITY;
  if (a.transform[j] == SIPNET_GPU_TF_LOG) return p;  // log |dtheta / dphi|
  if (a.transform[j] == SIPNET_GPU_TF_LOGIT) return log((t - a.lower[j]) * (a.upper[j] - t) / (a.upper[j] - a.lower[j]));
  return 0.0;
}

// member m's transformed rows; false when it does not take part (the MH move also needs a finite current
// log-likelihood and log prior)
__device__ __forceinline__ bool load_phi(const Args &a, int64_t m, double (&phi)[kMaxRows]) {
  bool in = (a.status[m] & kExcluded) == 0;
#pragma unroll
  for (int j = 0; j < kMaxRows; ++j)
    if (j < a.nrows) {
      const double t = a.params[(int64_t)a.rows[j] * a.ld + m];
      in = in && in_domain(t, a.transform[j], a.lower[j], a.upper[j]);
      phi[j] = in ? forward(t, a.transform[j], a.lower[j], a.upper[j]) : 0.0;
      if (a.scale) in = in && log_prior(a, j, t, phi[j]) > -INFINITY;
    }
  if (a.scale) in = in && isfinite(a.curLoglik[m]);
  return in;
}

// the move's (a, h) at site s: Liu-West (a = shrink, h = sqrt(1 - a^2)) or Metropolis-Hastings (a = 1, h = scale);
// h NaN: the site stays
__device__ __forceinline__ double2 move_ah(const Args &a, int s) {
  if (a.scale) return make_double2(1.0, a.scale[s]);
  const double sa = a.shrink[s];
  return make_double2(sa, sqrt(1.0 - sa * sa));
}

// the quantities of a pass inside a record: [q0, q0 + count)
__device__ __forceinline__ int2 quantities(int pass, int nrows) {
  if (pass == 1) return make_int2(0, 1 + nrows);
  if (pass == 2) return make_int2(kSum0, nrows * (nrows + 1) / 2);
  return make_int2(0, 2);
}

// One warp per chunk.  Passes 1 and 2 stage the chunk's (centred) phi in shared memory, zero for members that do not
// take part; lane q then sums quantity q over the chunk's members in index order.
template <int PASS>
__global__ void __launch_bounds__(kWarps * 32) members_kernel(const Args a) {
  __shared__ double sh[kWarps][kMaxRows][kChunk];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * kWarps + w;
  if (c >= a.nchunks) return;  // warp-uniform
  const int2 ch = a.chunk[c];
  const int32_t member0 = a.sites[ch.x].member0;
  const int cnt = min(kChunk, a.sites[ch.x].memberCount - ch.y);
  const int n = a.nrows;
  if (PASS == 3) {
    const double *cf = a.coef + (size_t)ch.x * kCoef;
    const bool mh = a.scale != nullptr;
    if (cf[0] == 0.0) {  // the site does not move
      if (mh)
        for (int i = lane; i < cnt; i += 32) a.valid[(int64_t)member0 + ch.y + i] = kMhNone;
      if (lane == 0) a.part[(size_t)c * kRec] = a.part[(size_t)c * kRec + 1] = 0.0;
      return;
    }
    const double sa = cf[1];
    int moved = 0, kept = 0;
    for (int i = lane; i < cnt; i += 32) {
      const int64_t m = (int64_t)member0 + ch.y + i;
      double phi[kMaxRows], zz[kMaxRows], th[kMaxRows];
      if (!load_phi(a, m, phi)) {
        if (mh) a.valid[m] = kMhNone;
        continue;
      }
      bool ok = true;
      double dl = 0.0;  // MH: sum_j lp_j(phi') - lp_j(phi)
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) zz[j] = a.z[(int64_t)j * a.nmembers + m];
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) {
          double s = 0.0;
#pragma unroll
          for (int l = 0; l <= j; ++l) s = s + cf[3 + kMaxRows + tri(j, l)] * zz[l];
          const double p = (sa * phi[j] + cf[3 + j]) + s;
          th[j] = inverse(p, a.transform[j], a.lower[j], a.upper[j]);
          ok = ok && in_domain(th[j], a.transform[j], a.lower[j], a.upper[j]);
          if (mh && ok) {
            const double l1 = log_prior(a, j, th[j], p);
            ok = l1 > -INFINITY;
            dl += l1 - log_prior(a, j, a.params[(int64_t)a.rows[j] * a.ld + m], phi[j]);
          }
        }
      auto P = [&](int k) -> double & { return a.params[(int64_t)k * a.ld + m]; };
      if (ok) {  // ensureAllocation on the proposed fractions, before anything is written
        double al[3] = {P(SIPNET_P_leafAllocation), P(SIPNET_P_woodAllocation), P(SIPNET_P_fineRootAllocation)};
        const int arow[3] = {SIPNET_P_leafAllocation, SIPNET_P_woodAllocation, SIPNET_P_fineRootAllocation};
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n)
            for (int q = 0; q < 3; ++q)
              if (a.rows[j] == arow[q]) al[q] = th[j];
        ok = !allocation_fails(al[0], al[1], al[2], 1 - al[0] - al[1] - al[2]);
      }
      if (!ok) {
        ++kept;
        if (mh) a.valid[m] = kMhInvalid;
        continue;
      }
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) P(a.rows[j]) = th[j];
      derive_dependent(P);
      ++moved;
      if (mh) {
        a.valid[m] = kMhValid;
        a.dlp[m] = dl;
      }
    }
    moved = __reduce_add_sync(kFull, moved);
    kept = __reduce_add_sync(kFull, kept);
    if (lane == 0) {
      a.part[(size_t)c * kRec] = (double)moved;
      a.part[(size_t)c * kRec + 1] = (double)kept;
    }
    return;
  }
  const double *mu = a.mom + (size_t)ch.x * kRec;
  int N = 0;
  for (int i = lane; i < kChunk; i += 32) {
    double phi[kMaxRows];
    bool in = false;
    if (i < cnt) in = load_phi(a, (int64_t)member0 + ch.y + i, phi);
    N += __popc(__ballot_sync(kFull, in));
#pragma unroll
    for (int j = 0; j < kMaxRows; ++j)
      if (j < n) sh[w][j][i] = !in ? 0.0 : PASS == 1 ? phi[j] : phi[j] - mu[1 + j];
  }
  __syncwarp();
  double *p = a.part + (size_t)c * kRec;
  if (PASS == 1) {
    if (lane == 0) p[0] = (double)N;
    if (lane < n) {
      double s = 0.0;
      for (int i = 0; i < cnt; ++i) s += sh[w][lane][i];
      p[1 + lane] = s;
    }
  } else {
    const int np = n * (n + 1) / 2;
    for (int q = lane; q < np; q += 32) {
      int j = 0;
      while (tri(j + 1, 0) <= q) ++j;
      const int l = q - tri(j, 0);
      double s = 0.0;
      for (int i = 0; i < cnt; ++i) s += sh[w][j][i] * sh[w][l][i];
      p[kSum0 + q] = s;
    }
  }
}

// pass `PASS` is complete for site s: `r` holds the site's sums over every rank (only the pass's quantities are set)
template <int PASS>
__device__ void finish(const Args &a, int s, const double *r) {
  double *mom = a.mom + (size_t)s * kRec;
  double *dg = a.diag + (size_t)s * 4;
  double *cf = a.coef + (size_t)s * kCoef;
  const int n = a.nrows;
  if (PASS == 1) {
    const double N = r[0];
    mom[0] = N;
    for (int j = 0; j < n; ++j) mom[1 + j] = N > 0.0 ? r[1 + j] / N : 0.0;
    dg[0] = N;
    dg[1] = -1.0;
    dg[2] = dg[3] = 0.0;
    return;
  }
  if (PASS == 3) {
    if (cf[0] != 0.0) {
      dg[2] = r[0];
      dg[3] = r[1];
    }
    return;
  }
  const double N = mom[0];
  const double2 ah = move_ah(a, s);
  cf[0] = 0.0;
  if (isnan(ah.y) || N < 2.0) return;
  // V (population covariance) and its semidefinite Cholesky factor, column by column
  double L[kTri];
  int rank = 0;
  for (int j = 0; j < n; ++j) {
    const double vjj = r[kSum0 + tri(j, j)] / N;
    double acc = 0.0;
    for (int m = 0; m < j; ++m) acc += L[tri(j, m)] * L[tri(j, m)];
    const double d = vjj - acc, mu = mom[1 + j];
    // a row whose spread is below 2^-40 of its mean is constant: its variance is the rounding of the mean, which
    // a summation of up to 2^23 members keeps below about 2^-42 |mean|, whatever the site's size or split
    if (d > 0x1p-40 * vjj && vjj > 0x1p-80 * (mu * mu)) {
      const double ljj = sqrt(d);
      L[tri(j, j)] = ljj;
      for (int i = j + 1; i < n; ++i) {
        double acc2 = 0.0;
        for (int m = 0; m < j; ++m) acc2 += L[tri(i, m)] * L[tri(j, m)];
        L[tri(i, j)] = (r[kSum0 + tri(i, j)] / N - acc2) / ljj;
      }
      ++rank;
    } else {
      for (int i = j; i < n; ++i) L[tri(i, j)] = 0.0;
    }
  }
  const double sa = ah.x, h = ah.y;
  cf[0] = 1.0;
  cf[1] = sa;
  cf[2] = (double)rank;
  for (int j = 0; j < n; ++j) {
    cf[3 + j] = (1.0 - sa) * mom[1 + j];
    for (int m = 0; m <= j; ++m) cf[3 + kMaxRows + tri(j, m)] = h * L[tri(j, m)];
  }
  dg[1] = (double)rank;
}

// One CTA per site: thread t sums quantity q0 + t over the site's chunks in chunk order.
template <int PASS>
__global__ void __launch_bounds__(kSiteThreads) site_kernel(const Args a) {
  __shared__ double r[kRec];
  const int s = blockIdx.x;
  const int2 sc = a.siteChunks[s];
  const int2 qs = quantities(PASS, a.nrows);
  for (int t = threadIdx.x; t < qs.y; t += kSiteThreads) {
    double acc = 0.0;
    for (int c = 0; c < sc.y; ++c) acc += a.part[(size_t)(sc.x + c) * kRec + qs.x + t];
    if (a.nranks == 1)
      r[qs.x + t] = acc;
    else
      a.rankRec[((size_t)a.rank * a.nsites + s) * kRec + qs.x + t] = acc;
  }
  if (a.nranks != 1) return;
  __syncthreads();
  if (threadIdx.x == 0) finish<PASS>(a, s, r);
}

// One CTA per site: rank 0's partial, then the others in rank order (identical on every rank).
template <int PASS>
__global__ void __launch_bounds__(kSiteThreads) combine_kernel(const Args a) {
  __shared__ double r[kRec];
  const int s = blockIdx.x;
  const int2 qs = quantities(PASS, a.nrows);
  for (int t = threadIdx.x; t < qs.y; t += kSiteThreads) {
    double acc = a.rankRec[(size_t)s * kRec + qs.x + t];
    for (int q = 1; q < a.nranks; ++q) acc += a.rankRec[((size_t)q * a.nsites + s) * kRec + qs.x + t];
    r[qs.x + t] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) finish<PASS>(a, s, r);
}

}  // namespace

int ensure_scratch(sipnet_gpu_handle *h) {
  if (int rc = ensure_chunks(h)) return rc;
  if (h->jtPart) return 0;
  const size_t S = (size_t)h->nsites, nc = (size_t)std::max<int64_t>(h->nchunks, 1);
  cudaError_t e = cudaMalloc((void **)&h->jtPart, nc * kRec * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->jtMom, S * kRec * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->jtCoef, S * kCoef * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->jtDiag, S * 4 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->jtShrink, S * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc((void **)&h->jtZ, (size_t)kMaxRows * h->nmembers * sizeof(double));
  if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "rejuvenation scratch: %s", cudaGetErrorString(e));
  return 0;
}

cudaError_t launch_members(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = (unsigned)std::max((a.nchunks + kWarps - 1) / kWarps, 1);
  if (pass == 1) {
    members_kernel<1><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 2) {
    members_kernel<2><<<g, kWarps * 32, 0, stream>>>(a);
  } else {
    members_kernel<3><<<g, kWarps * 32, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_site(const Args &a, int pass, cudaStream_t stream) {
  if (pass == 1) {
    site_kernel<1><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  } else if (pass == 2) {
    site_kernel<2><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  } else {
    site_kernel<3><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_combine(const Args &a, int pass, cudaStream_t stream) {
  if (pass == 1) {
    combine_kernel<1><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  } else if (pass == 2) {
    combine_kernel<2><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  } else {
    combine_kernel<3><<<a.nsites, kSiteThreads, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace jt
}  // namespace sip
