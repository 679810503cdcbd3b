// sip_assim.cu -- kernels of the ensemble adjustment Kalman filter (see sip_assim.cuh for the sequence of launches
// and the reduction order).  Compiled with -fmad=false like the rest of the model path: every product and sum below
// is rounded on its own, so the host reference can restate it.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>

#include "sip_assim.cuh"

namespace sip {
namespace as {
namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarps = 4;  // warps per CTA; one chunk (members kernel) or one site (site kernels) per warp

__device__ __forceinline__ bool finite(double x) { return isfinite(x); }

// the fixed tree: after it every lane holds the same sum of the 32 lane values
__device__ __forceinline__ void warp_sum(double (&v)[kRec]) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
#pragma unroll
    for (int i = 0; i < kRec; ++i) v[i] += __shfl_xor_sync(kFull, v[i], off);
}

// observation k's pass is complete for site s: `r` is the site's pass sum over every rank
template <int PASS>
__device__ void finish(const Args &a, int s, const double (&r)[kRec]) {
  double *mom = a.mom + (size_t)s * kRec;
  double *dg = a.diag + ((size_t)s * a.nobs + a.k) * 4;
  if (PASS == 1) {
    const double n = r[0];
    mom[0] = n;
    mom[1] = r[1] / n;
#pragma unroll
    for (int j = 0; j < kMaxRows; ++j)
      if (j < a.nrows) mom[2 + j] = r[2 + j] / n;
    dg[0] = n;
    return;
  }
  const double n = mom[0], ybar = mom[1];
  const double yo = a.value[(size_t)s * a.nobs + a.k], rv = a.variance[(size_t)s * a.nobs + a.k];
  const double syy = r[0];
  double *cf = a.coef + (size_t)s * kRec;
  const int before = (int)cf[0] & 2;
  if (!isnan(yo) && n >= 2.0 && syy != 0.0 && finite(syy)) {
    const double s2 = syy / (n - 1.0);
    const double ya = ybar + s2 / (s2 + rv) * (yo - ybar);
    const double alpha = sqrt(rv / (s2 + rv));
    cf[0] = 3.0;
    cf[1] = ya - ybar;
    cf[2] = alpha - 1.0;
    cf[3] = ybar;
#pragma unroll
    for (int j = 0; j < kMaxRows; ++j)
      if (j < a.nrows) cf[4 + j] = r[1 + j] / syy;
    dg[1] = ybar;
    dg[2] = s2;
    dg[3] = ya;
  } else {
    cf[0] = (double)before;
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    dg[1] = dg[2] = dg[3] = nanv;
  }
}

// One warp per chunk.  A member takes part iff its status has neither excluded bit and all its rows are finite;
// others are neither read into the sums nor written.
template <int PASS, bool APPLY, bool FLOOR>
__global__ void __launch_bounds__(kWarps * 32) members_kernel(const Args a) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (c >= a.nchunks) return;  // warp-uniform
  const int2 ch = a.chunk[c];
  const int32_t member0 = a.sites[ch.x].member0, count = a.sites[ch.x].memberCount;
  const int n = a.nrows;
  double cf[4 + kMaxRows];  // coefficients of observation k - 1
  int cflags = 0;
  if (APPLY) {
    const double *p = a.coef + (size_t)ch.x * kRec;
    cflags = (int)p[0];
#pragma unroll
    for (int i = 0; i < 4 + kMaxRows; ++i) cf[i] = p[i];
  }
  double mu[2 + kMaxRows];  // pass 2: means of observation k
  if (PASS == 2) {
    const double *p = a.mom + (size_t)ch.x * kRec;
#pragma unroll
    for (int i = 0; i < 2 + kMaxRows; ++i) mu[i] = p[i];
  }
  double acc[kRec];
#pragma unroll
  for (int i = 0; i < kRec; ++i) acc[i] = 0.0;

  for (int i = 0; i < kChunk / 32; ++i) {
    const int idx = ch.y + lane + 32 * i;
    if (idx >= count) break;
    const int64_t m = (int64_t)member0 + idx;
    uint32_t st = a.status[m];
    bool in = (st & kExcluded) == 0;
    double x[kMaxRows];
#pragma unroll
    for (int j = 0; j < kMaxRows; ++j)
      if (j < n) {
        x[j] = a.state[(int64_t)a.rows[j] * a.ld + m];
        in = in && finite(x[j]);
      }
    if (!in) continue;
    if (APPLY) {
      bool write = false;
      if (cflags & 1) {
        double y = 0.0;
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n) y = y + a.opPrev[j] * x[j];
        const double dy = cf[1] + cf[2] * (y - cf[3]);
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n) x[j] = x[j] + cf[4 + j] * dy;
        write = true;
      }
      if (FLOOR && (cflags & 2)) {
        bool floored = false;
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n && x[j] < 0.0) {
            x[j] = 0.0;
            floored = true;
          }
        if (floored) a.status[m] = st | SIPNET_GPU_ST_ANALYSIS_FLOORED;
        write = write || floored;
      }
      if (write)
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n) a.state[(int64_t)a.rows[j] * a.ld + m] = x[j];
    }
    if (PASS != 0) {
      double y = 0.0;
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) y = y + a.opCur[j] * x[j];
      if (PASS == 1) {
        acc[0] += 1.0;
        acc[1] += y;
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n) acc[2 + j] += x[j];
      } else {
        const double dy = y - mu[1];
        acc[0] += dy * dy;
#pragma unroll
        for (int j = 0; j < kMaxRows; ++j)
          if (j < n) acc[1 + j] += (x[j] - mu[2 + j]) * dy;
      }
    }
  }
  if (PASS == 0) return;
  warp_sum(acc);
  if (lane == 0) {
    double *p = a.part + (size_t)c * kRec;
#pragma unroll
    for (int i = 0; i < kRec; ++i) p[i] = acc[i];
  }
}

// One warp per site: its chunks in the fixed order.
template <int PASS>
__global__ void __launch_bounds__(kWarps * 32) site_reduce_kernel(const Args a) {
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (s >= a.nsites) return;
  const int2 sc = a.siteChunks[s];
  double acc[kRec];
#pragma unroll
  for (int i = 0; i < kRec; ++i) acc[i] = 0.0;
  for (int c = lane; c < sc.y; c += 32) {
    const double *p = a.part + (size_t)(sc.x + c) * kRec;
#pragma unroll
    for (int i = 0; i < kRec; ++i) acc[i] += p[i];
  }
  warp_sum(acc);
  if (lane != 0) return;
  if (a.nranks == 1) {
    finish<PASS>(a, s, acc);
  } else {
    double *p = a.rankRec + ((size_t)a.rank * a.nsites + s) * kRec;
#pragma unroll
    for (int i = 0; i < kRec; ++i) p[i] = acc[i];
  }
}

// One thread per site: rank 0's partial, then the others in rank order (identical on every rank).
template <int PASS>
__global__ void site_combine_kernel(const Args a) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.nsites) return;
  double r[kRec];
#pragma unroll
  for (int i = 0; i < kRec; ++i) r[i] = a.rankRec[(size_t)s * kRec + i];
  for (int q = 1; q < a.nranks; ++q) {
    const double *p = a.rankRec + ((size_t)q * a.nsites + s) * kRec;
#pragma unroll
    for (int i = 0; i < kRec; ++i) r[i] += p[i];
  }
  finish<PASS>(a, s, r);
}

unsigned blocks_for(int64_t units, int per) { return (unsigned)std::max<int64_t>((units + per - 1) / per, 1); }

}  // namespace

int ensure_scratch(sipnet_gpu_handle *h, int nobs) {
  if (int rc = ensure_chunks(h)) return rc;
  const size_t S = (size_t)h->nsites;
  if (!h->asPart) {
    cudaError_t e = cudaMalloc((void **)&h->asPart, (size_t)std::max<int64_t>(h->nchunks, 1) * kRec * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void **)&h->asMom, S * kRec * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void **)&h->asCoef, S * kRec * sizeof(double));
    if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "assimilation scratch: %s", cudaGetErrorString(e));
  }
  if (nobs > h->asObsCap) {
    cudaFree(h->asObs);
    cudaFree(h->asDiag);
    h->asObs = h->asDiag = nullptr;
    h->asObsCap = 0;
    cudaError_t e = cudaMalloc((void **)&h->asObs, 2 * S * (size_t)nobs * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void **)&h->asDiag, 4 * S * (size_t)nobs * sizeof(double));
    if (e != cudaSuccess) return fail(SIPNET_GPU_ERR_NO_DEVICE, "assimilation scratch: %s", cudaGetErrorString(e));
    h->asObsCap = nobs;
  }
  return 0;
}

cudaError_t launch_members(const Args &a, int pass, bool apply, bool floor, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nchunks, kWarps);
  if (pass == 1 && !apply && !floor) {
    members_kernel<1, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 1 && apply && !floor) {
    members_kernel<1, true, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 2 && !apply && !floor) {
    members_kernel<2, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 0 && apply && floor) {
    members_kernel<0, true, true><<<g, kWarps * 32, 0, stream>>>(a);
  } else {
    return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_site_reduce(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nsites, kWarps);
  if (pass == 1) {
    site_reduce_kernel<1><<<g, kWarps * 32, 0, stream>>>(a);
  } else {
    site_reduce_kernel<2><<<g, kWarps * 32, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_site_combine(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nsites, 128);
  if (pass == 1) {
    site_combine_kernel<1><<<g, 128, 0, stream>>>(a);
  } else {
    site_combine_kernel<2><<<g, 128, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace as
}  // namespace sip
