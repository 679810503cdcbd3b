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

// the log posterior g(l) of include/sipnet_gpu.h, and its derivative's numerator P(l) = -2 v w^2 g'(l), w = l sp2 + r
struct Posterior {
  double lp, v, sp2, r, d2;
  __device__ double g(double l) const {
    const double w = l * sp2 + r;
    return -((l - lp) * (l - lp)) / (2.0 * v) - 0.5 * log(w) - d2 / (2.0 * w);
  }
  __device__ double P(double l) const {
    const double w = l * sp2 + r;
    return 2.0 * (l - lp) * w * w + v * sp2 * (w - d2);
  }
};

// Anderson's adaptive update of f = {λ0, λ, σ} from one applied observation (include/sipnet_gpu.h).  P is a cubic
// with a positive leading term; the roots of P' cut [lo, hi] into pieces on which P is monotone, and each piece whose
// ends differ in sign holds one root, found by bisection to adjacent doubles.  Candidates in increasing order, a later
// one kept only when g is strictly larger: a tie takes the smaller λ.
__device__ void adapt(double *f, double s2, double d, double rv, double lo, double hi, double sdMin) {
  const double sd = f[2];
  const Posterior q = {f[1], sd * sd, s2 / f[0], rv, d * d};
  // P'(l) = A l^2 + B l + C
  const double a2 = q.sp2 * q.sp2;
  const double A = 6.0 * a2, B = 2.0 * (4.0 * q.sp2 * q.r - 2.0 * a2 * q.lp),
               C = 2.0 * q.r * q.r - 4.0 * q.sp2 * q.r * q.lp + q.v * a2;
  double c0 = lo, c1 = lo;  // the roots of P', clamped into [lo, hi]
  const double disc = B * B - 4.0 * A * C;
  if (disc > 0.0) {
    const double t = -0.5 * (B + copysign(sqrt(disc), B));
    const double u0 = t / A, u1 = t != 0.0 ? C / t : u0;
    c0 = fmin(fmax(fmin(u0, u1), lo), hi);
    c1 = fmin(fmax(fmax(u0, u1), lo), hi);
  }
  const double cut[4] = {lo, c0, c1, hi};
  double best = lo, gbest = q.g(lo);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double x0 = cut[i], x1 = cut[i + 1];
    double p0 = q.P(x0);
    const double p1 = q.P(x1);
    if (!((p0 < 0.0 && p1 > 0.0) || (p0 > 0.0 && p1 < 0.0))) continue;
    for (int it = 0; it < 2100; ++it) {  // enough halvings to reach adjacent doubles from any finite interval
      const double m = 0.5 * (x0 + x1);
      if (!(m > x0 && m < x1)) break;
      const double pm = q.P(m);
      if (pm == 0.0) {
        x0 = x1 = m;
        break;
      }
      if ((pm < 0.0) == (p0 < 0.0)) {
        x0 = m;
        p0 = pm;
      } else {
        x1 = m;
      }
    }
    const double gx = q.g(x0);
    if (gx > gbest) {
      best = x0;
      gbest = gx;
    }
  }
  if (q.g(hi) > gbest) {
    best = hi;
    gbest = q.g(hi);
  }
  const double D = gbest - q.g(best + sd);
  double sdNew = sd;
  if (D > 0.0 && finite(D)) sdNew = fmin(sd, sqrt(q.v / (2.0 * D)));
  f[1] = best;
  f[2] = fmax(sdMin, sdNew);
}

// observation k's pass is complete for site s: `r` is the site's pass sum over every rank
template <int PASS>
__device__ void finish(const Args &a, int s, const double (&r)[kRec]) {
  double *mom = a.mom + (size_t)s * kRec;
  double *dg = a.diag + ((size_t)s * a.nobs + a.k) * 4;
  if (PASS == kInflPass) {
    const double n = r[0], l0 = a.infl[(size_t)s * 3];
    const bool on = finite(l0) && l0 != 1.0 && n >= 2.0;
    mom[0] = on ? 1.0 : 0.0;
    mom[1] = sqrt(l0);
#pragma unroll
    for (int j = 0; j < kMaxRows; ++j)
      if (j < a.nrows) mom[2 + j] = r[2 + j] / n;
    if (on) a.coef[(size_t)s * kRec] = 2.0;  // an inflated site is floored as an updated one
    return;
  }
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
    if (a.infl) {
      double *f = a.infl + (size_t)s * 3;
      if (f[2] > 0.0 && finite(f[0])) adapt(f, s2, yo - ybar, rv, a.lamMin, a.lamMax, a.sdMin);
    }
  } else {
    cf[0] = (double)before;
    const double nanv = __longlong_as_double(0x7ff8000000000000ll);
    dg[1] = dg[2] = dg[3] = nanv;
  }
}

// One warp per chunk.  A member takes part iff its status has neither excluded bit and all its rows are finite;
// others are neither read into the sums nor written.
template <int PASS, bool APPLY, bool FLOOR, bool INFLATE>
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
  double mu[2 + kMaxRows];  // pass 2: means of observation k; INFLATE: the inflation record
  if (PASS == 2 || INFLATE) {
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
    bool write = false;
    if (INFLATE && mu[0] != 0.0) {
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) x[j] = mu[2 + j] + mu[1] * (x[j] - mu[2 + j]);
      write = true;
    }
    if (APPLY) {
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
    }
    if (write)
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) a.state[(int64_t)a.rows[j] * a.ld + m] = x[j];
    if (PASS == kInflPass) {
      acc[0] += 1.0;
#pragma unroll
      for (int j = 0; j < kMaxRows; ++j)
        if (j < n) acc[2 + j] += x[j];
    } else if (PASS != 0) {
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

int ensure_inflation(sipnet_gpu_handle *h) {
  if (h->asInfl) return 0;
  const cudaError_t e = cudaMalloc((void **)&h->asInfl, (size_t)h->nsites * 3 * sizeof(double));
  return e == cudaSuccess ? 0 : fail(SIPNET_GPU_ERR_NO_DEVICE, "inflation scratch: %s", cudaGetErrorString(e));
}

cudaError_t launch_members(const Args &a, int pass, bool apply, bool floor, bool inflate, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nchunks, kWarps);
  if (pass == 1 && !apply && !floor && !inflate) {
    members_kernel<1, false, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 1 && !apply && !floor && inflate) {
    members_kernel<1, false, false, true><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 1 && apply && !floor && !inflate) {
    members_kernel<1, true, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 2 && !apply && !floor && !inflate) {
    members_kernel<2, false, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 0 && apply && floor && !inflate) {
    members_kernel<0, true, true, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == kInflPass && !apply && !floor && !inflate) {
    members_kernel<kInflPass, false, false, false><<<g, kWarps * 32, 0, stream>>>(a);
  } else {
    return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_site_reduce(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nsites, kWarps);
  if (pass == 1) {
    site_reduce_kernel<1><<<g, kWarps * 32, 0, stream>>>(a);
  } else if (pass == 2) {
    site_reduce_kernel<2><<<g, kWarps * 32, 0, stream>>>(a);
  } else {
    site_reduce_kernel<kInflPass><<<g, kWarps * 32, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_site_combine(const Args &a, int pass, cudaStream_t stream) {
  const unsigned g = blocks_for(a.nsites, 128);
  if (pass == 1) {
    site_combine_kernel<1><<<g, 128, 0, stream>>>(a);
  } else if (pass == 2) {
    site_combine_kernel<2><<<g, 128, 0, stream>>>(a);
  } else {
    site_combine_kernel<kInflPass><<<g, 128, 0, stream>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace as
}  // namespace sip
