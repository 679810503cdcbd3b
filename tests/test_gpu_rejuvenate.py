"""Parameter rejuvenation: the Liu-West kernel-shrinkage move after a resample (sipnet_gpu_rejuvenate,
sipnet_gpu_comm_rejuvenate, sipnet_gpu_multi_rejuvenate; sip_jitter.cu) and the gather of the device parameter rows
(SIPNET_GPU_GATHER_PARAMS).

CPU: a numpy reference of the move (math.fsum for every sum, the header's Cholesky loop in its order) keeps the
ensemble's mean and population covariance for normals with sample mean 0 and covariance I that are orthogonal to the
centred phi, and tends to the identity as a -> 1; the ctypes mirror of sipnet_gpu_jitter_spec against the C layout.
GPU: moved phi within 1e-9 sqrt(V_jj) + 4 ulp of the reference (a bound that one dropped member breaks), and N, rank,
moved, kept exactly; rank-deficient sites made by resample; rejected proposals; the re-derived rows against
setupModel() through a fresh handle; what must not change; teams and multi-GPU partitions; launches per call;
rejected arguments; GATHER_PARAMS against the host's derivation.
"""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
from sipnet_b200 import _abi as A, api, synth

EXCLUDED = A.ST_BAD_ALLOCATION | A.ST_NONFINITE
P_ = A.P
RESCALED = [P_[n] for n in ("baseVegResp", "litterBreakdownRate", "baseSoilResp", "woodTurnoverRate", "leafTurnoverRate",
                            "fineRootTurnoverRate", "coarseRootTurnoverRate", "baseCoarseRootResp", "baseFineRootResp")]
ALLOC = [P_["leafAllocation"], P_["woodAllocation"], P_["fineRootAllocation"]]
I, L, G = A.TF_IDENTITY, A.TF_LOG, A.TF_LOGIT
# (row, transform, lower, upper): the 16 rows of the widest move
ROWS16 = [("psnTOpt", I, 0, 0), ("psnTMin", I, 0, 0), ("frozenSoilThreshold", I, 0, 0), ("aMax", I, 0, 0),
          ("halfSatPar", L, 0, 0), ("soilWHC", L, 0, 0), ("baseVegResp", L, 0, 0), ("vegRespQ10", L, 0, 0),
          ("wueConst", L, 0, 0), ("leafCSpWt", L, 0, 0), ("baseSoilResp", L, 0, 0), ("fAnoxia", G, 0.0, 0.55),
          ("leafAllocation", G, 0.0, 0.28), ("woodAllocation", G, 0.0, 0.28), ("dVpdSlope", G, 0.0, 1.0),
          ("baseFolRespFrac", G, 0.0, 1.0)]
SPECS = {1: [ROWS16[4]], 4: [ROWS16[0], ROWS16[5], ROWS16[11], ROWS16[12]], 16: ROWS16}


def unpack(rows):
    return ([P_[r[0]] for r in rows], [r[1] for r in rows], [float(r[2]) for r in rows], [float(r[3]) for r in rows])


# ---- the reference ---------------------------------------------------------------------------------------------------
def host_derive(P):
    """setupModel()'s unit changes and derived rows of the 80 rows, on the host (the device's own internal rows left out)."""
    Q = np.array(P, dtype=np.float64, copy=True)
    Q[RESCALED] /= 365.0
    derive_rows(Q)
    return Q


def derive_rows(Q, cols=slice(None)):
    Q[P_["coarseRootAllocation"], cols] = 1 - Q[P_["leafAllocation"], cols] - Q[P_["woodAllocation"], cols] - \
        Q[P_["fineRootAllocation"], cols]
    Q[P_["psnTMax"], cols] = Q[P_["psnTOpt"], cols] + (Q[P_["psnTOpt"], cols] - Q[P_["psnTMin"], cols])
    fa, ad = Q[P_["fAnoxia"], cols], Q[P_["anaerobicDecompRate"], cols]
    Q[P_["fAnoxia"], cols] = np.where(fa <= 0.0, 1e-6, np.where(fa >= 1.0, 1.0 - 1e-6, fa))
    Q[P_["anaerobicDecompRate"], cols] = np.where(ad <= 0.0, 1e-6, np.where(ad > 1.0, 1.0, ad))


def fwd(t, tf, lo, hi):
    with np.errstate(all="ignore"):
        return t if tf == I else np.log(t) if tf == L else np.log((t - lo) / (hi - t))


def inv(p, tf, lo, hi):
    with np.errstate(all="ignore"):
        return p if tf == I else np.exp(p) if tf == L else lo + (hi - lo) / (1.0 + np.exp(-p))


def in_domain(t, tf, lo, hi):
    t = np.asarray(t)
    ok = np.isfinite(t)
    return ok & (t > 0) if tf == L else ok & (t > lo) & (t < hi) if tf == G else ok


def cholesky(V):
    """The header's semidefinite Cholesky, column order; -> (L, rank)."""
    n = V.shape[0]
    Lm = np.zeros((n, n))
    rank = 0
    for j in range(n):
        d = V[j, j] - math.fsum(Lm[j, m] * Lm[j, m] for m in range(j))
        if d > 2.0 ** -40 * V[j, j]:
            Lm[j, j] = math.sqrt(d)
            for i in range(j + 1, n):
                Lm[i, j] = (V[i, j] - math.fsum(Lm[i, m] * Lm[j, m] for m in range(j))) / Lm[j, j]
            rank += 1
    return Lm, rank


def reference(params, status, ms, nsites, rows, tf, lo, hi, shrink, z):
    """include/sipnet_gpu.h sipnet_gpu_rejuvenate on device-unit params [80][M] ->
    (params', diag [nsites][4], phi' [n][M] (NaN where no proposal), moved mask, sd [n][nsites], margin)."""
    Q = np.array(params, dtype=np.float64, copy=True)
    n, M = len(rows), params.shape[1]
    diag = np.zeros((nsites, 4))
    phin = np.full((n, M), np.nan)
    moved = np.zeros(M, bool)
    sd = np.zeros((n, nsites))
    margin = np.inf
    for s in range(nsites):
        idx = np.nonzero(ms == s)[0]
        ok = (status[idx] & EXCLUDED) == 0
        for j in range(n):
            ok &= in_domain(params[rows[j], idx], tf[j], lo[j], hi[j])
        idx = idx[ok]
        N = idx.size
        diag[s] = N, -1, 0, 0
        a = shrink[s]
        if math.isnan(a) or N < 2:
            continue
        phi = np.array([fwd(params[rows[j], idx], tf[j], lo[j], hi[j]) for j in range(n)])
        mean = np.array([math.fsum(p) / N for p in phi])
        c = phi - mean[:, None]
        V = np.array([[math.fsum(c[j] * c[l]) / N for l in range(n)] for j in range(n)])
        sd[:, s] = np.sqrt(np.diag(V))
        Lm, rank = cholesky(V)
        h = math.sqrt(1 - a * a)
        pn = a * phi + ((1 - a) * mean)[:, None] + h * (Lm @ z[:, idx])
        th = np.array([inv(pn[j], tf[j], lo[j], hi[j]) for j in range(n)])
        acc = np.ones(N, bool)
        for j in range(n):
            acc &= in_domain(th[j], tf[j], lo[j], hi[j])
        al = [th[rows.index(r)] if r in rows else params[r, idx] for r in ALLOC]
        coarse = 1 - al[0] - al[1] - al[2]
        bad = (al[0] >= 1) | (al[1] >= 1) | (al[2] >= 1) | (coarse < 0)
        if any(r in rows for r in ALLOC):
            margin = min(margin, float(np.min(np.abs(coarse[acc]))) if acc.any() else np.inf)
        acc &= ~bad
        diag[s] = N, rank, acc.sum(), N - acc.sum()
        phin[:, idx] = pn
        for j in range(n):
            Q[rows[j], idx[acc]] = th[j][acc]
        derive_rows(Q, idx[acc])
        moved[idx[acc]] = True
    return Q, diag, phin, moved, sd, margin


def within_bound(got_params, phin, sd, ms, rows, tf, lo, hi, cols):
    for j in range(len(rows)):
        g = fwd(got_params[rows[j], cols], tf[j], lo[j], hi[j])
        w = phin[j, cols]
        tol = 1e-9 * sd[j, ms[cols]] + 4 * np.spacing(np.abs(w))
        if not np.all(np.abs(g - w) <= tol):
            return False
    return True


def centred_normals(phi, k, rng):
    """[k][N] normals with sample mean 0 and population covariance I, orthogonal to the centred rows of phi."""
    N = phi.shape[1]
    X = np.hstack([np.ones((N, 1)), (phi - phi.mean(axis=1, keepdims=True)).T, rng.standard_normal((N, k))])
    Qm, _ = np.linalg.qr(X)
    return (Qm[:, -k:] * math.sqrt(N)).T


def test_reference_keeps_mean_and_population_covariance():
    rng = np.random.default_rng(1)
    M, n = 400, 5
    rows = [P_[r] for r in ("psnTOpt", "psnTMin", "aMax", "frozenSoilThreshold", "wueConst")]
    P = host_derive(synth.synth_params(M, stream=3))
    P[rows] = rng.multivariate_normal(np.zeros(n), np.eye(n) + 0.6, size=M).T * 3 + 10
    phi = P[rows]
    z = centred_normals(phi, n, rng)
    assert np.allclose(z.mean(axis=1), 0, atol=1e-13) and np.allclose(z @ z.T / M, np.eye(n), atol=1e-12)
    for a in (0.5, 0.9, 0.98):
        Q, diag, phin, moved, _, _ = reference(P, np.zeros(M, np.uint32), np.zeros(M, np.int32), 1, rows, [I] * n,
                                              [0.0] * n, [0.0] * n, [a], z)
        assert moved.all() and diag[0].tolist() == [M, n, M, 0]
        new = Q[rows]
        np.testing.assert_allclose(new.mean(axis=1), phi.mean(axis=1), rtol=1e-13)
        np.testing.assert_allclose(np.cov(new, bias=True), np.cov(phi, bias=True), rtol=1e-11, atol=1e-12)
        assert not np.allclose(new, phi)
    # a -> 1: the identity
    Q, _, _, _, _, _ = reference(P, np.zeros(M, np.uint32), np.zeros(M, np.int32), 1, rows, [I] * n, [0.0] * n,
                                 [0.0] * n, [1 - 1e-12], z)
    np.testing.assert_allclose(Q[rows], phi, rtol=0, atol=1e-4 * np.std(phi))
    d = [np.max(np.abs(reference(P, np.zeros(M, np.uint32), np.zeros(M, np.int32), 1, rows, [I] * n, [0.0] * n,
                                 [0.0] * n, [1 - e], z)[0][rows] - phi)) for e in (1e-2, 1e-4, 1e-6)]
    assert d[0] > d[1] > d[2]


def test_ctypes_jitter_spec_matches_c_layout():
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "sipnet_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(sipnet_gpu_jitter_spec), offsetof(sipnet_gpu_jitter_spec, n_rows),
         offsetof(sipnet_gpu_jitter_spec, rows), offsetof(sipnet_gpu_jitter_spec, transform),
         offsetof(sipnet_gpu_jitter_spec, lower), offsetof(sipnet_gpu_jitter_spec, upper),
         offsetof(sipnet_gpu_jitter_spec, shrink), offsetof(sipnet_gpu_jitter_spec, z));
  printf("%d %d %d %d\n", SIPNET_GPU_TF_IDENTITY, SIPNET_GPU_TF_LOG, SIPNET_GPU_TF_LOGIT, SIPNET_GPU_GATHER_PARAMS);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        lines = subprocess.check_output([exe]).decode().split("\n")
    J = A.JitterSpec
    assert list(map(int, lines[0].split())) == [C.sizeof(J), J.n_rows.offset, J.rows.offset, J.transform.offset,
                                                J.lower.offset, J.upper.offset, J.shrink.offset, J.z.offset]
    assert list(map(int, lines[1].split())) == [A.TF_IDENTITY, A.TF_LOG, A.TF_LOGIT, A.GATHER_PARAMS]


def config(kind, seed=21):
    """'one': one site of 5 000 members; 'many': 40 sites of 100; ('c3', n, m): n sites of m.  The moved rows get a
    spread inside their LOGIT bounds; member 7 fails ensureAllocation and member 11 has fAnoxia outside its bounds."""
    n, m = (1, 5000) if kind == "one" else (40, 100) if kind == "many" else kind[1:]
    sites = [synth.synth_site(3 + s, 1, "half-daily") for s in range(n)]
    M = n * m
    P, ms = synth.synth_params(M, stream=seed), np.repeat(np.arange(n, dtype=np.int32), m)
    rng = np.random.default_rng(seed)
    P[P_["leafCSpWt"]] = rng.uniform(50, 90, M)
    P[P_["fAnoxia"]] = rng.uniform(0.05, 0.5, M)
    P[P_["leafAllocation"]] = rng.uniform(0.05, 0.25, M)
    P[P_["woodAllocation"]] = rng.uniform(0.05, 0.25, M)
    P[P_["leafAllocation"], 7] = 0.9
    P[P_["fAnoxia"], 11] = 0.6
    return sites, P, ms


def shrinks(nsites, seed=4):
    a = np.random.default_rng(seed).uniform(0.75, 0.97, nsites)
    a[3::7] = np.nan
    return a


def normals(k, M, seed=5):
    return np.random.default_rng(seed).standard_normal((k, M))


def test_reference_data_keeps_clear_of_the_allocation_boundary():
    """The GPU cases below compare moved / kept exactly: no proposal of theirs lies within 1e-12 of coarse = 0."""
    for kind in ("one", "many"):
        _, P, ms = config(kind)
        Q = host_derive(P)
        status = np.where(Q[P_["coarseRootAllocation"]] < 0, A.ST_BAD_ALLOCATION, 0).astype(np.uint32)
        rows, tf, lo, hi = unpack(ROWS16)
        nsites = int(ms.max()) + 1
        _, diag, _, _, _, margin = reference(Q, status, ms, nsites, rows, tf, lo, hi, shrinks(nsites), normals(16, ms.size))
        assert margin > 1e-12 and (diag[:, 2] > 0).any()
    _, _, margin = kept_case()
    assert margin > 1e-12


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
OUTS = A.OUT_FULL | A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS
KW = dict(outputs=OUTS, summary_cols=[A.O["nee"], A.O["plantWoodC"]], quantiles=[0.05, 0.5, 0.95], math=A.MATH_FAST,
          nee_sigma=0.5, max_event_records=16, out_steps_capacity=200)
SEG = 200                                    # steps of a forecast segment


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def forecast(kind, cls=api.Ensemble, **kw):
    sites, P, ms = config(kind)
    rng = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0, 1.5, s.nsteps))
    e = cls(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    e.run(0, SEG)
    return e, P, ms


def move(e, rows16, shrink, z):
    rows, tf, lo, hi = unpack(rows16)
    return e.rejuvenate(rows, tf, shrink, z, lo, hi)


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
@pytest.mark.parametrize("k", [1, 4, 16])
def test_matches_reference(kind, k):
    e, _, ms = forecast(kind)
    with e:
        p0, st0 = e.params(), e.status()
        shrink, z = shrinks(e.nsites), normals(k, e.nmembers)
        diag = move(e, SPECS[k], shrink, z)
        got = e.params()
        assert np.array_equal(e.status(), st0)
    rows, tf, lo, hi = unpack(SPECS[k])
    ref, rdiag, phin, moved, sd, _ = reference(p0, st0, ms, e.nsites, rows, tf, lo, hi, shrink, z)
    assert np.array_equal(diag, rdiag)
    assert moved.sum() > 0.8 * e.nmembers * (~np.isnan(shrink)).mean()
    assert within_bound(got, phin, sd, ms, rows, tf, lo, hi, np.nonzero(moved)[0])
    assert np.array_equal(got[:, ~moved], p0[:, ~moved])
    # every dependent row follows setupModel() from the moved rows (the host restates the 80-row part)
    chk = got.copy()
    derive_rows(chk)
    assert np.array_equal(chk, got)
    # the bound sees one member left out of the moments
    drop = int(np.nonzero(moved & (ms == 0))[0][0])
    st1 = st0.copy()
    st1[drop] |= A.ST_NONFINITE
    _, _, phin1, moved1, _, _ = reference(p0, st1, ms, e.nsites, rows, tf, lo, hi, shrink, z)
    assert not within_bound(got, phin1, sd, ms, rows, tf, lo, hi, np.nonzero(moved1)[0])


@gpu
def test_gather_params_is_the_host_derivation():
    e, P, _ = forecast("many")
    with e:
        got = e.params()
    ref = host_derive(P)
    other = [r for r in range(A.NPARAMS) if r not in RESCALED]
    assert np.array_equal(got[other], ref[other])
    np.testing.assert_allclose(got[RESCALED], ref[RESCALED], rtol=1e-15, atol=0)


ANCESTORS = np.array([20, 40, 60])


def rank_deficient_case():
    """Six sites of 100 whose ancestors' (psnTOpt, psnTMin) span the plane well: the factor's first two columns then
    hold the whole rank, and the remaining pivots are rounding noise far below 2^-40 of their diagonal."""
    sites, P, ms = config(("c3", 6, 100))
    for s in range(6):
        P[P_["psnTOpt"], ANCESTORS + 100 * s] = 15.0, 25.0, 20.0
        P[P_["psnTMin"], ANCESTORS + 100 * s] = -5.0, 0.0, 6.0
    return sites, P, ms


@gpu
def test_rank_deficient_sites_still_move():
    sites, P, ms = rank_deficient_case()
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **KW) as e:
        e.run(0, SEG)
        lw = np.full(e.nmembers, -1000.0)
        for s in range(6):
            lw[ANCESTORS[: 2 + s % 2] + 100 * s] = 0.0      # 2 or 3 ancestors per site
        anc, rdg = e.resample(np.full(6, 0.3), math.inf, lw)
        assert (rdg[:, 3] >= 2).all() and (rdg[:, 3] <= 3).all() and (anc >= 0).all()
        p0, st0 = e.params(), e.status()
        shrink, z = np.full(6, 0.9), normals(16, e.nmembers)
        diag = move(e, ROWS16, shrink, z)
        got = e.params()
    rows, tf, lo, hi = unpack(ROWS16)
    _, rdiag, phin, moved, sd, _ = reference(p0, st0, ms, 6, rows, tf, lo, hi, shrink, z)
    assert np.array_equal(diag, rdiag)
    assert (diag[:, 1] <= rdg[:, 3] - 1).all() and (diag[:, 2] > 0).all()
    assert within_bound(got, phin, sd, ms, rows, tf, lo, hi, np.nonzero(moved)[0])
    for s in range(6):                       # the move creates values no member had
        assert len(np.unique(got[rows[0], ms == s])) > rdg[s, 3]


def kept_case():
    """Allocation rows whose proposals sometimes fail ensureAllocation (fineRootAllocation is 0.4)."""
    sites, P, ms = config(("c3", 4, 100))
    rng = np.random.default_rng(12)
    total = np.where(rng.uniform(size=ms.size) < 0.85, rng.uniform(0.597, 0.5995, ms.size), rng.uniform(0.5, 0.56, ms.size))
    P[P_["leafAllocation"]] = rng.uniform(0.2, 0.3, ms.size)
    P[P_["woodAllocation"]] = total - P[P_["leafAllocation"]]      # leaf + wood mostly just below 1 - fineRoot
    P[P_["leafAllocation"], 7] = 0.9
    rows16 = [("leafAllocation", I, 0, 0), ("woodAllocation", G, 0.0, 0.6), ("aMax", I, 0, 0)]
    rows, tf, lo, hi = unpack(rows16)
    Q = host_derive(P)
    status = np.where(Q[P_["coarseRootAllocation"]] < 0, A.ST_BAD_ALLOCATION, 0).astype(np.uint32)
    _, diag, _, _, _, margin = reference(Q, status, ms, 4, rows, tf, lo, hi, np.full(4, 0.5), normals(3, ms.size, 13))
    return (sites, P, ms, rows16), diag, margin


@gpu
def test_rejected_proposals_keep_the_member():
    (sites, P, ms, rows16), _, _ = kept_case()
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **KW) as e:
        e.run(0, SEG)
        p0, st0 = e.params(), e.status()
        diag = move(e, rows16, np.full(4, 0.5), normals(3, e.nmembers, 13))
        got, st1 = e.params(), e.status()
    rows, tf, lo, hi = unpack(rows16)
    _, rdiag, _, moved, _, _ = reference(p0, st0, ms, 4, rows, tf, lo, hi, np.full(4, 0.5), normals(3, e.nmembers, 13))
    assert np.array_equal(diag, rdiag) and diag[:, 3].sum() >= 4 and (diag[:, 2] > 0).all()
    assert np.array_equal(got[:, ~moved], p0[:, ~moved])
    assert np.array_equal(st1, st0)
    assert not (st1 & A.ST_BAD_ALLOCATION)[np.arange(ms.size) != 7].any()
    assert (got[P_["coarseRootAllocation"]][moved] >= 0).all()


SETUP_ROWS = [("aMax", I, 0, 0), ("halfSatPar", L, 0, 0), ("psnTOpt", I, 0, 0), ("vegRespQ10", L, 0, 0),
              ("leafAllocation", G, 0.0, 0.28), ("woodAllocation", G, 0.0, 0.28), ("soilWHC", L, 0, 0),
              ("fAnoxia", G, 0.0, 1.0)]


@gpu
def test_rederivation_is_setup_models():
    kw = dict(outputs=A.OUT_FULL | A.OUT_LOGLIK, summary_cols=[], quantiles=[], math=A.MATH_VALIDATION,
              max_event_records=0)
    a, P, ms = forecast("many", **kw)
    sites, _, _ = config("many")
    with a, api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw)) as b:
        diag = move(a, SETUP_ROWS, shrinks(a.nsites), normals(len(SETUP_ROWS), a.nmembers))
        assert diag[:, 2].sum() > 0.5 * a.nmembers
        got = a.params()
        P2 = P.copy()
        rows = [P_[r[0]] for r in SETUP_ROWS]
        P2[rows] = got[rows]                   # none of these rows is rescaled by setupModel()
        b.set_params(P2)
        rv, rw = a.ring()
        b.set_state(a.state(), rv, rw, next_step=SEG)
        assert np.array_equal(b.params(), got)
        a.run(SEG, 2 * SEG)
        b.run(SEG, 2 * SEG)
        assert np.array_equal(a.output(), b.output(), equal_nan=True)
        assert np.array_equal(a.state(), b.state(), equal_nan=True)


def snapshot(e):
    rv, rw = e.ring()
    return dict(state=e.state(), status=e.status(), rv=rv, rw=rw, ll=e.loglik(), lln=e.loglik_n(),
                counts=e.event_counts(), recs=[[bytes(r) for r in m] for m in e.event_records()], out=e.output(),
                mean=e.mean(), var=e.variance(), q=e.quantiles())


@gpu
def test_nothing_else_changes():
    e, _, ms = forecast("many")
    with e:
        before, p0 = snapshot(e), e.params()
        shrink = shrinks(e.nsites)
        diag = move(e, ROWS16, shrink, normals(16, e.nmembers))
        after, got = snapshot(e), e.params()
    for key in before:
        if key == "recs":
            assert after[key] == before[key]
        else:
            assert np.array_equal(after[key], before[key], equal_nan=True), key
    skipped = np.isnan(shrink)[ms]
    assert np.array_equal(got[:, skipped], p0[:, skipped]) and (diag[np.isnan(shrink), 1] == -1).all()
    assert (diag[np.isnan(shrink), 2:] == 0).all()
    for m in (7, 11):                                     # bad allocation; fAnoxia outside its bounds
        assert np.array_equal(got[:, m], p0[:, m])
    assert diag[0, 0] <= 98                               # members 7 and 11 of site 0 do not take part


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_team_of_one_equals_handle(kind):
    res = []
    for team in (False, True):
        e, _, _ = forecast(kind)
        with e:
            rows, tf, lo, hi = unpack(ROWS16)
            args = (rows, tf, shrinks(e.nsites), normals(16, e.nmembers), lo, hi)
            if team:
                e.join_team(1, 0)
                diag = e.team_rejuvenate(*args)
            else:
                diag = e.rejuvenate(*args)
            res.append((diag, e.params()))
    for x, y in zip(*res):
        assert np.array_equal(x, y)


needs2 = pytest.mark.skipif("ngpus() < 2", reason="needs two GPUs on the box")
DEVICES = [pytest.param(None, marks=needs2, id="all-gpus"), pytest.param([0, 0], id="loopback2"),
           pytest.param([0, 0, 0], id="loopback3"), pytest.param([0] * 5, id="loopback5")]


@gpu
@pytest.mark.parametrize("devices", DEVICES)
@pytest.mark.parametrize("kind", ["one", ("c3", 11, 40)], ids=["split-site", "whole-sites"])
def test_multi_matches_one_gpu(devices, kind):
    one, _, ms = forecast(kind)
    multi, _, _ = forecast(kind, cls=api.MultiEnsemble, devices=devices)
    with one, multi:
        assert multi.ndevices >= 2
        assert np.array_equal(multi.params(), one.params())
        shrink, z = shrinks(one.nsites), normals(16, one.nmembers)
        p0, st0 = one.params(), one.status()
        d1 = move(one, ROWS16, shrink, z)
        dm = move(multi, ROWS16, shrink, z)
        g1, gm = one.params(), multi.params()
        assert np.array_equal(dm, d1) and (d1[:, 2] > 0).any()
        if kind != "one":
            assert np.array_equal(gm, g1)
        else:
            rows, tf, lo, hi = unpack(ROWS16)
            _, _, phin, moved, sd, _ = reference(p0, st0, ms, one.nsites, rows, tf, lo, hi, shrink, z)
            assert within_bound(gm, phin, sd, ms, rows, tf, lo, hi, np.nonzero(moved)[0])
            assert np.array_equal(gm[:, ~moved], g1[:, ~moved])
        assert np.array_equal(multi.status(), one.status())


@gpu
def test_launches_do_not_grow_with_sites():
    per_call = []
    for n in (3, 300):
        sites, P, ms, _ = synth.config_c3(nsites=n, members_per_site=10, nyears=1)
        with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=0, math=A.MATH_FAST) as e:
            z = normals(2, e.nmembers)
            c0 = e.launch_count()
            e.rejuvenate([P_["aMax"], P_["halfSatPar"]], [I, L], np.full(n, 0.9), z)
            c1 = e.launch_count()
            e.rejuvenate([P_["aMax"], P_["halfSatPar"]], [I, L], np.full(n, 0.9), z)
            per_call.append((c1 - c0, e.launch_count() - c1))
    assert per_call[0] == per_call[1] and per_call[0][0] == per_call[0][1] == 6


@gpu
def test_rejected_arguments_leave_everything_untouched():
    e, _, _ = forecast(("c3", 4, 50))
    twin, _, _ = forecast(("c3", 4, 50))
    with e, twin:
        p0 = e.params()
        lib = e.lib
        M = e.nmembers
        good = dict(rows=[P_["aMax"], P_["fAnoxia"]], tf=[I, G], lo=[0.0, 0.0], hi=[0.0, 0.55], shrink=np.full(4, 0.9),
                    z=normals(2, M))

        def rc_of(fn=lib.sipnet_gpu_rejuvenate, target=e.handle, null=None, n_rows=None, **kw):
            a = dict(good, **kw)
            spec, keep = e.jitter_spec(a["rows"], a["tf"], a["shrink"], a["z"], a["lo"], a["hi"])
            if n_rows is not None:
                spec.n_rows = n_rows
            if null:
                setattr(spec, null, None)
            return fn(target, None if null == "spec" else C.byref(spec), None)

        z_nan, z_inf = good["z"].copy(), good["z"].copy()
        z_nan[1, 17] = np.nan
        z_inf[0, 3] = -np.inf
        cases = {"NULL handle": lambda: rc_of(target=None), "NULL spec": lambda: rc_of(null="spec"),
                 "n_rows 0": lambda: rc_of(n_rows=0), "NaN z": lambda: rc_of(z=z_nan), "inf z": lambda: rc_of(z=z_inf),
                 "repeated row": lambda: rc_of(rows=[P_["aMax"], P_["aMax"]]),
                 "psnTMax": lambda: rc_of(rows=[P_["psnTMax"], P_["aMax"]]),
                 "coarseRootAllocation": lambda: rc_of(rows=[P_["coarseRootAllocation"], P_["aMax"]]),
                 "row 80": lambda: rc_of(rows=[80, P_["aMax"]]), "row -1": lambda: rc_of(rows=[-1, P_["aMax"]]),
                 "transform 3": lambda: rc_of(tf=[I, 3]), "lo = hi": lambda: rc_of(hi=[0.0, 0.0]),
                 "lo > hi": lambda: rc_of(lo=[0.0, 1.0]), "inf bound": lambda: rc_of(hi=[0.0, np.inf]),
                 "NaN bound": lambda: rc_of(lo=[0.0, np.nan]), "shrink 0": lambda: rc_of(shrink=np.array([0.9, 0, .9, .9])),
                 "shrink 1": lambda: rc_of(shrink=np.array([0.9, 1.0, .9, .9])),
                 "shrink -inf": lambda: rc_of(shrink=np.array([0.9, -np.inf, .9, .9]))}
        for f in ("rows", "transform", "shrink", "z", "lower", "upper"):
            cases[f"NULL {f}"] = lambda f=f: rc_of(null=f)
        for name, fn in cases.items():
            assert fn() == A.ERR_BAD_ARGUMENT, name
            assert np.array_equal(e.params(), p0), name
        e.join_team(1, 0)
        assert rc_of(fn=lib.sipnet_gpu_comm_rejuvenate, target=e.comm, z=z_nan) == A.ERR_BAD_ARGUMENT
        assert rc_of(fn=lib.sipnet_gpu_comm_rejuvenate, target=e.comm, n_rows=17) == A.ERR_BAD_ARGUMENT
        e.run(SEG, 2 * SEG)
        twin.run(SEG, 2 * SEG)
        for x, y in ((e.output(), twin.output()), (e.state(), twin.state()), (e.loglik(), twin.loglik()),
                     (e.status(), twin.status()), (e.params(), twin.params())):
            assert np.array_equal(x, y, equal_nan=True)
    multi, _, _ = forecast(("c3", 4, 50), cls=api.MultiEnsemble, devices=[0, 0])
    with multi:
        p0 = multi.params()
        spec, keep = multi.jitter_spec([P_["aMax"]], [I], np.full(4, 0.9), z_inf[:1])
        assert lib.sipnet_gpu_multi_rejuvenate(multi.multi, C.byref(spec), None) == A.ERR_BAD_ARGUMENT
        assert np.array_equal(multi.params(), p0)
