"""Parameter calibration: the tempered random-walk Metropolis-Hastings move (sipnet_gpu_mh_move,
sipnet_gpu_comm_mh_move, sipnet_gpu_multi_mh_move; proposal in sip_jitter.cu, snapshot and decision in
sip_resample.cu, driver in sip_comm.cu run_mh).

CPU: the ctypes mirror of sipnet_gpu_mh_spec against the C layout; a numpy reference of the log prior in phi (three
transforms, two priors) against closed-form densities, and a toy sampler (tau = 0) that keeps a prior sample at the
prior -- and fails to once the Jacobian term is dropped.
GPU: all-accepted moves against the Liu-West reference with a = 1 and a fresh handle's run; nothing accepted (invalid
proposals, negative delta) restores every gatherable field bit for bit; mixed decisions predicted from an all-accept
twin; a tempered resample-move loop against the exact posterior of a 512-point grid; teams and partitions; launches
and rejected arguments.
"""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy import stats

from conftest import ROOT
from sipnet_b200 import _abi as A, api, synth
from test_gpu_rejuvenate import ALLOC, cholesky, derive_rows, fwd, in_domain, inv

P_ = A.P
I, L, G = A.TF_IDENTITY, A.TF_LOG, A.TF_LOGIT
FLAT, NORMAL = A.PRIOR_FLAT, A.PRIOR_NORMAL
EXCLUDED = A.ST_BAD_ALLOCATION | A.ST_NONFINITE


# ---- the reference ---------------------------------------------------------------------------------------------------
def log_prior(theta, phi, tf, lo, hi, prior, a, b):
    """include/sipnet_gpu.h sipnet_gpu_mh_move: row j's log prior density in phi, constants dropped."""
    theta, phi = np.asarray(theta, np.float64), np.asarray(phi, np.float64)
    if prior == NORMAL:
        return -((phi - a) * (phi - a)) / (2.0 * (b * b))
    with np.errstate(all="ignore"):
        jac = np.zeros_like(phi) if tf == I else phi.copy() if tf == L else np.log((theta - lo) * (hi - theta) / (hi - lo))
    return np.where((theta >= a) & (theta <= b), jac, -np.inf)


def delta(tau, l_new, l_cur, lp_new, lp_cur):
    """delta_i = tau (L' - L) + sum_j [lp_j(phi') - lp_j(phi)]; lp_*: [n][M]; the tau term is 0 at tau = 0."""
    d = np.zeros(np.shape(l_new))
    for j in range(len(lp_new)):
        d = d + (lp_new[j] - lp_cur[j])
    with np.errstate(invalid="ignore"):
        return np.where(np.asarray(tau) == 0.0, 0.0, tau * (l_new - l_cur)) + d


def test_log_prior_matches_closed_form_densities():
    rng = np.random.default_rng(3)
    lo, hi = 2.0, 7.0
    # FLAT on theta: the density of phi is p_theta(g^-1(phi)) |dtheta/dphi|
    for tf, (a, b) in ((I, (-3.0, 4.0)), (L, (0.5, 9.0)), (G, (lo, hi))):
        th = rng.uniform(a, b, 200) if tf != G else rng.uniform(lo, hi, 200)
        ph = fwd(th, tf, lo, hi)
        got = log_prior(th, ph, tf, lo, hi, FLAT, a, b)
        dens = stats.uniform(a, b - a).logpdf(th)
        jac = 0.0 if tf == I else ph if tf == L else np.log((th - lo) * (hi - th) / (hi - lo))
        want = dens + jac
        np.testing.assert_allclose(got - got[0], want - want[0], rtol=0, atol=1e-12)
        out = np.array([a - 1.0, b + 1.0]) if tf != G else np.array([lo + 0.1, hi - 0.1])
        if tf != G:
            assert np.all(log_prior(out, fwd(out, tf, lo, hi), tf, lo, hi, FLAT, a, b) == -np.inf)
    assert np.all(log_prior(np.array([3.0, 6.0]), fwd(np.array([3.0, 6.0]), G, lo, hi), G, lo, hi, FLAT, 3.5, 5.0)
                  == -np.inf)
    # improper flat priors
    assert log_prior(1e300, 1e300, I, 0, 0, FLAT, -np.inf, np.inf) == 0.0
    assert log_prior(np.e, 1.0, L, 0, 0, FLAT, 0.0, np.inf) == 1.0
    # NORMAL on phi: lognormal (LOG), logit-normal (LOGIT), normal (IDENTITY)
    for tf in (I, L, G):
        ph = rng.normal(0.3, 1.7, 100)
        th = inv(ph, tf, lo, hi)
        got = log_prior(th, ph, tf, lo, hi, NORMAL, 0.3, 1.7)
        want = stats.norm(0.3, 1.7).logpdf(ph)
        np.testing.assert_allclose(got - got[0], want - want[0], rtol=0, atol=1e-12)
    th = np.exp(rng.normal(0.3, 1.7, 100))
    want = stats.lognorm(1.7, scale=np.exp(0.3)).logpdf(th) + np.log(th)  # density of phi = log theta
    got = log_prior(th, np.log(th), L, 0, 0, NORMAL, 0.3, 1.7)
    np.testing.assert_allclose(got - got[0], want - want[0], rtol=0, atol=1e-10)
    # delta
    assert delta(0.0, np.array([np.nan]), np.array([1.0]), [np.array([0.5])], [np.array([0.25])])[0] == 0.25
    assert delta(0.5, np.array([-3.0]), np.array([-1.0]), [np.array([0.5])], [np.array([0.25])])[0] == -0.75


def toy_sampler(jacobian: bool, moves=20, N=4000, seed=11):
    """Three independent rows under their priors (tau = 0): LOG with FLAT [1, 10], LOGIT (0, 1) with FLAT on the
    whole interval, IDENTITY with NORMAL(2, 0.5).  The random walk is the move's: phi + h L z with the population
    covariance's Cholesky factor.  Returns the theta sample."""
    rng = np.random.default_rng(seed)
    rows = [(L, 0.0, 0.0, FLAT, 1.0, 10.0), (G, 0.0, 1.0, FLAT, 0.0, 1.0), (I, 0.0, 0.0, NORMAL, 2.0, 0.5)]
    th = np.array([rng.uniform(1.0, 10.0, N), rng.uniform(0.0, 1.0, N), rng.normal(2.0, 0.5, N)])
    h = 2.38 / math.sqrt(3)

    def lps(t, p):
        out = []
        for j, (tf, lo, hi, pr, a, b) in enumerate(rows):
            lp = log_prior(t[j], p[j], tf, lo, hi, pr, a, b)
            if not jacobian and pr == FLAT:
                lp = np.where(np.isfinite(lp), 0.0, lp)
            out.append(lp)
        return out

    for _ in range(moves):
        ph = np.array([fwd(th[j], r[0], r[1], r[2]) for j, r in enumerate(rows)])
        V = np.cov(ph, bias=True)
        Lm, _ = cholesky(V)
        pn = ph + h * (Lm @ rng.standard_normal((3, N)))
        tn = np.array([inv(pn[j], r[0], r[1], r[2]) for j, r in enumerate(rows)])
        ok = np.ones(N, bool)
        for j, r in enumerate(rows):
            ok &= in_domain(tn[j], r[0], r[1], r[2])
        d = delta(0.0, np.zeros(N), np.zeros(N), lps(tn, pn), lps(th, ph))
        acc = ok & np.isfinite(d) & (np.log(rng.uniform(size=N)) < d)
        th[:, acc] = tn[:, acc]
    return th


def test_toy_sampler_keeps_the_prior_and_catches_a_dropped_jacobian():
    good = toy_sampler(True)
    p = [stats.kstest(good[0], stats.uniform(1, 9).cdf).pvalue, stats.kstest(good[1], stats.uniform(0, 1).cdf).pvalue,
         stats.kstest(good[2], stats.norm(2, 0.5).cdf).pvalue]
    assert min(p) > 0.01, p
    bad = toy_sampler(False)
    assert stats.kstest(bad[0], stats.uniform(1, 9).cdf).pvalue < 1e-6
    assert stats.kstest(bad[1], stats.uniform(0, 1).cdf).pvalue < 1e-6


def test_ctypes_mh_spec_matches_c_layout():
    fields = [f[0] for f in A.MHSpec._fields_]
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "sipnet_gpu.h"
int main(void) {
  printf("%zu", sizeof(sipnet_gpu_mh_spec));
''' + "".join(f'  printf(" %zu", offsetof(sipnet_gpu_mh_spec, {f}));\n' for f in fields) + r'''
  printf("\n%d %d\n", SIPNET_GPU_PRIOR_FLAT, SIPNET_GPU_PRIOR_NORMAL);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        lines = subprocess.check_output([exe]).decode().split("\n")
    assert list(map(int, lines[0].split())) == [C.sizeof(A.MHSpec)] + [getattr(A.MHSpec, f).offset for f in fields]
    assert list(map(int, lines[1].split())) == [A.PRIOR_FLAT, A.PRIOR_NORMAL]


def proposal_reference(params, status, cur, ms, nsites, rows, scale, z):
    """The proposal of the move (rejuvenate's reference with a = 1, h = scale) -> (phi' [n][M] NaN where no proposal,
    valid mask, diag[:, :2], sd [n][nsites]).  rows: (row, tf, lo, hi, prior, a, b)."""
    n, M = len(rows), params.shape[1]
    phin = np.full((n, M), np.nan)
    valid = np.zeros(M, bool)
    diag = np.zeros((nsites, 2))
    sd = np.zeros((n, nsites))
    for s in range(nsites):
        idx = np.nonzero(ms == s)[0]
        ok = ((status[idx] & EXCLUDED) == 0) & np.isfinite(cur[idx])
        for (r, tf, lo, hi, pr, a, b) in rows:
            t = params[r, idx]
            ok &= in_domain(t, tf, lo, hi)
            ok &= np.isfinite(log_prior(t, fwd(t, tf, lo, hi), tf, lo, hi, pr, a, b))
        idx = idx[ok]
        N = idx.size
        diag[s] = N, -1
        if math.isnan(scale[s]) or N < 2:
            continue
        phi = np.array([fwd(params[r[0], idx], r[1], r[2], r[3]) for r in rows])
        mean = np.array([math.fsum(p) / N for p in phi])
        c = phi - mean[:, None]
        V = np.array([[math.fsum(c[j] * c[l]) / N for l in range(n)] for j in range(n)])
        sd[:, s] = np.sqrt(np.diag(V))
        Lm, rank = cholesky(V, mean)
        diag[s, 1] = rank
        pn = phi + scale[s] * (Lm @ z[:, idx])
        th = np.array([inv(pn[j], r[1], r[2], r[3]) for j, r in enumerate(rows)])
        acc = np.ones(N, bool)
        for j, r in enumerate(rows):
            acc &= in_domain(th[j], r[1], r[2], r[3])
            acc &= np.isfinite(log_prior(th[j], pn[j], r[1], r[2], r[3], r[4], r[5], r[6]))
        rr = [r[0] for r in rows]
        al = [th[rr.index(x)] if x in rr else params[x, idx] for x in ALLOC]
        acc &= ~((al[0] >= 1) | (al[1] >= 1) | (al[2] >= 1) | (1 - al[0] - al[1] - al[2] < 0))
        phin[:, idx] = pn
        valid[idx[acc]] = True
    return phin, valid, diag, sd


def lp_rows(params, rows, cols):
    return [log_prior(params[r, cols], fwd(params[r, cols], tf, lo, hi), tf, lo, hi, pr, a, b)
            for (r, tf, lo, hi, pr, a, b) in rows]


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
OUTS = A.OUT_FULL | A.OUT_LOGLIK | A.OUT_EVENTS
KW = dict(outputs=OUTS, math=A.MATH_FAST, nee_sigma=0.5, max_event_records=16, out_steps_capacity=200)
SEG = 300                                    # the window: longer than the output capacity, so it runs in two pieces
# (row, transform, lower, upper, prior, prior_a, prior_b)
ROWS = [(P_["aMax"], I, 0.0, 0.0, FLAT, -np.inf, np.inf), (P_["halfSatPar"], L, 0.0, 0.0, NORMAL, 5.0, 2.0),
        (P_["fAnoxia"], G, 0.0, 0.55, FLAT, 0.0, 0.55), (P_["vegRespQ10"], L, 0.0, 0.0, FLAT, 0.0, np.inf)]


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def config(kind, seed=21):
    """'one': one site of 3 000 members; 'many': 24 sites of 100; ('c3', n, m): n sites of m.  Member 7 fails
    ensureAllocation and member 11 has fAnoxia outside its bounds."""
    n, m = (1, 3000) if kind == "one" else (24, 100) if kind == "many" else kind[1:]
    sites = [synth.synth_site(3 + s, 1, "half-daily", with_events=True) for s in range(n)]
    M = n * m
    P, ms = synth.synth_params(M, stream=seed), np.repeat(np.arange(n, dtype=np.int32), m)
    rng = np.random.default_rng(seed)
    P[P_["fAnoxia"]] = rng.uniform(0.05, 0.5, M)
    P[P_["leafAllocation"], 7] = 0.9
    P[P_["fAnoxia"], 11] = 0.6
    obs = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(obs.uniform(size=s.nsteps) < 0.3, np.nan, obs.normal(0, 1.5, s.nsteps))
    return sites, P, ms


def forecast(kind, cls=api.Ensemble, steps=SEG, **kw):
    sites, P, ms = config(kind)
    e = cls(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    for b in range(0, steps, 200):
        e.run(b, min(steps, b + 200))
    return e, P, ms


def scales(nsites, seed=4):
    h = np.random.default_rng(seed).uniform(0.3, 0.8, nsites)
    h[3::7] = np.nan
    return h


def normals(k, M, seed=5):
    return np.random.default_rng(seed).standard_normal((k, M))


def mh(e, rows, scale, tau, cur, z, log_u):
    r = [x[0] for x in rows]
    return e.mh_move(r, [x[1] for x in rows], [x[4] for x in rows], [x[5] for x in rows], [x[6] for x in rows], scale,
                     tau, cur, z, log_u, [x[2] for x in rows], [x[3] for x in rows])


def members(e):
    """Every gatherable per-member field."""
    rv, rw = e.ring()
    d = dict(params=e.params(), state=e.state(), rv=rv, rw=rw, status=e.status(), ll=e.loglik(), lln=e.loglik_n(),
             counts=e.event_counts(), recs=[[bytes(r) for r in m] for m in e.event_records()])
    if e.lib.sipnet_gpu_gather_bytes(e.handle, A.GATHER_COUNTERS):
        d["counters"] = e.counters()
    return d


def member_equal(a, b, m):
    for k in a:
        if k == "recs":
            if a[k][m] != b[k][m]:
                return False
        elif not np.array_equal(a[k][..., m], b[k][..., m], equal_nan=True):
            return False
    return True


def all_equal(a, b):
    for k in a:
        if k == "recs":
            assert a[k] == b[k]
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def within_bound(got, phin, sd, ms, rows, cols):
    for j, (r, tf, lo, hi, *_) in enumerate(rows):
        g = fwd(got[r, cols], tf, lo, hi)
        w = phin[j, cols]
        if not np.all(np.abs(g - w) <= 1e-9 * sd[j, ms[cols]] + 4 * np.spacing(np.abs(w))):
            return False
    return True


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_all_accepted_is_the_proposal_run(kind):
    e, P, ms = forecast(kind)
    sites, _, _ = config(kind)
    with e, api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **KW) as fresh:
        p0, st0, cur = e.params(), e.status(), e.loglik()
        scale, z = scales(e.nsites), normals(len(ROWS), e.nmembers)
        diag = mh(e, ROWS, scale, np.full(e.nsites, 0.7), cur, z, np.full(e.nmembers, -np.inf))
        assert e.nrun == 0
        got = members(e)
        phin, valid, rdiag, sd = proposal_reference(p0, st0, cur, ms, e.nsites, ROWS, scale, z)
        assert np.array_equal(diag[:, :2], rdiag)
        assert valid.sum() > 0.5 * e.nmembers
        moved = np.zeros(e.nmembers, bool)
        for s in range(e.nsites):
            if not math.isnan(scale[s]):
                moved |= (ms == s) & valid
        assert np.array_equal(diag[:, 3], np.bincount(ms[moved], minlength=e.nsites).astype(float))
        assert within_bound(got["params"], phin, sd, ms, ROWS, np.nonzero(moved)[0])
        chk = got["params"].copy()
        derive_rows(chk)
        assert np.array_equal(chk, got["params"])
        # every member equals a fresh handle that is given those rows and runs [0, s)
        P2 = P.copy()
        for r in ROWS:
            P2[r[0]] = got["params"][r[0]]             # none of these rows is rescaled by setupModel()
        fresh.set_params(P2)
        fresh.run(0, 200)
        fresh.run(200, SEG)
        want = members(fresh)
        for m in np.nonzero(moved)[0]:
            assert member_equal(got, want, m), m
        assert np.array_equal(got["params"][:, ~moved], p0[:, ~moved])


def resampled(kind, **kw):
    """A forecast, then a resample of every other site (members copied, log-likelihood zeroed)."""
    e, P, ms = forecast(kind, **kw)
    cur = e.loglik()
    u = np.where(np.arange(e.nsites) % 2 == 0, 0.37, np.nan)
    anc, _ = e.resample(u, math.inf, np.where(np.arange(e.nmembers) % 3 == 0, 0.0, -1.0))
    cur = np.where(anc >= 0, cur[np.maximum(anc, 0)], cur)
    return e, P, ms, cur


@gpu
@pytest.mark.parametrize("debug", [False, True], ids=["fast", "debug-dump"])
def test_nothing_accepted_restores_every_member(debug):
    kw = dict(outputs=OUTS | A.OUT_DEBUG, math=A.MATH_VALIDATION) if debug else {}
    e, P, ms, cur = resampled("many", **kw)
    with e:
        before = members(e)
        M, S = e.nmembers, e.nsites
        # (a) FLAT bounds on aMax at the members' own range and a huge scale: every proposal leaves them
        lo_a, hi_a = float(before["params"][P_["aMax"]].min()), float(before["params"][P_["aMax"]].max())
        rows = [(P_["aMax"], I, 0.0, 0.0, FLAT, lo_a, hi_a)] + ROWS[2:3]
        z = normals(2, M)
        phin, valid, rdiag, _ = proposal_reference(before["params"], before["status"], cur, ms, S, rows, np.full(S, 1e9), z)
        assert not valid.any()
        diag = mh(e, rows, np.full(S, 1e9), np.full(S, 1.0), cur, z, np.full(M, -np.inf))
        all_equal(members(e), before)
        assert np.array_equal(diag[:, :2], rdiag) and np.array_equal(diag[:, 2], rdiag[:, 0]) and (diag[:, 3] == 0).all()
        # (b) log u = 0 and a current log-likelihood no run reaches: delta < 0 for every member
        high = np.full(M, 1e12)
        z = normals(len(ROWS), M)
        phin, valid, rdiag, _ = proposal_reference(before["params"], before["status"], high, ms, S, ROWS, scales(S), z)
        diag = mh(e, ROWS, scales(S), np.full(S, 1.0), high, z, np.zeros(M))
        all_equal(members(e), before)
        assert np.array_equal(diag[:, :2], rdiag) and (diag[:, 3] == 0).all()
        assert diag[:, 2].sum() == rdiag[:, 0][~np.isnan(scales(S))].sum() - valid.sum()


@gpu
@pytest.mark.parametrize("tau", [0.0, 0.4, 1.0])
def test_mixed_decisions_follow_delta(tau):
    a, _, ms, cur = resampled("many")
    b, _, _, _ = resampled("many")
    with a, b:
        M, S = a.nmembers, a.nsites
        before = members(b)
        scale, z = scales(S), normals(len(ROWS), M)
        log_u = np.log(np.random.default_rng(9).uniform(size=M))
        da = mh(a, ROWS, scale, np.full(S, tau), cur, z, np.full(M, -np.inf))     # twin: every valid proposal run
        prop = members(a)
        db = mh(b, ROWS, scale, np.full(S, tau), cur, z, log_u)
        got = members(b)
        assert np.array_equal(da[:, :3], db[:, :3])
        _, valid, _, _ = proposal_reference(before["params"], before["status"], cur, ms, S, ROWS, scale, z)
        moving = valid & ~np.isnan(scale)[ms]
        # the twin keeps exactly the valid proposals whose run ends finite and not excluded
        ran_ok = (prop["params"] != before["params"]).any(axis=0)
        assert not (ran_ok & ~moving).any() and ran_ok.sum() > 0.9 * moving.sum()
        cols = np.arange(M)
        with np.errstate(all="ignore"):
            d = delta(tau, prop["ll"], cur, lp_rows(prop["params"], ROWS, cols), lp_rows(before["params"], ROWS, cols))
        clear = np.abs(log_u - d) >= 1e-9 * (1 + np.abs(d))
        accept = ran_ok & (log_u < d)
        assert accept.any() and (ran_ok & ~accept).any()
        for m in range(M):
            if ran_ok[m] and not clear[m]:
                continue
            assert member_equal(got, prop if accept[m] else before, m), m
        if clear[ran_ok].all():
            assert np.array_equal(db[:, 3], np.bincount(ms[accept], minlength=S).astype(float))


# ---- posterior correctness: a tempered resample-move loop against quadrature on a grid ------------------------------
AMAX = P_["aMax"]
A_LO, A_HI, A_TRUE = 20.0, 90.0, 53.2895432752984


def amax_site():
    s = synth.synth_site(5, 1, "half-daily")
    return s


def amax_handle(theta, sigma, obs=None, outputs=A.OUT_LOGLIK):
    site = amax_site()
    site.nee_obs = obs
    P = np.repeat(synth.base_param_vector()[:, None], theta.size, axis=1)
    P[AMAX] = theta
    return api.Ensemble([site], P, None, synth.SYNTH_FLAGS, outputs=outputs, math=A.MATH_FAST, nee_sigma=sigma)


def ess(lw):
    w = np.exp(lw - lw.max())
    return w.sum() ** 2 / (w * w).sum()


@gpu
def test_tempered_resample_move_reaches_the_grid_posterior():
    with amax_handle(np.array([A_TRUE]), 1.0, outputs=A.OUT_FULL) as t:
        t.run()
        obs = t.output()[A.O["nee"], :, 0].copy()
    T = obs.size
    obs[np.arange(T) % 3 == 1] = np.nan                       # a third of the steps unobserved
    # the grid: 512 values of theta; with sigma = 1 the log-likelihood is -SS / 2 + const, so any sigma follows
    grid = np.linspace(A_LO, A_HI, 514)[1:-1]
    with amax_handle(grid, 1.0, obs) as g:
        g.run()
        l1 = g.loglik()
    ss = -2.0 * (l1 - l1.max())
    # sigma that makes the posterior sd about a twelfth of the prior range (well resolved by the grid)
    sigma = 1.0
    for _ in range(60):
        w = np.exp(-ss / (2 * sigma * sigma))
        sd = math.sqrt(np.sum(w * grid * grid) / w.sum() - (np.sum(w * grid) / w.sum()) ** 2)
        sigma *= (((A_HI - A_LO) / 12) / sd) ** 0.5
    w = np.exp(-ss / (2 * sigma * sigma))
    g_mean = float(np.sum(w * grid) / w.sum())
    g_sd = math.sqrt(float(np.sum(w * grid * grid) / w.sum()) - g_mean ** 2)
    assert 20 * (grid[1] - grid[0]) < g_sd < (A_HI - A_LO) / 6
    # the sampler: N members from the prior (uniform theta), tempered to tau = 1
    N = 4096
    rng = np.random.default_rng(17)
    with amax_handle(rng.uniform(A_LO, A_HI, N), sigma, obs) as e:
        e.run()
        cur = e.loglik()
        tau, stage, rates = 0.0, 0, []
        rows = [(AMAX, G, A_LO, A_HI, FLAT, A_LO, A_HI)]
        while tau < 1.0:
            lo, hi = tau, 1.0                                  # ESS bisection: the next tau keeps half the ESS
            if ess((1.0 - tau) * cur) < N / 2:
                for _ in range(60):
                    mid = 0.5 * (lo + hi)
                    lo, hi = (mid, hi) if ess((mid - tau) * cur) >= N / 2 else (lo, mid)
            nxt = hi
            anc, _ = e.resample([rng.uniform()], math.inf, (nxt - tau) * cur)
            cur = cur[anc]
            tau = nxt
            for _ in range(3):
                th0 = e.params()[AMAX]
                diag = mh(e, rows, [2.38], [tau], cur, rng.standard_normal((1, N)), np.log(rng.uniform(size=N)))
                th1 = e.params()[AMAX]
                acc = th1 != th0
                assert diag[0, 3] == acc.sum()
                cur = np.where(acc, e.loglik(), cur)
                rates.append(acc.mean())
            stage += 1
            assert stage < 40
        theta = e.params()[AMAX]
    assert all(0.05 < r < 0.95 for r in rates), rates
    # Monte Carlo bound: with an SMC inefficiency below 16 (ESS >= N / 16), the posterior mean's standard error is at
    # most g_sd / 16; four of them are g_sd / 4.  The sd's relative error is bounded by the same 1/4.
    assert abs(theta.mean() - g_mean) < g_sd / 4, (theta.mean(), g_mean, g_sd)
    assert abs(theta.std() / g_sd - 1.0) < 0.25, (theta.std(), g_sd)


# ---- teams, partitions, launches, arguments ----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_team_of_one_equals_handle(kind):
    res = []
    for team in (False, True):
        e, _, ms = forecast(kind)
        with e:
            S, M, cur = e.nsites, e.nmembers, e.loglik()
            args = (ROWS, scales(S), np.full(S, 0.5), cur, normals(len(ROWS), M), np.log(np.random.default_rng(2).uniform(size=M)))
            if team:
                e.join_team(1, 0)
                r = [x[0] for x in ROWS]
                diag = e.team_mh_move(r, [x[1] for x in ROWS], [x[4] for x in ROWS], [x[5] for x in ROWS],
                                      [x[6] for x in ROWS], *args[1:], [x[2] for x in ROWS], [x[3] for x in ROWS])
            else:
                diag = mh(e, *args)
            res.append((diag, members(e)))
    assert np.array_equal(res[0][0], res[1][0])
    all_equal(res[0][1], res[1][1])


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
        S, M = one.nsites, one.nmembers
        cur = one.loglik()
        assert np.array_equal(multi.loglik(), cur)
        p0, st0 = one.params(), one.status()
        scale, z = scales(S), normals(len(ROWS), M)
        log_u = np.log(np.random.default_rng(6).uniform(size=M))
        d1 = mh(one, ROWS, scale, np.full(S, 1.0), cur, z, log_u)
        dm = mh(multi, ROWS, scale, np.full(S, 1.0), cur, z, log_u)
        g1, gm = one.params(), multi.params()
        assert np.array_equal(dm[:, :3], d1[:, :3]) and (d1[:, 3] > 0).any()
        acc1 = (g1 != p0).any(axis=0)
        accm = (gm != p0).any(axis=0)
        # Decisions agree member by member: a tie |log u - delta| below the proposals' 1e-9 relative difference has
        # probability near 1e-6 over these members and does not occur at these seeds.
        assert np.array_equal(acc1, accm) and np.array_equal(dm[:, 3], d1[:, 3])
        if kind != "one":
            assert np.array_equal(gm, g1)
            for x, y in ((multi.state(), one.state()), (multi.loglik(), one.loglik()), (multi.status(), one.status())):
                assert np.array_equal(x, y, equal_nan=True)
        else:
            phin, _, _, sd = proposal_reference(p0, st0, cur, ms, S, ROWS, scale, z)
            assert within_bound(gm, phin, sd, ms, ROWS, np.nonzero(acc1)[0])
            assert np.array_equal(gm[:, ~acc1], g1[:, ~acc1])
            assert np.array_equal(multi.status(), one.status())


@gpu
def test_launches_do_not_grow_with_sites():
    per_call = []
    for n in (3, 300):
        sites, P, ms, _ = synth.config_c3(nsites=n, members_per_site=10, nyears=1)
        with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK, math=A.MATH_FAST) as e:
            e.run(0, 100)
            M = e.nmembers
            args = ([P_["aMax"], P_["halfSatPar"]], [I, L], [FLAT, FLAT], [-np.inf, 0.0], [np.inf, np.inf],
                    np.full(n, 0.5), np.full(n, 1.0), e.loglik(), normals(2, M), np.zeros(M))
            c0 = e.launch_count()
            e.mh_move(*args)
            c1 = e.launch_count()
            e.mh_move(*args)
            per_call.append((c1 - c0, e.launch_count() - c1))
            # every scale NaN: nothing is launched and the run range stays
            out = e.loglik()
            c2 = e.launch_count()
            diag = e.mh_move(*args[:5], np.full(n, np.nan), *args[6:])
            assert e.launch_count() == c2 and np.array_equal(e.loglik(), out)
            assert np.isnan(diag[:, 0]).all() and (diag[:, 1] == -1).all() and (diag[:, 2:] == 0).all()
    # moments (4), snapshot, proposal, reset, the optimistic run and its replay, accept, counts
    assert per_call[0] == per_call[1] and per_call[0][0] == per_call[0][1] == 11


@gpu
def test_rejected_arguments_leave_everything_untouched():
    e, _, _ = forecast(("c3", 4, 50))
    twin, _, _ = forecast(("c3", 4, 50))
    with e, twin:
        before = members(e)
        lib = e.lib
        M = e.nmembers
        good = dict(rows=[P_["aMax"], P_["fAnoxia"]], tf=[I, G], lo=[0.0, 0.0], hi=[0.0, 0.55], prior=[FLAT, NORMAL],
                    pa=[-np.inf, 0.0], pb=[np.inf, 1.0], scale=np.full(4, 0.5), tau=np.full(4, 0.5), cur=e.loglik(),
                    z=normals(2, M), lu=np.zeros(M))

        def rc_of(fn=lib.sipnet_gpu_mh_move, target=e.handle, null=None, n_rows=None, **kw):
            a = dict(good, **kw)
            spec, keep = e.mh_spec(a["rows"], a["tf"], a["prior"], a["pa"], a["pb"], a["scale"], a["tau"], a["cur"],
                                   a["z"], a["lu"], a["lo"], a["hi"])
            if n_rows is not None:
                spec.n_rows = n_rows
            if null:
                setattr(spec, null, None)
            return fn(target, None if null == "spec" else C.byref(spec), None)

        def with_(name, i, v):
            x = np.array(good[name], dtype=np.float64 if name not in ("rows", "prior", "tf") else np.int32)
            x.flat[i] = v
            return {name: x}

        cases = {"NULL handle": lambda: rc_of(target=None), "NULL spec": lambda: rc_of(null="spec"),
                 "n_rows 0": lambda: rc_of(n_rows=0), "n_rows 17": lambda: rc_of(n_rows=17),
                 "NaN z": lambda: rc_of(**with_("z", 17, np.nan)), "inf z": lambda: rc_of(**with_("z", 3, -np.inf)),
                 "repeated row": lambda: rc_of(rows=[P_["aMax"], P_["aMax"]]),
                 "psnTMax": lambda: rc_of(rows=[P_["psnTMax"], P_["aMax"]]),
                 "row 80": lambda: rc_of(rows=[80, P_["aMax"]]), "transform 3": lambda: rc_of(tf=[I, 3]),
                 "lo = hi": lambda: rc_of(hi=[0.0, 0.0]), "prior 2": lambda: rc_of(prior=[FLAT, 2]),
                 "prior -1": lambda: rc_of(prior=[-1, NORMAL]),
                 "FLAT a = b": lambda: rc_of(pa=[1.0, 0.0], pb=[1.0, 1.0]),
                 "FLAT a > b": lambda: rc_of(pa=[2.0, 0.0], pb=[1.0, 1.0]),
                 "FLAT NaN": lambda: rc_of(pa=[np.nan, 0.0]),
                 "FLAT outside LOGIT": lambda: rc_of(prior=[FLAT, FLAT], pa=[-np.inf, 0.0], pb=[np.inf, 0.6]),
                 "FLAT inf on LOGIT": lambda: rc_of(prior=[FLAT, FLAT], pa=[-np.inf, -np.inf], pb=[np.inf, 0.5]),
                 "NORMAL sd 0": lambda: rc_of(pb=[np.inf, 0.0]), "NORMAL sd -1": lambda: rc_of(pb=[np.inf, -1.0]),
                 "NORMAL sd inf": lambda: rc_of(pb=[np.inf, np.inf]),
                 "NORMAL mean inf": lambda: rc_of(pa=[-np.inf, np.inf]),
                 "scale 0": lambda: rc_of(**with_("scale", 1, 0.0)), "scale -1": lambda: rc_of(**with_("scale", 1, -1.0)),
                 "scale inf": lambda: rc_of(**with_("scale", 1, np.inf)),
                 "tau NaN": lambda: rc_of(**with_("tau", 2, np.nan)), "tau 1.5": lambda: rc_of(**with_("tau", 2, 1.5)),
                 "tau -0.1": lambda: rc_of(**with_("tau", 2, -0.1)),
                 "tau NaN at a site left alone": lambda: rc_of(scale=np.array([0.5, np.nan, .5, .5]),
                                                               tau=np.array([0.5, np.nan, .5, .5])),
                 "log_u NaN": lambda: rc_of(**with_("lu", 5, np.nan)), "log_u inf": lambda: rc_of(**with_("lu", 5, np.inf)),
                 "log_u > 0": lambda: rc_of(**with_("lu", 5, 1e-300))}
        for f in ("rows", "transform", "prior", "prior_a", "prior_b", "scale", "tempering", "current_loglik", "z",
                  "log_u", "lower", "upper"):
            cases[f"NULL {f}"] = lambda f=f: rc_of(null=f)
        for name, fn in cases.items():
            assert fn() == A.ERR_BAD_ARGUMENT, name
            all_equal(members(e), before)
        assert e.nrun == SEG - 200
        e.join_team(1, 0)
        assert rc_of(fn=lib.sipnet_gpu_comm_mh_move, target=e.comm, **with_("z", 1, np.nan)) == A.ERR_BAD_ARGUMENT
        assert rc_of(fn=lib.sipnet_gpu_comm_mh_move, target=e.comm, n_rows=17) == A.ERR_BAD_ARGUMENT
        e.run(SEG, SEG + 100)
        twin.run(SEG, SEG + 100)
        all_equal(members(e), members(twin))
        assert np.array_equal(e.output(), twin.output(), equal_nan=True)
    # s = 0, and tau > 0 without a log-likelihood
    sites, P, ms = config(("c3", 2, 20))
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK) as f, \
            api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_FULL, out_steps_capacity=50) as g:
        args = ([P_["aMax"]], [I], [FLAT], [-np.inf], [np.inf], np.full(2, 0.5), np.full(2, 0.5), np.zeros(40),
                normals(1, 40), np.zeros(40))
        with pytest.raises(api.SipnetGpuError):
            f.mh_move(*args)
        g.run(0, 50)
        p0 = g.params()
        with pytest.raises(api.SipnetGpuError):
            g.mh_move(*args)
        assert np.array_equal(g.params(), p0) and g.nrun == 50
        g.mh_move(*args[:6], np.array([0.0, 0.0]), *args[7:])          # tau = 0 needs no log-likelihood
    multi, _, _ = forecast(("c3", 4, 50), cls=api.MultiEnsemble, devices=[0, 0])
    with multi:
        p0 = multi.params()
        M = multi.nmembers
        lu = np.zeros(M)
        lu[3] = np.nan
        spec, keep = multi.mh_spec([P_["aMax"]], [I], [FLAT], [-np.inf], [np.inf], np.full(4, 0.5), np.full(4, 0.5),
                                   np.zeros(M), normals(1, M), lu)
        assert lib.sipnet_gpu_multi_mh_move(multi.multi, C.byref(spec), None) == A.ERR_BAD_ARGUMENT
        assert np.array_equal(multi.params(), p0)
