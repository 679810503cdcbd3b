"""Prior covariance inflation before the EAKF, fixed or adaptive per site (sipnet_gpu_assimilate_inflated and its comm /
multi variants; sip_assim.cu).

CPU: a numpy reference of the inflation (math.fsum means) and of Anderson's adaptive update (the cubic through
numpy.roots, Newton-polished, plus the bounds; the density-ratio rule for the spread), on top of the EAKF reference of
test_gpu_assimilate; its properties; a seeded scalar random walk in which the EAKF without inflation is overconfident
and the adaptive scheme is not; the ctypes mirror of sipnet_gpu_inflation_spec against the C layout.
GPU: synth ensembles after a one-year forecast, against the reference (state within 1e-9 x prior sd + 4 ulp, N and
the floor bit exact, lambda and its sd within 1e-10 relative); calls that inflate nothing are bit-identical to
sipnet_gpu_assimilate; what must not change stays bit-identical; inflation of unobserved sites and its floor; three
forecast -> analysis cycles; teams and multi-GPU partitions; launches per call; rejected arguments.
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
from test_gpu_assimilate import eakf_reference, obs_for, prior_sd, within_bound

POOLS = list(range(12))
EXCLUDED = A.ST_BAD_ALLOCATION | A.ST_NONFINITE
S = A.S


# ---- the reference ---------------------------------------------------------------------------------------------------
def log_posterior(lam, lp, v, sp2, r, d2):
    """g(lambda) of include/sipnet_gpu.h."""
    w = lam * sp2 + r
    return -(lam - lp) ** 2 / (2 * v) - 0.5 * math.log(w) - d2 / (2 * w)


def adapt_reference(lam, sd, sp2, d, r, lo, hi, sd_min):
    """One adaptive update -> (lambda, sd): the argmax of g over the cubic's real roots in [lo, hi] and the bounds."""
    v, d2 = sd * sd, d * d

    def P(x):
        w = x * sp2 + r
        return 2 * (x - lam) * w * w + v * sp2 * (w - d2)

    def dP(x):
        w = x * sp2 + r
        return 2 * w * w + 4 * sp2 * (x - lam) * w + v * sp2 * sp2

    coef = [2 * sp2 * sp2, 4 * sp2 * r - 2 * sp2 * sp2 * lam, 2 * r * r - 4 * sp2 * r * lam + v * sp2 * sp2,
            -2 * lam * r * r + v * sp2 * r - v * sp2 * d2]
    cands = [lo, hi]
    for z in np.roots(coef):
        if abs(z.imag) > 1e-6 * max(1.0, abs(z.real)):
            continue
        x = float(z.real)
        for _ in range(4):                                    # polish: numpy.roots is good to a few ulp of the scale
            q = dP(x)
            if q == 0:
                break
            x -= P(x) / q
        if lo <= x <= hi:
            cands.append(x)
    best, gbest = None, -math.inf
    for x in sorted(cands):
        gx = log_posterior(x, lam, v, sp2, r, d2)
        if gx > gbest:
            best, gbest = x, gx
    delta = gbest - log_posterior(best + sd, lam, v, sp2, r, d2)
    sd_new = min(sd, math.sqrt(v / (2 * delta))) if delta > 0 and math.isfinite(delta) else sd
    return best, max(sd_min, sd_new)


def takers(X, st, member_site, s, rows):
    idx = np.nonzero(member_site == s)[0]
    ok = ((st[idx] & EXCLUDED) == 0) & np.all(np.isfinite(X[rows][:, idx]), axis=0)
    return idx[ok]


def inflate_reference(state, status, member_site, nsites, rows, lam):
    """The prior inflation alone: -> (state, inflated[nsites])."""
    X = np.array(state, dtype=np.float64, copy=True)
    inflated = np.zeros(nsites, bool)
    for s in range(nsites):
        idx = takers(X, status, member_site, s, rows)
        l0 = lam[s]
        if not (math.isfinite(l0) and l0 != 1.0 and idx.size >= 2):
            continue
        f = math.sqrt(l0)
        for row in rows:
            x = X[row, idx]
            xbar = math.fsum(x) / idx.size
            X[row, idx] = xbar + f * (x - xbar)
        inflated[s] = True
    return X, inflated


def inflated_reference(state, status, member_site, nsites, rows, op, value, variance, lam, lam_sd=None,
                       bounds=(1.0, 100.0), sd_min=0.0, floor=True):
    """sipnet_gpu_assimilate_inflated of include/sipnet_gpu.h -> (state, status, diag, lambda, lambda_sd)."""
    lam = np.array(lam, dtype=np.float64)
    sd = None if lam_sd is None else np.array(lam_sd, dtype=np.float64)
    X, inflated = inflate_reference(state, status, member_site, nsites, rows, lam)
    X, st, diag = eakf_reference(X, status, member_site, nsites, rows, op, value, variance, floor=False)
    updated = inflated | np.isfinite(diag[:, :, 1]).any(axis=1)
    for s in np.nonzero(updated)[0] if floor else []:
        idx = takers(X, st, member_site, s, rows)
        sub = X[rows][:, idx]
        neg = sub < 0
        sub[neg] = 0.0
        X[np.ix_(rows, idx)] = sub
        st[idx[neg.any(axis=0)]] |= A.ST_ANALYSIS_FLOORED
    lam0 = lam.copy()
    for s in range(nsites) if sd is not None else []:
        if not (sd[s] > 0 and math.isfinite(lam0[s])):
            continue
        for k in range(diag.shape[1]):
            if math.isfinite(diag[s, k, 1]):
                lam[s], sd[s] = adapt_reference(lam[s], sd[s], diag[s, k, 2] / lam0[s], value[s, k] - diag[s, k, 1],
                                                variance[s, k], bounds[0], bounds[1], sd_min)
    return X, st, diag, lam, sd


def random_walk(cycles=400, members=50, seed=1, adaptive=True):
    """The scalar toy: truth x += N(0, q), members x += N(0, (sqrt(q) / 4)^2) (a quarter of the truth's noise sd),
    y = x + N(0, r), q = r = 1; each cycle one EAKF analysis through the reference, adaptive from lambda = 1, sd = 1
    (sd_min 0.1) or without inflation.  -> (d^2 / (s2 + r) per cycle, lambda per cycle)."""
    rng = np.random.default_rng(seed)
    q = r = 1.0
    truth = 0.0
    X = np.zeros((1, members))
    X[0] = rng.normal(0.0, 1.0, members)
    status = np.zeros(members, np.uint32)
    ms = np.zeros(members, np.int32)
    lam, sd = np.array([1.0]), (np.array([1.0]) if adaptive else None)
    nis, lams = [], []
    for _ in range(cycles):
        truth += rng.normal(0.0, math.sqrt(q))
        X[0] += rng.normal(0.0, 0.25 * math.sqrt(q), members)
        y = truth + rng.normal(0.0, math.sqrt(r))
        X, _, diag, lam, sd = inflated_reference(X, status, ms, 1, [0], np.ones((1, 1)), np.array([[y]]),
                                                 np.array([[r]]), lam, sd, sd_min=0.1, floor=False)
        _, ybar, s2, _ = diag[0, 0]
        nis.append((y - ybar) ** 2 / (s2 + r))
        lams.append(lam[0])
    return np.array(nis), np.array(lams)


def toy_state(seed=5, M=300, nsites=2):
    rng = np.random.default_rng(seed)
    state = np.zeros((A.NSTATE, M))
    state[POOLS] = rng.normal(50.0, 4.0, (12, M))
    state[S["soilC"]] += 0.7 * state[S["plantWoodC"]]
    return state, np.zeros(M, np.uint32), np.repeat(np.arange(nsites, dtype=np.int32), M // nsites)


def test_fixed_inflation_scales_the_covariance_and_keeps_the_means():
    state, status, ms = toy_state()
    lam = np.array([1.7, np.nan])
    X, inflated = inflate_reference(state, status, ms, 2, POOLS, lam)
    assert list(inflated) == [True, False]
    a, b = state[POOLS][:, ms == 0], X[POOLS][:, ms == 0]
    np.testing.assert_allclose(np.cov(b), 1.7 * np.cov(a), rtol=1e-12)
    np.testing.assert_allclose(b.mean(axis=1), a.mean(axis=1), rtol=1e-13)
    assert np.array_equal(X[:, ms == 1], state[:, ms == 1])
    # and the EAKF after it sees the inflated variance
    op = np.eye(12)[[S["plantWoodC"]]]
    _, _, diag, lam1, sd1 = inflated_reference(state, status, ms, 2, POOLS, op, np.array([[50.0], [50.0]]),
                                               np.array([[4.0], [4.0]]), lam)
    np.testing.assert_allclose(diag[0, 0, 2], 1.7 * np.var(a[S["plantWoodC"]], ddof=1), rtol=1e-12)
    assert np.array_equal(lam1, lam, equal_nan=True) and sd1 is None


def test_large_sd_approaches_the_clamped_maximum_likelihood():
    sp2, r = 2.0, 1.0
    for d, want in ((3.0, (9.0 - 1.0) / 2.0), (10.0, 20.0), (0.1, 1.0)):     # interior, clamped above, below
        lam, sd = adapt_reference(1.5, 1e4, sp2, d, r, 1.0, 20.0, 0.0)
        assert lam == pytest.approx(want, rel=1e-3), d
        assert sd <= 1e4


def test_zero_sd_keeps_lambda():
    state, status, ms = toy_state()
    op = np.eye(12)[[S["plantWoodC"]]]
    value, var = np.array([[80.0], [20.0]]), np.array([[1.0], [1.0]])
    for sd in (np.zeros(2), None):
        _, _, _, lam, sd1 = inflated_reference(state, status, ms, 2, POOLS, op, value, var, [1.3, 2.0], sd)
        assert list(lam) == [1.3, 2.0]
        assert sd1 is None if sd is None else list(sd1) == [0.0, 0.0]


def test_lambda_follows_the_innovation():
    sp2, r, lam = 3.0, 2.0, 2.0
    expect = lam * sp2 + r                                                   # 8
    for d2, up in ((30.0, True), (20.0, True), (4.0, False), (0.5, False)):
        new, _ = adapt_reference(lam, 0.5, sp2, math.sqrt(d2), r, 0.5, 10.0, 0.0)
        assert (new > lam) if up else (new < lam), (d2, new)
        assert (d2 > expect) == up


def test_sd_never_grows_and_the_clamps_hold():
    rng = np.random.default_rng(11)
    for _ in range(2000):
        lo = rng.uniform(0.2, 1.0)
        hi = lo + rng.uniform(0.0, 5.0)
        lam = rng.uniform(lo, hi)
        sd = rng.uniform(0.01, 3.0)
        sd_min = rng.uniform(0.0, sd)
        new, sd1 = adapt_reference(lam, sd, rng.uniform(0.01, 10.0), rng.normal(0, 5.0), rng.uniform(0.01, 5.0), lo,
                                   hi, sd_min)
        assert lo <= new <= hi
        assert sd_min <= sd1 <= sd


def test_adaptive_inflation_keeps_a_random_walk_consistent():
    nis, lams = random_walk()
    nis0, _ = random_walk(adaptive=False)
    assert abs(nis.mean() - 1.0) < 0.1, nis.mean()
    assert nis0.mean() > 1.5, nis0.mean()
    assert lams[-100:].mean() > 1.2


def test_ctypes_inflation_spec_matches_c_layout():
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "sipnet_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu\n", sizeof(sipnet_gpu_inflation_spec), offsetof(sipnet_gpu_inflation_spec, lambda),
         offsetof(sipnet_gpu_inflation_spec, lambda_sd), offsetof(sipnet_gpu_inflation_spec, lambda_min),
         offsetof(sipnet_gpu_inflation_spec, lambda_max), offsetof(sipnet_gpu_inflation_spec, sd_min));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        got = list(map(int, subprocess.check_output([exe]).decode().split()))
    F = A.InflationSpec
    assert got == [C.sizeof(F), F.lambda_.offset, F.lambda_sd.offset, F.lambda_min.offset, F.lambda_max.offset,
                   F.sd_min.offset]


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
OUTS = A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS
KW = dict(outputs=OUTS, summary_cols=[A.O["nee"], A.O["plantWoodC"]], quantiles=[0.05, 0.5, 0.95], math=A.MATH_FAST,
          nee_sigma=0.5, max_event_records=16)
YEAR = 730
BOUNDS = (1.0, 100.0)


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def config(kind, nyears=1):
    """'one': one site of 5 000 members; 'many': 40 sites of 100; ('c3', n, m): n sites of m (as test_gpu_assimilate)."""
    n, m = (1, 5000) if kind == "one" else (40, 100) if kind == "many" else kind[1:]
    sites = [synth.synth_site(3 + s, nyears, "half-daily") for s in range(n)]
    P, ms = synth.synth_params(n * m, stream=21), np.repeat(np.arange(n, dtype=np.int32), m)
    rng = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0, 1.5, s.nsteps))
    P[A.P["leafAllocation"], 7] = 0.9                            # bad allocation: never integrated, never assimilated
    return sites, P, ms


def forecast(kind, cls=api.Ensemble, nyears=1, steps=YEAR, **kw):
    sites, P, ms = config(kind, nyears)
    e = cls(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    e.run(0, steps)
    return e, ms


def ops(nobs):
    op = np.zeros((nobs, 12))
    picks = [S["plantWoodC"], S["soilC"], S["soilWater"], S["litterC"]]
    for k in range(nobs):
        op[k, picks[k]] = 1.0
    op[0, [S["plantWoodC"], S["coarseRootC"], S["fineRootC"]]] = 1.0
    return op


def lambdas(nsites, mode, seed=4):
    """Per-site (lambda, lambda_sd): fixed -- values in [1.1, 2.5], one site NaN, one at 1; adaptive -- the same
    with sd 0.4 at most sites, 0 (fixed) at one."""
    rng = np.random.default_rng(seed)
    lam = rng.uniform(1.1, 2.5, nsites)
    if nsites > 2:
        lam[1], lam[2] = np.nan, 1.0
    if mode == "fixed":
        return lam, None
    sd = np.full(nsites, 0.4)
    if nsites > 3:
        sd[3] = 0.0
    return lam, sd


def check_against_reference(got, gstatus, gdiag, glam, gsd, st0, status0, ms, nsites, rows, op, value, var, lam, sd,
                            sd_min=0.0):
    ref, rstatus, rdiag, rlam, rsd = inflated_reference(st0, status0, ms, nsites, rows, op, value, var, lam, sd, BOUNDS,
                                                        sd_min)
    assert within_bound(got, ref, prior_sd(st0, status0, ms, nsites), ms, rows)
    assert np.array_equal(gstatus, rstatus)
    assert np.array_equal(gdiag[..., 0], rdiag[..., 0])
    np.testing.assert_allclose(gdiag[..., 1:], rdiag[..., 1:], rtol=1e-9, equal_nan=True)
    np.testing.assert_allclose(glam, rlam, rtol=1e-10, equal_nan=True)
    if sd is None:
        assert gsd is None
    else:
        np.testing.assert_allclose(gsd, rsd, rtol=1e-10)
    return rlam, rsd


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
@pytest.mark.parametrize("mode", ["fixed", "adaptive"])
def test_matches_reference(kind, mode):
    e, ms = forecast(kind)
    with e:
        st0, status0 = e.state(), e.status()
        op = ops(4)
        value, var = obs_for(st0, ms, e.nsites, op, shift=1.5)
        lam, sd = lambdas(e.nsites, mode)
        lam_in, sd_in = lam.copy(), None if sd is None else sd.copy()
        diag, glam, gsd = e.assimilate_inflated(POOLS, op, value, var, lam, sd, BOUNDS)
        assert np.array_equal(lam, lam_in, equal_nan=True)                   # the inputs are not modified
        assert sd is None or np.array_equal(sd, sd_in)
        rlam, _ = check_against_reference(e.state(), e.status(), diag, glam, gsd, st0, status0, ms, e.nsites, POOLS,
                                          op, value, var, lam, sd)
    if mode == "adaptive":
        moved = np.isfinite(lam) & (sd > 0)
        assert (rlam[moved] != lam[moved]).mean() > 0.5
        assert np.array_equal(glam[~moved], lam[~moved], equal_nan=True)
        assert np.array_equal(gsd[~moved], sd[~moved])


@gpu
def test_inflating_nothing_is_assimilate():
    nsites = 40
    cases = {"lambda 1, sd 0": (np.ones(nsites), np.zeros(nsites)), "lambda NaN": (np.full(nsites, np.nan), None),
             "lambda 1, no sd": (np.ones(nsites), None)}
    e, ms = forecast("many")
    with e:
        op = ops(4)
        value, var = obs_for(e.state(), ms, nsites, op)
        c0 = e.launch_count()
        d0 = e.assimilate(POOLS, op, value, var)
        want = (e.state(), e.status(), d0, e.launch_count() - c0)
    for name, (lam, sd) in cases.items():
        e, _ = forecast("many")
        with e:
            c0 = e.launch_count()
            diag, glam, gsd = e.assimilate_inflated(POOLS, op, value, var, lam, sd)
            got = (e.state(), e.status(), diag, e.launch_count() - c0)
        for x, y in zip(got, want):
            assert np.array_equal(x, y, equal_nan=True), name
        assert np.array_equal(glam, lam, equal_nan=True), name
        assert (gsd is None) == (sd is None), name


def snapshot(e):
    return dict(state=e.state(), status=e.status(), ring=e.ring(), ll=e.loglik(), counts=e.event_counts(),
                mean=e.mean(), var=e.variance(), q=e.quantiles())


@gpu
def test_untouched_data():
    e, ms = forecast("many")
    with e:
        before = snapshot(e)
        st = before["state"]
        rows = [S["plantWoodC"], S["soilC"], S["litterC"], S["minN"]]
        op = np.array([[1.0, 0.0, 0.0, 0.0]])
        value, var = obs_for(st, ms, e.nsites, np.eye(12)[[S["plantWoodC"]]])
        value[1] = np.nan                                                     # site 1: lambda NaN and unobserved
        lam, sd = lambdas(e.nsites, "adaptive")
        lam[[5, 9]] = np.nan
        diag, glam, gsd = e.assimilate_inflated(rows, op, value, var, lam, sd)
        after = snapshot(e)
    unlisted = [r for r in range(A.NSTATE) if r not in rows]
    assert np.array_equal(after["state"][unlisted], before["state"][unlisted], equal_nan=True)
    for key in ("ll", "counts", "mean", "var", "q"):
        assert np.array_equal(after[key], before[key], equal_nan=True), key
    for a, b in zip(after["ring"], before["ring"]):
        assert np.array_equal(a, b)
    floor = np.uint32(A.ST_ANALYSIS_FLOORED)
    assert np.array_equal(after["status"] & ~floor, before["status"])
    keep = ((before["status"] & EXCLUDED) != 0) | (ms == 1)
    assert keep[7]                                                            # bad allocation: does not take part
    assert np.array_equal(after["state"][:, keep], before["state"][:, keep], equal_nan=True)
    assert not (after["status"][keep] & floor).any()
    for s in (5, 9):                                                          # lambda NaN: no inflation, no update
        assert np.isnan(glam[s]) and gsd[s] == sd[s]
    check_against_reference(after["state"], after["status"], diag, glam, gsd, before["state"], before["status"], ms,
                            e.nsites, rows, op, value, var, lam, sd)


@gpu
def test_unobserved_sites_are_inflated_and_floored():
    e, ms = forecast("many")
    with e:
        st, status = e.state(), e.status()
        rv, rw = e.ring()
        row = S["litterC"]
        zero = int(np.nonzero((ms == 2) & ((status & EXCLUDED) == 0))[0][3])
        st[row, zero] = 0.0                                                   # a pool at 0, the site mean above 0
        e.set_state(st, rv, rw, next_step=YEAR)
        status = e.status()
        op = ops(2)
        value, var = obs_for(st, ms, e.nsites, op)
        value[2] = value[4] = np.nan                                          # sites 2 and 4: no observation
        lam = np.ones(e.nsites)
        lam[2], lam[4] = 1.8, 1.0
        diag, glam, _ = e.assimilate_inflated(POOLS, op, value, var, lam)
        got, gstatus = e.state(), e.status()
    assert st[row, ms == 2].mean() > 0
    assert got[row, zero] == 0.0 and not np.signbit(got[row, zero])
    assert gstatus[zero] & A.ST_ANALYSIS_FLOORED
    site2 = (ms == 2) & ((status & EXCLUDED) == 0)
    wood = S["plantWoodC"]
    assert (got[wood, site2] != st[wood, site2]).mean() > 0.9                # inflated though unobserved
    assert np.array_equal(got[:, ms == 4], st[:, ms == 4], equal_nan=True)   # lambda 1 and unobserved: untouched
    assert np.array_equal(gstatus[ms == 4], status[ms == 4])
    assert np.isnan(diag[[2, 4], :, 1:]).all()
    check_against_reference(got, gstatus, diag, glam, None, st, status, ms, e.nsites, POOLS, op, value, var, lam, None)


@gpu
def test_three_cycles():
    kind, seg = ("c3", 10, 100), 180
    kw = dict(outputs=A.OUT_FULL, out_steps_capacity=seg)
    sites, P, ms = config(kind)
    a = api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    b = api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    with a, b:
        lam, sd = np.full(10, 1.0), np.full(10, 0.6)
        a.run(0, seg)
        op = ops(4)
        for cycle in range(3):
            st0, status0 = a.state(), a.status()
            value, var = obs_for(st0, ms, 10, op, shift=2.0, seed=cycle)
            diag, glam, gsd = a.assimilate_inflated(POOLS, op, value, var, lam, sd, BOUNDS, sd_min=0.05)
            check_against_reference(a.state(), a.status(), diag, glam, gsd, st0, status0, ms, 10, POOLS, op, value,
                                    var, lam, sd, sd_min=0.05)
            if cycle > 0:
                assert (glam != lam).any()
            lam, sd = glam, gsd
            rv, rw = a.ring()
            t = (cycle + 1) * seg
            b.set_state(a.state(), rv, rw, next_step=t)
            a.run(t, t + seg)
            b.run(t, t + seg)
            assert np.array_equal(a.output(), b.output(), equal_nan=True), cycle
            assert np.array_equal(a.state(), b.state(), equal_nan=True), cycle
        assert (lam > 1.0).mean() > 0.5


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_team_of_one_equals_handle(kind):
    res = []
    for team in (False, True):
        e, ms = forecast(kind)
        with e:
            op = ops(4)
            value, var = obs_for(e.state(), ms, e.nsites, op, shift=1.5)
            lam, sd = lambdas(e.nsites, "adaptive")
            if team:
                e.join_team(1, 0)
                out = e.team_assimilate_inflated(POOLS, op, value, var, lam, sd)
            else:
                out = e.assimilate_inflated(POOLS, op, value, var, lam, sd)
            res.append((e.state(), e.status()) + out)
    for x, y in zip(*res):
        assert np.array_equal(x, y, equal_nan=True)


needs2 = pytest.mark.skipif("ngpus() < 2", reason="needs two GPUs on the box")
DEVICES = [pytest.param(None, marks=needs2, id="all-gpus"), pytest.param([0, 0], id="loopback2"),
           pytest.param([0, 0, 0], id="loopback3"), pytest.param([0] * 5, id="loopback5")]


@gpu
@pytest.mark.parametrize("devices", DEVICES)
def test_multi_split_site(devices):
    kw = dict(outputs=A.OUT_FULL, out_steps_capacity=YEAR)
    one, ms = forecast("one", nyears=2, **kw)
    multi, _ = forecast("one", cls=api.MultiEnsemble, nyears=2, devices=devices, **kw)
    with one, multi:
        assert multi.ndevices >= 2
        st0, status0 = one.state(), one.status()
        op = ops(4)
        value, var = obs_for(st0, ms, 1, op, shift=1.5)
        lam, sd = np.array([1.4]), np.array([0.5])
        d1, l1, s1 = one.assimilate_inflated(POOLS, op, value, var, lam, sd)
        dm, lm, sm = multi.assimilate_inflated(POOLS, op, value, var, lam, sd)
        got = multi.state()
        sdp = prior_sd(st0, status0, ms, 1)
        assert within_bound(got, one.state(), sdp, ms, POOLS)
        check_against_reference(got, multi.status(), dm, lm, sm, st0, status0, ms, 1, POOLS, op, value, var, lam, sd)
        assert np.array_equal(multi.status(), one.status())
        assert np.array_equal(dm[..., 0], d1[..., 0])
        np.testing.assert_allclose(dm, d1, rtol=1e-12)
        np.testing.assert_allclose(lm, l1, rtol=1e-10)
        np.testing.assert_allclose(sm, s1, rtol=1e-10)
        assert lm[0] != lam[0]


@gpu
@pytest.mark.parametrize("devices", DEVICES)
def test_multi_whole_sites_bit_identical(devices):
    kw = dict(outputs=A.OUT_FULL, out_steps_capacity=YEAR)
    one, ms = forecast(("c3", 11, 40), nyears=2, **kw)
    multi, _ = forecast(("c3", 11, 40), cls=api.MultiEnsemble, nyears=2, devices=devices, **kw)
    with one, multi:
        st0 = one.state()
        op = ops(4)
        value, var = obs_for(st0, ms, 11, op, shift=1.5)
        value[4, 1] = np.nan
        value[6] = np.nan
        lam, sd = lambdas(11, "adaptive")
        r1 = one.assimilate_inflated(POOLS, op, value, var, lam, sd)
        rm = multi.assimilate_inflated(POOLS, op, value, var, lam, sd)
        for x, y in zip(rm, r1):
            assert np.array_equal(x, y, equal_nan=True)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        assert np.array_equal(multi.status(), one.status())
        one.run(YEAR, 2 * YEAR)
        multi.run(YEAR, 2 * YEAR)
        assert np.array_equal(multi.output(), one.output(), equal_nan=True)


@gpu
def test_launches_do_not_grow_with_sites():
    nobs = 2
    for n in (3, 300):
        sites, P, ms, _ = synth.config_c3(nsites=n, members_per_site=10, nyears=1)
        with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK, math=A.MATH_FAST) as e:
            e.run(0, 20)
            op = ops(nobs)
            value, var = obs_for(e.state(), ms, n, op)
            counts = []
            for call in (lambda: e.assimilate(POOLS, op, value, var),
                         lambda: e.assimilate_inflated(POOLS, op, value, var, np.ones(n), np.full(n, 0.5)),
                         lambda: e.assimilate_inflated(POOLS, op, value, var, np.full(n, 1.2)),
                         lambda: e.assimilate_inflated(POOLS, op, value, var, np.full(n, 1.2), np.full(n, 0.5))):
                c0 = e.launch_count()
                call()
                counts.append(e.launch_count() - c0)
        assert counts == [4 * nobs + 1, 4 * nobs + 1, 4 * nobs + 3, 4 * nobs + 3], (n, counts)


@gpu
def test_rejected_arguments_leave_everything_untouched():
    e, ms = forecast(("c3", 4, 50))
    with e:
        before = (e.state(), e.status())
        op = ops(2)
        value, var = obs_for(before[0], ms, 4, op)
        lib = e.lib
        good = dict(lam=np.array([1.2, 1.0, np.nan, 2.0]), sd=np.array([0.3, 0.0, 0.5, 0.2]), bounds=(1.0, 10.0),
                    sd_min=0.1)

        def rc_of(fn=lib.sipnet_gpu_assimilate_inflated, target=e.handle, value=value, patch=None, **kw):
            a = dict(good, **kw)
            spec, _k, _n = e.obs_spec(POOLS, op, value, var)
            infl, (lam, sd) = e.inflation_spec(a["lam"], a["sd"], a["bounds"], a["sd_min"])
            lam0, sd0 = lam.copy(), None if sd is None else sd.copy()
            if patch:
                patch(infl)
            rc = fn(target, C.byref(spec), C.byref(infl), None)
            if rc != 0:
                assert np.array_equal(lam, lam0, equal_nan=True)
                assert sd is None or np.array_equal(sd, sd0, equal_nan=True)
            return rc

        def lam_with(i, v):
            lam = good["lam"].copy()
            lam[i] = v
            return lam

        def sd_with(i, v):
            sd = good["sd"].copy()
            sd[i] = v
            return sd

        spec_ok, keep_ok, _n = e.obs_spec(POOLS, op, value, var)
        bad_value = value.copy()
        bad_value[1, 0] = np.inf
        cases = {
            "bad obs spec": lambda: rc_of(value=bad_value),
            "NULL infl": lambda: lib.sipnet_gpu_assimilate_inflated(e.handle, C.byref(spec_ok), None, None),
            "NULL lambda": lambda: rc_of(patch=lambda f: setattr(f, "lambda_", None)),
            "lambda 0": lambda: rc_of(lam=lam_with(1, 0.0)),
            "lambda negative": lambda: rc_of(lam=lam_with(1, -1.0)),
            "lambda inf": lambda: rc_of(lam=lam_with(1, np.inf)),
            "lambda_min 0": lambda: rc_of(bounds=(0.0, 10.0)),
            "lambda_min > lambda_max": lambda: rc_of(bounds=(3.0, 2.0)),
            "lambda_max inf": lambda: rc_of(bounds=(1.0, np.inf)),
            "lambda_min NaN": lambda: rc_of(bounds=(np.nan, 10.0)),
            "sd_min negative": lambda: rc_of(sd_min=-0.1),
            "sd_min inf": lambda: rc_of(sd_min=np.inf),
            "sd NaN": lambda: rc_of(sd=sd_with(1, np.nan)),
            "sd inf": lambda: rc_of(sd=sd_with(1, np.inf)),
            "sd negative": lambda: rc_of(sd=sd_with(1, -0.2)),
            "sd below sd_min": lambda: rc_of(sd=sd_with(0, 0.05)),
            "adaptive lambda below the bounds": lambda: rc_of(lam=lam_with(0, 0.5)),
            "adaptive lambda above the bounds": lambda: rc_of(lam=lam_with(3, 11.0)),
        }
        for name, fn in cases.items():
            assert fn() == A.ERR_BAD_ARGUMENT, name
            assert np.array_equal(e.state(), before[0], equal_nan=True), name
            assert np.array_equal(e.status(), before[1]), name
        # fixed sites may lie outside the bounds; NaN lambda with sd > 0 is fine
        assert rc_of(lam=np.array([0.5, 1.0, np.nan, 20.0]), sd=np.array([0.0, 0.0, 0.5, 0.0])) == 0
        e.join_team(1, 0)
        assert rc_of(fn=lib.sipnet_gpu_comm_assimilate_inflated, target=e.comm, lam=lam_with(1, -1.0)) == \
            A.ERR_BAD_ARGUMENT
    multi, _ = forecast(("c3", 4, 50), cls=api.MultiEnsemble, devices=[0, 0])
    with multi:
        s0 = multi.state()
        spec, _k, _n = multi.obs_spec(POOLS, op, value, var)
        infl, _keep = multi.inflation_spec(good["lam"], good["sd"], (1.0, 10.0), 0.5)   # sd below sd_min
        assert lib.sipnet_gpu_multi_assimilate_inflated(multi.multi, C.byref(spec), C.byref(infl), None) == \
            A.ERR_BAD_ARGUMENT
        assert np.array_equal(multi.state(), s0, equal_nan=True)
