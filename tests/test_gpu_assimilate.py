"""Sequential data assimilation: the ensemble adjustment Kalman filter on the carried pools (sipnet_gpu_assimilate,
sipnet_gpu_comm_assimilate, sipnet_gpu_multi_assimilate; sip_assim.cu).

CPU: a numpy reference of the update (math.fsum for every sum) against the Kalman closed form; the ctypes mirror of
sipnet_gpu_obs_spec against the C layout.
GPU: synth ensembles after a one-year forecast (fast math policy), against the reference within 1e-9 x the row's
prior ensemble standard deviation at its site + 4 ulp -- a bound that one dropped member breaks; what must not change
stays bit-identical; the floor; the next segment; determinism; teams and multi-GPU partitions; launches per call;
rejected arguments.
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

POOLS = list(range(12))                      # SIPNET_S_plantWoodC .. SIPNET_S_plantStorageN
EXCLUDED = A.ST_BAD_ALLOCATION | A.ST_NONFINITE
S = A.S


# ---- the reference ---------------------------------------------------------------------------------------------------
def eakf_reference(state, status, member_site, nsites, rows, op, value, variance, floor=True):
    """The update of include/sipnet_gpu.h on a [NSTATE][M] state: -> (state, status, diag).  floor=False leaves out
    the final floor (to see which values went below 0)."""
    X = np.array(state, dtype=np.float64, copy=True)
    st = np.array(status, dtype=np.uint32, copy=True)
    rows = list(rows)
    op = np.asarray(op, np.float64).reshape(-1, len(rows))
    nobs = op.shape[0]
    diag = np.full((nsites, nobs, 4), np.nan)
    applied = np.zeros(nsites, bool)

    def takers(s):
        idx = np.nonzero(member_site == s)[0]
        ok = ((st[idx] & EXCLUDED) == 0) & np.all(np.isfinite(X[rows][:, idx]), axis=0)
        return idx[ok]

    for k in range(nobs):
        for s in range(nsites):
            idx = takers(s)
            n = idx.size
            diag[s, k, 0] = n
            yo, r = value[s, k], variance[s, k]
            if n == 0:
                continue
            x = X[rows][:, idx]
            y = np.array([math.fsum(col) for col in (op[k][:, None] * x).T])
            ybar = math.fsum(y) / n
            dy = y - ybar
            syy = math.fsum(dy * dy)
            if np.isnan(yo) or n < 2 or syy == 0 or not math.isfinite(syy):
                continue
            xbar = np.array([math.fsum(x[j]) / n for j in range(len(rows))])
            sjy = np.array([math.fsum((x[j] - xbar[j]) * dy) for j in range(len(rows))])
            s2 = syy / (n - 1)
            ya = ybar + s2 / (s2 + r) * (yo - ybar)
            alpha = math.sqrt(r / (s2 + r))
            diag[s, k, 1:] = ybar, s2, ya
            d = (ya - ybar) + (alpha - 1) * (y - ybar)
            for j, row in enumerate(rows):
                X[row, idx] = x[j] + (sjy[j] / syy) * d
            applied[s] = True
    for s in np.nonzero(applied)[0] if floor else []:
        idx = takers(s)
        sub = X[rows][:, idx]
        neg = sub < 0
        sub[neg] = 0.0
        X[np.ix_(rows, idx)] = sub
        st[idx[neg.any(axis=0)]] |= A.ST_ANALYSIS_FLOORED
    return X, st, diag


def prior_sd(state, status, member_site, nsites):
    """[NSTATE][nsites] sample standard deviation of every row over the members that take part."""
    sd = np.zeros((state.shape[0], nsites))
    for s in range(nsites):
        idx = np.nonzero(member_site == s)[0]
        ok = ((status[idx] & EXCLUDED) == 0) & np.all(np.isfinite(state[POOLS][:, idx]), axis=0)
        if ok.sum() > 1:
            sd[:, s] = np.std(state[:, idx[ok]], axis=1, ddof=1)
    return sd


def within_bound(got, ref, sd, member_site, rows, cols=None):
    cols = np.arange(got.shape[1]) if cols is None else cols
    for r in rows:
        g, w = got[r, cols], ref[r, cols]
        if not np.array_equal(np.isnan(g), np.isnan(w)):
            return False
        tol = 1e-9 * sd[r, member_site[cols]] + 4 * np.spacing(np.abs(w))
        fin = ~np.isnan(w)
        if not np.all(np.abs(g[fin] - w[fin]) <= tol[fin]):
            return False
    return True


def test_reference_single_direct_observation_is_the_kalman_closed_form():
    rng = np.random.default_rng(3)
    M = 257
    state = np.zeros((A.NSTATE, M))
    state[POOLS] = rng.normal(50.0, 4.0, (12, M))
    state[S["soilC"]] += 0.7 * state[S["plantWoodC"]]               # correlated with the observed row
    status = np.zeros(M, np.uint32)
    ms = np.zeros(M, np.int32)
    yo, r = 55.0, 9.0
    op = np.zeros((1, 12))
    op[0, S["plantWoodC"]] = 1.0
    X, st, diag = eakf_reference(state, status, ms, 1, POOLS, op, np.array([[yo]]), np.array([[r]]))
    x = state[S["plantWoodC"]]
    s2 = np.var(x, ddof=1)
    ya = x.mean() + s2 / (s2 + r) * (yo - x.mean())
    assert diag[0, 0, 0] == M
    np.testing.assert_allclose(diag[0, 0, 1:], [x.mean(), s2, ya], rtol=1e-13)
    xa = X[S["plantWoodC"]]
    np.testing.assert_allclose(xa.mean(), ya, rtol=1e-13)
    np.testing.assert_allclose(np.var(xa, ddof=1), r / (s2 + r) * s2, rtol=1e-12)
    # a correlated row moves by its regression on the observed one
    b = np.cov(state[S["soilC"]], x)[0, 1] / s2
    np.testing.assert_allclose(X[S["soilC"]].mean() - state[S["soilC"]].mean(), b * (ya - x.mean()), rtol=1e-11)
    assert not (st & A.ST_ANALYSIS_FLOORED).any()
    # the Kalman posterior covariance of the pair
    c = np.cov(X[[S["soilC"], S["plantWoodC"]]], ddof=1)
    c0 = np.cov(state[[S["soilC"], S["plantWoodC"]]], ddof=1)
    k = c0[:, 1] / (c0[1, 1] + r)
    np.testing.assert_allclose(c, c0 - np.outer(k, c0[1, :]), rtol=1e-10)


def test_ctypes_obs_spec_matches_c_layout():
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "sipnet_gpu.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(sipnet_gpu_obs_spec), offsetof(sipnet_gpu_obs_spec, n_rows),
         offsetof(sipnet_gpu_obs_spec, rows), offsetof(sipnet_gpu_obs_spec, n_obs), offsetof(sipnet_gpu_obs_spec, op),
         offsetof(sipnet_gpu_obs_spec, value), offsetof(sipnet_gpu_obs_spec, variance));
  printf("%u\n", (unsigned)SIPNET_GPU_ST_ANALYSIS_FLOORED);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        lines = subprocess.check_output([exe]).decode().split("\n")
    O = A.ObsSpec
    assert list(map(int, lines[0].split())) == [C.sizeof(O), O.n_rows.offset, O.rows.offset, O.n_obs.offset,
                                                O.op.offset, O.value.offset, O.variance.offset]
    assert int(lines[1]) == A.ST_ANALYSIS_FLOORED


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
OUTS = A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS
KW = dict(outputs=OUTS, summary_cols=[A.O["nee"], A.O["plantWoodC"]], quantiles=[0.05, 0.5, 0.95], math=A.MATH_FAST,
          nee_sigma=0.5, max_event_records=16)
YEAR = 730                                   # half-daily steps of 2011


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def config(kind, nyears=1):
    """'one': one site of 5 000 members; 'many': 40 sites of 100; ('c3', n, m): n sites of m.  No event schedule:
    the C3 schedule harvests every plant pool to 0 before the year ends, which would leave nothing to observe."""
    n, m = (1, 5000) if kind == "one" else (40, 100) if kind == "many" else kind[1:]
    sites = [synth.synth_site(3 + s, nyears, "half-daily") for s in range(n)]
    P, ms = synth.synth_params(n * m, stream=21), np.repeat(np.arange(n, dtype=np.int32), m)
    rng = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0, 1.5, s.nsteps))
    P[A.P["leafAllocation"], 7] = 0.9                            # bad allocation: never integrated, never assimilated
    return sites, P, ms


def forecast(kind, cls=api.Ensemble, nyears=1, **kw):
    sites, P, ms = config(kind, nyears)
    e = cls(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    e.run(0, YEAR)
    return e, ms


def obs_for(state, ms, nsites, op, shift=0.5, rel_var=0.25, seed=1):
    """Observations near the prior: y° = prior mean + shift sd, r = rel_var x prior variance (per site, per obs)."""
    rng = np.random.default_rng(seed)
    nobs = op.shape[0]
    value = np.empty((nsites, nobs))
    var = np.empty((nsites, nobs))
    for s in range(nsites):
        y = op @ state[POOLS][:, ms == s]
        y = y[:, np.isfinite(y).all(axis=0)]
        for k in range(nobs):
            sd = max(float(np.std(y[k])), 1e-3 * abs(float(np.mean(y[k]))), 1e-6)
            value[s, k] = np.mean(y[k]) + shift * sd * (1 + 0.2 * rng.standard_normal())
            var[s, k] = rel_var * sd * sd
    return value, var


def ops(nobs, combined):
    op = np.zeros((nobs, 12))
    picks = [S["plantWoodC"], S["soilC"], S["soilWater"], S["litterC"]]
    for k in range(nobs):
        op[k, picks[k]] = 1.0
    if combined:
        op[0, [S["plantWoodC"], S["coarseRootC"], S["fineRootC"]]] = 1.0
    return op


def snapshot(e):
    return dict(state=e.state(), status=e.status(), ring=e.ring(), ll=e.loglik(), counts=e.event_counts(),
                mean=e.mean(), var=e.variance(), q=e.quantiles())


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
@pytest.mark.parametrize("nobs,combined", [(1, False), (1, True), (4, False), (4, True)])
def test_matches_reference(kind, nobs, combined):
    e, ms = forecast(kind)
    with e:
        st0, status0 = e.state(), e.status()
        op = ops(nobs, combined)
        value, var = obs_for(st0, ms, e.nsites, op)
        diag = e.assimilate(POOLS, op, value, var)
        got = e.state()
    ref, _, rdiag = eakf_reference(st0, status0, ms, e.nsites, POOLS, op, value, var)
    sd = prior_sd(st0, status0, ms, e.nsites)
    assert within_bound(got, ref, sd, ms, POOLS)
    assert np.array_equal(diag[..., 0], rdiag[..., 0])
    np.testing.assert_allclose(diag[..., 1:], rdiag[..., 1:], rtol=1e-9, equal_nan=True)
    assert (rdiag[..., 0] > 1).all() and np.isfinite(rdiag[..., 3]).all()
    # the bound is tight enough to see one member left out of the statistics
    drop = int(np.nonzero(((status0 & EXCLUDED) == 0) & (ms == 0))[0][0])
    status1 = status0.copy()
    status1[drop] |= A.ST_BAD_ALLOCATION
    ref1, _, _ = eakf_reference(st0, status1, ms, e.nsites, POOLS, op, value, var)
    others = np.setdiff1d(np.arange(e.nmembers), [drop])
    assert not within_bound(got, ref1, sd, ms, POOLS, others)


@gpu
def test_closed_form_and_two_halves():
    e, ms = forecast("one")
    with e:
        st0 = e.state()
        row = S["plantWoodC"]
        op1 = np.zeros((1, 12))
        op1[0, row] = 1.0
        value, var = obs_for(st0, ms, 1, op1, shift=0.5)
        sd = prior_sd(st0, e.status(), ms, 1)
        diag = e.assimilate(POOLS, op1, value, var)
        xa = e.state()[row][(e.status() & EXCLUDED) == 0]
        assert (xa > 0).all()
    n, ybar, s2, ya = diag[0, 0]
    alpha2 = var[0, 0] / (s2 + var[0, 0])
    np.testing.assert_allclose(xa.mean(), ya, rtol=1e-12)
    np.testing.assert_allclose(np.var(xa, ddof=1), alpha2 * s2, rtol=1e-12)
    # (y°, r) twice on the same row == (y°, r / 2) once
    outs = []
    for twice in (True, False):
        e, _ = forecast("one")
        with e:
            if twice:
                e.assimilate(POOLS, np.vstack([op1, op1]), np.hstack([value, value]), np.hstack([var, var]))
            else:
                e.assimilate(POOLS, op1, value, var / 2)
            outs.append(e.state())
    assert within_bound(outs[0], outs[1], sd, ms, POOLS)


@gpu
def test_untouched_outputs_rows_and_bad_members():
    e, ms = forecast("many")
    with e:
        before = snapshot(e)
        op = ops(4, True)
        value, var = obs_for(before["state"], ms, e.nsites, op)
        diag = e.assimilate(POOLS, op, value, var)
        after = snapshot(e)
    unlisted = [r for r in range(A.NSTATE) if r not in POOLS]
    assert np.array_equal(after["state"][unlisted], before["state"][unlisted], equal_nan=True)
    for key in ("ll", "counts", "mean", "var", "q"):
        assert np.array_equal(after[key], before[key], equal_nan=True), key
    for a, b in zip(after["ring"], before["ring"]):
        assert np.array_equal(a, b)
    floor = np.uint32(A.ST_ANALYSIS_FLOORED)
    assert np.array_equal(after["status"] & ~floor, before["status"])
    bad = (before["status"] & EXCLUDED) != 0
    assert bad[7]                                                    # leafAllocation = 0.9: bad allocation
    assert np.array_equal(after["state"][:, bad], before["state"][:, bad], equal_nan=True)
    assert not (after["status"][bad] & floor).any()
    n = np.array([(~bad & (ms == s)).sum() for s in range(e.nsites)])
    assert np.array_equal(diag[:, 0, 0], n) and n[0] == 99


@gpu
def test_nonparticipants_and_skipped_sites_do_not_change():
    e, ms = forecast("many")
    with e:
        st, status = e.state(), e.status()
        rv, rw = e.ring()
        st[S["plantWoodC"], 11] = np.nan                            # a member that does not take part
        st[S["soilC"], ms == 5] = np.nan                            # site 5: one member left, N < 2
        st[S["soilC"], 503] = e.state()[S["soilC"], 503]
        live6 = (ms == 6) & ((status & EXCLUDED) == 0)
        st[S["plantWoodC"], live6] = 1234.5                          # site 6: the observed row has zero variance
        e.set_state(st, rv, rw, next_step=YEAR)
        rows = [S["plantWoodC"], S["soilC"], S["litterC"], S["minN"]]
        op = np.array([[1.0, 0.0, 0.0, 0.0]])
        value, var = obs_for(st, ms, e.nsites, np.eye(12)[[S["plantWoodC"]]])
        value[3] = np.nan                                            # site 3: not observed
        diag = e.assimilate(rows, op, value, var)
        after, astatus = e.state(), e.status()
        ring = e.ring()
    for a, b in zip(ring, (rv, rw)):
        assert np.array_equal(a, b)
    ref, _, rdiag = eakf_reference(st, status, ms, e.nsites, rows, op, value, var)
    floor = np.uint32(A.ST_ANALYSIS_FLOORED)
    assert np.array_equal(astatus & ~floor, status)
    keep = ((status & EXCLUDED) != 0) | np.isin(ms, [3, 5, 6])
    keep[11] = True
    assert np.array_equal(after[:, keep], st[:, keep], equal_nan=True)
    assert not (astatus[keep] & floor).any()
    assert (after[S["plantWoodC"], ~keep] != st[S["plantWoodC"], ~keep]).mean() > 0.9
    # N counts only the members that take part
    n = np.array([(((status & EXCLUDED) == 0) & (ms == s) & np.isfinite(st[rows]).all(axis=0)).sum()
                  for s in range(e.nsites)])
    assert np.array_equal(diag[:, 0, 0], n) and np.array_equal(rdiag[:, 0, 0], n)
    assert n[5] == 1 and n[0] == 98                                  # member 7 (bad allocation) and 11 (NaN) excluded
    for s in (3, 5, 6):
        assert np.isnan(diag[s, 0, 1:]).all(), s
    assert np.isfinite(diag[[0, 1, 2, 4], 0, 1:]).all()
    assert within_bound(after, ref, prior_sd(st, status, ms, e.nsites), ms, rows)


@gpu
def test_floor_sets_zero_and_the_status_bit():
    e, ms = forecast("one")
    with e:
        st0, status0 = e.state(), e.status()
        row = S["plantWoodC"]
        op = np.eye(12)[[row]]
        sd = float(np.std(st0[row][(status0 & EXCLUDED) == 0]))
        value, var = np.array([[0.0]]), np.array([[(0.05 * sd) ** 2]])
        e.assimilate(POOLS, op, value, var)
        got, status = e.state(), e.status()
    # the reference without its floor: which values went below 0 (and by more than the bound)
    nofloor, _, _ = eakf_reference(st0, status0, ms, 1, POOLS, op, value, var, floor=False)
    sd = prior_sd(st0, status0, ms, 1)
    tol = 1e-9 * sd[POOLS, 0][:, None] + 4 * np.spacing(np.abs(nofloor[POOLS]))
    ref, rstatus, _ = eakf_reference(st0, status0, ms, 1, POOLS, op, value, var)
    assert within_bound(got, ref, sd, ms, POOLS)
    below = nofloor[POOLS] < -tol
    assert below.sum() > 100
    assert np.all(got[POOLS][below] == 0) and not np.signbit(got[POOLS][below]).any()
    flagged = (status & A.ST_ANALYSIS_FLOORED) != 0
    assert np.array_equal(status & ~np.uint32(A.ST_ANALYSIS_FLOORED), status0)
    clear = np.all(np.abs(nofloor[POOLS]) > tol, axis=0) | ((status0 & EXCLUDED) != 0)
    assert np.array_equal(flagged[clear], ((rstatus & A.ST_ANALYSIS_FLOORED) != 0)[clear])
    assert flagged.sum() > 100
    assert not flagged[7]


@gpu
def test_next_segment_equals_set_state():
    kw = dict(outputs=A.OUT_FULL, out_steps_capacity=YEAR)
    a, ms = forecast(("c3", 10, 100), nyears=2, **kw)
    sites, P, _ = config(("c3", 10, 100), nyears=2)
    with a, api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw)) as b:
        st0 = a.state()
        op = ops(4, True)
        value, var = obs_for(st0, ms, a.nsites, op)
        a.assimilate(POOLS, op, value, var)
        rv, rw = a.ring()
        b.set_state(a.state(), rv, rw, next_step=YEAR)
        a.run(YEAR, 2 * YEAR)
        b.run(YEAR, 2 * YEAR)
        assert np.array_equal(a.output(), b.output(), equal_nan=True)
        assert np.array_equal(a.state(), b.state(), equal_nan=True)
        assert not np.array_equal(a.state(), st0, equal_nan=True)


@gpu
def test_deterministic():
    outs = []
    for _ in range(2):
        e, ms = forecast("many")
        with e:
            op = ops(4, True)
            value, var = obs_for(e.state(), ms, e.nsites, op)
            diag = e.assimilate(POOLS, op, value, var)
            outs.append((e.state(), e.status(), diag))
    for x, y in zip(*outs):
        assert np.array_equal(x, y, equal_nan=True)


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_team_of_one_equals_handle(kind):
    res = []
    for team in (False, True):
        e, ms = forecast(kind)
        with e:
            op = ops(4, True)
            value, var = obs_for(e.state(), ms, e.nsites, op)
            if team:
                e.join_team(1, 0)
                diag = e.team_assimilate(POOLS, op, value, var)
            else:
                diag = e.assimilate(POOLS, op, value, var)
            res.append((e.state(), e.status(), diag))
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
        assert np.array_equal(multi.state(), st0, equal_nan=True)
        op = ops(4, True)
        value, var = obs_for(st0, ms, 1, op)
        d1 = one.assimilate(POOLS, op, value, var)
        dm = multi.assimilate(POOLS, op, value, var)
        got = multi.state()
        ref, _, _ = eakf_reference(st0, status0, ms, 1, POOLS, op, value, var)
        sd = prior_sd(st0, status0, ms, 1)
        assert within_bound(got, one.state(), sd, ms, POOLS)
        assert within_bound(got, ref, sd, ms, POOLS)
        assert np.array_equal(multi.status(), one.status())
        assert np.array_equal(dm[..., 0], d1[..., 0])
        np.testing.assert_allclose(dm, d1, rtol=1e-12)
        # the next segment from the team's analysis: what one GPU computes from the same state
        rv, rw = one.ring()
        one.set_state(got, rv, rw, next_step=YEAR)
        one.run(YEAR, 2 * YEAR)
        multi.run(YEAR, 2 * YEAR)
        assert np.array_equal(multi.output(), one.output(), equal_nan=True)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)


@gpu
@pytest.mark.parametrize("devices", DEVICES)
def test_multi_whole_sites_bit_identical(devices):
    kw = dict(outputs=A.OUT_FULL, out_steps_capacity=YEAR)
    one, ms = forecast(("c3", 11, 40), nyears=2, **kw)
    multi, _ = forecast(("c3", 11, 40), cls=api.MultiEnsemble, nyears=2, devices=devices, **kw)
    with one, multi:
        st0 = one.state()
        op = ops(4, True)
        value, var = obs_for(st0, ms, 11, op)
        value[4, 1] = np.nan
        d1 = one.assimilate(POOLS, op, value, var)
        dm = multi.assimilate(POOLS, op, value, var)
        assert np.array_equal(dm, d1, equal_nan=True)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        assert np.array_equal(multi.status(), one.status())
        one.run(YEAR, 2 * YEAR)
        multi.run(YEAR, 2 * YEAR)
        assert np.array_equal(multi.output(), one.output(), equal_nan=True)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)


@gpu
def test_launches_do_not_grow_with_sites():
    per_call = []
    for n in (3, 300):
        sites, P, ms, _ = synth.config_c3(nsites=n, members_per_site=10, nyears=1)
        with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK, math=A.MATH_FAST) as e:
            e.run(0, 20)
            op = ops(2, True)
            value, var = obs_for(e.state(), ms, n, op)
            c0 = e.launch_count()
            e.assimilate(POOLS, op, value, var)
            c1 = e.launch_count()
            e.assimilate(POOLS, op, value, var)
            per_call.append((c1 - c0, e.launch_count() - c1))
    assert per_call[0] == per_call[1] and per_call[0][0] == per_call[0][1] > 0


@gpu
def test_rejected_arguments_leave_state_untouched():
    e, ms = forecast(("c3", 4, 50))
    with e:
        before = (e.state(), e.status())
        op = ops(2, False)
        value, var = obs_for(before[0], ms, 4, op)
        lib = e.lib

        def rc_of(rows=POOLS, op=op, value=value, var=var, patch=None, fn=lib.sipnet_gpu_assimilate, target=e.handle):
            spec, keep, _ = e.obs_spec(rows, op, value, var)
            if patch:
                patch(spec)
            return fn(target, C.byref(spec), None)

        def setp(field, v):
            return lambda sp: setattr(sp, field, v)

        bad_op = [op.copy() for _ in range(3)]
        bad_op[0][0, 0] = np.nan
        bad_op[1][1, 3] = np.inf
        bad_op[2][1] = 0.0
        cases = {
            "NULL spec": lambda: lib.sipnet_gpu_assimilate(e.handle, None, None),
            "NULL rows": lambda: rc_of(patch=setp("rows", None)),
            "NULL op": lambda: rc_of(patch=setp("op", None)),
            "NULL value": lambda: rc_of(patch=setp("value", None)),
            "NULL variance": lambda: rc_of(patch=setp("variance", None)),
            "n_rows 0": lambda: rc_of(patch=setp("n_rows", 0)),
            "n_obs 0": lambda: rc_of(patch=setp("n_obs", 0)),
            "repeated row": lambda: rc_of(rows=[0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 0]),
            "plantCAccountingDelta": lambda: rc_of(rows=POOLS[:11] + [S["plantCAccountingDelta"]]),
            "tracker row": lambda: rc_of(rows=POOLS[:11] + [S["yearlyGpp"]]),
            "ring cursor": lambda: rc_of(rows=POOLS[:11] + [S["meanStart"]]),
            "phenology flag": lambda: rc_of(rows=POOLS[:11] + [S["didLeafGrowth"]]),
            "negative row": lambda: rc_of(rows=POOLS[:11] + [-1]),
            "NaN op": lambda: rc_of(op=bad_op[0]),
            "inf op": lambda: rc_of(op=bad_op[1]),
            "all-zero op row": lambda: rc_of(op=bad_op[2]),
        }
        for name, v in (("+inf", np.inf), ("-inf", -np.inf)):
            val = value.copy()
            val[2, 1] = v
            cases[f"{name} value"] = lambda val=val: rc_of(value=val)
        for name, v in (("NaN", np.nan), ("inf", np.inf), ("zero", 0.0), ("negative", -1.0)):
            vv = var.copy()
            vv[1, 0] = v
            cases[f"{name} variance"] = lambda vv=vv: rc_of(var=vv)
        for name, fn in cases.items():
            assert fn() == A.ERR_BAD_ARGUMENT, name
            assert np.array_equal(e.state(), before[0], equal_nan=True), name
            assert np.array_equal(e.status(), before[1]), name
        # a missing variance where the value is missing too is fine
        vv = var.copy()
        value2 = value.copy()
        value2[1, 0] = vv[1, 0] = np.nan
        assert rc_of(value=value2, var=vv) == 0
        # the team and multi entry points check the same way
        e.join_team(1, 0)
        assert rc_of(op=bad_op[2], fn=lib.sipnet_gpu_comm_assimilate, target=e.comm) == A.ERR_BAD_ARGUMENT
    multi, _ = forecast(("c3", 4, 50), cls=api.MultiEnsemble, devices=[0, 0])
    with multi:
        s0 = multi.state()
        spec, keep, _ = multi.obs_spec(POOLS, op, value, var * -1.0)
        assert lib.sipnet_gpu_multi_assimilate(multi.multi, C.byref(spec), None) == A.ERR_BAD_ARGUMENT
        assert np.array_equal(multi.state(), s0, equal_nan=True)
