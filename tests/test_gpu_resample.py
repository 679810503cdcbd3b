"""Sequential Monte Carlo: per-site systematic resampling of the members (sipnet_gpu_resample,
sipnet_gpu_comm_resample, sipnet_gpu_multi_resample; sip_resample.cu).

CPU: a reference in Python integers and math.exp against the properties of systematic resampling, on random and
adversarial weights; the push form K(C) against the per-slot definition.
GPU: ancestors and diagnostics against the reference (on the handle's NEE log-likelihood and on caller weights);
copies bit for bit, and the next segment against a fresh handle given the copied parameters and state; what must not
change; teams and multi-GPU partitions bit-identical to one GPU; launches per call; rejected arguments.
"""
import bisect
import ctypes as C
import math

import numpy as np
import pytest

from sipnet_b200 import _abi as A, api, synth

EXCLUDED = A.ST_BAD_ALLOCATION | A.ST_NONFINITE
NEXT_BELOW_1 = float(np.nextafter(1.0, 0.0))


# ---- the reference ---------------------------------------------------------------------------------------------------
def systematic(W, u):
    """Ancestors (site-local) of the n slots for integer weights W and u in [0, 1)."""
    n, T, U = len(W), sum(W), int(math.ldexp(u, 32))
    C = [0]
    for x in W[:-1]:
        C.append(C[-1] + x)
    return [bisect.bisect_right(C, ((k << 32) + U) * T // (n << 32)) - 1 for k in range(n)]


def first_slot(Cv, T, U, n):
    """K(C) = clamp(ceil((ceil(C n 2^32 / T) - U) / 2^32), 0, n): the first slot k with t_k >= C."""
    a = -(-(Cv * n << 32) // T)
    return min(max(-(-(a - U) // (1 << 32)), 0), n)


def weights(l, part):
    lmax = max(x for x, p in zip(l, part) if p)
    w = [math.exp(x - lmax) if p else 0.0 for x, p in zip(l, part)]
    return lmax, w


def reference(l, status, member_site, nsites, u, ess_fraction=math.inf):
    """include/sipnet_gpu.h sipnet_gpu_resample: -> (ancestors [M], diag [nsites][4])."""
    anc = np.full(len(l), -1, np.int64)
    diag = np.zeros((nsites, 4))
    for s in range(nsites):
        idx = np.nonzero(member_site == s)[0]
        ls = [float(l[i]) for i in idx]
        part = [(int(status[i]) & EXCLUDED) == 0 and math.isfinite(x) for i, x in zip(idx, ls)]
        N = sum(part)
        diag[s] = N, np.nan, np.nan, 0
        if N == 0:
            continue
        lmax, w = weights(ls, part)
        s1 = math.ldexp(float(sum(int(math.ldexp(x, 100)) for x in w)), -100)
        s2 = math.ldexp(float(sum(int(math.ldexp(x * x, 100)) for x in w)), -100)
        ess = s1 * s1 / s2
        diag[s, 1:3] = ess, lmax + math.log(s1 / N)
        if math.isnan(u[s]) or not ess < ess_fraction * idx.size:
            continue
        a = systematic([int(math.ldexp(x, 40)) for x in w], float(u[s]))
        anc[idx] = idx[a]
        diag[s, 3] = len(set(a))
    return anc, diag


def adversarial_weights(rng):
    """(name, log-weights) rows, NaN / -inf = not taking part."""
    n = 257
    rows = [("ties", np.zeros(n)), ("spread 1e300", -rng.uniform(0, 1e300, n)),
            ("one dominant", np.r_[0.0, np.full(n - 1, -800.0)]),
            ("all W = 0 but one", np.r_[np.full(100, -30.0), 0.0, np.full(n - 101, -29.0)]),
            ("single participant", np.r_[np.full(50, -np.inf), 3.0, np.full(n - 51, np.nan)]),
            ("random", rng.normal(0, 3, n)), ("random wide", rng.normal(0, 40, n))]
    mixed = rng.normal(0, 2, n)
    mixed[rng.uniform(size=n) < 0.3] = -np.inf
    mixed[rng.uniform(size=n) < 0.2] = np.nan
    rows.append(("-inf and NaN", mixed))
    return rows


@pytest.mark.parametrize("u", [0.0, 0.3, 0.5, NEXT_BELOW_1])
def test_reference_is_systematic_resampling(u):
    rng = np.random.default_rng(5)
    for name, l in adversarial_weights(rng):
        part = [math.isfinite(x) for x in l]
        _, w = weights(list(l), part)
        W = [int(math.ldexp(x, 40)) for x in w]
        n, T = len(W), sum(W)
        a = systematic(W, u)
        assert all(x <= y for x, y in zip(a, a[1:])), name
        counts = np.bincount(a, minlength=n)
        for i in range(n):
            lo, hi = (n * W[i]) // T, -(-(n * W[i]) // T)
            assert lo <= counts[i] <= hi, (name, i)
        assert all(W[i] > 0 for i in a), name
        if name == "single participant":
            assert set(a) == {50}
        if name == "all W = 0 but one":
            assert set(a) == {100}


def test_equal_weights_give_the_identity():
    for n in (1, 2, 3, 100, 128, 257, 5000):
        for u in (0.0, 1e-9, 0.25, 0.5, 0.999, NEXT_BELOW_1):
            for wv in (1 << 40, 12345):
                assert systematic([wv] * n, u) == list(range(n)), (n, u)


def test_push_form_equals_per_slot_definition():
    rng = np.random.default_rng(11)
    cases = [[int(x) for x in rng.integers(0, 1 << 40, size=int(n))] for n in rng.integers(1, 300, size=40)]
    cases += [[1 << 40] * 7, [0, 0, 1 << 40, 0], [1] * 5 + [1 << 40], [3, 1 << 40, 0, 0, 5]]
    for W in cases:
        if sum(W) == 0:
            continue
        n, T = len(W), sum(W)
        for u in (0.0, 0.5, NEXT_BELOW_1, float(rng.uniform())):
            U = int(math.ldexp(u, 32))
            a = systematic(W, u)
            Cv = 0
            for i, x in enumerate(W):
                got = list(range(first_slot(Cv, T, U, n), first_slot(Cv + x, T, U, n)))
                assert got == [k for k in range(n) if a[k] == i], (W, u, i)
                Cv += x
            assert first_slot(0, T, U, n) == 0 and first_slot(T, T, U, n) == n


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
OUTS = A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS
KW = dict(outputs=OUTS, summary_cols=[A.O["nee"], A.O["plantWoodC"]], quantiles=[0.05, 0.5, 0.95], math=A.MATH_FAST,
          nee_sigma=0.5, max_event_records=16)
YEAR = 730                                   # half-daily steps of 2011


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def config(kind, nyears=1, events=False):
    """'one': one site of 5 000 members; 'many': 40 sites of 100 (mixed blocks); ('c3', n, m): n sites of m."""
    n, m = (1, 5000) if kind == "one" else (40, 100) if kind == "many" else kind[1:]
    sites = [synth.synth_site(3 + s, nyears, "half-daily", with_events=events) for s in range(n)]
    P, ms = synth.synth_params(n * m, stream=21), np.repeat(np.arange(n, dtype=np.int32), m)
    rng = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0, 1.5, s.nsteps))
    P[A.P["leafAllocation"], 7] = 0.9                            # bad allocation: never integrated
    return sites, P, ms


def forecast(kind, cls=api.Ensemble, nyears=1, events=False, **kw):
    sites, P, ms = config(kind, nyears, events)
    e = cls(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    e.run(0, YEAR)
    return e, ms


def site_u(nsites, seed=2):
    u = np.random.default_rng(seed).uniform(size=nsites)
    u[::5] = 0.0
    u[1::5] = NEXT_BELOW_1
    return u


def check_against_reference(anc, diag, ref_anc, ref_diag):
    assert np.array_equal(anc, ref_anc)
    assert np.array_equal(diag[:, [0, 3]], ref_diag[:, [0, 3]])
    np.testing.assert_allclose(diag[:, 1:3], ref_diag[:, 1:3], rtol=1e-12, atol=0, equal_nan=True)


def record(e):
    rv, rw = e.ring()
    recs = e.event_records() if e.max_event_records else None
    return dict(state=e.state(), rv=rv, rw=rw, status=e.status(), counts=e.event_counts(), recs=recs)


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
@pytest.mark.parametrize("ess_fraction", [math.inf, 0.5])
def test_loglik_matches_reference(kind, ess_fraction):
    e, ms = forecast(kind)
    with e:
        ll, status = e.loglik(), e.status()
        u = site_u(e.nsites)
        anc, diag = e.resample(u, ess_fraction)
    ref_anc, ref_diag = reference(ll, status, ms, e.nsites, u, ess_fraction)
    check_against_reference(anc, diag, ref_anc, ref_diag)
    assert (ref_anc >= 0).any()


@gpu
def test_caller_weights_match_reference():
    e, ms = forecast(("c3", 18, 257))
    rng = np.random.default_rng(4)
    rows = adversarial_weights(rng)
    lw = np.concatenate([r[1] for r in rows] + [rng.normal(0, 1, 257) for _ in range(18 - len(rows))])
    lw[ms == 17] = np.nan                                        # no participant: never resampled
    with e:
        status = e.status()
        for u in (np.zeros(18), np.full(18, NEXT_BELOW_1), site_u(18)):
            u = u.copy()
            u[16] = np.nan
            anc, diag = e.resample(u, math.inf, lw)
            ref_anc, ref_diag = reference(lw, status, ms, 18, u)
            check_against_reference(anc, diag, ref_anc, ref_diag)
            assert diag[17, 0] == 0 and np.isnan(diag[17, 1:3]).all() and (anc[ms == 17] == -1).all()
            assert (anc[ms == 16] == -1).all() and diag[16, 0] > 0
            status = e.status()
        assert diag[0, 3] == 257                                 # ties: every member once


@gpu
def test_copies_are_exact_and_the_next_segment_matches_a_fresh_handle():
    kw = dict(outputs=A.OUT_FULL | A.OUT_LOGLIK | A.OUT_EVENTS | A.OUT_DEBUG, out_steps_capacity=YEAR, math=A.MATH_VALIDATION,
              summary_cols=[], quantiles=[])
    kind = ("c3", 6, 64)
    a, ms = forecast(kind, nyears=2, events=True, **kw)
    sites, P, _ = config(kind, nyears=2, events=True)
    with a, api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw)) as b:
        prior, cnt0 = record(a), a.counters()
        assert prior["counts"].sum() > 0 and cnt0.sum() > 0
        lw = np.random.default_rng(9).normal(0, 2, a.nmembers)
        anc, diag = a.resample(site_u(6), math.inf, lw)
        assert (anc >= 0).all() and len(set(anc.tolist())) < a.nmembers
        got = record(a)
        for key in ("state", "rv", "rw", "counts"):
            assert np.array_equal(got[key], prior[key][..., anc], equal_nan=True), key
        assert np.array_equal(a.counters(), cnt0[:, anc])
        assert np.array_equal(got["status"], prior["status"][anc])
        assert all(bytes(x) == bytes(y) for i, j in enumerate(anc) for x, y in zip(got["recs"][i], prior["recs"][j]))
        assert (a.loglik() == 0).all() and (a.loglik_n() == 0).all()
        assert got["status"][7] == prior["status"][anc[7]]
        # a fresh handle given the copied parameters and state runs the same next segment
        b.set_params(P[:, anc])
        b.set_state(prior["state"][:, anc], prior["rv"][:, anc], prior["rw"][:, anc], next_step=YEAR)
        a.run(YEAR, 2 * YEAR)
        b.run(YEAR, 2 * YEAR)
        assert np.array_equal(a.output(), b.output(), equal_nan=True)
        assert np.array_equal(a.state(), b.state(), equal_nan=True)
        assert np.array_equal(a.loglik(), b.loglik(), equal_nan=True)


@gpu
def test_skipped_sites_and_other_data_stay_bit_identical():
    e, ms = forecast("many", nyears=2, outputs=OUTS | A.OUT_FULL, out_steps_capacity=YEAR)
    with e:
        before = record(e)
        out0, mean0, var0, q0 = e.output(), e.mean(), e.variance(), e.quantiles()
        ll0, n0 = e.loglik(), e.loglik_n()
        lw = np.random.default_rng(3).normal(0, 0.3, e.nmembers)  # ESS ~ 0.9 n: kept at 0.6
        for s in (0, 3):                                          # ESS ~ 1: resampled
            lw[ms == s] = np.where(np.arange(100) == 1, 0.0, -50.0)
        u = site_u(e.nsites)
        u[[2, 5]] = np.nan
        anc, diag = e.resample(u, 0.6, lw)
        ref_anc, ref_diag = reference(lw, before["status"], ms, e.nsites, u, 0.6)
        check_against_reference(anc, diag, ref_anc, ref_diag)
        skipped = anc < 0
        assert skipped[ms == 2].all() and skipped[ms == 5].all() and not skipped[ms == 3].any()
        assert (diag[:, 1] >= 0.6 * 100).any()                   # some sites skipped by the threshold
        after = record(e)
        for key in ("state", "rv", "rw", "status", "counts"):
            assert np.array_equal(after[key][..., skipped], before[key][..., skipped], equal_nan=True), key
        assert np.array_equal(e.loglik()[skipped], ll0[skipped]) and (e.loglik()[~skipped] == 0).all()
        assert np.array_equal(e.loglik_n()[skipped], n0[skipped])
        for x, y in ((e.output(), out0), (e.mean(), mean0), (e.variance(), var0), (e.quantiles(), q0)):
            assert np.array_equal(x, y, equal_nan=True)
        # the bad-allocation member of site 0 takes its ancestor's record, status included
        assert not skipped[7] and after["status"][7] == before["status"][anc[7]]
        assert (before["status"][7] & A.ST_BAD_ALLOCATION) and not (after["status"][7] & A.ST_BAD_ALLOCATION)
        # skipped members keep accumulating their likelihood
        e.run(YEAR, YEAR + 40)
        ll1 = e.loglik()
        assert (ll1[skipped & (before["status"] & EXCLUDED == 0)] != ll0[skipped & (before["status"] & EXCLUDED == 0)]).any()


@gpu
@pytest.mark.parametrize("kind", ["one", "many"])
def test_team_of_one_equals_handle(kind):
    res = []
    for team in (False, True):
        e, ms = forecast(kind)
        with e:
            u = site_u(e.nsites)
            if team:
                e.join_team(1, 0)
                anc, diag = e.team_resample(u, 0.9)
            else:
                anc, diag = e.resample(u, 0.9)
            res.append((anc, diag, e.state(), e.status(), e.loglik()))
    for x, y in zip(*res):
        assert np.array_equal(x, y, equal_nan=True)


needs2 = pytest.mark.skipif("ngpus() < 2", reason="needs two GPUs on the box")
DEVICES = [pytest.param(None, marks=needs2, id="all-gpus"), pytest.param([0, 0], id="loopback2"),
           pytest.param([0, 0, 0], id="loopback3"), pytest.param([0] * 5, id="loopback5")]


@gpu
@pytest.mark.parametrize("devices", DEVICES)
@pytest.mark.parametrize("kind", ["one", ("c3", 11, 40)], ids=["split-site", "whole-sites"])
def test_multi_bit_identical_to_one_gpu(devices, kind):
    kw = dict(outputs=A.OUT_FULL | A.OUT_LOGLIK | A.OUT_EVENTS, out_steps_capacity=YEAR)
    one, ms = forecast(kind, nyears=2, **kw)
    multi, _ = forecast(kind, cls=api.MultiEnsemble, nyears=2, devices=devices, **kw)
    with one, multi:
        assert multi.ndevices >= 2
        u = site_u(one.nsites)
        for ess in (math.inf, 0.7):
            a1, d1 = one.resample(u, ess)
            am, dm = multi.resample(u, ess)
            assert np.array_equal(am, a1) and np.array_equal(dm, d1, equal_nan=True)
            lw = np.random.default_rng(6).normal(0, 1, one.nmembers)
            a1, d1 = one.resample(u, ess, lw)
            am, dm = multi.resample(u, ess, lw)
            assert np.array_equal(am, a1) and np.array_equal(dm, d1, equal_nan=True)
            assert (a1 >= 0).any()
        for x, y in ((multi.state(), one.state()), (multi.status(), one.status()), (multi.loglik(), one.loglik()),
                     (multi.event_counts(), one.event_counts())):
            assert np.array_equal(x, y, equal_nan=True)
        one.run(YEAR, 2 * YEAR)
        multi.run(YEAR, 2 * YEAR)
        assert np.array_equal(multi.output(), one.output(), equal_nan=True)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        assert np.array_equal(multi.status(), one.status())


@gpu
def test_launches_do_not_grow_with_sites():
    per_call = []
    for n in (3, 300):
        sites, P, ms, _ = synth.config_c3(nsites=n, members_per_site=10, nyears=1)
        with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK, math=A.MATH_FAST) as e:
            e.run(0, 20)
            lw = np.random.default_rng(1).normal(0, 1, e.nmembers)
            c0 = e.launch_count()
            e.resample(np.full(n, 0.5), math.inf, lw)
            c1 = e.launch_count()
            e.resample(np.full(n, 0.5), math.inf, lw)
            per_call.append((c1 - c0, e.launch_count() - c1))
    assert per_call[0] == per_call[1] and per_call[0][0] == per_call[0][1] > 0


@gpu
def test_rejected_arguments_leave_everything_untouched():
    e, ms = forecast(("c3", 4, 50), nyears=2)
    twin, _ = forecast(("c3", 4, 50), nyears=2)
    with e, twin:
        def snap():
            return record(e), e.loglik(), e.loglik_n()

        before = snap()
        lib = e.lib
        u = np.full(4, 0.5)
        lw = np.zeros(e.nmembers)

        def rc_of(u=u, ess=math.inf, lw=lw, fn=lib.sipnet_gpu_resample, target=e.handle):
            return fn(target, None if u is None else u.ctypes.data, ess, None if lw is None else lw.ctypes.data, None, None)

        cases = {"NULL handle": lambda: rc_of(target=None), "NULL u": lambda: rc_of(u=None),
                 "NaN ess_fraction": lambda: rc_of(ess=math.nan), "negative ess_fraction": lambda: rc_of(ess=-0.1)}
        for name, v in (("u = 1", 1.0), ("u < 0", -1e-300), ("u = inf", math.inf), ("u = -inf", -math.inf)):
            uu = u.copy()
            uu[2] = v
            cases[name] = lambda uu=uu: rc_of(u=uu)
        lwi = lw.copy()
        lwi[130] = math.inf
        cases["+inf log-weight"] = lambda: rc_of(lw=lwi)
        ll = e.loglik()
        for name, fn in cases.items():
            assert fn() == A.ERR_BAD_ARGUMENT, name
            now = snap()
            for key in before[0]:
                if key != "recs":
                    assert np.array_equal(now[0][key], before[0][key], equal_nan=True), (name, key)
            assert np.array_equal(now[1], before[1]) and np.array_equal(now[2], before[2]), name
        assert np.array_equal(e.loglik(), ll)
        e.join_team(1, 0)
        assert rc_of(ess=-1.0, fn=lib.sipnet_gpu_comm_resample, target=e.comm) == A.ERR_BAD_ARGUMENT
        assert rc_of(lw=lwi, fn=lib.sipnet_gpu_comm_resample, target=e.comm) == A.ERR_BAD_ARGUMENT
        # parameters (and everything else) untouched: the next segment is the one of a handle that saw no call
        e.run(YEAR, YEAR + 200)
        twin.run(YEAR, YEAR + 200)
        for x, y in ((e.state(), twin.state()), (e.loglik(), twin.loglik()), (e.mean(), twin.mean()),
                     (e.status(), twin.status())):
            assert np.array_equal(x, y, equal_nan=True)
    # no log-weights and no log-likelihood
    sites, P, ms = config(("c3", 2, 20))
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_FULL) as f:
        f.run(0, 10)
        s0 = f.state()
        assert f.lib.sipnet_gpu_resample(f.handle, np.full(2, 0.5).ctypes.data, math.inf, None, None, None) == A.ERR_BAD_ARGUMENT
        assert np.array_equal(f.state(), s0, equal_nan=True)
    multi, _ = forecast(("c3", 4, 50), cls=api.MultiEnsemble, devices=[0, 0])
    with multi:
        s0, p0 = multi.state(), multi.status()
        assert lib.sipnet_gpu_multi_resample(multi.multi, u.ctypes.data, math.inf, lwi.ctypes.data, None, None) == \
            A.ERR_BAD_ARGUMENT
        assert np.array_equal(multi.state(), s0, equal_nan=True) and np.array_equal(multi.status(), p0)
