"""GPU: the multi-GPU layer of the C ABI (sipnet_gpu_comm_*, sipnet_gpu_multi_*; SURVEY 8e).

* a team of ONE rank runs the cross-rank summary kernels (sip_gsum.cu) without any exchange: its results must equal
  the single-GPU row summaries (sip_reduce.cu) -- quantiles bit for bit (both pick exact order statistics and use the
  same lerp), moments to rounding;
* sipnet_gpu_multi_* (one process, all GPUs of a box with two or more; or a loopback team of several ranks on
  GPU 0) must deliver exactly what one GPU delivers -- per-member output bit for bit in both partitions (whole sites per device / one site's members split),
  split-site summaries through the NCCL team select, log-likelihoods, event records.
"""
import numpy as np
import pytest

from sipnet_b200 import _abi as A, api, synth

pytestmark = pytest.mark.gpu

COLS = [A.O["nee"], A.O["gpp"], A.O["snow"]]       # snow: heavy ties (exact zeros) ; gpp: constant night rows
QS = [0.05, 0.5, 0.95, 1.0]


def ngpus() -> int:
    import torch
    return torch.cuda.device_count()


def _ensemble(nmembers, nyears=2, stream=11, nsites=1):
    if nsites == 1:
        site = synth.synth_site(3, nyears, "half-daily", with_events=True)
        P = synth.synth_params(nmembers, stream=stream)
        return [site], P, None
    sites, P, ms, _ = synth.config_c3(nsites=nsites, members_per_site=nmembers // nsites, nyears=nyears)
    return sites, P, ms


@pytest.mark.parametrize("nmembers,nsites", [(9000, 1), (300, 3), (40, 1)])
def test_team_of_one_equals_local_summaries(nmembers, nsites):
    sites, P, ms = _ensemble(nmembers, nsites=nsites)
    P[A.P["leafAllocation"], 7] = 0.9                          # a failed member (bad allocation): NaN rows, excluded
    kw = dict(outputs=A.OUT_MOMENTS | A.OUT_QUANTILES, summary_cols=COLS, quantiles=QS, math=A.MATH_FAST)
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **kw) as ens:
        ens.run()
        mean, var, q = ens.mean(), ens.variance(), ens.quantiles()
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **kw) as ens:
        ens.join_team(1, 0)
        ens.run()
        ens.team_summaries()
        tmean, tvar, tq = ens.mean(), ens.variance(), ens.quantiles()
        levels = ens.team_last_levels()
    assert np.array_equal(q, tq, equal_nan=True), f"quantiles differ (levels {levels})"
    np.testing.assert_allclose(tmean, mean, rtol=1e-14, atol=1e-300)
    np.testing.assert_allclose(tvar, var, rtol=1e-12, atol=1e-24)
    assert np.isfinite(q).any()


def test_team_select_handles_ties_and_tiny_rows():
    """Order statistics inside large groups of equal values (exact zeros, duplicated members) need every key bit."""
    sites, P, ms = _ensemble(2048, nyears=1)
    P[:, 1024:] = P[:, :1024]                                  # every member twice: ties everywhere
    kw = dict(outputs=A.OUT_FULL | A.OUT_QUANTILES, summary_cols=COLS, quantiles=[0.0, 0.3, 0.5, 1.0], math=A.MATH_FAST)
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **kw) as ens:
        ens.join_team(1, 0)
        ens.run()
        out = ens.output()
        ens.team_summaries()
        tq = ens.quantiles()
    for i, c in enumerate(COLS):
        want = np.quantile(out[c], [0.0, 0.3, 0.5, 1.0], axis=1)
        np.testing.assert_allclose(tq[0, i], want, rtol=4e-16, atol=1e-300)


needs2 = pytest.mark.skipif("ngpus() < 2", reason="needs two GPUs on the box")
# every GPU of the box, or a loopback team of 2 / 3 ranks on GPU 0 (the same collectives done by device copies)
DEVICES = [pytest.param(None, marks=needs2, id="all-gpus"), pytest.param([0, 0], id="loopback2"),
           pytest.param([0, 0, 0], id="loopback3")]


@pytest.mark.parametrize("devices", DEVICES)
def test_multi_split_site_equals_one_gpu(devices):
    sites, P, ms = _ensemble(5000)
    site = sites[0]
    rng = np.random.default_rng(5)
    site.nee_obs = np.where(rng.uniform(size=site.nsteps) < 0.2, np.nan, rng.normal(0, 1.5, site.nsteps))
    kw = dict(outputs=A.OUT_FULL | A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS, summary_cols=COLS,
              quantiles=QS, math=A.MATH_FAST, nee_sigma=0.5, max_event_records=64)
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, **kw) as ens:
        ens.run()
        ref = dict(out=ens.output(), mean=ens.mean(), var=ens.variance(), q=ens.quantiles(), ll=ens.loglik(),
                   state=ens.state(), status=ens.status(), counts=ens.event_counts(), recs=ens.event_records())
    with api.MultiEnsemble(sites, P, ms, synth.SYNTH_FLAGS, devices=devices, **kw) as me:
        assert me.ndevices == (min(ngpus(), 8) if devices is None else len(devices)) and me.ndevices >= 2
        me.run()
        assert np.array_equal(me.output(), ref["out"], equal_nan=True)
        assert np.array_equal(me.state(), ref["state"], equal_nan=True)
        assert np.array_equal(me.status(), ref["status"])
        assert np.array_equal(me.loglik(), ref["ll"])
        assert np.array_equal(me.event_counts(), ref["counts"])
        got = me.event_records()
        for a, b in zip(got, ref["recs"]):
            assert [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in a] == \
                   [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in b]
        assert np.array_equal(me.quantiles(), ref["q"], equal_nan=True)      # exact order statistics, same lerp
        np.testing.assert_allclose(me.mean(), ref["mean"], rtol=1e-13, atol=1e-300)
        np.testing.assert_allclose(me.variance(), ref["var"], rtol=1e-11, atol=1e-24)


@pytest.mark.parametrize("devices", DEVICES)
def test_multi_whole_sites_equal_one_gpu(devices):
    # more sites than GPUs on any box: whole sites per device (fewer sites than devices would split them instead)
    sites, P, ms, flags = synth.config_c3(nsites=11, members_per_site=40, nyears=2)
    kw = dict(outputs=A.OUT_FULL | A.OUT_MOMENTS | A.OUT_EVENTS, summary_cols=[A.O["nee"]], math=A.MATH_FAST,
              max_event_records=64)
    with api.Ensemble(sites, P, ms, flags, **kw) as ens:
        ens.run()
        ref = dict(out=ens.output(), mean=ens.mean(), var=ens.variance(), status=ens.status(), counts=ens.event_counts())
    with api.MultiEnsemble(sites, P, ms, flags, devices=devices, **kw) as me:
        assert me.ndevices <= 11 and (devices is None or me.ndevices == len(devices))
        me.run()
        assert np.array_equal(me.output(), ref["out"], equal_nan=True)
        assert np.array_equal(me.mean(), ref["mean"], equal_nan=True)        # whole sites: the same local kernels
        assert np.array_equal(me.variance(), ref["var"], equal_nan=True)
        assert np.array_equal(me.status(), ref["status"])
        assert np.array_equal(me.event_counts(), ref["counts"])
