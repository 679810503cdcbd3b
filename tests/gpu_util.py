"""Shared helpers for the GPU parity tests."""
import numpy as np

from sipnet_b200 import _abi as A

RTOL = 1e-10  # north_star: "all state pools and fluxes within 1e-10 relative"

# fields that must match EXACTLY (branch / event / clamp decisions)
EXACT_DEBUG = ("t.lastYear", "pt.didLeafGrowth", "pt.didLeafFall", "pt.lastYear", "s.isAlive")


def column_scales(ref: np.ndarray) -> np.ndarray:
    """Per-column magnitude over the run: max_t |col| (>= tiny).  ref is [T][ncol]."""
    s = np.nanmax(np.abs(ref), axis=0)
    return np.where(s > 0, s, 1.0)


# Error metric (SURVEY 7 hard part 2): |a-b| <= rtol * max(|a|, |b|, floor), floor per column.
#  * default floor = 1e-6 x the column's own magnitude over the run, i.e. strict
#    relative error except for values six orders below the column's scale;
#  * plantCAccountingDelta (printed as nppStorage) is a CANCELLATION ACCUMULATOR:
#    |value| ~ 1e-2 while the terms it sums are ~ plantWoodC ~ 1e3, so 1-ulp
#    differences of pow/exp between CUDA's libm and glibc show up as ~1e-9 of its
#    own value although they are ~1e-15 of the quantities involved.  The survey
#    measured the same amplification inside the reference itself (+-1 ulp libm
#    perturbation => 1.3e-8 relative on this field only, no branch flips) and
#    prescribes plantWoodC as its floor; the printed column plantWoodC =
#    plantWoodC + delta (sipnet.c:455-456) is held to the strict default.
def debug_scales(ref_dbg: np.ndarray) -> np.ndarray:
    s = 1e-6 * column_scales(ref_dbg)
    s[A.D["envi.plantCAccountingDelta"]] = column_scales(ref_dbg)[A.D["envi.plantWoodC"]]
    return s


def out_scales(ref_out: np.ndarray) -> np.ndarray:
    s = 1e-6 * column_scales(ref_out)
    s[A.O["nppStorage"]] = column_scales(ref_out)[A.O["plantWoodC"]]
    return s


def max_rel(a: np.ndarray, b: np.ndarray, scale: np.ndarray) -> np.ndarray:
    """max over time of |a-b| / max(|a|,|b|,floor) per column (floor: see above)."""
    den = np.maximum(np.maximum(np.abs(a), np.abs(b)), scale[None, :])
    err = np.abs(a - b) / den
    err = np.where(np.isnan(a) & np.isnan(b), 0.0, err)
    return np.nanmax(err, axis=0)


def assert_close(a, b, scale, names, rtol=RTOL, what=""):
    e = max_rel(a, b, scale)
    bad = np.argwhere(~(e <= rtol)).ravel()
    assert bad.size == 0, what + " " + ", ".join(f"{names[i]}={e[i]:.3e}" for i in bad[:8])
    return float(np.nanmax(e)) if e.size else 0.0


# the pool columns: their empty / non-empty pattern is a clamp or mortality decision
POOL_COLS = [A.O[n] for n in ("plantWoodC", "plantLeafC", "soilC", "coarseRootC", "fineRootC", "litterC", "soilWater", "snow",
                              "minN", "soilOrgN", "litterN", "plantStorageN")]


def check_throughput(got, o_out, got_recs, o_recs, tag, cols=None):
    """The throughput policy's bar (tests/test_gpu_throughput.py): `got` [T'][len(cols)] holds one member's values of
    the output columns `cols` (all 32 by default) from a MATH_THROUGHPUT run, `o_out` [T][32] the oracle's.
      * every column within RTOL, except nLeaching (the drainage of a nearly saturated soil) within 10 * RTOL;
      * the empty / non-empty pattern of the pool columns exact ("empty" = below 1e-12 of the column's magnitude);
      * event records (when `o_recs` is not None): steps, types, variants exact, values within RTOL.
    Returns (worst error of the RTOL columns, worst nLeaching error)."""
    cols = list(range(A.NOUT)) if cols is None else list(cols)
    T = o_out.shape[0]
    g, ref = got[:T], o_out[:, cols]
    scale = out_scales(o_out)[cols]
    names = [A.OUT_NAMES[c] for c in cols]
    keep = [i for i, c in enumerate(cols) if c != A.O["nLeaching"]]
    nl = [i for i, c in enumerate(cols) if c == A.O["nLeaching"]]
    err = assert_close(g[:, keep], ref[:, keep], scale[keep], [names[i] for i in keep], RTOL, tag) if keep else 0.0
    err_nl = assert_close(g[:, nl], ref[:, nl], scale[nl], ["nLeaching"], 10 * RTOL, tag) if nl else 0.0
    pools = [i for i, c in enumerate(cols) if c in POOL_COLS]
    if pools:
        tiny = 1e-12 * np.maximum(np.nanmax(np.abs(ref[:, pools]), axis=0), 1e-300)
        assert np.array_equal(np.abs(g[:, pools]) <= tiny, np.abs(ref[:, pools]) <= tiny), \
            f"{tag}: pool clamp / mortality pattern differs"
    if o_recs is not None:
        assert [(r.step, r.type, r.variant, r.nval) for r in got_recs] == [(r.step, r.type, r.variant, r.nval) for r in o_recs], \
            f"{tag}: event rows differ"
        for a, b in zip(got_recs, o_recs):
            for k in range(b.nval):
                assert abs(a.val[k] - b.val[k]) <= RTOL * max(abs(a.val[k]), abs(b.val[k]), 1e-6), (tag, b.type, k)
    return err, err_nl


def random_flag_cases(ntrials=30, members=6, seed=2026):
    """Seeded random combinations of the 12 model flags that pass validateContext() (context.c:195-223), each with a
    synthetic two-year site (alternating step patterns, event schedule when EVENTS is on) and a few wide-prior members."""
    import numpy as np

    from sipnet_b200 import _abi as A, synth
    rng = np.random.default_rng(seed)
    for trial in range(ntrials):
        f = dict(A.DEFAULT_FLAGS)
        f.update(events=int(rng.integers(0, 2)), gdd=int(rng.integers(0, 2)), growthResp=int(rng.integers(0, 2)),
                 leafWater=int(rng.integers(0, 2)), litterPool=int(rng.integers(0, 2)), snow=int(rng.integers(0, 2)),
                 waterHResp=int(rng.integers(0, 2)), flooding=int(rng.integers(0, 2)))
        if not f["gdd"]:
            f["soilPhenol"] = int(rng.integers(0, 2))
        f["anaerobic"] = int(rng.integers(0, 2))
        if f["litterPool"]:
            f["carbonSaturation"] = int(rng.integers(0, 2))
            if f["anaerobic"]:
                f["nitrogenCycle"] = int(rng.integers(0, 2))
        site = synth.synth_site(100 + trial, 2, ["half-daily", "unequal"][trial % 2], with_events=bool(f["events"]),
                                gdd_flag=f["gdd"])
        P = synth.synth_params(members, stream=1000 + trial)
        P[A.P["soilCSaturation"], :] = rng.uniform(500, 5000)
        P[A.P["waterDrainFrac"], :] = rng.uniform(0.1, 2.0)
        yield trial, f, site, P
