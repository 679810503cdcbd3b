"""GPU: both quantile selects and the moment kernels against an exact reference, on adversarial rows.

The reference has no ensemble code (SURVEY 8c), so the definitions are this library's (sip_reduce.cu), restated
plainly here over the FINITE values of a row -- NaN and +-inf are not members of a summary (`finite_hi`):
  * quantile: numpy's "linear" rule on the sorted finite values, pos = p (n - 1), evaluated with the same lerp as the
    kernels (sip_reduce.cu); compared BIT FOR BIT (-0.0 == +0.0), and cross-checked with np.quantile;
  * mean and population variance: exact rational values (integer arithmetic on the doubles' significands), against
    error bounds that any summation order meets, but that a dropped or doubled member breaks by orders of magnitude:
      |mean - mu| <= (n + 1) u mean|x|,   |var - v| <= (n + 3) u v + 2 ((n + 1) u mean|x|)^2 + (n + 1) 2^-1074
    (u = 2^-53; the last term allows for squares that underflow below the subnormal range).
Rows are injected into the handle's column buffer after a short run (summaries are computed lazily, on the first
gather), so the model's own numbers do not limit what is tested.  Paths: sipnet_gpu_rows_summary, the per-site row
kernel and the warp moments kernel behind a handle, the cross-rank select as a team of one and as loopback teams of
2..8 ranks on one GPU (sipnet_gpu_multi_init with one device listed repeatedly).
"""
import warnings
from fractions import Fraction

import numpy as np
import pytest

from sipnet_b200 import _abi as A, api, synth

pytestmark = pytest.mark.gpu

U = Fraction(1, 2 ** 53)
TINY = Fraction(1, 2 ** 1074)
DMAX = float(np.finfo(np.float64).max)
COL = A.O["nee"]

QSETS = [[0.5], [0.05, 0.25, 0.75, 0.95], [0.0, 0.05, 0.5, 0.95, 1.0], [0.0, 0.001, 0.05, 0.25, 0.5, 0.75, 0.999, 1.0]]
# out of ascending order, repeated, and two probabilities inside one order-statistic interval (lo, lo+1, lo, lo+1)
UNSORTED = [[0.95, 0.05], [0.5, 0.95, 0.55], [0.5, 0.5], [1.0, 0.0, 0.5, 0.25, 0.75], [0.05, 0.95, 0.05],
            [0.3, 0.3], [0.3000001, 0.3]]


# ---- reference ----------------------------------------------------------------------------------------------------
def ref_quantiles(rows, probs):
    """rows [R][n] (NaN / inf = not a member) -> [len(probs)][R]."""
    rows = np.asarray(rows, np.float64)
    fin = np.isfinite(rows)
    v = np.sort(np.where(fin, rows, np.inf), axis=1)
    n = fin.sum(axis=1)
    has = n > 0
    out = np.full((len(probs), rows.shape[0]), np.nan)
    if rows.shape[1] == 0:                                # a site without members
        return out
    with np.errstate(over="ignore", invalid="ignore"):
        for i, p in enumerate(probs):
            pos = np.float64(p) * (n - 1.0)
            lo = np.floor(pos)
            fr = pos - lo
            hi = np.where(fr > 0, lo + 1.0, lo)
            a = np.take_along_axis(v, np.where(has, lo, 0).astype(np.int64)[:, None], 1)[:, 0]
            b = np.take_along_axis(v, np.where(has, hi, 0).astype(np.int64)[:, None], 1)[:, 0]
            q = np.where(fr >= 0.5, b - (b - a) * (1.0 - fr), a + (b - a) * fr)
            out[i] = np.where(has, q, np.nan)
    return out


def same(got, want):
    """bit for bit, NaN == NaN, -0.0 == +0.0"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return got.shape == want.shape and np.array_equal(np.where(got == 0, 0.0, got), np.where(want == 0, 0.0, want),
                                                      equal_nan=True)


def check_quantiles(rows, probs, got, what):
    want = ref_quantiles(rows, probs)
    bad = [(i, r) for i in range(len(probs)) for r in range(len(rows)) if not same(got[i, r], want[i, r])]
    assert not bad, f"{what}: {len(bad)} quantiles differ, first (q {bad[0][0]}, row {bad[0][1]}): " \
                    f"{got[bad[0]]!r} vs {want[bad[0]]!r}"
    for r, row in enumerate(rows):                        # numpy agrees where it can ((b - a) 0 = NaN past DBL_MAX)
        x = np.sort(row[np.isfinite(row)])
        with np.errstate(over="ignore"):
            if x.size == 0 or (x.size > 1 and np.any(np.diff(x) > DMAX)):
                continue
        with warnings.catch_warnings(), np.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            npq = np.quantile(x, probs)
        np.testing.assert_allclose(got[:, r], npq, rtol=4e-16, atol=0, err_msg=f"{what}: numpy, row {r}")


def exact_sums(x):
    """(sum x, sum x^2, sum |x|) of finite doubles, exactly: as integers in units of 2^-1074 (2^-2148 for squares)."""
    m, e = np.frexp(x)
    M = (m * 2.0 ** 53).astype(np.int64)
    sh = (e.astype(np.int64) - 53 + 1074)
    def scaled(v, k):                                     # v 2^k; k < 0 only where v is a multiple of 2^-k (subnormals)
        return v << k if k >= 0 else v >> -k
    s1 = s2 = sa = 0
    for k in np.unique(sh):
        g = M[sh == k].astype(object)
        s1 += scaled(int(g.sum()), int(k))
        s2 += scaled(int((g * g).sum()), 2 * int(k))
        sa += scaled(int(abs(g).sum()), int(k))
    return s1, s2, sa


def check_moments(row, mean, var, what):
    x = row[np.isfinite(row)]
    n = x.size
    if n == 0:
        assert np.isnan(mean) and np.isnan(var), f"{what}: empty row gives {mean}, {var}"
        return
    big = float(np.abs(x).max())                          # Python floats: n big overflows to inf quietly
    if (np.all(x > 0) or np.all(x < 0)) and n * float(np.abs(x).min()) > DMAX * (1 + 2 ** -50):
        assert not np.isfinite(mean) and not np.isfinite(var), f"{what}: the sum overflows, got {mean}, {var}"
        return
    if n * big > DMAX / 2:
        return                                            # partial sums may or may not overflow, depending on order
    s1, s2, sa = exact_sums(x)
    mu = Fraction(s1, n << 1074)
    mabs = Fraction(sa, n << 1074)
    assert np.isfinite(mean), f"{what}: mean {mean}"
    t = (n + 1) * U * mabs
    assert abs(Fraction(float(mean)) - mu) <= t + TINY, f"{what}: mean {mean!r} vs {float(mu)!r} (n {n})"
    v = Fraction(n * s2 - s1 * s1, (n * n) << 2148)
    if v >= DMAX:
        assert var == np.inf, f"{what}: variance {var} (exact {float(v)})"
    elif n * 4 * big * big < DMAX:                        # no square of a deviation overflows
        assert np.isfinite(var), f"{what}: variance {var}"
        bound = (n + 3) * U * v + 2 * t * t + (n + 1) * TINY
        assert abs(Fraction(float(var)) - v) <= bound, f"{what}: variance {var!r} vs {float(v)!r} (n {n})"


def check_all(rows, probs, mean, var, quant, what):
    if quant is not None:
        check_quantiles(rows, probs, quant, what)
    if mean is not None:
        for r, row in enumerate(rows):
            check_moments(row, mean[r], var[r], f"{what}, row {r}")


# ---- rows -----------------------------------------------------------------------------------------------------------
KINDS = ["normal", "wide", "subnormal", "dblmax", "dblmax+", "infnan", "adjacent", "zeros", "constant", "rankconst",
         "nan1", "allnan", "two"]


def gen(kind, M, rng, R=3):
    """One row: the whole ensemble of a (site, step).  R: the ranks a loopback team splits it over (rankconst)."""
    if kind == "normal":
        return rng.normal(3.0, 2.0, M)
    if kind == "wide":                                    # 10^-300 .. 10^300, both signs, +-0
        x = rng.choice([-1.0, 1.0], M) * 10.0 ** rng.uniform(-300, 300, M)
        x[::11] = 0.0
        x[5::13] = -0.0
        return x
    if kind == "subnormal":
        return np.ldexp(rng.integers(-2 ** 52 + 1, 2 ** 52, M).astype(np.float64), -1074)
    if kind in ("dblmax", "dblmax+"):                     # within 8 ulps of +-DBL_MAX
        b = (np.uint64(0x7FEFFFFFFFFFFFFF) - rng.integers(0, 8, M).astype(np.uint64)).view(np.float64)
        return b if kind == "dblmax+" else b * rng.choice([-1.0, 1.0], M)
    if kind == "infnan":
        x = rng.normal(size=M)
        u = rng.uniform(size=M)
        x[u < 0.1] = np.nan
        x[(u >= 0.1) & (u < 0.15)] = np.inf
        x[(u >= 0.15) & (u < 0.2)] = -np.inf
        return x
    if kind == "adjacent":                                # x and nextafter(x), differing in the key's last bit only
        v = float(np.float32(abs(rng.normal()) + 0.1))
        return np.where(rng.uniform(size=M) < 0.5, v, np.nextafter(v, np.inf))
    if kind == "zeros":                                   # a group of > 1024 exact zeros holds the 5 % statistic
        nneg = int(0.03 * M)
        nz = max(min(1100, M - nneg), M // 20)
        x = np.concatenate([-1.0 - rng.uniform(size=nneg), np.zeros(nz), 1.0 + rng.uniform(size=M - nneg - nz)])
        return rng.permutation(x)
    if kind == "constant":
        return np.full(M, -7.25)
    if kind == "rankconst":                               # constant on each rank, different between ranks
        return -2.0 + 1.5 * np.repeat(np.arange(R), np.diff([(M * d) // R for d in range(R + 1)])).astype(np.float64)
    if kind == "nan1":                                    # the first ranks of a team hold only NaN
        x = rng.normal(size=M)
        x[: M // 2 + 1] = np.nan
        return x
    if kind == "allnan":
        return np.full(M, np.nan)
    if kind == "two":                                     # two distinct values, many of each
        return np.where(rng.uniform(size=M) < 0.3, -1.5, 2.5)
    raise ValueError(kind)


def rows_of(M, seed, R=3, kinds=KINDS):
    rng = np.random.default_rng(seed)
    return np.stack([gen(k, M, rng, R) for k in kinds])


def emit_row(M, inner, rng):
    """`inner` keys in one level-0 bin ([1, 1.5)) hold the median; the rest lie far below and above."""
    h = (M - inner) // 2
    x = np.concatenate([-5.0 - rng.uniform(size=h), 1.0 + 0.5 * rng.uniform(size=inner), 100 + rng.uniform(size=M - h - inner)])
    return rng.permutation(x)


def dense_row(M, rng):
    """M distinct values agreeing in the top 40 key bits: only the 64-bit levels tell them apart."""
    base = np.uint64(np.float64(1.7).view(np.uint64)) & ~np.uint64(2 ** 24 - 1)
    return (base | rng.choice(2 ** 24, size=M, replace=False).astype(np.uint64)).view(np.float64)


# ---- running the paths --------------------------------------------------------------------------------------------
_TINY_SITE = None


def tiny_site(nsteps):
    """A site of `nsteps` steps of real forcing (the first steps of a synthetic site)."""
    global _TINY_SITE
    if _TINY_SITE is None or _TINY_SITE[0] < nsteps:
        s = synth.synth_site(0, max(1, -(-nsteps // 730)), "half-daily")
        _TINY_SITE = (s.nsteps, s)
    s = _TINY_SITE[1]
    return api.SiteData(s.year[:nsteps], s.day[:nsteps], {k: v[:nsteps] for k, v in s.clim.items()})


def _setup(sizes, nsteps):
    site = tiny_site(nsteps)
    sites = [site] * len(sizes)
    P = synth.synth_params(int(sum(sizes)), stream=3)
    ms = np.repeat(np.arange(len(sizes)), sizes).astype(np.int32)
    return sites, P, ms


def _inject(lib, handle, nsteps, cols, X):
    """X [ncols][nsteps][M_local] -> the handle's column buffer ([slot][nsteps][ld], slot = column with OUT_FULL)."""
    import torch
    from sipnet_b200 import distributed as D
    assert lib.sipnet_gpu_sync(handle) == 0
    M = X.shape[2]
    assert lib.sipnet_gpu_gather_bytes(handle, A.GATHER_STATUS) == 4 * M
    ld = (M + 15) // 16 * 16
    view = D.DeviceArray(lib.sipnet_gpu_device_ptr(handle, A.GATHER_FULL), (A.NOUT, nsteps, ld)).tensor()
    for i, c in enumerate(cols):
        view[c, :, :M] = torch.from_numpy(np.ascontiguousarray(X[i])).cuda()
    torch.cuda.synchronize()


def run_handle(sizes, rows_per_site, probs, moments=True, team=False, cols=(COL,), want_levels=False):
    """rows_per_site[s]: [ncols][nsteps][sizes[s]].  -> mean/var [site][col][n], quant [site][col][q][n] (, levels)"""
    nsteps = rows_per_site[0].shape[1]
    sites, P, ms = _setup(sizes, nsteps)
    outputs = A.OUT_FULL | (A.OUT_MOMENTS if moments else 0) | (A.OUT_QUANTILES if probs else 0)
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=outputs, summary_cols=list(cols), quantiles=probs,
                      math=A.MATH_FAST) as ens:
        if team:
            ens.join_team(1, 0)
        ens.run(0, nsteps)
        _inject(ens.lib, ens.handle, nsteps, cols, np.concatenate(rows_per_site, axis=2))
        if team:
            ens.team_summaries()
        res = (ens.mean() if moments else None, ens.variance() if moments else None, ens.quantiles() if probs else None)
        return res + ((ens.team_last_levels(),) if want_levels else ())


def loopback_shares(sizes, R):
    """Global member columns held by each rank of sipnet_gpu_multi_init(devices = [0] * R): the library's partition,
    without the devices that would get no member."""
    m0 = np.concatenate([[0], np.cumsum(sizes)])
    D = min(R, int(m0[-1]))
    shares = []
    for d in range(D):
        if len(sizes) < D:                                 # split sites: a contiguous share of every site
            idx = np.concatenate([np.arange(m0[s] + (n * d) // D, m0[s] + (n * (d + 1)) // D) for s, n in enumerate(sizes)])
        else:                                              # whole sites
            idx = np.arange(m0[(len(sizes) * d) // D], m0[(len(sizes) * (d + 1)) // D])
        if idx.size:
            shares.append(idx.astype(np.int64))
    return shares


def run_loopback(sizes, rows_per_site, probs, R, moments=True, cols=(COL,)):
    nsteps = rows_per_site[0].shape[1]
    sites, P, ms = _setup(sizes, nsteps)
    outputs = A.OUT_FULL | (A.OUT_MOMENTS if moments else 0) | (A.OUT_QUANTILES if probs else 0)
    X = np.concatenate(rows_per_site, axis=2)
    with api.MultiEnsemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=outputs, summary_cols=list(cols), quantiles=probs,
                           math=A.MATH_FAST, devices=[0] * R) as me:
        shares = loopback_shares(sizes, R)
        assert me.ndevices == len(shares)
        me.run(0, nsteps)
        for i, idx in enumerate(shares):
            _inject(me.lib, me.lib.sipnet_gpu_multi_handle(me.multi, i), nsteps, cols, X[:, :, idx])
        return (me.mean() if moments else None, me.variance() if moments else None, me.quantiles() if probs else None)


def per_site(sizes, seed, R=3, kinds=KINDS, ncols=1):
    rng = np.random.default_rng(seed)
    return [np.stack([np.stack([gen(k, n, rng, R) for k in kinds]) for _ in range(ncols)]) for n in sizes]


def check_handle_result(sizes, data, probs, res, what):
    mean, var, quant = res[:3]
    for s in range(len(sizes)):
        for c in range(data[s].shape[0]):
            check_all(data[s][c], probs, None if mean is None else mean[s, c], None if var is None else var[s, c],
                      None if quant is None else quant[s, c], f"{what}, site {s} ({sizes[s]} members), column {c}")


# ---- sipnet_gpu_rows_summary --------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 4000, 8192, 8193, 9000, 70001])
@pytest.mark.parametrize("probs", QSETS + UNSORTED, ids=str)
def test_rows_summary_exact(M, probs):
    import torch
    from sipnet_b200 import distributed as D
    rows = rows_of(M, seed=M)
    mean, var, q = D.rows_summary(torch.from_numpy(rows).cuda(), probs)
    check_all(rows, probs, mean.cpu().numpy(), var.cpu().numpy(), q.cpu().numpy(), f"rows_summary M={M}")


def test_rows_summary_rejects_bad_probabilities():
    import torch
    from sipnet_b200 import distributed as D
    x = torch.zeros((2, 5), dtype=torch.float64, device="cuda")
    for probs in ([0.5, np.nan], [1.5], [-0.25]):
        with pytest.raises(api.SipnetGpuError, match="out of"):
            D.rows_summary(x, probs)


# ---- the per-site row kernel and the warp moments kernel behind a handle ------------------------------------------
RAGGED = [1, 2, 8192, 8193, 70001, 9000]                  # the last site gets a NaN tail (a ragged site)


@pytest.mark.parametrize("probs", QSETS + UNSORTED, ids=str)
def test_handle_row_kernel_exact(probs):
    data = per_site(RAGGED, seed=21)
    data[-1][:, :, 6000:] = np.nan
    res = run_handle(RAGGED, data, probs)
    check_handle_result(RAGGED, data, probs, res, "handle")


@pytest.mark.parametrize("sizes", [[1, 31, 32, 33, 255, 256], [257, 1, 32]], ids=["warp", "falls-back-to-row-kernel"])
def test_handle_moments_only_exact(sizes):
    data = per_site(sizes, seed=22)
    res = run_handle(sizes, data, [])
    check_handle_result(sizes, data, [], res, "moments")


def test_grid_tiling_of_steps_and_sites():
    """More than 65 535 steps (the warp moments kernel tiles grid.y over steps) and more than 65 535 sites (the row
    kernel tiles grid.y over sites).  Row t / site s gets values that identify it, so a tile written to the wrong
    place, or read from it, shows."""
    rng = np.random.default_rng(4)
    nsteps = 65535 + 70
    X = (np.arange(nsteps)[:, None] * 8 + rng.integers(0, 8, size=(nsteps, 4))).astype(np.float64)
    mean, var, _ = run_handle([4], [X[None]], [])
    want_mean = X.sum(axis=1) / 4                          # integers: the sums are exact in any order
    assert np.array_equal(mean[0, 0], want_mean)
    for t in list(range(65530, 65545)) + [0, nsteps - 1]:
        check_moments(X[t], mean[0, 0, t], var[0, 0, t], f"step {t}")
    nsites = 65535 + 37
    sizes = [2] * nsites
    vals = (np.arange(nsites)[:, None] * 4 + rng.integers(0, 4, size=(nsites, 2))).astype(np.float64)
    data = [vals[s].reshape(1, 1, 2) for s in range(nsites)]
    mean, var, q = run_handle(sizes, data, [0.5, 0.0])
    assert np.array_equal(mean[:, 0, 0], vals.sum(axis=1) / 2)
    assert np.array_equal(q[:, 0, 0, 0], vals.sum(axis=1) / 2)  # the median of two integers below 2^53
    assert np.array_equal(q[:, 0, 1, 0], vals.min(axis=1))


# ---- the cross-rank select: a team of one -------------------------------------------------------------------------
TEAM_SIZES = [1, 2, 17, 8193, 70001]


@pytest.mark.parametrize("probs", [QSETS[3], QSETS[2]] + UNSORTED, ids=str)
def test_team_of_one_exact(probs):
    data = per_site(TEAM_SIZES, seed=23)
    res = run_handle(TEAM_SIZES, data, probs, team=True)
    check_handle_result(TEAM_SIZES, data, probs, res, "team of one")


@pytest.mark.parametrize("case,probs,M,levels", [
    ("adjacent", [0.5], 20000, 7),      # two adjacent doubles: all eight histogram levels, the last one 5 bits wide
    ("zeros", [0.05], 40000, 2),        # > 1024 equal keys hold the statistic: the tie test ends the select early
    ("emit16", [0.5], 4001, 0),         # 16 keys in the statistic's level-0 bin: finished by gathering them
    ("emit17", [0.5], 4001, 1),         # 17 keys: one more level first
    ("dense", [0.05, 0.5, 0.95], 2 ** 20, 6),  # 2^20 distinct keys sharing 40 bits: the 64-bit levels
])
def test_team_select_reaches_its_paths(case, probs, M, levels):
    rng = np.random.default_rng(31)
    if case.startswith("emit"):
        x = emit_row(M, int(case[4:]), rng)
    elif case == "dense":
        x = dense_row(M, rng)
    else:
        x = gen(case, M, rng)
    data = [np.stack([x, rng.permutation(x)])[None]]
    mean, var, q, got_levels = run_handle([M], data, probs, team=True, want_levels=True)
    check_handle_result([M], data, probs, (mean, var, q), case)
    assert got_levels == levels, f"{case}: the select used {got_levels} levels"
    # and the local row kernel on the same rows
    res = run_handle([M], data, probs)
    assert same(res[2], q)


# ---- the cross-rank select: loopback teams of R ranks on one GPU --------------------------------------------------
def _team_sizes(R):
    # one split site for R = 2; otherwise a small site too (fewer sites than ranks: every site is split), whose
    # R + 1 members leave most ranks with one member
    return [70001] if R == 2 else [R + 1, 70001]


@pytest.mark.parametrize("R", [2, 3, 5, 8])
@pytest.mark.parametrize("probs", [QSETS[3], [0.95, 0.05], [0.5, 0.95, 0.55], [0.05, 0.95, 0.05], [0.3, 0.3]], ids=str)
def test_loopback_team_exact(R, probs):
    sizes = _team_sizes(R)
    data = per_site(sizes, seed=40 + R, R=R)
    got = run_loopback(sizes, data, probs, R)
    check_handle_result(sizes, data, probs, got, f"team of {R}")
    one = run_handle(sizes, data, probs, team=True)
    assert same(got[2], one[2]), "quantiles differ from the team of one"


@pytest.mark.parametrize("ncols", [1, 8, 9])
def test_loopback_team_summary_columns(ncols):
    sizes = [9001]
    kinds = ["normal", "zeros", "nan1", "adjacent"]
    data = per_site(sizes, seed=50, R=3, kinds=kinds, ncols=ncols)
    cols = list(range(ncols))
    if ncols > 8:
        with pytest.raises(api.SipnetGpuError, match="1..8 summary columns"):
            run_loopback(sizes, data, [0.05, 0.5], 3, cols=cols)
        return
    got = run_loopback(sizes, data, [0.05, 0.5], 3, cols=cols)
    check_handle_result(sizes, data, [0.05, 0.5], got, f"{ncols} columns")


def test_multi_init_rejects_a_repeated_device_mixed_with_others():
    sites, P, ms = _setup([8], 4)
    with pytest.raises(api.SipnetGpuError, match="one device repeatedly"):
        api.MultiEnsemble(sites, P, ms, synth.SYNTH_FLAGS, devices=[0, 0, 1])


# ---- loopback partitions against one GPU: real model output -------------------------------------------------------
def _compare_multi_with_one_gpu(sites, P, ms, flags, R, probs, ndev):
    site_obs = np.random.default_rng(5)
    for s in {id(x): x for x in sites}.values():
        s.nee_obs = np.where(site_obs.uniform(size=s.nsteps) < 0.2, np.nan, site_obs.normal(0, 1.5, s.nsteps))
    kw = dict(outputs=A.OUT_FULL | A.OUT_MOMENTS | A.OUT_QUANTILES | A.OUT_LOGLIK | A.OUT_EVENTS,
              summary_cols=[A.O["nee"], A.O["gpp"], A.O["snow"]], quantiles=probs, math=A.MATH_FAST, nee_sigma=0.5,
              max_event_records=64)
    with api.Ensemble(sites, P, ms, flags, **kw) as ens:
        ens.run()
        ref = dict(out=ens.output(), mean=ens.mean(), var=ens.variance(), q=ens.quantiles(), ll=ens.loglik(),
                   state=ens.state(), status=ens.status(), counts=ens.event_counts(), recs=ens.event_records())
    with api.MultiEnsemble(sites, P, ms, flags, devices=[0] * R, **kw) as me:
        assert me.ndevices == ndev
        me.run()
        out = me.output()
        assert np.array_equal(out, ref["out"], equal_nan=True)
        assert np.array_equal(me.state(), ref["state"], equal_nan=True)
        assert np.array_equal(me.status(), ref["status"])
        assert np.array_equal(me.loglik(), ref["ll"])
        assert np.array_equal(me.event_counts(), ref["counts"])
        for a, b in zip(me.event_records(), ref["recs"]):
            assert [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in a] == \
                   [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in b]
        q, mean, var = me.quantiles(), me.mean(), me.variance()
    assert np.array_equal(q, ref["q"], equal_nan=True)
    for s in range(len(sites)):
        sel = ms == s
        for i, c in enumerate(kw["summary_cols"]):
            rows = out[c][:, sel]                          # [T][members of the site]
            check_quantiles(rows, probs, q[s, i], f"site {s}, column {c}")
            for t in range(0, rows.shape[0], 97):
                check_moments(rows[t], mean[s, i, t], var[s, i, t], f"site {s}, column {c}, step {t}")


def test_loopback_split_with_fewer_members_than_ranks():
    """Two sites of 1 and 2 members over 3 ranks: split sites, and the rank that would get no member is left out."""
    site = synth.synth_site(3, 1, "half-daily", with_events=True)
    P = synth.synth_params(3, stream=12)
    ms = np.array([0, 1, 1], np.int32)
    _compare_multi_with_one_gpu([site, site], P, ms, synth.SYNTH_FLAGS, 3, [0.05, 0.5, 1.0], 2)


@pytest.mark.parametrize("nsites,occupied,R,ndev", [(4, [0, 1], 2, 1), (6, [0, 1, 4, 5], 3, 2)])
def test_loopback_whole_sites_with_an_empty_site_range(nsites, occupied, R, ndev):
    """Whole sites per rank where a rank's site range holds no member: that rank is left out, and the rank before
    it takes its (empty) sites, so the summaries still cover every site in order."""
    sites = [synth.synth_site(i, 1, "half-daily", with_events=True) for i in range(nsites)]
    P = synth.synth_params(15 * len(occupied), stream=13)
    ms = np.repeat(occupied, 15).astype(np.int32)
    _compare_multi_with_one_gpu(sites, P, ms, synth.SYNTH_FLAGS, R, [0.95, 0.05], ndev)
