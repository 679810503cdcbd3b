"""The ensemble filters against their references on the shapes the model's own states never reach: ragged site tables
(empty sites, 1 and 2 participants, member counts at and one past the 128-member chunk edges, sites of more than 32
chunks), adversarial values, loopback teams whose even split cuts sites mid-chunk or leaves a rank with no or one
member, and whole-sites partitions that leave devices out (so every per-site argument is sliced at a site offset).

References are imported, not restated: eakf_reference (test_gpu_assimilate), inflated_reference / the inflation check
(test_gpu_inflation), the resampler's integer reference and adversarial weight rows (test_gpu_resample), and the
Liu-West reference with the header's semidefinite Cholesky (test_gpu_rejuvenate).

Comparisons and why their tolerances hold:
  * EAKF.  N exactly; a skipped observation (NaN value, n < 2, S_yy = 0 or not finite) leaves the site bit for bit
    and its diagnostics NaN.  The analysis, and ybar, s2, ya, within E = 1e-9 sd + 4 ulp (test_gpu_assimilate's
    bound) plus 2 B, where B is a first-order bound on what any order of naive sums can change (eakf_bound below),
    with u = 2^-53 and eta = 2^-1074:
        y_i     e_i   = (nrows + 1) u sum_j |op_j x_ij| + sum_j |op_j| E_ij     (E_ij: the bound on the input member)
        ybar    e_y   = n u mean|y| + mean e_i + u |ybar|
        xbar_j  e_x   = n u mean|x_j| + mean E_j + u |xbar_j|
        S_yy    e_S   = (n + 2) u S_yy + 2 sum |dy_i| e_i + sum (e_i + e_y)^2 + n eta
        S_jy    e_Sj  = (n + 2) u sum |cx_ij dy_i| + sum |cx_ij| e_i + sum |dy_i| E_ij + sum (E_ij + e_x)(e_i + e_y) + n eta
    (a constant shift of every dy_i or cx_ij changes S_yy and S_jy only at second order, because sum dy = sum cx = 0
    for the exact means); then s2 = S_yy / (n - 1), k = s2 / (s2 + r), alpha = sqrt(r / (s2 + r)), b_j = S_jy / S_yy,
    d_i = k (y° - ybar) + (alpha - 1) dy_i, each with its first-order propagated error plus a few u of its own
    rounding, and the analysis x_ij + b_j d_i gets E_ij + |b_j| e_d + |d_i| e_b + e_b e_d + 2 u (|x_ij| + |b_j d_i|).  The
    squares and products of first-order errors are kept (in e_S, e_Sj and the analysis' e_b e_d); the factor 2
    covers the remaining higher-order terms (of e_S / S_yy in 1 / S_yy and in alpha).  A
    dropped member moves the site's means by ~ sd / n, far outside this bound on the model-like sites.  The floor bit
    is compared for members whose every row is clear of 0 by more than the bound.
  * Inflation: test_gpu_inflation's check (state as above with its 1e-9 sd bound, N and the floor exact, lambda and
    its sd within 1e-10 relative) on model-like values; sites with n < 2 keep lambda.
  * Resampling: ancestors, N and the distinct-ancestor count exactly, ESS and log-evidence within 1e-12 relative (as
    test_gpu_resample: integer sums, so only exp and the final divisions round); copies bit for bit.
  * Liu-West: N and rank exactly; phi' within test_gpu_rejuvenate's bound (1e-9 sqrt(V_jj) + 4 ulp), compared in
    theta: the bound's interval mapped through the monotone inverse transform, plus 4 ulp of theta (near a LOGIT
    bound the round trip theta -> phi loses exactly the digits the bound is about).  A member whose
    reference proposal lies within that bound of a domain or allocation edge may take either verdict; there must be
    at most 1 % of a site's participants of them, and moved / kept must match up to their count.
  * MH: N and rank as test_gpu_mh's proposal reference; verdicts follow delta from an all-accept twin outside a
    margin of 1e-9 (1 + |delta|) (as test_gpu_mh); rejected members bit for bit; on teams log u = -inf, so the
    verdicts must agree exactly.
  * The Liu-West bound adds, per member, e ((1 - a) + h sum|z|) with e = N u mean|phi|: the kernel's mean of a
    constant row is a naive sum's rounding away from the row (see mean_slack).
  * Resampling at its size limit: a site of 2^23 members with equal weights (T = 2^63) resamples to the identity.
  * Teams: a loopback team against one GPU -- resampling bit for bit (integer sums), the floating-point filters
    within the bounds above; whole-sites partitions bit for bit against one GPU, each site's diagnostics in its row.
"""
import math

import numpy as np
import pytest

from sipnet_b200 import _abi as A, api, synth
from test_gpu_assimilate import eakf_reference, prior_sd
from test_gpu_inflation import check_against_reference as check_inflated
from test_gpu_mh import ROWS as MH_ROWS, delta, log_prior, member_equal, mh, proposal_reference
from test_gpu_rejuvenate import EXCLUDED, SPECS, cholesky, fwd, in_domain, inv, reference as lw_reference, unpack
from test_gpu_rejuvenate import within_bound as lw_within_bound
from test_gpu_resample import NEXT_BELOW_1, adversarial_weights, reference as rs_reference

POOLS = list(range(12))
S, P_ = A.S, A.P
U, ETA = 2.0 ** -53, 2.0 ** -1074
CHUNK = 128                                           # kChunk, sipnet_b200/csrc/sip_handle.h
SIZES = [1, 2, 3, 31, 32, 33, 127, 128, 129, 0, 256, 4096, 4097, 4225]
OBSERVED = [S["plantWoodC"], S["soilC"], S["soilWater"], S["litterC"], S["coarseRootC"], S["fineRootC"]]
UNOBSERVED = S["minN"]
CLASSES = ["model", "offset", "const", "huge", "subnormal", "negative", "nan_row", "nan_obs"]


# ---- the EAKF's reduction-order bound (see the module docstring) ------------------------------------------------------
def eakf_bound(state, status, ms, nsites, rows, op, value, variance):
    """-> (B [NSTATE][M], Bd [nsites][nobs][3]): bounds on |kernel - reference| for the analysis and (ybar, s2, ya)."""
    rows = list(rows)
    op = np.asarray(op, np.float64).reshape(-1, len(rows))
    nobs, nr = op.shape[0], len(rows)
    E = np.zeros((nr, state.shape[1]))
    Bd = np.zeros((nsites, nobs, 3))
    ok = ((status & EXCLUDED) == 0) & np.all(np.isfinite(state[rows]), axis=0)
    for k in range(nobs):
        X, _, _ = eakf_reference(state, status, ms, nsites, rows, op[:k], value[:, :k], variance[:, :k], floor=False)
        for s in range(nsites):
            idx = np.nonzero((ms == s) & ok)[0]
            n, yo, r = idx.size, value[s, k], variance[s, k]
            if n < 2 or math.isnan(yo):
                continue
            x, Ein, a = X[rows][:, idx], E[:, idx], np.abs(op[k])
            y = op[k] @ x
            ei = (nr + 1) * U * (a @ np.abs(x)) + a @ Ein
            ybar = math.fsum(y) / n
            ey = n * U * np.mean(np.abs(y)) + ei.mean() + U * abs(ybar)
            dy = y - ybar
            syy = math.fsum(dy * dy)
            if syy == 0 or not math.isfinite(syy):
                continue
            xbar = np.array([math.fsum(v) / n for v in x])
            ex = n * U * np.mean(np.abs(x), axis=1) + Ein.mean(axis=1) + U * np.abs(xbar)
            cx = x - xbar[:, None]
            eS = (n + 2) * U * syy + 2 * np.sum(np.abs(dy) * ei) + np.sum((ei + ey) ** 2) + n * ETA
            sjy = np.array([math.fsum(c * dy) for c in cx])
            eSj = ((n + 2) * U * (np.abs(cx) @ np.abs(dy)) + np.abs(cx) @ ei + Ein @ np.abs(dy)
                   + (Ein + ex[:, None]) @ (ei + ey) + n * ETA)
            s2 = syy / (n - 1)
            es2 = eS / (n - 1) + U * s2
            kk, alpha = s2 / (s2 + r), math.sqrt(r / (s2 + r))
            ek = r / (s2 + r) ** 2 * es2 + 2 * U * kk
            eal = alpha / (2 * (s2 + r)) * es2 + 2 * U * alpha
            g = kk * (yo - ybar)
            eg = abs(yo - ybar) * ek + kk * ey + 2 * U * abs(g)
            b = sjy / syy
            eb = (eSj + np.abs(b) * eS) / syy + U * np.abs(b)
            d = g + (alpha - 1) * dy
            ed = eg + np.abs(dy) * eal + abs(alpha - 1) * (ei + ey) + 3 * U * (abs(g) + np.abs(alpha - 1) * np.abs(dy))
            E[:, idx] = (Ein + np.abs(b)[:, None] * ed[None, :] + np.abs(d)[None, :] * eb[:, None] + np.outer(eb, ed)
                         + 2 * U * (np.abs(x) + np.abs(np.outer(b, d))))
            Bd[s, k] = ey, es2, ey + eg + U * abs(ybar + g)
    B = np.zeros_like(state)
    B[rows] = 2 * E
    return B, 2 * Bd


def test_reference_two_member_site_is_the_closed_form():
    """n = 2: s2 = (y1 - y2)^2 / 2, and the analysis puts the pair at ya -+ alpha |y1 - y2| / 2."""
    state = np.zeros((A.NSTATE, 2))
    state[POOLS] = 10.0
    row = S["plantWoodC"]
    state[row] = 7.0, 11.0
    state[S["soilC"]] = 3.0, 5.0                                          # exactly collinear with the observed row
    op = np.eye(12)[[row]]
    yo, r = 12.0, 2.0
    X, st, diag = eakf_reference(state, np.zeros(2, np.uint32), np.zeros(2, np.int32), 1, POOLS, op,
                                 np.array([[yo]]), np.array([[r]]))
    s2 = 8.0
    ya = 9.0 + s2 / (s2 + r) * (yo - 9.0)
    alpha = math.sqrt(r / (s2 + r))
    assert diag[0, 0].tolist() == [2.0, 9.0, s2, ya]
    np.testing.assert_allclose(X[row], [ya - 2 * alpha, ya + 2 * alpha], rtol=1e-15)
    np.testing.assert_allclose(X[S["soilC"]], 4.0 + (X[row] - 9.0) / 2, rtol=1e-15)
    B, Bd = eakf_bound(state, np.zeros(2, np.uint32), np.zeros(2, np.int32), 1, POOLS, op, np.array([[yo]]),
                       np.array([[r]]))
    assert (B[row] > 0).all() and (B[row] < 1e3 * U * 10).all() and (Bd[0, 0] < 1e3 * U * 10).all()
    assert (B[S["snow"]] < 1e-13).all()


def test_cholesky_rank_of_constant_and_collinear_rows():
    rng = np.random.default_rng(2)
    phi = rng.normal(size=(4, 300))
    cases = {"full": (phi, 4)}
    c = phi.copy()
    c[1] = 0.0                                                            # a constant row
    cases["constant"] = (c, 3)
    c = phi.copy()
    c[2] = 3.0 * c[0] - 1.5                                               # two exactly collinear rows
    cases["collinear"] = (c, 3)
    c = phi.copy()
    c[3] = 2.0 * np.log(np.exp(c[1])) + 7.0                              # collinear up to rounding
    cases["collinear, rounded"] = (c, 3)
    c = phi.copy()
    c[1], c[3] = 0.0, -c[0]
    cases["both"] = (c, 2)
    for name, (p, want) in cases.items():
        cc = p - np.array([math.fsum(v) / p.shape[1] for v in p])[:, None]
        V = np.array([[math.fsum(cc[j] * cc[l]) / p.shape[1] for l in range(4)] for j in range(4)])
        Lm, rank = cholesky(V)
        assert rank == want, name
        np.testing.assert_allclose(Lm @ Lm.T, V, rtol=0, atol=1e-9 * np.max(np.diag(V)))


# ---- GPU ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
KW = dict(outputs=A.OUT_LOGLIK, math=A.MATH_FAST, nee_sigma=0.5)


def excluded_members(sizes):
    """Global indices given leafAllocation = 0.9 (ST_BAD_ALLOCATION): the first and last member of a site's first two
    chunks, one whole interior chunk of a site of 32 k + 1 members, all but one member of a site of 33, every member
    of a site of 3."""
    out = []
    m0 = 0
    for n in sizes:
        loc = set()
        if n >= CHUNK:
            loc |= {0, CHUNK - 1, CHUNK, n - 1}
            if n > 9 * CHUNK and n % CHUNK == 1:
                loc |= set(range(8 * CHUNK, 9 * CHUNK))
        if n == 33:
            loc |= set(range(n)) - {16}
        if n == 3:
            loc |= set(range(n))
        out += [m0 + i for i in sorted(loc)]
        m0 += n
    return np.array(sorted(set(out)), np.int64)


def table(sizes, seed=21):
    nsites = len(sizes)
    sites = [synth.synth_site(3 + s % 6, 1, "half-daily") for s in range(nsites)]
    ms = np.repeat(np.arange(nsites, dtype=np.int32), sizes)
    P = synth.synth_params(ms.size, stream=seed)
    rng = np.random.default_rng(seed)
    P[P_["leafCSpWt"]] = rng.uniform(50, 90, ms.size)
    P[P_["fAnoxia"]] = rng.uniform(0.05, 0.5, ms.size)
    P[P_["leafAllocation"]] = rng.uniform(0.05, 0.25, ms.size)
    P[P_["woodAllocation"]] = rng.uniform(0.05, 0.25, ms.size)
    P[P_["leafAllocation"], excluded_members(sizes)] = 0.9
    obs = np.random.default_rng(8)
    for s in sites:
        s.nee_obs = np.where(obs.uniform(size=s.nsteps) < 0.3, np.nan, obs.normal(0, 1.5, s.nsteps))
    return sites, P, ms


def handle(sizes, P=None, cls=api.Ensemble, **kw):
    sites, P0, ms = table(sizes)
    e = cls(sites, P0 if P is None else P, ms, synth.SYNTH_FLAGS, **dict(KW, **kw))
    e.run(0, 2)
    return e, ms


def eakf_values(state, ms, nsites, rng, classes=CLASSES):
    """The pools of each site in one value class (site s: classes[s % len(classes)])."""
    X = state.copy()
    for s in range(nsites):
        idx = np.nonzero(ms == s)[0]
        z = rng.standard_normal((12, idx.size))
        z[S["soilC"]] += 0.7 * z[S["plantWoodC"]]
        z[S["litterC"]] -= 0.4 * z[S["soilWater"]]
        c = classes[s % len(classes)]
        v = {"offset": 1e6 + 1e-3 * z, "huge": 1e160 * (1.0 + 0.2 * z), "subnormal": 1e-310 * z,
             "negative": 3.0 + 4.0 * z,
             "const": np.repeat(32.5 * (1 + np.arange(12.0))[:, None], idx.size, axis=1)}.get(c, 50.0 + 4.0 * z)
        X[np.ix_(POOLS, idx)] = v
        if c == "nan_row" and idx.size:
            X[UNOBSERVED, idx[:: 5]] = np.nan
    return X


def eakf_obs(state, status, ms, nsites, op, classes=CLASSES, seed=1):
    rng = np.random.default_rng(seed)
    value, var = np.zeros((nsites, op.shape[0])), np.ones((nsites, op.shape[0]))
    for s in range(nsites):
        idx = np.nonzero((ms == s) & ((status & EXCLUDED) == 0))[0]
        y = op @ state[POOLS][:, idx]
        y = y[:, np.isfinite(y).all(axis=0)]
        c = classes[s % len(classes)]
        for k in range(op.shape[0]):
            if y.shape[1] < 2:
                continue
            with np.errstate(over="ignore", invalid="ignore"):
                mu, sd = float(np.mean(y[k])), float(np.std(y[k]))
            sd = sd if math.isfinite(sd) else 0.0                # the class near 1e160: its spread overflows
            shift = -3.0 if c == "negative" else 0.5 * (1 + 0.2 * rng.standard_normal())
            value[s, k] = mu + shift * sd
            v = (0.05 if c == "negative" else 0.5) * sd
            var[s, k] = v * v if 0 < v * v < 1e300 else 1.0
        if c == "nan_obs":
            value[s] = np.nan
    return value, var


def ops(nobs, combined):
    op = np.zeros((nobs, 12))
    for k in range(nobs):
        op[k, OBSERVED[k]] = 1.0
    if combined:
        op[0, [S["plantWoodC"], S["coarseRootC"], S["fineRootC"]]] = 1.0
    return op


def check_eakf(got, gstatus, diag, st0, status0, ms, nsites, op, value, var, cols=None):
    ref, rstatus, rdiag = eakf_reference(st0, status0, ms, nsites, POOLS, op, value, var)
    B, Bd = eakf_bound(st0, status0, ms, nsites, POOLS, op, value, var)
    sd = prior_sd(st0, status0, ms, nsites)
    cols = np.arange(st0.shape[1]) if cols is None else cols
    assert np.array_equal(diag[..., 0], rdiag[..., 0])
    assert np.array_equal(np.isnan(diag[..., 1:]), np.isnan(rdiag[..., 1:]))
    fin = ~np.isnan(rdiag[..., 1:])
    tol_d = 1e-9 * np.abs(rdiag[..., 1:]) + Bd
    assert np.all(np.abs(diag[..., 1:] - rdiag[..., 1:])[fin] <= tol_d[fin])
    g, w = got[POOLS][:, cols], ref[POOLS][:, cols]
    assert np.array_equal(np.isnan(g), np.isnan(w))
    tol = 1e-9 * sd[POOLS][:, ms[cols]] + 4 * np.spacing(np.abs(w)) + B[POOLS][:, cols]
    ok = ~np.isnan(w)
    bad = ok & ~(np.abs(g - w) <= tol)
    assert not bad.any(), (np.nonzero(bad.any(axis=0))[0][:10], np.max(np.abs(g - w)[ok] / tol[ok]))
    clear = np.all(np.abs(w) > tol, axis=0) | ~np.isfinite(w).all(axis=0)
    assert np.array_equal(gstatus[cols][clear], rstatus[cols][clear])
    return ref, rdiag


@gpu
@pytest.mark.parametrize("nobs,combined", [(1, False), (1, True), (4, False), (4, True)])
def test_eakf_ragged_sites(nobs, combined):
    e, ms = handle(SIZES)
    with e:
        rv, rw = e.ring()
        status0 = e.status()
        st0 = eakf_values(e.state(), ms, e.nsites, np.random.default_rng(3))
        e.set_state(st0, rv, rw, next_step=2)
        op = ops(nobs, combined)
        value, var = eakf_obs(st0, status0, ms, e.nsites, op)
        diag = e.assimilate(POOLS, op, value, var)
        got, gstatus = e.state(), e.status()
    ref, rdiag = check_eakf(got, gstatus, diag, st0, status0, ms, e.nsites, op, value, var)
    cls = np.array([CLASSES[s % len(CLASSES)] for s in range(e.nsites)])
    n = rdiag[:, 0, 0]
    assert n[[0, 1, 2, 5, 9]].tolist() == [1, 2, 0, 1, 0] and n[12] == 4097 - 4 - CHUNK
    # the skipped classes and the sites with n < 2 stay bit for bit, with NaN diagnostics
    skip = np.isin(cls, ["const", "huge", "subnormal", "nan_obs"]) | (n < 2)
    keep = skip[ms] | ((status0 & EXCLUDED) != 0) | ~np.isfinite(st0[POOLS]).all(axis=0)
    assert np.array_equal(got[:, keep], st0[:, keep], equal_nan=True)
    assert np.array_equal(gstatus[keep], status0[keep])
    assert np.isnan(diag[skip, :, 1:]).all()
    assert np.isfinite(diag[~skip, :, 1:]).all()
    # the floor happened on the negative class only, and everywhere else nothing went below 0
    floored = (gstatus & A.ST_ANALYSIS_FLOORED) != 0
    assert floored[cls[ms] == "negative"].sum() > 50 and not floored[cls[ms] != "negative"].any()
    # the bound is tight enough to see one member left out (site 13: 34 chunks, class 'negative')
    drop = int(np.nonzero(((status0 & EXCLUDED) == 0) & (ms == 13))[0][-1])
    status1 = status0.copy()
    status1[drop] |= A.ST_BAD_ALLOCATION
    ref1, _, _ = eakf_reference(st0, status1, ms, e.nsites, POOLS, op, value, var)
    B, _ = eakf_bound(st0, status1, ms, e.nsites, POOLS, op, value, var)
    tol = 1e-9 * prior_sd(st0, status0, ms, e.nsites)[POOLS][:, ms] + 4 * np.spacing(np.abs(ref1[POOLS])) + B[POOLS]
    site = (ms == 13) & (np.arange(ms.size) != drop)
    assert not np.all(np.abs(got[POOLS] - ref1[POOLS])[:, site] <= tol[:, site])


@gpu
@pytest.mark.parametrize("mode", ["fixed", "adaptive"])
def test_inflation_ragged_sites(mode):
    e, ms = handle(SIZES)
    with e:
        rv, rw = e.ring()
        status0 = e.status()
        st0 = eakf_values(e.state(), ms, e.nsites, np.random.default_rng(4), ["model", "negative"])
        e.set_state(st0, rv, rw, next_step=2)
        op = ops(4, True)
        value, var = eakf_obs(st0, status0, ms, e.nsites, op, ["model", "negative"])
        lam = np.random.default_rng(5).uniform(1.1, 2.5, e.nsites)
        sd = np.full(e.nsites, 0.4) if mode == "adaptive" else None
        diag, glam, gsd = e.assimilate_inflated(POOLS, op, value, var, lam, sd)
        got, gstatus = e.state(), e.status()
    check_inflated(got, gstatus, diag, glam, gsd, st0, status0, ms, e.nsites, POOLS, op, value, var, lam, sd)
    n = diag[:, 0, 0]
    small = n < 2
    assert small.sum() == 4                                      # n = 1, 0, 1 and the empty site
    assert np.array_equal(glam[small], lam[small]) and (sd is None or np.array_equal(gsd[small], sd[small]))
    assert np.array_equal(got[:, small[ms]], st0[:, small[ms]], equal_nan=True)
    if mode == "adaptive":
        assert not np.array_equal(glam[~small], lam[~small])


def resample_weights(ms, sizes, rng):
    """Per-site log-weights: the adversarial rows of test_gpu_resample cut or tiled to the site, and W = 0 runs (log
    weight -800 against a maximum of 0) that end exactly at a chunk edge."""
    rows = [r for _, r in adversarial_weights(rng)]
    lw = np.empty(ms.size)
    m0 = 0
    for s, n in enumerate(sizes):
        r = rows[s % len(rows)]
        lw[m0:m0 + n] = np.resize(r, n)
        if n > CHUNK and s % 2 == 0:
            lw[m0:m0 + CHUNK] = -800.0
            lw[m0 + CHUNK + 1] = 0.0                     # (members CHUNK - 1 and CHUNK do not take part)
        elif n > CHUNK:
            lw[m0 + n - 1 - CHUNK:m0 + n] = -800.0
            lw[m0 + 1] = 0.0
        m0 += n
    return lw


def site_u(nsites):
    u = np.random.default_rng(2).uniform(size=nsites)
    u[::3] = 0.0
    u[1::3] = NEXT_BELOW_1
    return u


@gpu
def test_resample_ragged_sites():
    e, ms = handle(SIZES)
    with e:
        lw = resample_weights(ms, SIZES, np.random.default_rng(4))
        status = e.status()
        st0 = e.state()
        for u in (site_u(e.nsites), np.zeros(e.nsites), np.full(e.nsites, NEXT_BELOW_1)):
            anc, diag = e.resample(u, math.inf, lw)
            ref_anc, ref_diag = rs_reference(lw, status, ms, e.nsites, u)
            assert np.array_equal(anc, ref_anc)
            assert np.array_equal(diag[:, [0, 3]], ref_diag[:, [0, 3]])
            np.testing.assert_allclose(diag[:, 1:3], ref_diag[:, 1:3], rtol=1e-12, atol=0, equal_nan=True)
            assert diag[9, 0] == 0 and diag[2, 0] == 0 and np.isnan(diag[[2, 9], 1:3]).all()
            moved = anc >= 0
            got = e.state()
            assert np.array_equal(got[:, moved], st0[:, anc[moved]], equal_nan=True)
            assert np.array_equal(e.status()[moved], status[anc[moved]])
            st0, status = got, e.status()


def lw_params(P, ms, nsites, rows, tf, lo, hi):
    """Site s gets a parameter class: model-like (the table's values), one constant row (a value whose phi has a full
    significand, so no naive sum of it is exact and the mean comes back rounded), rows 0 and 1 collinear (row 0 =
    2 phi_1 + 1), N = 2, N = 1, and members on and just inside the LOGIT bounds."""
    P = P.copy()
    for s in range(nsites):
        idx = np.nonzero(ms == s)[0]
        c = s % 6
        if c == 1:
            P[rows[0], idx] = {A.TF_IDENTITY: 20.1, A.TF_LOG: 0.1}.get(tf[0], lo[0] + 0.1 * (hi[0] - lo[0]))
        elif c == 2 and len(rows) > 1 and tf[0] == A.TF_IDENTITY:
            P[rows[0], idx] = 2.0 * fwd(P[rows[1], idx], tf[1], lo[1], hi[1]) + 1.0
        elif c in (3, 4):
            P[P_["leafAllocation"], idx[5 - c:]] = 0.9         # N = 2 and N = 1 (fewer where an edge member is out)
        elif c == 5:
            f = P_["fAnoxia"]
            P[f, idx[1::9]] = 0.55
            P[f, idx[2::9]] = np.nextafter(0.55, 0.0)
            P[f, idx[3::9]] = 0.0
            P[f, idx[4::9]] = 0.55 * (1 - 2.0 ** -30)
            P[f, idx[5::9]] = 1e-9
    return P


def lw_ambiguous(p0, phin, sd, ms, rows, tf, lo, hi):
    """Members whose reference proposal lies within the bound (1e-9 sd + 4 ulp in phi) of a domain edge, or whose
    coarse-root allocation is within the corresponding theta interval of 0."""
    cand = np.nonzero(~np.isnan(phin).any(axis=0))[0]
    amb = np.zeros(cand.size, bool)
    alloc = [P_["leafAllocation"], P_["woodAllocation"], P_["fineRootAllocation"]]
    al = [p0[r, cand].copy() for r in alloc]
    width = np.zeros(cand.size)
    for j in range(len(rows)):
        w = phin[j, cand]
        tol = 1e-9 * sd[j, ms[cand]] + 4 * np.spacing(np.abs(w))
        a, b = inv(w - tol, tf[j], lo[j], hi[j]), inv(w + tol, tf[j], lo[j], hi[j])
        amb |= in_domain(a, tf[j], lo[j], hi[j]) != in_domain(b, tf[j], lo[j], hi[j])
        if rows[j] in alloc:
            al[alloc.index(rows[j])] = inv(w, tf[j], lo[j], hi[j])
            width += np.abs(b - a)
    with np.errstate(invalid="ignore"):
        amb |= np.abs(1 - al[0] - al[1] - al[2]) <= width
    out = np.zeros(p0.shape[1], bool)
    out[cand[amb]] = True
    return out


def mean_slack(p0, ms, nsites, rows, tf, lo, hi, shrink, z, cand):
    """A derived slack for the moved phi on top of the reference's bound, which scales with the site's spread: where a
    row is constant, its spread is 0 and what is left is the rounding of the kernel's mean.  A naive sum of N values
    is within N u sum|phi| of the exact one, so |mean - mu| <= e = N u mean|phi|; the centred values, and so the row's
    entries of L below the diagonal, are at most e; phi' = a phi + (1 - a) mean + h L z then moves by at most
    e ((1 - a) + h sum_m |z_m|).  -> [n][M]."""
    extra = np.zeros((len(rows), p0.shape[1]))
    for s in range(nsites):
        idx = cand[ms[cand] == s]
        if idx.size == 0 or math.isnan(shrink[s]):
            continue
        a = shrink[s]
        h = math.sqrt(1 - a * a)
        for j in range(len(rows)):
            e = idx.size * U * np.mean(np.abs(fwd(p0[rows[j], idx], tf[j], lo[j], hi[j])))
            extra[j, idx] = e * ((1 - a) + h * np.sum(np.abs(z[:, idx]), axis=0))
    return extra


def check_lw(got, p0, phin, sd, moved, either, ms, rows, tf, lo, hi, extra):
    """Moved members within the bound (compared in theta), kept ones bit for bit; a member in `either` may be one or
    the other."""
    sure = ~either
    assert lw_within_bound(got, phin, sd, ms, rows, tf, lo, hi, np.nonzero(moved & sure)[0], True, extra)
    assert np.array_equal(got[:, ~moved & sure], p0[:, ~moved & sure])
    for m in np.nonzero(either)[0]:
        assert np.array_equal(got[:, m], p0[:, m]) or lw_within_bound(got, phin, sd, ms, rows, tf, lo, hi, [m], True,
                                                                      extra)


@gpu
@pytest.mark.parametrize("k", [1, 4, 16])
def test_liu_west_ragged_sites(k):
    rows, tf, lo, hi = unpack(SPECS[k])
    sites, P, ms = table(SIZES)
    P = lw_params(P, ms, len(SIZES), rows, tf, lo, hi)
    e, _ = handle(SIZES, P)
    with e:
        p0, st0 = e.params(), e.status()
        shrink = np.random.default_rng(4).uniform(0.75, 0.97, e.nsites)
        z = np.random.default_rng(5).standard_normal((k, e.nmembers))
        diag = e.rejuvenate(rows, tf, shrink, z, lo, hi)
        got = e.params()
    ref, rdiag, phin, moved, sd, _ = lw_reference(p0, st0, ms, e.nsites, rows, tf, lo, hi, shrink, z)
    assert np.array_equal(diag[:, :2], rdiag[:, :2])
    assert rdiag[9, 0] == 0 and rdiag[9, 1] == -1 and rdiag[5, 0] == 1 and rdiag[5, 1] == -1
    assert rdiag[3, 0] == 2 and rdiag[4, 0] == 1 and rdiag[4, 1] == -1
    cls = np.arange(e.nsites) % 6
    big = rdiag[:, 0] >= 2 * k
    assert (rdiag[(cls == 1) & big, 1] <= k - 1).all() and ((cls == 1) & big & (np.array(SIZES) > 32 * CHUNK)).any()
    if k > 1:
        assert (rdiag[(cls == 2) & big, 1] <= k - 1).all()
    either = lw_ambiguous(p0, phin, sd, ms, rows, tf, lo, hi)
    for s in range(e.nsites):
        assert either[ms == s].sum() <= 0.01 * rdiag[s, 0], s
        assert abs(diag[s, 2] - rdiag[s, 2]) <= either[ms == s].sum(), s
        assert diag[s, 2] + diag[s, 3] == rdiag[s, 2] + rdiag[s, 3], s
    assert moved.sum() > 0.5 * ms.size
    cand = np.nonzero(~np.isnan(phin).any(axis=0))[0]
    check_lw(got, p0, phin, sd, moved, either, ms, rows, tf, lo, hi,
             mean_slack(p0, ms, e.nsites, rows, tf, lo, hi, shrink, z, cand))
    print(f"k={k}: {int(either.sum())} member(s) within the bound of an edge")


# ---- loopback teams that split sites unevenly --------------------------------------------------------------------------
SPLITS = [(2, [4097]), (3, [2, 4097]), (5, [1, 3, 129, 4097]), (8, [1, 2, 9, 129, 257, 4097, 4225])]


def shares(sizes, R):
    """Global member indices of each rank of the library's even split (sites split: a contiguous share of each)."""
    m0 = np.concatenate([[0], np.cumsum(sizes)])
    return [np.concatenate([np.arange(m0[s] + n * d // R, m0[s] + n * (d + 1) // R) for s, n in enumerate(sizes)])
            .astype(np.int64) for d in range(R)]


def inject(me, R, sizes, st, P=None):
    """Every rank's members get their columns of st (and of P): the C set_state / set_params on each rank's handle."""
    lib = me.lib
    for d, idx in enumerate(shares(sizes, R)):
        h = lib.sipnet_gpu_multi_handle(me.multi, d)
        if P is not None:
            Pd = np.ascontiguousarray(P[:, idx])
            assert lib.sipnet_gpu_set_params(h, Pd.ctypes.data, idx.size) == 0
        if st is not None:
            sd = np.ascontiguousarray(st[:, idx])
            assert lib.sipnet_gpu_set_state(h, sd.ctypes.data, idx.size, None, None, idx.size, 2) == 0


@gpu
@pytest.mark.parametrize("R,sizes", SPLITS, ids=[f"R{r}" for r, _ in SPLITS])
def test_uneven_team_splits(R, sizes):
    part = [np.diff(np.r_[n * np.arange(R) // R, n]) for n in sizes]
    assert any((p == 0).any() or (p == 1).any() or (p % CHUNK != 0).any() for p in part)
    one, ms = handle(sizes)
    multi, _ = handle(sizes, cls=api.MultiEnsemble, devices=[0] * R)
    with one, multi:
        assert multi.ndevices == R
        nsites = len(sizes)
        classes = ["model", "offset", "negative"]
        status0 = one.status()
        assert np.array_equal(multi.status(), status0)
        rv, rw = one.ring()
        st0 = eakf_values(one.state(), ms, nsites, np.random.default_rng(3), classes)
        one.set_state(st0, rv, rw, next_step=2)
        inject(multi, R, sizes, st0)
        assert np.array_equal(multi.state(), st0, equal_nan=True)
        # EAKF: both against the reference, and against each other within twice the bound
        op = ops(4, True)
        value, var = eakf_obs(st0, status0, ms, nsites, op, classes)
        d1 = one.assimilate(POOLS, op, value, var)
        dm = multi.assimilate(POOLS, op, value, var)
        check_eakf(one.state(), one.status(), d1, st0, status0, ms, nsites, op, value, var)
        check_eakf(multi.state(), multi.status(), dm, st0, status0, ms, nsites, op, value, var)
        assert np.array_equal(dm[..., 0], d1[..., 0])
        # inflation, fixed and adaptive, from the same model-like prior on both
        stI = eakf_values(st0, ms, nsites, np.random.default_rng(9), ["model", "negative"])
        for lam_sd in (None, np.full(nsites, 0.4)):
            one.set_state(stI, rv, rw, next_step=2)
            inject(multi, R, sizes, stI)
            sI = one.status()
            valI, varI = eakf_obs(stI, sI, ms, nsites, op, ["model", "negative"])
            lam = np.linspace(1.3, 2.2, nsites)
            r1 = one.assimilate_inflated(POOLS, op, valI, varI, lam, lam_sd)
            rm = multi.assimilate_inflated(POOLS, op, valI, varI, lam, lam_sd)
            for e, (dg, gl, gs) in ((one, r1), (multi, rm)):
                check_inflated(e.state(), e.status(), dg, gl, gs, stI, sI, ms, nsites, POOLS, op, valI, varI, lam, lam_sd)
            assert np.array_equal(rm[0][..., 0], r1[0][..., 0])
        # Liu-West on 4 rows: N and rank exact, phi' within the bound, verdicts equal
        rows, tf, lo, hi = unpack(SPECS[4])
        p0, st2 = one.params(), one.status()
        assert np.array_equal(multi.params(), p0)
        shrink = np.random.default_rng(4).uniform(0.75, 0.97, nsites)
        z = np.random.default_rng(5).standard_normal((4, ms.size))
        j1 = one.rejuvenate(rows, tf, shrink, z, lo, hi)
        jm = multi.rejuvenate(rows, tf, shrink, z, lo, hi)
        ref, rdiag, phin, moved, sd, _ = lw_reference(p0, st2, ms, nsites, rows, tf, lo, hi, shrink, z)
        either = lw_ambiguous(p0, phin, sd, ms, rows, tf, lo, hi)
        assert not either.any()
        assert np.array_equal(j1, rdiag) and np.array_equal(jm, rdiag)
        extra = mean_slack(p0, ms, nsites, rows, tf, lo, hi, shrink, z, np.nonzero(~np.isnan(phin).any(axis=0))[0])
        for got in (one.params(), multi.params()):
            check_lw(got, p0, phin, sd, moved, either, ms, rows, tf, lo, hi, extra)
        # resampling: bit for bit against one GPU and against the reference
        lw = resample_weights(ms, sizes, np.random.default_rng(7))
        u = site_u(nsites)
        st1, status1, stm = one.state(), one.status(), multi.state()
        a1, g1 = one.resample(u, math.inf, lw)
        am, gm = multi.resample(u, math.inf, lw)
        ref_anc, ref_diag = rs_reference(lw, status1, ms, nsites, u)
        assert np.array_equal(a1, ref_anc) and np.array_equal(am, ref_anc)
        assert np.array_equal(gm, g1, equal_nan=True)
        assert np.array_equal(g1[:, [0, 3]], ref_diag[:, [0, 3]])
        np.testing.assert_allclose(g1[:, 1:3], ref_diag[:, 1:3], rtol=1e-12, atol=0, equal_nan=True)
        assert np.array_equal(multi.state()[:, am >= 0], stm[:, am[am >= 0]], equal_nan=True)
        assert np.array_equal(one.state()[:, a1 >= 0], st1[:, a1[a1 >= 0]], equal_nan=True)
        # MH on the resampled members (some sites collapsed onto one ancestor): log u = -inf accepts every valid
        # proposal whose run ends finite; N and rank as the reference, the same verdicts on both, members that do not
        # move (invalid proposals, NaN current log-likelihood, the site with scale NaN) restored bit for bit
        rng = np.random.default_rng(12)
        befores = [fields(one), fields(multi)]
        p0, stp, cur = one.params(), one.status(), one.loglik()
        cur = np.where(rng.uniform(size=ms.size) < 0.05, np.nan, cur)
        scale = rng.uniform(0.3, 0.8, nsites)
        if nsites > 1:
            scale[-1] = np.nan
        tau = np.where(np.arange(nsites) % 2 == 0, 0.0, 0.7)
        zz = rng.standard_normal((len(MH_ROWS), ms.size))
        log_u = np.full(ms.size, -np.inf)
        h1 = mh(one, MH_ROWS, scale, tau, cur, zz, log_u)
        hm = mh(multi, MH_ROWS, scale, tau, cur, zz, log_u)
        _, valid, pdiag, _ = proposal_reference(p0, stp, cur, ms, nsites, MH_ROWS, scale, zz)
        assert np.array_equal(h1[:, :2], pdiag) and np.array_equal(hm[:, :2], pdiag)
        assert np.array_equal(hm, h1)
        acc = []
        for e, before in zip((one, multi), befores):
            after = fields(e)
            # a member of a collapsed site (rank 0) is accepted with its own parameters: a verdict is any change
            a = np.array([not member_equal(after, before, m) for m in range(ms.size)])
            assert not (a & ~valid).any()
            acc.append(a)
        assert np.array_equal(acc[0], acc[1]) and acc[0].sum() == h1[:, 3].sum() > 0


# ---- whole-sites partitions that leave devices out ---------------------------------------------------------------------
# (4 sites, [0, 1], 2 devices) keeps one device, which then takes over every site from site 0: only the 6-site case
# slices per-site arguments at a non-zero first site (4); the 4-site one checks that a partition of one kept device
# leaves the empty sites' rows in place.
WHOLE = [(4, [0, 1], 2), (6, [0, 1, 4, 5], 3)]


def fields(e):
    """The per-member fields a filter may change."""
    return dict(params=e.params(), state=e.state(), status=e.status(), ll=e.loglik(), lln=e.loglik_n(),
                recs=[[] for _ in range(e.nmembers)])


@gpu
@pytest.mark.parametrize("nsites,occupied,R", WHOLE, ids=["4-sites-R2", "6-sites-R3"])
def test_whole_sites_with_left_out_devices(nsites, occupied, R):
    sizes = [129 + 64 * s if s in occupied else 0 for s in range(nsites)]
    one, ms = handle(sizes)
    multi, _ = handle(sizes, cls=api.MultiEnsemble, devices=[0] * R)
    with one, multi:
        assert multi.ndevices == len(occupied) // 2
        one.run(2, 200)
        multi.run(2, 200)
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        sid = np.arange(nsites, dtype=np.float64)
        op = ops(2, True)
        st = one.state()
        value = np.empty((nsites, 2))
        for s in range(nsites):
            y = op @ st[POOLS][:, (ms == s) & ((one.status() & EXCLUDED) == 0)]
            value[s] = y.mean(axis=1) * (1 + 0.01 * (s + 1)) if y.size else 1.0 + s
        var = np.outer(1.0 + sid, [0.5, 2.0])
        lam, lam_sd = 1.2 + 0.1 * sid, 0.1 + 0.05 * sid
        r1 = one.assimilate_inflated(POOLS, op, value, var, lam, lam_sd)
        rm = multi.assimilate_inflated(POOLS, op, value, var, lam, lam_sd)
        for a, b in zip(r1, rm):
            assert np.array_equal(a, b, equal_nan=True)
        assert np.isfinite(r1[0][occupied, :, 1:]).all() and (r1[0][occupied, :, 0] > 0).all()
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        assert np.array_equal(multi.status(), one.status())
        u = 0.1 + 0.8 * sid / nsites
        u[occupied[-1]] = np.nan
        lw = -np.abs(np.random.default_rng(3).normal(0, 1, ms.size)) * (1 + ms)
        a1, g1 = one.resample(u, math.inf, lw)
        am, gm = multi.resample(u, math.inf, lw)
        assert np.array_equal(am, a1) and np.array_equal(gm, g1, equal_nan=True)
        assert (a1[ms == occupied[-1]] == -1).all() and (a1[ms == occupied[0]] >= 0).all()
        assert np.array_equal(multi.state(), one.state(), equal_nan=True)
        rows, tf, lo, hi = unpack(SPECS[4])
        shrink = 0.8 + 0.02 * sid
        shrink[occupied[0]] = np.nan
        z = np.random.default_rng(5).standard_normal((4, ms.size))
        j1 = one.rejuvenate(rows, tf, shrink, z, lo, hi)
        jm = multi.rejuvenate(rows, tf, shrink, z, lo, hi)
        assert np.array_equal(jm, j1)
        assert j1[occupied[0], 1] == -1 and (j1[occupied[1:], 2] > 0).all()
        assert np.array_equal(multi.params(), one.params())
        scale = 0.3 + 0.05 * sid
        scale[occupied[1]] = np.nan
        tau = 0.1 * (1 + sid)
        cur = one.loglik()
        zz = np.random.default_rng(6).standard_normal((len(MH_ROWS), ms.size))
        log_u = np.log(np.random.default_rng(7).uniform(size=ms.size))
        log_u[::2] = -np.inf
        h1 = mh(one, MH_ROWS, scale, tau, cur, zz, log_u)
        hm = mh(multi, MH_ROWS, scale, tau, cur, zz, log_u)
        assert np.array_equal(hm, h1)
        assert h1[occupied[1], 1] == -1 and (h1[[occupied[0]] + occupied[2:], 3] > 0).all()
        f1, fm = fields(one), fields(multi)
        for key in f1:
            assert np.array_equal(fm[key], f1[key], equal_nan=True), key


# ---- MH on the ragged table --------------------------------------------------------------------------------------------
@gpu
def test_mh_ragged_sites():
    """Per-member log u = -inf on every 7th member, a NaN current log-likelihood (not a participant) on every 37th,
    tau = 0 on some sites, scale NaN on one.  Verdicts follow delta from an all-accept twin (as test_gpu_mh), outside
    a margin of 1e-9 (1 + |delta|); rejected members are restored bit for bit; N and rank as the reference."""
    a, ms = handle(SIZES)
    b, _ = handle(SIZES)
    with a, b:
        for e in (a, b):
            e.run(2, 40)
        M, S = a.nmembers, a.nsites
        rng = np.random.default_rng(13)
        cur = a.loglik()
        cur[::37] = np.nan
        scale = rng.uniform(0.3, 0.8, S)
        scale[6] = np.nan
        tau = rng.uniform(0.3, 1.0, S)
        tau[[3, 8, 12]] = 0.0
        z = rng.standard_normal((len(MH_ROWS), M))
        log_u = np.log(rng.uniform(size=M))
        log_u[::7] = -np.inf
        before = fields(b)
        da = mh(a, MH_ROWS, scale, tau, cur, z, np.full(M, -np.inf))
        prop = fields(a)
        db = mh(b, MH_ROWS, scale, tau, cur, z, log_u)
        got = fields(b)
    _, valid, pdiag, _ = proposal_reference(before["params"], before["status"], cur, ms, S, MH_ROWS, scale, z)
    assert np.array_equal(da[:, :2], pdiag) and np.array_equal(db[:, :3], da[:, :3])
    assert pdiag[9].tolist() == [0, -1] and pdiag[2].tolist() == [0, -1] and pdiag[6, 1] == -1
    ran_ok = (prop["params"] != before["params"]).any(axis=0)
    assert not (ran_ok & ~valid).any() and ran_ok.sum() > 0.5 * valid.sum()
    cols = np.arange(M)

    def lp(P):
        return [log_prior(P[r, cols], fwd(P[r, cols], tf, lo, hi), tf, lo, hi, pr, pa, pb)
                for (r, tf, lo, hi, pr, pa, pb) in MH_ROWS]
    with np.errstate(all="ignore"):
        d = delta(tau[ms], prop["ll"], cur, lp(prop["params"]), lp(before["params"]))
    clear = np.abs(log_u - d) >= 1e-9 * (1 + np.abs(d))
    accept = ran_ok & (log_u < d)
    assert accept.any() and (ran_ok & ~accept).any() and accept[::7].sum() == ran_ok[::7].sum()
    for m in range(M):
        if ran_ok[m] and not clear[m]:
            continue
        assert member_equal(got, prop if accept[m] else before, m), m
    if clear[ran_ok].all():
        assert np.array_equal(db[:, 3], np.bincount(ms[accept], minlength=S).astype(float))


# ---- the resampler's size limit ----------------------------------------------------------------------------------------
@gpu
def test_resample_size_limit():
    """kMaxSiteMembers = 2^23: with equal weights T = 2^23 2^40 = 2^63 exactly, the largest total the resampler's
    unsigned 64-bit table takes.  One site of 2^23 members resamples to the identity with N = ESS = 2^23; one of
    2^23 + 1 is refused and nothing changes.  outputs = 0, no event records, the default (smallest) ring of 13 slots
    for half-daily steps, no run.  A member's record is record_words = 106 device parameters + 38 state + 2 x 13 ring
    + 1 + 2 counter words + 0 events + 1 = 174 doubles; on the device the handle's parameters, state and ring take
    about (106 + 38 + 26) 8 B = 1.4 KB a member and the resampler's send and receive records 2 x 174 x 8 B = 2.8 KB,
    so at most about 35 GB for 2^23 members if both exchange buffers are allocated at full size.  On the host the [80][M]
    parameter array is 5.4 GB and a gathered state 2.5 GB.  Measured on one NVIDIA B200 (1 000 W power limit): 26.5 GiB
    of device memory in use after the 2^23-member resample, including the CUDA context; host peak RSS 5.8 GiB."""
    import gc
    import resource
    import torch
    M = 1 << 23
    site = synth.synth_site(3, 1, "half-daily")
    for n, ok in ((M, True), (M + 1, False)):
        P = np.repeat(synth.synth_params(1, stream=21), n, axis=1)
        e = api.Ensemble([site], P, np.zeros(n, np.int32), synth.SYNTH_FLAGS, outputs=0, math=A.MATH_FAST)
        del P
        gc.collect()
        with e:
            lw = np.zeros(n)
            if ok:
                anc, diag = e.resample(np.array([0.5]), math.inf, lw)
                assert np.array_equal(anc, np.arange(n))
                assert diag[0].tolist() == [n, n, 0.0, n]
                free, total = torch.cuda.mem_get_info()
                print(f"2^23 members: device in use {(total - free) / 2**30:.1f} GiB, host peak RSS "
                      f"{resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2**20:.1f} GiB")
            else:
                st0, status0 = e.state(), e.status()
                with pytest.raises(api.SipnetGpuError) as err:
                    e.resample(np.array([0.5]), math.inf, lw)
                assert err.value.code == A.ERR_BAD_ARGUMENT
                assert np.array_equal(e.state(), st0, equal_nan=True)
                assert np.array_equal(e.status(), status0)
                del st0
        gc.collect()
