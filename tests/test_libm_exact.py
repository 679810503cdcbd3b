"""The restated exp/pow (sipnet_b200/csrc/sip_libm.cuh) against the live glibc libm.

CPU: the product header is compiled in host mode by tests/native/libm_check.cpp
and compared bit for bit on ~10^7 inputs (model-shaped ranges, raw random bit
patterns, every special branch: zeros, infinities, NaN, subnormal bases,
negative bases, overflow / underflow / subnormal results).
GPU: the device build is compared bit for bit with numpy/glibc on the host."""
import os
import subprocess
import tempfile

from fractions import Fraction

import numpy as np
import pytest

from conftest import ROOT


def test_host_restatement_is_bit_exact():
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "libm_check")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-mfma", "-I", os.path.join(ROOT, "sipnet_b200", "csrc"),
                               os.path.join(ROOT, "tests", "native", "libm_check.cpp"), "-lm", "-o", exe])
        out = subprocess.run([exe, "700000"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert "0 mismatches; pow" in out.stdout and out.stdout.strip().endswith("0 mismatches")


def test_tables_match_system_libm():
    """The committed table header equals what tools/gen_libm_tables.py extracts from this box's libm."""
    hdr = os.path.join(ROOT, "sipnet_b200", "csrc", "sip_libm_tables.h")
    before = open(hdr).read()
    subprocess.check_call(["python", os.path.join(ROOT, "tools", "gen_libm_tables.py")], stdout=subprocess.DEVNULL)
    after = open(hdr).read()
    if before != after:
        open(hdr, "w").write(before)
    assert before == after, "system libm tables differ from the committed ones (different glibc?)"


@pytest.mark.gpu
def test_device_libm_is_bit_exact():
    from sipnet_b200 import api
    rng = np.random.default_rng(12345)
    n = 400000
    xs = np.concatenate([rng.uniform(-60, 20, n), rng.uniform(-750, 710, n), rng.uniform(-1100, 1100, n // 4),
                         np.array([0.0, -0.0, 1e-300, -1e-17, 709.78, -745.13, 512.0, -512.0, np.inf, -np.inf, np.nan])])
    got = api.device_libm("exp", xs)
    # numpy's exp may use its own SIMD kernels; the expected values come from the C library itself
    import ctypes
    libm = ctypes.CDLL("libm.so.6")
    libm.exp.restype = ctypes.c_double
    libm.exp.argtypes = [ctypes.c_double]
    libm.pow.restype = ctypes.c_double
    libm.pow.argtypes = [ctypes.c_double, ctypes.c_double]
    idx = np.concatenate([rng.choice(xs.size - 11, 60000, replace=False), np.arange(xs.size - 11, xs.size)])
    want = np.array([libm.exp(float(xs[i])) for i in idx])
    ok = ~np.isnan(want)
    assert np.array_equal(np.isnan(got[idx]), np.isnan(want))
    assert np.array_equal(got[idx][ok].view(np.uint64), want[ok].view(np.uint64))
    bx = np.concatenate([np.full(n, 2.0), rng.uniform(1, 6, n), rng.uniform(1e-6, 6, n), rng.uniform(0, 1, n),
                         rng.uniform(0, 2, n // 4), -rng.uniform(0, 10, n // 4)])
    by = np.concatenate([rng.uniform(-300, 10, n), rng.uniform(-6, 6, n), rng.uniform(0.5, 4, n), rng.uniform(0, 4, n),
                         rng.uniform(-1100, 1100, n // 4), np.round(rng.uniform(-40, 40, n // 4))])
    gotp = api.device_libm("pow", bx, by)
    idx = rng.choice(bx.size, 60000, replace=False)
    wantp = np.array([libm.pow(float(bx[i]), float(by[i])) for i in idx])
    ok = ~np.isnan(wantp)
    assert np.array_equal(np.isnan(gotp[idx]), np.isnan(wantp))
    assert np.array_equal(gotp[idx][ok].view(np.uint64), wantp[ok].view(np.uint64))


# the edges of every guard of the optimistic policy (sip_num.cuh FastNum) and the special values of exp / pow / division
SPECIALS = np.array([0.0, -0.0, 5e-324, -5e-324, 1e-320, 2.0 ** -1022, 2.0 ** -1000, -2.0 ** -970, 2.0 ** -969, 2.0 ** -901,
                     2.0 ** -900, -2.0 ** -899, 2.0 ** -65, 2.0 ** -64, 2.0 ** -63, 2.0 ** -55, -2.0 ** -55, 2.0 ** -54,
                     np.nextafter(2.0 ** -54, 0), -np.nextafter(2.0 ** -54, 0), 2.0 ** -53, 1e-17, -1e-17, 0.5, 1.0,
                     -1.0, np.nextafter(1.0, 2), np.nextafter(1.0, 0), 1.5, 2.0, 3.0, 10.0, 511.9999, np.nextafter(512.0, 0),
                     512.0, -512.0, 709.0, -745.0, 1024.0, 2.0 ** 62, 2.0 ** 63, 2.0 ** 64, np.nextafter(2.0 ** 64, 0),
                     2.0 ** 899, 2.0 ** 900, 2.0 ** 964, 1e300, 1.7e308, np.inf, -np.inf, np.nan])


def _glibc():
    import ctypes
    libm = ctypes.CDLL("libm.so.6")
    for f, n in (("exp", 1), ("pow", 2)):
        getattr(libm, f).restype = ctypes.c_double
        getattr(libm, f).argtypes = [ctypes.c_double] * n
    return libm


def _same_bits(got, want):
    return np.array_equal(np.asarray(got).view(np.uint64), np.asarray(want).view(np.uint64))


@pytest.mark.gpu
def test_optimistic_policy_is_exact_or_flags():
    """FastNum (sip_num.cuh), the production kernel's numerics: every value it does not flag for a replay equals
    glibc's exp / pow and the IEEE quotient bit for bit -- signed zeros, subnormals and the edges of every guard
    included -- and the inputs the model actually produces are not flagged."""
    from sipnet_b200 import api
    libm = _glibc()
    rng = np.random.default_rng(2024)
    flagged = np.uint64(api.EVAL_FLAGGED)
    specials = SPECIALS

    # ---- exp
    xs = np.concatenate([rng.uniform(-60, 20, 200000), rng.uniform(-511, 511, 100000), rng.uniform(-1e-15, 1e-15, 20000),
                         rng.uniform(-600, 600, 20000), specials, -specials])
    got = api.device_libm("fast_exp", xs)
    fl = got.view(np.uint64) == flagged
    assert not fl[np.abs(xs) < 512].any() and fl[~(np.abs(xs) < 512)].all()
    idx = np.concatenate([rng.choice(xs.size - 2 * specials.size, 30000, replace=False),
                          np.arange(xs.size - 2 * specials.size, xs.size)])
    idx = idx[~fl[idx]]
    assert _same_bits(got[idx], np.array([libm.exp(float(v)) for v in xs[idx]]))

    # ---- pow, varying base (the model: a clipped [0, 1] base, a positive parameter as exponent)
    bx = np.concatenate([rng.uniform(0, 1, 100000), np.zeros(2000), np.ones(2000), rng.uniform(1e-6, 6, 100000),
                         np.repeat(specials, specials.size), np.repeat(-specials, specials.size)])
    by = np.concatenate([rng.uniform(0, 4, 100000), rng.uniform(0, 4, 2000), rng.uniform(-4, 4, 2000), rng.uniform(-6, 6, 100000),
                         np.tile(specials, specials.size), np.tile(-specials, specials.size)])
    got = api.device_libm("fast_pow", bx, by)
    fl = got.view(np.uint64) == flagged
    assert not fl[:204000].any()                          # model-shaped inputs take the fast path
    idx = np.concatenate([rng.choice(204000, 30000, replace=False), np.arange(204000, bx.size)])
    idx = idx[~fl[idx]]
    want = np.array([libm.pow(float(a), float(b)) for a, b in zip(bx[idx], by[idx])])
    assert not np.isnan(want).any()                       # a NaN result is always flagged
    assert _same_bits(got[idx], want)

    # ---- pow through the cached log of the base (Q10 factors, 2^x of the canopy integral, vpd^exponent)
    bx = np.concatenate([np.full(100000, 2.0), rng.uniform(1, 6, 100000), rng.uniform(1e-64, 3, 50000),
                         np.repeat(specials, specials.size)])
    by = np.concatenate([rng.uniform(-300, 10, 100000), rng.uniform(-6, 6, 100000), rng.uniform(0.5, 4, 50000),
                         np.tile(specials, specials.size)])
    by[:64] = 0.0
    by[64:128] = -0.0
    by[128:256] = rng.uniform(-1e-20, 1e-20, 128)         # |y| < 2^-65: glibc's 1 + y branch
    got = api.device_libm("fast_powc", bx, by)
    fl = got.view(np.uint64) == flagged
    assert not fl[100000:250000].any() and not fl[:256].any()
    idx = np.concatenate([np.arange(256), rng.choice(250000, 30000, replace=False), np.arange(250000, bx.size)])
    idx = idx[~fl[idx]]
    want = np.array([libm.pow(float(a), float(b)) for a, b in zip(bx[idx], by[idx])])
    assert not np.isnan(want).any()
    assert _same_bits(got[idx], want)

    # ---- division: numerators of every kind over ordinary positive divisors; other divisors must be flagged
    a = np.concatenate([rng.normal(0, 100, 200000), rng.uniform(0, 1e-9, 50000), np.zeros(1000), -np.zeros(1000),
                        np.repeat(specials, specials.size), np.repeat(-specials, specials.size)])
    b = np.concatenate([rng.uniform(1e-6, 1e6, 200000), rng.uniform(0.1, 50, 50000), rng.uniform(0.1, 50, 2000),
                        np.tile(specials, specials.size), np.tile(specials, specials.size)])
    got = api.device_libm("fast_div", a, b)
    fl = got.view(np.uint64) == flagged
    assert not fl[:252000].any()
    ordinary = (b >= 2.0 ** -64) & (b < 2.0 ** 64)
    assert fl[~ordinary].all()                            # zero, negative, tiny, huge, inf, nan divisors
    with np.errstate(all="ignore"):
        want = a / b
    assert _same_bits(got[~fl], want[~fl])
    q = np.abs(want[ordinary])
    inside = (q == 0) | ((q >= 2.0 ** -900) & (q < 2.0 ** 900))
    assert np.array_equal(~fl[ordinary], inside)          # the guard is exactly "zero or 2^-900 <= |q| < 2^900"


def _exponent(x):
    """floor(log2 |x|) of a nonzero Fraction"""
    n, d = abs(x.numerator), x.denominator
    e = n.bit_length() - d.bit_length()
    return e if (n >= d << e if e >= 0 else n << -e >= d) else e - 1


def _significand(x):
    """|x| / 2^floor(log2 |x|), in [1, 2)"""
    return abs(x) / Fraction(2) ** _exponent(x)


@pytest.mark.gpu
def test_throughput_quotients_against_exact_rationals():
    """The throughput policy's divisions (sip_num.cuh ThroughNum), op by op against fractions.Fraction.

    div(a, b) = RN(a * y) with y = seed(b), the refined reciprocal.  Write Q = a / b = m_q 2^e_q and 1/b = m_r 2^e_r
    (m in [1, 2)).  Then |q - Q| <= |RN(a y) - a y| + |a| |y - 1/b|, and |a| = m_q 2^e_q / (m_r 2^e_r), so in ulps of Q
    (2^(e_q - 52)):
      * y correctly rounded, |y - 1/b| <= 2^(e_r - 53):  |q - Q| <= 1/2 + m_q / (2 m_r) < 1.5 ulp.  (When a y crosses
        into the next binade, RN(a y) is that power of two, no farther from Q than a y is; the bound stands.)
      * y only faithful, |y - 1/b| < 2^(e_r - 52):  |q - Q| < m_q / m_r + 1 (the rounding may then be a full ulp of Q).
    The test checks which of the two the seed is for every sampled divisor, against RN(1/b), and asserts the bound that
    follows for that element."""
    from sipnet_b200 import api
    rng = np.random.default_rng(2026)
    n = 100000
    b = np.concatenate([rng.uniform(1, 2, n // 4), np.exp(rng.uniform(-44, 44, n // 4)),
                        rng.integers(2 ** 52, 2 ** 53, n // 4).astype(np.float64) * 2.0 ** rng.integers(-116, 11, n // 4),
                        rng.uniform(0.1, 50, n // 4)])
    a = np.concatenate([rng.normal(0, 100, n // 2), np.exp(rng.uniform(-40, 40, n // 2)) * rng.choice([-1.0, 1.0], n // 2)])
    a[: n // 8] = rng.integers(2 ** 52, 2 ** 53, n // 8).astype(np.float64) * 2.0 ** -52   # both significands random

    # ---- op 8: the refined reciprocal against RN(1/b)
    y = api.device_libm("seed", b)
    rn = 1.0 / b
    cr = y == rn
    for i in np.flatnonzero(~cr):                      # faithful: y and RN(1/b) are the two neighbours of 1/b
        r = 1 / Fraction(float(b[i]))
        lo, hi = sorted((Fraction(float(y[i])), Fraction(float(rn[i]))))
        assert np.nextafter(rn[i], y[i]) == y[i] and lo < r < hi, (b[i].hex(), y[i].hex())

    # ---- op 6: the quotient, in ulps of the exact quotient
    q = api.device_libm("thr_div", a, b)
    assert not (q.view(np.uint64) == np.uint64(api.EVAL_FLAGGED)).any()
    worst, worst_bound = 0.0, 0.0
    for i in range(a.size):
        Q = Fraction(float(a[i])) / Fraction(float(b[i]))
        ulp = Fraction(2) ** (_exponent(Q) - 52)
        err = abs(Fraction(float(q[i])) - Q) / ulp
        ratio = _significand(Q) / _significand(1 / Fraction(float(b[i])))
        bound = Fraction(1, 2) + ratio / 2 if cr[i] else 1 + ratio
        assert err <= bound, (a[i].hex(), b[i].hex(), float(err), float(bound), bool(cr[i]))
        worst, worst_bound = max(worst, float(err)), max(worst_bound, float(bound))
    if cr.all():
        assert worst_bound < 1.5                        # sip_num.cuh: "<= 1.5 ulp instead of correctly rounded"
    print(f"throughput division: seed correctly rounded for {int(cr.sum())} of {cr.size} divisors; worst error "
          f"{worst:.4f} ulp of the exact quotient, largest proved bound of the sample {worst_bound:.4f} ulp")

    # ---- flags: the divisor check and nothing else (no quotient-range guard); op 7 = IEEE a / b where op 5 is unflagged
    sa = np.concatenate([np.repeat(SPECIALS, SPECIALS.size), np.repeat(-SPECIALS, SPECIALS.size), a[:2000]])
    sb = np.concatenate([np.tile(SPECIALS, SPECIALS.size), np.tile(SPECIALS, SPECIALS.size), b[:2000]])
    ordinary = (sb >= 2.0 ** -64) & (sb < 2.0 ** 64)
    flag = np.uint64(api.EVAL_FLAGGED)
    f5, f6, f7 = ((api.device_libm(op, sa, sb).view(np.uint64) == flag) for op in ("fast_div", "thr_div", "thr_divw"))
    assert np.array_equal(f6, ~ordinary) and np.array_equal(f7, ~ordinary)
    assert (f5 | ~f6).all() and (f5 & ordinary).any()   # op 5 flags more: its quotient-range guard
    for x, z in ((a, b), (sa[~f5], sb[~f5])):
        with np.errstate(all="ignore"):
            assert _same_bits(api.device_libm("thr_divw", x, z), x / z)

    # ---- edges, unflagged: quotients in the subnormal range and past DBL_MAX
    m1, m2 = rng.uniform(1, 2, 2000), rng.uniform(1, 2, 2000)
    sub_a, sub_b = m1 * 2.0 ** -1000 * rng.choice([-1.0, 1.0], 2000), m2 * 2.0 ** rng.integers(23, 64, 2000)
    q6, q7 = api.device_libm("thr_div", sub_a, sub_b), api.device_libm("thr_divw", sub_a, sub_b)
    assert not (q6.view(np.uint64) == flag).any() and not (q7.view(np.uint64) == flag).any() and np.isfinite(q7).all()
    tiny = Fraction(2) ** -1074
    for i in range(sub_a.size):   # rounding to the subnormal grid (<= 2^-1075) + the seed's share (< |Q| 2^-52 < 2^-1074)
        assert abs(Fraction(float(q6[i])) - Fraction(float(sub_a[i])) / Fraction(float(sub_b[i]))) < Fraction(3, 2) * tiny
    big_a, big_b = m1 * 2.0 ** 1000 * rng.choice([-1.0, 1.0], 2000), m2 * 2.0 ** -rng.integers(26, 64, 2000)
    q6, q7 = api.device_libm("thr_div", big_a, big_b), api.device_libm("thr_divw", big_a, big_b)
    assert np.array_equal(q6, np.copysign(np.inf, big_a))   # a y > DBL_MAX: RN(a y) overflows
    assert np.isnan(q7).all() and not (q7.view(np.uint64) == flag).any()   # q0 = inf, r = -inf: q0 + y r = NaN
