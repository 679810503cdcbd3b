"""GPU: the cross-rank select's candidate lists (sip_gsum.cu) against the exact reference.

A level pass whose filter -- the slots in play plus the bins of the statistics waiting for the emit -- holds at most
kGsListCap (4 096) keys over all ranks copies each rank's members inside it to a list, and the later levels and the
emit scan that list instead of the row.  Lists are kept by a rank whose members per site are at least 4 x kGsListCap,
so the rows here have >= 16 384 members per rank.  The rows are built so that the filter population is known:
  * `cap` / `cap+1`: the median's 19-bit bin holds exactly 4 096 / 4 097 keys and its 11-bit bin more than 4 096, so
    the level-2 pass compacts the first row and not the second;
  * `narrow`: 3 000 keys of two adjacent doubles hold the median inside a bin of 3 000 keys: compacted at level 2,
    then five more levels (the last 64-bit ones) from the list;
  * `dense` and `zeros`: filters that stay too wide to compact.
Quantiles must match the reference bit for bit and the moments stay inside the bounds of check_moments, whichever
rank holds the candidates; the select must take as many levels as the route without lists (the histograms are the
same).
"""
import numpy as np
import pytest

from sipnet_b200 import _abi as A, api, synth
from test_gpu_summaries_exact import (QSETS, check_handle_result, dense_row, gen, loopback_shares, run_handle,
                                      run_loopback, same)

pytestmark = pytest.mark.gpu

CAP = 4096
M1 = 20000                                                # one rank: lists from 16 384 members per site on


def bin_row(M, inner, rng, lo_mid=1000, low=None):
    """The median in a 19-bit key bin ([1, 1 + 2^-7)) of `inner` distinct keys; its 11-bit bin ([0.5, 2)) also holds
    `lo_mid` keys below it; the rest lie far below and above (other 11-bit bins)."""
    low = M // 2 - lo_mid - inner // 4 if low is None else low
    high = M - low - lo_mid - inner
    assert low + lo_mid <= (M - 1) // 2 < low + lo_mid + inner and high >= 0
    x = np.concatenate([-5.0 + rng.uniform(size=low), 0.5 + 0.49 * rng.uniform(size=lo_mid),
                        1.0 + np.sort(rng.choice(2 ** 45, size=inner, replace=False)) * 2.0 ** -52,
                        100.0 + rng.uniform(size=high)])
    return rng.permutation(x)


def narrow_row(M, rng, inner=3000, lo_mid=2000):
    """`inner` keys of two adjacent doubles in [1, 1 + 2^-7) hold the median: every level, the last from the list."""
    x = bin_row(M, inner, rng, lo_mid)
    v = 1.0 + 2.0 ** -9
    inside = (x >= 1.0) & (x < 1.0 + 2.0 ** -7)
    x[inside] = np.where(rng.uniform(size=int(inside.sum())) < 0.5, v, np.nextafter(v, np.inf))
    return x


@pytest.mark.parametrize("inner", [CAP, CAP + 1], ids=["cap", "cap+1"])
@pytest.mark.parametrize("probs", [[0.5], [0.05, 0.5, 0.95]], ids=str)
def test_filter_at_the_capacity(inner, probs):
    rng = np.random.default_rng(inner)
    x = bin_row(M1, inner, rng)
    data = [np.stack([x, rng.permutation(x)])[None]]      # two steps: the same members in another order
    res = run_handle([M1], data, probs, team=True, want_levels=True)
    check_handle_result([M1], data, probs, res, f"{inner} keys in the bin")
    local = run_handle([M1], data, probs)
    assert same(local[2], res[2]), "team of one vs the local row kernel"


@pytest.mark.parametrize("case,probs,levels", [
    ("narrow", [0.5], 7),                # compacted at level 2, levels 3..7 and the emit from the list
    ("dense", [0.05, 0.5, 0.95], 6),     # every key shares 40 bits: too wide until the 64-bit levels
    ("zeros", [0.05], 2),                # a slot of > 4 096 equal keys: too wide, ended by the tie test
])
def test_levels_unchanged_by_the_lists(case, probs, levels):
    rng = np.random.default_rng(77)
    M = 2 ** 17 if case != "narrow" else M1
    if case == "narrow":
        x = narrow_row(M, rng)
    elif case == "dense":
        x = dense_row(M, rng)
    else:
        x = gen("zeros", M, rng)
    data = [np.stack([x, rng.permutation(x)])[None]]
    mean, var, q, got = run_handle([M], data, probs, team=True, want_levels=True)
    check_handle_result([M], data, probs, (mean, var, q), case)
    assert got == levels, f"{case}: the select used {got} levels"


# ---- loopback teams: one rank holds every candidate, the others none --------------------------------------------
MT = 8 * 16400                                            # >= 16 384 members per rank for up to 8 ranks


def _gather_to(x, idx, rng):
    """x with its members inside [1, 1 + 2^-7) moved to the member columns `idx` (same multiset of values)."""
    inside = (x >= 1.0) & (x < 1.0 + 2.0 ** -7)
    cand, rest = x[inside], x[~inside]
    assert cand.size <= idx.size
    out = np.empty_like(x)
    mask = np.zeros(x.size, bool)
    mask[idx[:cand.size]] = True
    out[mask] = cand
    out[~mask] = rng.permutation(rest)
    return out


def _team_rows(R, rng):
    shares = loopback_shares([MT], R)
    first, last = shares[0], shares[-1]
    rows = []
    for inner in (CAP, CAP + 1):
        x = bin_row(MT, inner, rng)
        rows += [_gather_to(x, first, rng), _gather_to(x, last, rng), x]
    y = narrow_row(MT, rng)
    rows += [_gather_to(y, first, rng), _gather_to(y, last, rng)]
    rows += [dense_row(MT, rng), gen("zeros", MT, rng), gen("normal", MT, rng)]
    return np.stack(rows)


@pytest.mark.parametrize("R", [2, 3, 5, 8])
@pytest.mark.parametrize("probs", [[0.5], QSETS[3]], ids=["median", "two-groups"])
def test_loopback_lists_with_uneven_candidates(R, probs):
    """QSETS[3] has 8 probabilities: two groups of kGsMaxQ, so a list made for the first group must not serve the
    second."""
    rng = np.random.default_rng(100 + R)
    data = [_team_rows(R, rng)[None]]
    got = run_loopback([MT], data, probs, R)
    check_handle_result([MT], data, probs, got, f"team of {R}")
    one = run_handle([MT], data, probs, team=True)
    assert same(got[2], one[2]), "quantiles differ from the team of one"
