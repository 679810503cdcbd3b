"""Every instantiation of the step kernel under test, each confirmed by the name the profiler records.

The step kernel is 78 instantiations of `run_kernel` (sip_run.cuh): for the optimistic (FastNum) and the throughput
(ThroughNum) numerics, 3 flag policies x {32-member blocks, 128-member blocks, 128 with two sites per block (MIX)} x
{all 32 columns in place (FULL), only the kept summary columns} x {one CTA per block, persistent grid (DYN)}; and 6
general (ExactNum) ones: validation, debug dump and replay, at both block sizes.

CPU: the ledger.  The instantiations in the built library (cuobjdump + cu++filt) are exactly the rows of MATRIX and
EXACT_ROWS below, so a kernel added without a case fails before anyone reaches a GPU.

GPU: one case per row.  Each case runs inside torch.profiler and asserts that the optimistic / throughput kernel it
names was launched, and no other one (the replay and the validation reference are the only other run_kernel
launches).  Every case runs three segments [0, 300), [300, 600), [600, T) -- not multiples of the 256-step work item
of the persistent grid -- against the same configuration under MATH_VALIDATION:
  * FastNum: bit for bit -- every kept column of every step, state, ring, status (ST_REPLAY masked), log-likelihood
    and its observation count, event counts and records -- and bit for bit against the oracle on sampled members
    (first and last member of every site and of every mixed block, the last member, the replayed members);
  * ThroughNum: the oracle under the throughput bar (gpu_util.check_throughput) on the same sampled members; against
    the validation run the pools of the final state within RTOL, and status, observation counts, event counts and
    event steps / types / variants exactly.
Two members of every case leave the optimistic exp guard (a 2000 m2/m2 canopy): ST_REPLAY is set on exactly those.
The first segment, where they leave it, is integrated by the replay, the ExactNum kernel, so their columns there equal
the oracle's bit for bit under both numerics.  The site's first mortality event clears the canopy; from then on the
kernel under test integrates them like any other member (under ThroughNum: within the throughput bar)."""
import json
import os
import re
import shutil
import subprocess
import tempfile
from collections import namedtuple

import numpy as np
import pytest

from conftest import ROOT
from gpu_util import RTOL, check_throughput

LIB = os.path.join(ROOT, "sipnet_b200", "libsipnet_gpu.so")

Inst = namedtuple("Inst", "num policy block full dyn mix debug replay")

# StaticFlags masks (sip_run.cuh kMaskDefault / kMaskCropN); RuntimeFlags = the generic policy
POLICY_OF_MASK = {163: "default", 947: "cropn"}


def _split_top(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    return out + [cur.strip()]


def _num(tok):
    """`(bool)0`, `false`, `(int)128`, `128`, `(unsigned int)163`, `163u` -> int"""
    t = re.sub(r"\((?:unsigned int|int|bool)\)", "", tok).strip()
    return {"false": 0, "true": 1}[t] if t in ("false", "true") else int(t.rstrip("uU"))


def parse_run_kernel(name):
    """A demangled run_kernel name, in cu++filt's or the profiler's spelling -> Inst (None for any other kernel)."""
    i = name.find("run_kernel<")
    if i < 0:
        return None
    start, depth = i + len("run_kernel<"), 0
    for j in range(start, len(name)):
        if name[j] == "<":
            depth += 1
        elif name[j] == ">":
            if depth == 0:
                break
            depth -= 1
    fl, debug, num, block, replay, full, dyn, tune = _split_top(name[start:j])
    m = re.search(r"StaticFlags<([^>]*)>", fl)
    policy = POLICY_OF_MASK[_num(m.group(1))] if m else "generic"
    mix = _num(_split_top(tune[tune.index("<") + 1:tune.rindex(">")])[1])
    return Inst(num.split("::")[-1], policy, _num(block), _num(full), _num(dyn), mix, _num(debug), _num(replay))


# ---- the matrix: one row per optimistic / throughput instantiation ------------------------------------------------
# layout (member counts per site, see LAYOUTS): `sites` = 5 sites whose counts leave tails of every size and one site
# small enough to sit inside a block (MIX at 128), `aligned` = multiples of 128 (no mixed block), `dyn32` / `dyn128` /
# `dynmix` = more block descriptors than resident CTAs (persistent grid), the last with mixed blocks.
# columns: FULL = OUT_FULL; a tuple = the kept summary columns in slot order (every Emitter path: NEE and GPP alone in
# both slot orders, NEE or GPP with a column of the switch, GPP alone, switch columns only); () = no column buffer
# (log-likelihood and events only).
FULL = "full"
NG, GN, NW, G, WOOD, NONE, NGW = (("nee", "gpp"), ("gpp", "nee"), ("nee", "soilWater"), ("gpp",), ("plantWoodC",), (),
                                  ("nee", "gpp", "soilWater"))
MATRIX = [
    # numerics  flags      block layout     columns
    ("fast", "default", 32, "sites", FULL),
    ("fast", "default", 32, "sites", NG),
    ("fast", "default", 32, "dyn32", FULL),
    ("fast", "default", 32, "dyn32", GN),
    ("fast", "default", 128, "aligned", FULL),
    ("fast", "default", 128, "aligned", NW),
    ("fast", "default", 128, "sites", FULL),
    ("fast", "default", 128, "sites", G),
    ("fast", "default", 128, "dyn128", FULL),
    ("fast", "default", 128, "dyn128", WOOD),
    ("fast", "default", 128, "dynmix", FULL),
    ("fast", "default", 128, "dynmix", NONE),
    ("fast", "cropn", 32, "sites", FULL),
    ("fast", "cropn", 32, "sites", NGW),
    ("fast", "cropn", 32, "dyn32", FULL),
    ("fast", "cropn", 32, "dyn32", WOOD),
    ("fast", "cropn", 128, "aligned", FULL),
    ("fast", "cropn", 128, "aligned", G),
    ("fast", "cropn", 128, "sites", FULL),
    ("fast", "cropn", 128, "sites", NW),
    ("fast", "cropn", 128, "dyn128", FULL),
    ("fast", "cropn", 128, "dyn128", NONE),
    ("fast", "cropn", 128, "dynmix", FULL),
    ("fast", "cropn", 128, "dynmix", NG),
    ("fast", "generic", 32, "sites", FULL),
    ("fast", "generic", 32, "sites", NONE),
    ("fast", "generic", 32, "dyn32", FULL),
    ("fast", "generic", 32, "dyn32", NW),
    ("fast", "generic", 128, "aligned", FULL),
    ("fast", "generic", 128, "aligned", GN),
    ("fast", "generic", 128, "sites", FULL),
    ("fast", "generic", 128, "sites", WOOD),
    ("fast", "generic", 128, "dyn128", FULL),
    ("fast", "generic", 128, "dyn128", G),
    ("fast", "generic", 128, "dynmix", FULL),
    ("fast", "generic", 128, "dynmix", NGW),
    ("thr", "default", 32, "sites", FULL),
    ("thr", "default", 32, "sites", GN),
    ("thr", "default", 32, "dyn32", FULL),
    ("thr", "default", 32, "dyn32", NG),
    ("thr", "default", 128, "aligned", FULL),
    ("thr", "default", 128, "aligned", G),
    ("thr", "default", 128, "sites", FULL),
    ("thr", "default", 128, "sites", NW),
    ("thr", "default", 128, "dyn128", FULL),
    ("thr", "default", 128, "dyn128", NONE),
    ("thr", "default", 128, "dynmix", FULL),
    ("thr", "default", 128, "dynmix", WOOD),
    ("thr", "cropn", 32, "sites", FULL),
    ("thr", "cropn", 32, "sites", WOOD),
    ("thr", "cropn", 32, "dyn32", FULL),
    ("thr", "cropn", 32, "dyn32", NONE),
    ("thr", "cropn", 128, "aligned", FULL),
    ("thr", "cropn", 128, "aligned", NG),
    ("thr", "cropn", 128, "sites", FULL),
    ("thr", "cropn", 128, "sites", NGW),
    ("thr", "cropn", 128, "dyn128", FULL),
    ("thr", "cropn", 128, "dyn128", GN),
    ("thr", "cropn", 128, "dynmix", FULL),
    ("thr", "cropn", 128, "dynmix", G),
    ("thr", "generic", 32, "sites", FULL),
    ("thr", "generic", 32, "sites", G),
    ("thr", "generic", 32, "dyn32", FULL),
    ("thr", "generic", 32, "dyn32", NW),
    ("thr", "generic", 128, "aligned", FULL),
    ("thr", "generic", 128, "aligned", WOOD),
    ("thr", "generic", 128, "sites", FULL),
    ("thr", "generic", 128, "sites", NONE),
    ("thr", "generic", 128, "dyn128", FULL),
    ("thr", "generic", 128, "dyn128", NG),
    ("thr", "generic", 128, "dynmix", FULL),
    ("thr", "generic", 128, "dynmix", GN),
]
# cases that add no instantiation: ctx.snow has no arithmetic effect, so DEFAULT_FLAGS with snow = 0 must still run
# the default policy's kernel (and stay bit-identical); the debug dump at both block sizes
EXTRA = [
    ("fast", "default-nosnow", 32, "sites", FULL),
    ("thr", "default-nosnow", 128, "aligned", NG),
    ("debug", "cropn", 32, "sites", FULL),
    ("debug", "generic", 128, "sites", FULL),
]


def case_id(row):
    num, flags, block, layout, cols = row
    return f"{num}-{flags}-{block}-{layout}-" + (cols if cols == FULL else "+".join(cols) or "nocols")


POLICY_OF_FLAGS = {"default": "default", "default-nosnow": "default", "cropn": "cropn", "generic": "generic"}
NUMERICS = {"fast": "FastNum", "thr": "ThroughNum"}
DYN_LAYOUTS = ("dyn32", "dyn128", "dynmix")
MIX_LAYOUTS = ("sites", "dynmix")


def expected_inst(row):
    num, flags, block, layout, cols = row
    return Inst(NUMERICS[num], POLICY_OF_FLAGS[flags], block, int(cols == FULL), int(layout in DYN_LAYOUTS),
                int(block == 128 and layout in MIX_LAYOUTS), 0, 0)


# the general kernels: the validation reference of every case, the replay after every optimistic / throughput run,
# the debug cases (MIX: the general kernels always take the two-site path at 128, sip_run_exact.cu)
EXACT_ROWS = {f"{what}-{b}": Inst("ExactNum", "generic", b, 0, 0, int(b == 128), int(what == "debug"), int(what == "replay"))
              for what in ("validation", "replay", "debug") for b in (32, 128)}

LEDGER = {case_id(r): expected_inst(r) for r in MATRIX} | EXACT_ROWS


def binary_instantiations():
    if not (os.path.exists(LIB) and shutil.which("cuobjdump") and shutil.which("cu++filt")):
        pytest.skip("library, cuobjdump or cu++filt missing")
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(m for m in re.findall(r"Function (\S+):", out) if "run_kernel" in m))
    dem = subprocess.run(["cu++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.split("\n")
    return {parse_run_kernel(d): d for d in dem if "run_kernel" in d}


def test_ledger_names_every_instantiation_in_the_library():
    insts = binary_instantiations()
    assert len(insts) == 78, len(insts)
    assert None not in insts
    rows = set(LEDGER.values())
    assert len(rows) == len(LEDGER), "two rows name the same instantiation"
    missing = [insts[i] for i in insts if i not in rows]
    assert not missing, "instantiations without a case: " + "; ".join(missing)
    extra = [name for name, i in LEDGER.items() if i not in insts]
    assert not extra, "rows naming an instantiation the library lacks: " + ", ".join(extra)


def test_name_parser_reads_both_spellings():
    """cu++filt writes `(bool)0`, `(unsigned int)947`; the profiler (CUPTI) writes `false`, `947u`."""
    a = ("void sip::k1::run_kernel<sip::StaticFlags<(unsigned int)947>, (bool)0, sip::ThroughNum, (int)128, (bool)0, "
         "(bool)1, (bool)1, sip::k1::Tune<(int)128, (bool)1, (int)1, (int)16>>(sip::RunArgs)")
    b = ("void sip::k1::run_kernel<sip::StaticFlags<947u>, false, sip::ThroughNum, 128, false, true, true, "
         "sip::k1::Tune<128, true, 1, 16> >(sip::RunArgs)")
    want = Inst("ThroughNum", "cropn", 128, 1, 1, 1, 0, 0)
    assert parse_run_kernel(a) == want and parse_run_kernel(b) == want
    assert parse_run_kernel("void sip::k1::run_kernel<sip::RuntimeFlags, true, sip::ExactNum, 32, false, false, false, "
                            "sip::k1::Tune<32, false, 1, 32> >(sip::RunArgs)") == Inst("ExactNum", "generic", 32, 0, 0, 0, 1, 0)
    assert parse_run_kernel("void sip::gs::gs_pass0<4>(sip::gs::Args)") is None


def test_persistent_layouts_exceed_resident_ctas():
    for layout, resident in (("dyn32", RESIDENT_32), ("dyn128", RESIDENT_128), ("dynmix", RESIDENT_128)):
        assert len(block_layout(LAYOUTS[layout], 32 if layout == "dyn32" else 128)) > resident, layout
    assert sum(1 for m0, c0, c in block_layout(LAYOUTS["dynmix"], 128) if c > c0) == 2
    assert sum(1 for m0, c0, c in block_layout(LAYOUTS["sites"], 128) if c > c0) == 3
    assert all(sum(c) % 16 == 0 for c in LAYOUTS.values())            # ld == M: kept columns are [ncols][n][M]


# ---- GPU ------------------------------------------------------------------------------------------------------------
# Resident CTAs of the persistent launches (their grid = cudaOccupancyMaxActiveBlocksPerMultiprocessor x SMs).  32-member
# blocks: 5 per SM, read on one B200 (148 SMs) as the grid of all twelve persistent 32-member launches in the profiler
# trace (253-255 registers, 40.6 KB of shared memory per block); 128-member blocks ask for 2 per SM.  The dyn* layouts
# have more block descriptors; should the occupancy change, the kernel-name assertion of those cases fails instead of
# quietly testing the static kernel.
RESIDENT_32 = 148 * 5
RESIDENT_128 = 148 * 2
SEGMENT = 300
MAXREC = 16


LAYOUTS = {
    "sites": [100, 37, 5, 150, 28],                       # 320 members; tails 100, 37+5 (one site inside), 22, 28
    "aligned": [256, 128, 384],
    "dyn128": [128 * 100, 128 * 100, 128 * 100],          # 300 blocks of 128 > 296 resident
    "dynmix": [128 * 100 + 37, 5, 128 * 101 + 22, 128 * 100],   # 303 blocks, two of them mixed
    "dyn32": [32 * 300 + 21, 32 * 300 + 7, 32 * (RESIDENT_32 - 540) - 28],   # 802 blocks of 32 > 740 resident
}


def block_layout(counts, B):
    """The host's block descriptors (sipnet_gpu.cu): (member0, count0, count) per block, a site's tail sharing its block
    with the next site's head at 128."""
    blocks, starts = [], np.concatenate([[0], np.cumsum(counts)])
    taken = 0
    for s, n in enumerate(counts):
        off, taken_next = taken, 0
        while off < n:
            m0 = starts[s] + off
            c0 = min(B, n - off)
            c = c0
            if B == 128 and c0 < B and s + 1 < len(counts):
                taken_next = min(B - c0, counts[s + 1])
                c = c0 + taken_next
            blocks.append((int(m0), int(c0), int(c)))
            off += B
        taken = taken_next
    return blocks


def _flags(name):
    from sipnet_b200 import _abi as A, synth
    return {"default": dict(A.DEFAULT_FLAGS), "default-nosnow": dict(A.DEFAULT_FLAGS, snow=0),
            "cropn": dict(synth.SYNTH_FLAGS), "generic": dict(synth.SYNTH_FLAGS, flooding=1, growthResp=1)}[name]


def _kernel_launches(prof):
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    out = []
    for e in trace.get("traceEvents", []):
        if e.get("cat") == "kernel" and "run_kernel" in e.get("name", ""):
            out.append((parse_run_kernel(e["name"]), e.get("args", {}).get("grid")))
    return out


def _kept(ens, ncols, n, M):
    import torch
    from sipnet_b200 import _abi as A
    from sipnet_b200.distributed import DeviceArray
    return DeviceArray(ens.device_ptr(A.GATHER_FULL), (ncols, n, M), (n * M, M, 1)).tensor(torch.cuda.current_device())


def _first_diff(got, want, cols):
    """where two [T][ncols] series first differ in bits: (step, column name, got, want)"""
    t, c = np.argwhere(got.view(np.int64) != want.view(np.int64))[0]
    from sipnet_b200 import _abi as A
    return f"(step {t}, {A.OUT_NAMES[cols[c]]}: {got[t, c]!r} != {want[t, c]!r})"


def _status_diff(got, want):
    bad = np.flatnonzero(got != want)
    return ", ".join(f"member {m}: {got[m]:#x} != {want[m]:#x}" for m in bad[:4])


def _records(ens):
    """[M][MAXREC] record array of the event records (slots past a member's count are cleared)"""
    from sipnet_b200 import _abi as A
    buf = np.zeros(ens.nmembers * MAXREC, dtype=np.dtype(A.EventRecord))
    ens.gather_raw(A.GATHER_EVENT_RECORDS, buf.ctypes.data, buf.nbytes)
    buf = buf.reshape(ens.nmembers, MAXREC)
    cnt = np.minimum(ens.event_counts(), MAXREC)
    buf[np.arange(MAXREC)[None, :] >= cnt[:, None]] = np.zeros((), dtype=buf.dtype)
    return np.rec.array(buf), cnt


LAUNCHED = {}   # Inst -> (case, grid) confirmed by the profiler
WORST = {}      # throughput instantiation -> worst relative error against the oracle


def _setup(row):
    from sipnet_b200 import _abi as A, synth
    num, flags, block, layout, cols = row
    counts = LAYOUTS[layout]
    M = int(sum(counts))
    assert M % 16 == 0
    sites = [synth.synth_site(40 + i, 1, ["half-daily", "unequal"][i % 2], with_events=True) for i in range(len(counts))]
    rng = np.random.default_rng(M + len(counts))
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0, 1.5, s.nsteps))
    ms = np.repeat(np.arange(len(counts), dtype=np.int32), counts)
    P = synth.synth_params(M, stream=7 + len(counts))
    blocks = block_layout(counts, block)
    mixed = [b for b in blocks if b[2] > b[1]]
    # replayed members: the first member of the second 128-member block, and the head of the second site of a mixed
    # block (else the last member).  Their canopy leaves the exp guard in the first segment and is gone before the
    # second (the site's mortality events), so they are replayed in the first segment only.
    replay = [128, mixed[-1][0] + mixed[-1][1] if mixed else M - 1]
    for m in replay:
        P[A.P["laiInit"], m] = 2000.0
        P[A.P["leafTurnoverRate"], m] = 0.01
    starts = np.concatenate([[0], np.cumsum(counts)])
    sample = {0, M - 1, *replay}
    for s in range(len(counts)):
        sample |= {int(starts[s]), int(starts[s + 1] - 1)}
    for m0, c0, c in mixed:
        sample |= {m0, m0 + c0 - 1, m0 + c0, m0 + c - 1}
    sample |= set(rng.choice(M, 6, replace=False).tolist())
    return sites, ms, P, sorted(replay), np.array(sorted(sample)), mixed


def run_case(row, oracle):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from sipnet_b200 import _abi as A, api
    num, flags_name, block, layout, cols = row
    tag = case_id(row)
    flags = _flags(flags_name)
    sites, ms, P, replay, sample, mixed = _setup(row)
    M = P.shape[1]
    if cols == FULL:
        outputs, colidx, kw = A.OUT_FULL, list(range(A.NOUT)), {}
    elif cols:
        colidx = [A.O[c] for c in cols]
        outputs, kw = A.OUT_MOMENTS, dict(summary_cols=colidx)
    else:
        outputs, colidx, kw = 0, [], {}
    debug = num == "debug"
    outputs |= A.OUT_LOGLIK | A.OUT_EVENTS | (A.OUT_DEBUG if debug else 0)
    math = {"fast": A.MATH_FAST, "thr": A.MATH_THROUGHPUT, "debug": A.MATH_VALIDATION}[num]
    common = dict(outputs=outputs, block_threads=block, out_steps_capacity=SEGMENT, nee_sigma=0.5, max_event_records=MAXREC,
                  **kw)
    ncols = len(colidx)
    T = max(s.nsteps for s in sites)
    cuts = [0, SEGMENT, 2 * SEGMENT, T]
    got_s, dbg_s = [], []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with api.Ensemble(sites, P, ms, flags, math=math, **common) as ens, \
                api.Ensemble(sites, P, ms, flags, math=A.MATH_VALIDATION, **dict(common, outputs=outputs & ~A.OUT_DEBUG)) as ref:
            idx = torch.as_tensor(sample, device="cuda")
            for a, b in zip(cuts[:-1], cuts[1:]):
                ens.run(a, b)
                ref.run(a, b)
                ens.sync()
                ref.sync()
                if ncols:
                    g, w = _kept(ens, ncols, b - a, M), _kept(ref, ncols, b - a, M)
                    if num != "thr":
                        assert torch.equal(g.view(torch.int64), w.view(torch.int64)), f"{tag}: kept columns of [{a}, {b})"
                    got_s.append(g.index_select(2, idx).cpu().numpy())
                if debug:
                    dbg_s.append(ens.debug()[:, :, sample])
            res = {k: (getattr(ens, k)(), getattr(ref, k)()) for k in ("state", "status", "loglik", "loglik_n", "event_counts")}
            res["ring"] = (ens.ring(), ref.ring())
            res["recs"] = (_records(ens), _records(ref))
        torch.cuda.synchronize()

    # ---- which kernels ran
    launches = _kernel_launches(prof)
    kinds = {i for i, _ in launches}
    want = {EXACT_ROWS[f"validation-{block}"]}
    if num == "debug":
        want.add(EXACT_ROWS[f"debug-{block}"])
    else:
        want |= {expected_inst(row), EXACT_ROWS[f"replay-{block}"]}
    assert kinds == want, f"{tag}: launched {sorted(kinds)}, expected {sorted(want)}"
    for i, grid in launches:
        LAUNCHED.setdefault(i, (tag, grid))

    # ---- against the validation run
    (st, st_r), (status, status_r) = res["state"], res["status"]
    # ST_REPLAY is the optimistic kernels' alone, ST_BALANCE (the mass-balance check) the debug dump's alone
    assert np.array_equal(status & ~np.uint32(A.ST_REPLAY | A.ST_BALANCE), status_r), \
        f"{tag}: status {_status_diff(status & ~np.uint32(A.ST_REPLAY | A.ST_BALANCE), status_r)}"
    if num != "debug":
        assert np.flatnonzero(status & A.ST_REPLAY).tolist() == replay, f"{tag}: replayed members"
    assert np.array_equal(res["loglik_n"][0], res["loglik_n"][1]), f"{tag}: observation counts"
    assert np.array_equal(res["event_counts"][0], res["event_counts"][1]), f"{tag}: event counts"
    (rg, rg_r), ((rec, rec_n), (rec_r, _)) = res["ring"], res["recs"]
    recs_list = lambda m: list(rec[m][:rec_n[m]])  # noqa: E731
    if num != "thr":
        # the debug kernel also carries the yearly / total trackers and the harvest fractions
        rows = [k for k, n in enumerate(A.STATE_NAMES) if not (debug and n.startswith(("yearly", "totGpp", "totR", "totNpp", "harvest")))]
        assert np.array_equal(st[rows], st_r[rows], equal_nan=True), f"{tag}: state"
        assert np.array_equal(rg[0], rg_r[0]) and np.array_equal(rg[1], rg_r[1]), f"{tag}: ring"
        assert np.array_equal(res["loglik"][0], res["loglik"][1]), f"{tag}: log-likelihood"
        assert rec.tobytes() == rec_r.tobytes(), f"{tag}: event records"
    else:
        for f in ("step", "type", "variant", "nval"):
            assert np.array_equal(rec[f], rec_r[f]), f"{tag}: event record {f}"
        pools = [A.S[n] for n in ("plantWoodC", "plantLeafC", "soilC", "soilWater", "litterC", "snow", "coarseRootC",
                                  "fineRootC", "minN", "soilOrgN", "litterN", "plantStorageN")]
        x, y = st[pools], st_r[pools]
        floor = 1e-6 * np.maximum(np.nanmax(np.abs(y), axis=1), 1e-300)[:, None]
        err = np.abs(x - y) / np.maximum(np.maximum(np.abs(x), np.abs(y)), floor)
        assert np.nanmax(err) <= RTOL, f"{tag}: final pools {np.nanmax(err):.3e}"

    # ---- against the oracle on the sampled members
    kept = np.concatenate(got_s, axis=1) if ncols else None            # [ncols][T][k]
    dbg = np.concatenate(dbg_s, axis=1) if debug else None
    inst = expected_inst(row) if num != "debug" else EXACT_ROWS[f"debug-{block}"]
    worst = WORST.setdefault(inst, [0.0, 0.0]) if num == "thr" else None
    for j, m in enumerate(sample):
        site = sites[ms[m]]
        rc, done, o_out, o_dbg, o_all = oracle.run(flags, P[:, m], site, want_debug=debug, max_event_records=4096)
        o_recs = o_all[:MAXREC]                                          # the kernel keeps a member's first MAXREC
        if status[m] & A.ST_BAD_ALLOCATION:
            assert rc == 3, f"{tag}: member {m}"
            continue
        assert rc == 0 and done == site.nsteps, f"{tag}: member {m}"
        n = site.nsteps
        if ncols:
            assert np.isnan(kept[:, n:, j]).all(), f"{tag}: member {m} past its site's end"
        if num == "thr":
            if ncols:
                if m in replay:   # the first segment is the replay's: the ExactNum kernel, the oracle's bits
                    g, w = kept[:, :SEGMENT, j].T, o_out[:SEGMENT, colidx]
                    assert np.array_equal(g, w, equal_nan=True), f"{tag}: replayed member {m} vs the oracle {_first_diff(g, w, colidx)}"
                e, e_nl = check_throughput(kept[:, :n, j].T, o_out, recs_list(m), o_recs, f"{tag} m{m}", cols=colidx)
                worst[0], worst[1] = max(worst[0], e), max(worst[1], e_nl)
            assert bool(status[m] & A.ST_DIED) == any(r.type == 7 for r in o_all), f"{tag}: member {m} DIED"
            continue
        if ncols:
            g, w = kept[:, :n, j].T, o_out[:, colidx]
            assert np.array_equal(g, w, equal_nan=True), f"{tag}: member {m} vs the oracle {_first_diff(g, w, colidx)}"
        if debug:
            assert np.array_equal(dbg[:, :n, j].T, o_dbg, equal_nan=True), f"{tag}: member {m} debug rows vs the oracle"
        assert [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in recs_list(m)] == \
               [(r.step, r.type, r.variant, r.nval, tuple(r.val)) for r in o_recs], f"{tag}: member {m} event records"
    nblocks = len(block_layout(LAYOUTS[layout], block))
    print(f"{tag}: {M} members, {nblocks} blocks ({len(mixed)} mixed), {len(sample)} members vs the oracle, "
          f"replayed {replay}" + (f", worst {worst[0]:.2e} (nLeaching {worst[1]:.2e})" if worst else ""))


@pytest.mark.gpu
@pytest.mark.parametrize("row", MATRIX + EXTRA, ids=case_id)
def test_instantiation(oracle, row):
    run_case(row, oracle)


@pytest.mark.gpu
def test_zz_every_instantiation_was_launched():
    want = set(LEDGER.values())
    got = set(LAUNCHED) & want
    for i in sorted(WORST, key=str):
        print(f"throughput {i.policy}/{i.block}/{'full' if i.full else 'kept'}/{'dyn' if i.dyn else 'static'}/"
              f"{'mix' if i.mix else 'one'}: worst {WORST[i][0]:.3e}, nLeaching {WORST[i][1]:.3e}")
    dyn32 = sorted({tuple(g) for i, (_, g) in LAUNCHED.items() if i.dyn and i.block == 32 and g})
    print(f"instantiations launched and confirmed by name: {len(got)} of {len(want)}; persistent 32-member grids {dyn32}")
    missing = sorted(str(i) for i in want - got)
    assert not missing, missing
    assert set(LAUNCHED) <= want
