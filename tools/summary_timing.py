#!/usr/bin/env python
"""Device time of the cross-rank team summaries (sip_gsum.cu, driven by sip_comm.cu) on one GPU's C4 share, and
where the select's rows end.

    python tools/summary_timing.py [--libs a.so,b.so] [--rounds 3] [--passes 20] [--members 131072] [--years 10]
                                   [--no-profile] [--no-rows] [--out DIR]

Workload: the bench's C4 share (1 site x 131 072 members x 10 years of half-daily steps, NEE and GPP kept, mean /
variance / quantiles 0.05, 0.5, 0.95) through api.Ensemble as a team of one; the forecast runs once, then
team_summaries() is timed alone.  Each pass reads 15.3 GB of kept values, far more than the 126 MB L2.

  * `team_summaries()`: CUDA events around each of `--passes` calls (after one warm-up call); median and spread.  With
    several `--libs` the builds are alternated `--rounds` times, one child process per (round, build), so a before
    and an after are measured in one invocation under the same conditions.
  * per kernel: torch.profiler (CUDA activities) in a child of its own per build, over 5 calls; launches are named
    by their place in a call (pass0, level1, level2, level3+, emit, finish).
  * rows (once, with the first build): how far the exact select has to go on this data, from the kept values
    themselves (sorted on the device): the level whose resolve decides each row, and the population of each level
    pass's filter -- the slots in play plus the bins of statistics waiting for the emit -- which decides whether the
    pass compacts the row's candidates (<= kGsListCap keys).  The tie shortcut (a slot of > 1 024 equal keys) is
    modelled; nothing here reads library internals.

Every child prints one JSON line; they carry the GPU name and power limit (read-only nvidia-smi query) and a digest
of the results (quantiles, mean, variance), which must agree between builds that compute the same thing.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QUANTILES = [0.05, 0.5, 0.95]
LIST_CAP = 4096  # kGsListCap (sip_gsum.cuh)
EMIT = 16        # kGsEmit


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the timing stands without it, but say so
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def make_ensemble(args):
    sys.path.insert(0, ROOT)
    from sipnet_b200 import _abi as A, api, synth
    site = synth.synth_site(0, args.years, "half-daily")
    params = synth.synth_params(args.members, stream=100)
    ens = api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), math=A.MATH_FAST, device=0,
                       outputs=A.OUT_MOMENTS | A.OUT_QUANTILES, summary_cols=[A.O["nee"], A.O["gpp"]], quantiles=QUANTILES)
    ens.join_team(1, 0)
    ens.run(0, site.nsteps)
    ens.sync()
    return ens, site.nsteps


def digest(ens) -> str:
    h = hashlib.sha1()
    for a in (ens.quantiles(), ens.mean(), ens.variance()):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def child_events(args):
    ens, _ = make_ensemble(args)
    ens.team_summaries()
    ms = []
    for _ in range(args.passes):
        ens.sync()
        ens.timer_start()
        ens.team_summaries()
        ms.append(ens.timer_stop_ms())
    ms = np.array(ms)
    out = {"what": "team_summaries", "lib": os.environ.get("SIPNET_GPU_LIB", "default"), "passes": len(ms),
           "median_ms": round(float(np.median(ms)), 3), "mean_ms": round(float(ms.mean()), 3),
           "min_ms": round(float(ms.min()), 3), "max_ms": round(float(ms.max()), 3),
           "select_levels": ens.team_last_levels(), "digest": digest(ens), **gpu_info()}
    ens.close()
    print(json.dumps(out), flush=True)


def child_profile(args):
    from torch.profiler import ProfilerActivity, profile
    ens, _ = make_ensemble(args)
    ens.team_summaries()
    ens.sync()
    calls = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            ens.team_summaries()
        ens.sync()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    kern = sorted((e for e in trace.get("traceEvents", []) if e.get("cat") == "kernel" and "gs::" in e.get("name", "")),
                  key=lambda e: e["ts"])
    ms, level = {}, 0
    for e in kern:
        name = e["name"]
        if "gs_pass0" in name:
            tag, level = "pass0", 0
        elif "gs_level" in name:
            level += 1
            tag = f"level{level}" if level < 3 else "level3+"
        elif "gs_emit" in name:
            tag = "emit"
        elif "gs_finish" in name:
            tag = "finish"
        else:
            tag = "other"
        ms[tag] = ms.get(tag, 0.0) + e["dur"] * 1e-3 / calls
    ms = {k: round(v, 3) for k, v in ms.items()}
    ens.close()
    print(json.dumps({"what": "kernels_ms_per_call", "lib": os.environ.get("SIPNET_GPU_LIB", "default"), **ms,
                      "sum": round(sum(ms.values()), 3), **gpu_info()}), flush=True)


def row_stats(K, n, probs):
    """K [R][M] int64 keys (signed order, non-finite = int64 max, sorted), n [R] finite counts -> per row and order
    statistic: pop[R][S][8] (keys sharing its prefix after each level's bits), pre[R][S][8], eq[R][S] (keys equal to it)."""
    import torch
    ks = []
    for p in probs:
        pos = p * (n.double() - 1.0)
        lo = torch.floor(pos)
        hi = torch.where(pos - lo > 0, lo + 1, lo)
        ks += [lo, hi]
    ks = torch.stack(ks, 1).clamp(min=0).long()                     # [R][S]
    ks = torch.minimum(ks, (n - 1).clamp(min=0)[:, None])
    key = K.gather(1, ks)                                            # [R][S]
    pops, pres = [], []
    for level in range(8):
        bits = 11 + 8 * level if level < 7 else 64
        P = K >> (64 - bits) if bits < 64 else K
        pre = key >> (64 - bits) if bits < 64 else key
        right = torch.minimum(torch.searchsorted(P, pre, right=True), n[:, None])
        pops.append(right - torch.searchsorted(P, pre))
        pres.append(pre)
    eq = torch.minimum(torch.searchsorted(K, key, right=True), n[:, None]) - torch.searchsorted(K, key)
    return torch.stack(pops, 2), torch.stack(pres, 2), eq


def decide(pop, pre, eq):
    """One row (numpy, [S][8] / [S]): the level whose resolve makes each statistic final (pop <= kGsEmit, all 64 bits,
    or the tie shortcut: the level-l pass, l >= 2, watches slots of > 1 024 keys, and a slot whose keys are all equal
    makes its statistics final before the resolve of level l), whether it then needs the emit, and the filter
    population of every level pass."""
    S = pop.shape[0]
    fin, emitted = [], []
    for s in range(S):
        f, e = 7, False
        for level in range(8):
            if level >= 2 and pop[s][level - 1] > 1024 and pop[s][level - 1] == eq[s]:
                f, e = level, False
                break
            if pop[s][level] <= EMIT:
                f, e = level, level < 7
                break
        fin.append(f)
        emitted.append(e)
    done = max(fin)
    filt = {}
    for level in range(1, done + 1):  # the level-l pass runs while some statistic is open after resolve l - 1
        seen, tot = set(), 0
        for s in range(S):
            if fin[s] > level - 1:
                k = ("slot", int(pre[s][level - 1]))
                p = int(pop[s][level - 1])
            elif emitted[s]:
                k = ("emit", fin[s], int(pre[s][fin[s]]))
                p = int(pop[s][fin[s]])
            else:
                continue
            if k not in seen:
                seen.add(k)
                tot += p
        filt[level] = tot
    return done, filt


def child_rows(args):
    import torch
    ens, T = make_ensemble(args)
    sys.path.insert(0, ROOT)
    from sipnet_b200 import _abi as A
    from sipnet_b200.distributed import DeviceArray
    M = args.members
    ld = (M + 15) // 16 * 16
    cols = DeviceArray(ens.device_ptr(A.GATHER_FULL), (2, T, M), (T * ld, ld, 1)).tensor(0)
    done_hist, filt_by_level, compact_at = {}, {}, {}
    imax = torch.iinfo(torch.int64).max
    for c in range(2):
        for t0 in range(0, T, 256):
            x = cols[c, t0:t0 + 256]
            b = x.view(torch.int64)
            fin = torch.isfinite(x)
            key = torch.where(b < 0, b ^ torch.tensor(imax, device=b.device), b)   # signed-order key
            key = torch.where(fin, key, torch.full_like(key, imax))
            K, _ = torch.sort(key, dim=1)
            n = fin.sum(1)
            const = (K[:, 0] == K.gather(1, (n - 1).clamp(min=0)[:, None])[:, 0]) & (n > 0)
            pop, pre, eq = (t.cpu().numpy() for t in row_stats(K, n, QUANTILES))
            nn, cc = n.cpu().numpy(), const.cpu().numpy()
            for r in range(K.shape[0]):
                if nn[r] == 0 or cc[r]:
                    tag = "empty" if nn[r] == 0 else "constant"
                    done_hist[tag] = done_hist.get(tag, 0) + 1
                    continue
                done, filt = decide(pop[r], pre[r], eq[r])
                done_hist[f"after_level{done}"] = done_hist.get(f"after_level{done}", 0) + 1
                first = None
                for level, f in filt.items():
                    filt_by_level.setdefault(level, []).append(f)
                    if first is None and f <= LIST_CAP:
                        first = level
                compact_at[str(first or "never")] = compact_at.get(str(first or "never"), 0) + 1
    ens.close()
    out = {"what": "rows", "rows": 2 * T, "decided": dict(sorted(done_hist.items())),
           "compacted_at_level_pass": dict(sorted(compact_at.items())), "filter_population": {}, **gpu_info()}
    for level, f in sorted(filt_by_level.items()):
        f = np.array(f)
        out["filter_population"][f"level{level}_pass"] = {
            "rows": int(f.size), "p10": int(np.percentile(f, 10)), "median": int(np.median(f)),
            "p90": int(np.percentile(f, 90)), "max": int(f.max()), f"le_{LIST_CAP}": int((f <= LIST_CAP).sum())}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", default="", help="comma-separated libsipnet_gpu.so builds to alternate (default: in-tree)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--members", type=int, default=131072)
    ap.add_argument("--years", type=int, default=10)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-rows", action="store_true")
    ap.add_argument("--out", default="", help="also append every JSON line to DIR/summary_timing.jsonl")
    ap.add_argument("--mode", default="", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.mode:
        return {"events": child_events, "profile": child_profile, "rows": child_rows}[args.mode](args)
    libs = [os.path.abspath(x) for x in args.libs.split(",") if x] or [""]
    lines = []

    def run(mode, lib):
        env = dict(os.environ)
        if lib:
            env["SIPNET_GPU_LIB"] = lib
        cmd = [sys.executable, os.path.abspath(__file__), "--mode", mode, "--members", str(args.members),
               "--years", str(args.years), "--passes", str(args.passes)]
        out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, text=True)
        sys.stdout.write(out.stdout)
        sys.stdout.flush()
        if out.returncode != 0:
            raise SystemExit(f"summary_timing: child {mode} {lib or 'default'} exited {out.returncode}")
        lines.extend(x for x in out.stdout.splitlines() if x.startswith("{"))

    for _ in range(args.rounds):
        for lib in libs:
            run("events", lib)
    if not args.no_profile:
        for lib in libs:
            run("profile", lib)
    if not args.no_rows:
        run("rows", libs[0])
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "summary_timing.jsonl"), "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
