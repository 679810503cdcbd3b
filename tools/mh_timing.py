"""Device time of sipnet_gpu_mh_move (the tempered Metropolis-Hastings move: sip_jitter.cu proposes, sip_resample.cu
snapshots and decides) on one GPU's share of the C4 and C3 workloads, beside a plain reset() + run(0, s) of the same
handle.

    python tools/mh_timing.py [--rows 4] [--calls 10] [--warmup 2] [--out FILE.json]

Shapes: C4 share = 1 site x 131 072 members over its 10-year window (7 306 steps); C3 share = 2 500 sites x 100 members
over a 1-year window; synthetic forcing and NEE observations, SIPNET_GPU_OUT_LOGLIK only.  The move takes `--rows` rows
(IDENTITY and LOG rows, improper FLAT priors) with scale h = 0.5 and tau = 1 at every site, the handle's log-likelihood
as the current one, and fresh seeded normals and log-uniforms per call (drawn outside the timed region).  Each call is
timed with CUDA events on the handle's stream and includes the uploads and the download of the diagnostics; the
reset + run pair is timed the same way, alternating with the moves.  The figures are medians after `--warmup`.
Prints one JSON line per shape with the GPU name and power limit (read-only nvidia-smi query).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sipnet_b200 import _abi as A, api, synth  # noqa: E402
from tools.assimilate_timing import gpu_info  # noqa: E402

ROWS = [("psnTOpt", A.TF_IDENTITY), ("aMax", A.TF_IDENTITY), ("halfSatPar", A.TF_LOG), ("vegRespQ10", A.TF_LOG),
        ("soilWHC", A.TF_LOG), ("baseVegResp", A.TF_LOG), ("wueConst", A.TF_LOG), ("leafCSpWt", A.TF_LOG)]


def with_obs(sites, seed=3):
    rng = np.random.default_rng(seed)
    for s in sites:
        s.nee_obs = np.where(rng.uniform(size=s.nsteps) < 0.3, np.nan, rng.normal(0.0, 1.5, s.nsteps))
    return sites


def measure(name, sites, P, ms, k, calls, warmup) -> dict:
    nsites = len(sites)
    rows = [A.P[r] for r, _ in ROWS[:k]]
    tf = [t for _, t in ROWS[:k]]
    lo = [-np.inf if t == A.TF_IDENTITY else 0.0 for t in tf]
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=A.OUT_LOGLIK, math=A.MATH_FAST, nee_sigma=2.0) as e:
        s = max(x.nsteps for x in sites)
        e.run(0, s)
        rng = np.random.default_rng(7)
        M = e.nmembers
        move_ms, run_ms, acc = [], [], []
        launches = 0
        for i in range(warmup + calls):
            cur = e.loglik()
            z, lu = rng.standard_normal((k, M)), np.log(rng.uniform(size=M))
            c0 = e.launch_count()
            e.timer_start()
            diag = e.mh_move(rows, tf, [A.PRIOR_FLAT] * k, lo, [np.inf] * k, np.full(nsites, 0.5), np.ones(nsites), cur,
                             z, lu)
            t_move = e.timer_stop_ms()
            launches = e.launch_count() - c0
            e.timer_start()
            e.reset()
            e.run(0, s)
            t_run = e.timer_stop_ms()
            if i >= warmup:
                move_ms.append(t_move)
                run_ms.append(t_run)
                acc.append(float(diag[:, 3].sum() / max(diag[:, 0].sum(), 1)))
    med, base = float(np.median(move_ms)), float(np.median(run_ms))
    return {"shape": name, "sites": nsites, "members": M, "steps": s, "rows": k, "mh_move_ms_median": med,
            "mh_move_ms_min": float(np.min(move_ms)), "mh_move_ms_max": float(np.max(move_ms)),
            "reset_run_ms_median": base, "reset_run_ms_min": float(np.min(run_ms)),
            "reset_run_ms_max": float(np.max(run_ms)), "move_minus_run_ms": med - base,
            "move_over_run": med / base if base > 0 else None, "calls": calls, "warmup": warmup,
            "launches_per_call": int(launches), "accepted_fraction_median": float(np.median(acc)),
            "upload_bytes": 8 * M * (k + 2) + 16 * nsites}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=4)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    if not 1 <= args.rows <= len(ROWS):
        ap.error(f"--rows must be 1..{len(ROWS)}")
    info = gpu_info()
    lines = []
    M = 131072
    lines.append(measure("c4_share", with_obs([synth.synth_site(0, 10, "half-daily")]), synth.synth_params(M, stream=1),
                         np.zeros(M, np.int32), args.rows, args.calls, args.warmup))
    sites = with_obs([synth.synth_site(s, 1, "half-daily") for s in range(2500)])
    P, ms = synth.synth_params(250000, stream=1), np.repeat(np.arange(2500, dtype=np.int32), 100)
    lines.append(measure("c3_share", sites, P, ms, args.rows, args.calls, args.warmup))
    for line in lines:
        line.update(info)
        print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
