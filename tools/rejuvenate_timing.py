"""Device time of sipnet_gpu_rejuvenate (the Liu-West parameter move, sip_jitter.cu) on one GPU's share of the C4 and
C3 workloads, beside the forecast pass of the same handle.

    python tools/rejuvenate_timing.py [--rows 8] [--calls 20] [--warmup 3] [--out FILE.json]

Shapes: C4 share = 1 site x 131 072 members (the bench workload per GPU, 10-year forecast); C3 share = 2 500 sites x
100 members (1-year forecast); synthetic forcing.  The move takes `--rows` rows (four IDENTITY, then LOG rows) with
shrink a = 0.95 at every site and fresh seeded normals per call (drawn outside the timed region).  Each call is timed
with CUDA events on the handle's stream; it includes the upload of z (rows x members doubles) and of shrink and the
download of the diagnostics.  The figure is the median of `--calls` calls after `--warmup`.  Bytes are computed from the shapes: the two moment passes and the
proposal pass each read the listed rows, the proposal pass also reads z and writes the listed and dependent rows.
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

ROWS = [("psnTOpt", A.TF_IDENTITY), ("psnTMin", A.TF_IDENTITY), ("aMax", A.TF_IDENTITY),
        ("frozenSoilThreshold", A.TF_IDENTITY), ("halfSatPar", A.TF_LOG), ("soilWHC", A.TF_LOG),
        ("baseVegResp", A.TF_LOG), ("vegRespQ10", A.TF_LOG), ("wueConst", A.TF_LOG), ("leafCSpWt", A.TF_LOG),
        ("baseSoilResp", A.TF_LOG), ("soilRespQ10", A.TF_LOG), ("fineRootQ10", A.TF_LOG), ("coarseRootQ10", A.TF_LOG),
        ("baseFineRootResp", A.TF_LOG), ("baseCoarseRootResp", A.TF_LOG)]
DEPENDENT_ROWS = 2 + 2 + 26          # coarseRootAllocation, psnTMax, the two clamps, the internal rows


def measure(name, sites, P, ms, k, calls, warmup) -> dict:
    nsites = len(sites)
    rows = [A.P[r] for r, _ in ROWS[:k]]
    tf = [t for _, t in ROWS[:k]]
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=0, math=A.MATH_FAST) as e:
        e.run()
        forecast_ms = e.last_run_ms()
        rng = np.random.default_rng(7)
        shrink = np.full(nsites, 0.95)
        times = []
        launches = e.launch_count()
        for i in range(warmup + calls):
            z = rng.standard_normal((k, e.nmembers))   # fresh normals per call, as a filter draws them
            e.timer_start()
            diag = e.rejuvenate(rows, tf, shrink, z)
            ms_ = e.timer_stop_ms()
            if i >= warmup:
                times.append(ms_)
        launches = (e.launch_count() - launches) // (warmup + calls)
        M = e.nmembers
    med = float(np.median(times))
    return {"shape": name, "sites": nsites, "members": M, "rows": k, "rejuvenate_ms_median": med,
            "rejuvenate_ms_min": float(np.min(times)), "rejuvenate_ms_max": float(np.max(times)), "calls": calls,
            "warmup": warmup, "launches_per_call": int(launches), "forecast_pass_ms": forecast_ms,
            "forecast_steps": int(max(s.nsteps for s in sites)),
            "rejuvenate_over_forecast": med / forecast_ms if forecast_ms > 0 else None,
            "z_upload_bytes": 8 * k * M, "read_bytes": 8 * M * (4 * k + 1), "write_bytes": 8 * M * (k + DEPENDENT_ROWS),
            "moved": int(diag[:, 2].sum()), "kept": int(diag[:, 3].sum()),
            "note": "bytes computed from the shapes (z upload: host to device; rows: status and the listed rows read by "
                    "three passes, z once; listed and dependent rows written once)"}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=8)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    if not 1 <= args.rows <= len(ROWS):
        ap.error(f"--rows must be 1..{len(ROWS)}")
    info = gpu_info()
    lines = []
    site = synth.synth_site(0, 10, "half-daily")
    M = 131072
    lines.append(measure("c4_share", [site], synth.synth_params(M, stream=1), np.zeros(M, np.int32), args.rows,
                         args.calls, args.warmup))
    sites = [synth.synth_site(s, 1, "half-daily") for s in range(2500)]
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
