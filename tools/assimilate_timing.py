"""Device time of sipnet_gpu_assimilate (the ensemble adjustment Kalman filter, sip_assim.cu) on one GPU's share of
the C4 and C3 workloads, beside the forecast pass of the same handle.

    python tools/assimilate_timing.py [--calls 20] [--warmup 3] [--inflation none,fixed,adaptive] [--out FILE.json]

--inflation times sipnet_gpu_assimilate_inflated as well, on the same handle after the same forecast: `fixed` inflates
every site by lambda = 1.5 (two more launches), `adaptive` also updates lambda (sd 0.5, bounds [1, 100]); every call
gets the same inputs.  `none` is the plain call.

Shapes: C4 share = 1 site x 131 072 members (the bench workload per GPU, 10-year forecast); C3 share = 2 500 sites x
100 members (1-year forecast); synthetic forcing without an event schedule (its harvest would leave the plant pools
at 0, and a skipped observation writes nothing).  12 pool rows, 4 observations per site: plantWoodC + coarseRootC +
fineRootC, soilC, soilWater, litterC.  Each call is timed with CUDA events on the handle's stream (it includes the upload of the
observations and the download of the diagnostics); the figure is the median of `--calls` calls after `--warmup`.
The analysis follows a forecast, so the 12 rows (12.6 MB at 131 072 members) are read from L2, as they would be in a
forecast-analysis cycle; the figure is an L2-resident one.  Bytes are computed from the shapes: every pass reads the
rows and the status word of every member, the updates write the rows.  Prints one JSON line per shape with the GPU
name and power limit (read-only nvidia-smi query).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sipnet_b200 import _abi as A, api, synth  # noqa: E402

NROWS, NOBS = 12, 4


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the timing stands without it, but say so
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def operator() -> np.ndarray:
    op = np.zeros((NOBS, NROWS))
    op[0, [A.S["plantWoodC"], A.S["coarseRootC"], A.S["fineRootC"]]] = 1.0
    op[1, A.S["soilC"]] = op[2, A.S["soilWater"]] = op[3, A.S["litterC"]] = 1.0
    return op


def observations(state, ms, nsites, op):
    """y° = prior site mean + 0.5 sd, r = (0.5 sd)^2."""
    y = op @ state[:NROWS]
    value = np.empty((nsites, NOBS))
    var = np.empty((nsites, NOBS))
    for k in range(NOBS):
        cnt = np.bincount(ms, minlength=nsites)
        mean = np.bincount(ms, y[k], minlength=nsites) / cnt
        sq = np.bincount(ms, (y[k] - mean[ms]) ** 2, minlength=nsites) / cnt
        sd = np.maximum(np.sqrt(sq), 1e-6)
        value[:, k] = mean + 0.5 * sd
        var[:, k] = (0.5 * sd) ** 2
    return value, var


MODES = ("none", "fixed", "adaptive")


def analysis(e, mode, rows, op, value, var):
    """One call of the mode, as a function of nothing."""
    n = e.nsites
    if mode == "none":
        return lambda: e.assimilate(rows, op, value, var)
    sd = np.full(n, 0.5) if mode == "adaptive" else None
    return lambda: e.assimilate_inflated(rows, op, value, var, np.full(n, 1.5), sd)


def measure(name, sites, P, ms, calls, warmup, modes) -> list:
    nsites = len(sites)
    lines = []
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=0, math=A.MATH_FAST) as e:
        e.run()
        forecast_ms = e.last_run_ms()
        op = operator()
        value, var = observations(e.state(), ms, nsites, op)
        rows = list(range(NROWS))
        M = e.nmembers
        for mode in modes:
            call = analysis(e, mode, rows, op, value, var)
            times = []
            launches = e.launch_count()
            for i in range(warmup + calls):
                e.timer_start()
                call()
                ms_ = e.timer_stop_ms()
                if i >= warmup:
                    times.append(ms_)
            launches = (e.launch_count() - launches) // (warmup + calls)
            passes = 2 * NOBS + 1 + (1 if mode != "none" else 0)     # members passes; the inflation adds one
            per_member_read = NROWS * 8 + 4
            read = passes * per_member_read * M
            written = (NOBS + (1 if mode != "none" else 0)) * NROWS * 8 * M
            med = float(np.median(times))
            lines.append({"shape": name, "inflation": mode, "sites": nsites, "members": M, "rows": NROWS,
                          "observations": NOBS, "assimilate_ms_median": med, "assimilate_ms_min": float(np.min(times)),
                          "assimilate_ms_max": float(np.max(times)), "calls": calls, "warmup": warmup,
                          "launches_per_call": int(launches), "forecast_pass_ms": forecast_ms,
                          "forecast_steps": int(max(s.nsteps for s in sites)),
                          "analysis_over_forecast": med / forecast_ms if forecast_ms > 0 else None,
                          "rows_bytes": NROWS * 8 * M, "bytes_read": read, "bytes_written": written,
                          "note": "rows L2-resident after the forecast; bytes computed from the shapes"})
    return lines


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--inflation", default="none",
                    help="comma-separated modes to time, each of none, fixed, adaptive (default: none)")
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    modes = args.inflation.split(",")
    if not modes or any(m not in MODES for m in modes):
        ap.error(f"--inflation takes a comma-separated list of {', '.join(MODES)}")
    info = gpu_info()
    lines = []
    site = synth.synth_site(0, 10, "half-daily")
    M = 131072
    lines += measure("c4_share", [site], synth.synth_params(M, stream=1), np.zeros(M, np.int32), args.calls,
                     args.warmup, modes)
    sites = [synth.synth_site(s, 1, "half-daily") for s in range(2500)]
    P, ms = synth.synth_params(250000, stream=1), np.repeat(np.arange(2500, dtype=np.int32), 100)
    lines += measure("c3_share", sites, P, ms, args.calls, args.warmup, modes)
    for line in lines:
        line.update(info)
        print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
