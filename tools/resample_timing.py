"""Device time of sipnet_gpu_resample (the per-site systematic particle filter, sip_resample.cu) on one GPU's share of
the C4 and C3 workloads, beside the forecast pass of the same handle.

    python tools/resample_timing.py [--calls 20] [--warmup 3] [--out FILE.json]

Shapes: C4 share = 1 site x 131 072 members (the bench workload per GPU, 10-year forecast); C3 share = 2 500 sites x
100 members (1-year forecast); synthetic forcing.  Log-weights are seeded normals with sd 2 passed by the caller, so
every call resamples every site (ess_fraction = inf) from the same weights.  Each call is timed with CUDA events on
the handle's stream; it includes the upload of the weights and the tables, the two host round trips of the per-site
records and the download of the ancestors and diagnostics.  The figure is the median of `--calls` calls after
`--warmup`.  Bytes are computed from the shapes: the record of a member (its parameter, state and ring rows and its
status) is read and written once by the pack and once by the unpack.  Prints one JSON line per shape with the GPU
name and power limit (read-only nvidia-smi query).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sipnet_b200 import _abi as A, api, synth  # noqa: E402
from tools.assimilate_timing import gpu_info  # noqa: E402

# The record layout of sip_resample.cu rs::record_words: device parameter rows (sip_types.cuh kNParamDev), state,
# both ring rows, status and event count, the counters (two per word), the event records, the ancestor's index.
# Keep this in step with rs::record_words; the handles timed here keep no event records (outputs = 0).
NPARAM_DEV = A.NPARAMS + 26
EVREC_WORDS = C.sizeof(A.EventRecord) // 8


def record_words(ring_slots: int, max_event_records: int) -> int:
    return NPARAM_DEV + A.NSTATE + 2 * ring_slots + 1 + (A.NCOUNTERS + 1) // 2 + EVREC_WORDS * max_event_records + 1


def measure(name, sites, P, ms, calls, warmup) -> dict:
    nsites = len(sites)
    with api.Ensemble(sites, P, ms, synth.SYNTH_FLAGS, outputs=0, math=A.MATH_FAST) as e:
        e.run()
        forecast_ms = e.last_run_ms()
        lw = np.random.default_rng(7).normal(0.0, 2.0, e.nmembers)
        u = np.random.default_rng(8).uniform(size=nsites)
        times = []
        launches = e.launch_count()
        for i in range(warmup + calls):
            e.timer_start()
            anc, diag = e.resample(u, math.inf, lw)
            ms_ = e.timer_stop_ms()
            if i >= warmup:
                times.append(ms_)
        launches = (e.launch_count() - launches) // (warmup + calls)
        M, ring = e.nmembers, e.ring_slots
    record = record_words(ring, 0) * 8
    med = float(np.median(times))
    return {"shape": name, "sites": nsites, "members": M, "ring_slots": ring, "record_bytes": record,
            "resample_ms_median": med, "resample_ms_min": float(np.min(times)), "resample_ms_max": float(np.max(times)),
            "calls": calls, "warmup": warmup, "launches_per_call": int(launches), "forecast_pass_ms": forecast_ms,
            "forecast_steps": int(max(s.nsteps for s in sites)),
            "resample_over_forecast": med / forecast_ms if forecast_ms > 0 else None,
            "record_traffic_bytes": 4 * record * M, "mean_distinct_ancestors_per_site": float(np.mean(diag[:, 3])),
            "note": "bytes computed from the shapes; pack + unpack each read and write every record once"}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    info = gpu_info()
    lines = []
    site = synth.synth_site(0, 10, "half-daily")
    M = 131072
    lines.append(measure("c4_share", [site], synth.synth_params(M, stream=1), np.zeros(M, np.int32), args.calls,
                         args.warmup))
    sites = [synth.synth_site(s, 1, "half-daily") for s in range(2500)]
    P, ms = synth.synth_params(250000, stream=1), np.repeat(np.arange(2500, dtype=np.int32), 100)
    lines.append(measure("c3_share", sites, P, ms, args.calls, args.warmup))
    for line in lines:
        line.update(info)
        print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
