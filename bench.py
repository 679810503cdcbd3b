#!/usr/bin/env python
"""bench.py -- ensemble member-timesteps/sec of the SIPNET integration loop on 1..8 B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU)

Workload (BASELINE.json configs[3], "C4", the north-star target; weak scaling): ONE synthetic site, 10 years of
half-daily forcing (T = 7306), flags litter+anaerobic+nitrogen, a parameter ensemble of 131072 members PER GPU
(8 GPUs = the 1M-member target), reduced on the device to the ensemble mean, variance and exact 5/50/95 %
quantiles of NEE and GPP per step -- over the members of ALL ranks.  One "step" = one pass of the hot path over
that batch: state reset, all 7306 model steps of every member (reference loop sipnet.c:1969-1982), and the team
summaries (sipnet_gpu_comm_summaries: NCCL all-reduce of key histograms, no member value leaves its GPU).

value   : member-timesteps/s over all ranks, inputs resident in HBM, CUDA events on the library's stream (the NCCL
          exchange runs on that stream), max over ranks.
e2e     : the same pass through the C ABI with HOST buffers: parameter upload from pinned host memory + run +
          summaries + gather of the summaries into host memory, inside the timed region.
roofline: dominant kernel = the fused step kernel (sip::k1::run_kernel), FP64-issue bound.  Two bases side by side:
          `frac` = SURVEY 8(d)'s algorithmic 3200 flop/member-step against the FP64 FMA peak measured live;
          `frac_executed` = FP64-pipe instructions the kernel actually executes per member-step (from this round's
          ncu capture, file named in the line) x member-steps/s against the measured FP64 issue rate -- the number
          ncu reports as sm__inst_executed_pipe_fp64.
extras  : `c5` (32768 draws per GPU scored by NEE log-likelihood, NCCL all-gather through the C ABI) at every N;
          `c2` (BASELINE.json configs[1]: 4096 members, full per-step output, device + host-delivered) at N = 1.
cpu_baseline / --impl reference: the unmodified reference (oracle/_ref) on the host cores, a bounded sample of the
          same ensemble, one process per core.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ensemble member-timesteps/sec"
UNIT = "member-timesteps/s"
FLOP_PER_MEMBER_STEP = 3200.0   # SURVEY 8d / BASELINE.md 4: ~630 FP64 ops + ~19 libm calls (an estimate; kept for continuity)
FP64_INST_PER_MEMBER_STEP_FALLBACK = 800.0   # executed FP64-pipe instructions per member-step if the facts file is missing
MEMBERS_PER_GPU = 131072        # C4: 1M members / 8 GPUs
C5_DRAWS_PER_GPU = 32768        # C5: 256k draws / 8 GPUs
QUANTILES = [0.05, 0.5, 0.95]
KERNEL_FACTS = os.path.join(ROOT, "profiles", "r02_kernel_facts.json")   # written from this round's ncu capture


def workload_name(members_per_gpu: int, years: int) -> str:
    return (f"C4 (weak scaling): 1 site x {members_per_gpu} members per GPU x {years} yr half-daily, "
            "litter+anaerobic+nitrogen, on-device ensemble mean/variance + exact 5/50/95% quantiles of NEE and GPP "
            "over all ranks")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members", type=int, default=MEMBERS_PER_GPU, help="members per GPU")
    ap.add_argument("--years", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the c5 / c2 sections and the oracle spot check")
    ap.add_argument("--workload", default="c4", choices=["c4", "c3"],
                    help="c4 = the bench workload; c3 = BASELINE.json configs[2] as one extra line (10k sites x 100 members)")
    ap.add_argument("--sites", type=int, default=0, help="c3: sites per GPU (default 10000 / n_gpus)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="c4 workload of --impl ours only: rank 0 writes what the last timed pass returned as "
                         "DIR/<name>.npy (float64, under 64 MB in all), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c4"):
        ap.error("--dump-outputs applies to the c4 workload of --impl ours only")
    return args


# ---------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------- CPU arms
def _ref_worker(args):
    """One process = a slice of members through the UNMODIFIED reference (oracle/_ref shim)."""
    flags, params, site_npz, idx, text_dir = args
    from oracle.pyoracle import RefShim
    from sipnet_b200 import _abi as A
    from sipnet_b200.api import SiteData
    shim = RefShim()
    site = SiteData(site_npz["year"], site_npz["day"], {k: site_npz[k] for k in A.CLIM_COLS})
    t0 = time.perf_counter()
    steps = 0
    for m in idx:
        main_out = os.path.join(text_dir, f"sipnet.out.{os.getpid()}.{m}") if text_dir else None
        rc, done, _, _ = shim.run(flags, params[:, m], site, want_debug=False, main_out=main_out)
        steps += done
    return steps, time.perf_counter() - t0


class CpuReference:
    """The reference CPU implementation on all host cores (one process per core, each running members through
    oracle/_ref -- the unmodified reference -- or, if that build is absent, the oracle port on threads)."""

    def __init__(self, site, params, flags, cores: int):
        from oracle import pyoracle
        from sipnet_b200 import _abi as A
        self.site = site
        self.params = params
        self.flags = flags
        self.cores = cores
        self.kind = "reference" if pyoracle.have_ref() else "port"
        self.pool = None
        if self.kind == "reference":
            self.site_npz = dict(year=self.site.year, day=self.site.day, **{k: self.site.clim[k] for k in A.CLIM_COLS})
            self.pool = mp.get_context("spawn").Pool(cores)
            # warm: import, load the .so, page in
            self.pool.map(_ref_worker, [(flags, params, self.site_npz, [i % params.shape[1]], None) for i in range(cores)])
        else:
            self.oracle = pyoracle.Oracle()

    def sample(self, members_per_core: int, text_dir: str | None = None):
        """-> (member-steps/s, description)"""
        from sipnet_b200 import _abi as A
        site, cores = self.site, self.cores
        nm = min(self.params.shape[1], members_per_core * cores)
        if self.kind == "reference":
            chunks = [list(range(i, nm, cores)) for i in range(cores)]
            t0 = time.perf_counter()
            res = self.pool.map(_ref_worker, [(self.flags, self.params, self.site_npz, c, text_dir) for c in chunks])
            wall = time.perf_counter() - t0
            how = "every member writes its sipnet.out text file (outputState, sipnet.c:453-473)" if text_dir else "no text output"
            return sum(r[0] for r in res) / wall, (f"{nm} members x {site.nsteps} steps, one process per core, "
                                                    f"unmodified reference (oracle/_ref), {how}")
        from sipnet_b200.api import flags_array
        out = np.zeros((nm, A.NOUT))
        fl = flags_array(self.flags)
        clim = (C.POINTER(C.c_double) * 11)(*[site.clim[k].ctypes.data_as(C.POINTER(C.c_double)) for k in A.CLIM_COLS])
        arr, nev = site.event_array()
        P = np.ascontiguousarray(self.params[:, :nm])
        lib = self.oracle.lib
        lib.sipnet_oracle_run_ensemble.restype = C.c_int
        t0 = time.perf_counter()
        lib.sipnet_oracle_run_ensemble(
            fl.ctypes.data_as(C.POINTER(C.c_int32)), P.ctypes.data_as(C.POINTER(C.c_double)), C.c_int64(nm),
            C.c_int64(nm), C.c_int64(site.nsteps), site.year.ctypes.data_as(C.POINTER(C.c_int32)),
            site.day.ctypes.data_as(C.POINTER(C.c_int32)), clim, C.c_int64(nev), arr, C.c_int(cores),
            out.ctypes.data_as(C.POINTER(C.c_double)))
        wall = time.perf_counter() - t0
        return nm * site.nsteps / wall, f"{nm} members x {site.nsteps} steps, {cores} threads, oracle port"

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def bench_config(args, T: int) -> dict:
    """The `config` object -- identical in both arms."""
    return {"workload": workload_name(args.members, args.years), "members_per_gpu": args.members, "model_steps": T,
            "summaries": "mean, variance, quantiles 0.05/0.5/0.95 of NEE and GPP per step",
            "l2": "every pass writes 15.3 GB of summary columns per GPU (>> 126 MB L2); inputs are re-read from HBM"}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation on the host cores, same config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sipnet_b200 import synth
    site = synth.synth_site(0, args.years, "half-daily")
    cores = os.cpu_count() or 1
    per_core = 48                                  # bounded sample per step: ~1-2 s of work per core
    params = synth.synth_params(min(args.members, per_core * cores), stream=100)   # the first members of rank 0's ensemble
    flags = dict(synth.SYNTH_FLAGS)
    cpu = CpuReference(site, params, flags, cores)
    vals = []
    sample = ""
    for i in range(args.warmup + args.steps):
        v, sample = cpu.sample(per_core)
        if i >= args.warmup:
            vals.append(v)
    cpu.close()
    value = float(np.mean(vals))
    T = site.nsteps
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * (params.shape[1] * T) / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args, T),
        "note": "each step is a bounded sample of the workload's members on the host cores; the reference has no "
                "ensemble code, so the summaries are not part of this arm",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": cpu.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------- GPU arm
class Dist:
    """torch.distributed is plumbing here: rendezvous, barrier, max over ranks, broadcast of the NCCL id that the
    library's own communicator (sipnet_gpu_comm_init_rank) is built from."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.affinity = self._bind_to_gpu_node()
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def _bind_to_gpu_node(self) -> str:
        """Run this rank (and first-touch its pinned buffers) on the CPU cores NVML lists as local to its GPU, so that
        eight ranks' device<->host copies do not all cross one socket."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.local)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                return f"nvml: {len(cpus)} cores local to GPU {self.local}"
        except Exception as exc:  # no NVML / not permitted: stay where the launcher put us
            return f"unchanged ({type(exc).__name__})"
        return "unchanged"

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def comm_id(self, api) -> bytes | None:
        if self.world == 1:
            return None
        t = self.torch.zeros(128, dtype=self.torch.uint8, device="cuda")
        if self.rank == 0:
            t.copy_(self.torch.frombuffer(bytearray(api.unique_comm_id()), dtype=self.torch.uint8))
        self.dist.broadcast(t, src=0)
        return bytes(t.cpu().numpy().tobytes())

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def pinned(lib, nbytes: int) -> int:
    p = lib.sipnet_gpu_host_alloc(nbytes)
    if not p:
        raise SystemExit("bench.py: pinned host allocation failed")
    return p


def section_throughput_policy(args, D: Dist, site):
    """The same C4 pass under the tolerance-budgeted numerics (SIPNET_GPU_MATH_THROUGHPUT: reciprocal-multiply
    division, -fmad=true; within 1e-10 of the reference, not bit-identical) -- reported beside the headline."""
    from sipnet_b200 import _abi as A, api, synth
    M, T = args.members, site.nsteps
    params = synth.synth_params(M, stream=100 + D.rank)
    ens = api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), math=A.MATH_THROUGHPUT, device=D.local,
                       outputs=A.OUT_MOMENTS | A.OUT_QUANTILES, summary_cols=[A.O["nee"], A.O["gpp"]], quantiles=QUANTILES)
    ens.join_team(D.world, D.rank, D.comm_id(api))

    def one_pass():
        ens.reset()
        ens.run(0, T)
        ens.team_summaries()

    one_pass()
    ens.sync()
    D.barrier()
    n = 3
    ens.timer_start()
    kern = []
    for _ in range(n):
        one_pass()
        kern.append(ens.last_run_ms())
    ms = D.max(ens.timer_stop_ms() / n)
    kern_ms = D.max(float(np.mean(kern)))
    D.barrier()
    ens.close()
    return {"math": "throughput (SIPNET_GPU_MATH_THROUGHPUT): division = multiplication by the refined reciprocal, model "
                    "arithmetic with -fmad=true; 1e-10 relative of the reference on every test ensemble "
                    "(tests/test_gpu_throughput.py), not bit-identical",
            "value": D.world * M * T / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "step_kernel_ms": kern_ms,
            "step_kernel_member_steps_per_s_per_gpu": M * T / (kern_ms * 1e-3)}


def section_c4(args, D: Dist, lib, site, fp64_peak_tflops):
    """The headline: C4 share per rank + team summaries over all ranks."""
    from sipnet_b200 import _abi as A, api, synth
    M = args.members
    T = site.nsteps
    params = synth.synth_params(M, stream=100 + D.rank)
    cid = D.comm_id(api)
    # cold start, on the books: sipnet_gpu_init (site preparation, uploads, setupModel on the device), the team, the
    # first pass with cold caches / first-use allocations, and the summaries delivered to the host
    D.barrier()
    t_cold = time.perf_counter()
    ens = api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), math=A.MATH_FAST, device=D.local,
                       outputs=A.OUT_MOMENTS | A.OUT_QUANTILES, summary_cols=[A.O["nee"], A.O["gpp"]], quantiles=QUANTILES)
    ens.join_team(D.world, D.rank, cid)
    t_init = time.perf_counter() - t_cold

    def one_pass():
        ens.reset()
        ens.run(0, T)
        ens.team_summaries()

    one_pass()
    cold_q = ens.quantiles()
    cold_m, cold_v = ens.mean(), ens.variance()
    t_cold = D.max(time.perf_counter() - t_cold)
    del cold_q, cold_m, cold_v

    for _ in range(max(args.warmup, 3)):
        one_pass()
    ens.sync()
    sampler = ClockSampler(D.local)
    launches0 = ens.launch_count()
    D.barrier()
    sampler.start()
    ens.timer_start()
    for _ in range(args.steps):
        one_pass()
    total_ms = ens.timer_stop_ms()
    D.barrier()
    clocks = sampler.stop()
    launches = ens.launch_count() - launches0
    ms_per_step = D.max(total_ms / args.steps)
    levels = ens.team_last_levels()
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, ens, M, T)

    # phases of one pass (an extra, untimed pass with a stopwatch around each phase)
    kern, summ = [], []
    for _ in range(3):
        ens.reset()
        ens.run(0, T)
        kern.append(ens.last_run_ms())
        ens.sync()
        D.barrier()
        ens.timer_start()
        ens.team_summaries()
        summ.append(ens.timer_stop_ms())
    kern_ms = D.max(float(np.mean(kern)))
    summ_ms = D.max(float(np.mean(summ)))
    q_dev = ens.quantiles()
    mean_dev = ens.mean()
    assert np.isfinite(q_dev).all() and np.isfinite(mean_dev).all()
    replayed = int((ens.status() & A.ST_REPLAY).astype(bool).sum())

    # ---- end to end: pinned host params -> device, run, team summaries, summaries -> pinned host
    par_bytes = A.NPARAMS * M * 8
    nsum = 2 * T
    out_bytes = (2 * nsum + len(QUANTILES) * nsum) * 8
    hpar = pinned(lib, par_bytes)
    hout = pinned(lib, out_bytes)
    C.memmove(hpar, params.ctypes.data, par_bytes)

    def e2e_pass():
        ens.set_params(hpar, M)                               # H2D of the ensemble + setupModel()
        ens.run(0, T)
        ens.team_summaries()
        ens.gather_raw(A.GATHER_MEAN, hout, nsum * 8)
        ens.gather_raw(A.GATHER_VARIANCE, hout + nsum * 8, nsum * 8)
        ens.gather_raw(A.GATHER_QUANTILES, hout + 2 * nsum * 8, len(QUANTILES) * nsum * 8)

    e2e_pass()
    D.barrier()
    n_e2e = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    ens.timer_start()
    for _ in range(n_e2e):
        e2e_pass()
    e2e_dev_ms = ens.timer_stop_ms() / n_e2e
    e2e_wall_ms = 1e3 * (time.perf_counter() - t0) / n_e2e
    e2e_ms = D.max(max(e2e_dev_ms, e2e_wall_ms))              # the gathers block the host: wall clock is the honest one
    D.barrier()
    host_mean = np.ctypeslib.as_array((C.c_double * nsum).from_address(hout)).copy()
    assert np.array_equal(host_mean.reshape(mean_dev.shape), mean_dev), "the summaries really are in host memory"
    lib.sipnet_gpu_host_free(hout)
    lib.sipnet_gpu_host_free(hpar)

    # ---- seeded oracle spot check of bench members, outside the timed region (rank 0)
    spot = None
    if D.rank == 0 and not args.no_extras:
        spot = oracle_spot_check(site, params, ens)
    ens.close()
    return dict(cold_s=t_cold, init_s=t_init, M=M, T=T, ms_per_step=ms_per_step, kern_ms=kern_ms, summ_ms=summ_ms, clocks=clocks, launches=launches,
                e2e_ms=e2e_ms, h2d=par_bytes, d2h=out_bytes, levels=levels, replayed=replayed, spot=spot)


def kept_columns(ens, M: int, T: int):
    """Zero-copy torch view [2][T][M] of the per-member NEE and GPP columns the summaries are taken over."""
    import torch
    from sipnet_b200 import _abi as A
    from sipnet_b200.distributed import DeviceArray
    ld = (M + 15) // 16 * 16
    return DeviceArray(ens.device_ptr(A.GATHER_FULL), (2, T, M), (T * ld, ld, 1)).tensor(torch.cuda.current_device())


DUMP_MEMBERS = 64       # per-member columns are 16 B per member-step (15 GB at the default size): the dump keeps a sample
DUMP_BYTES = 60 << 20   # data of all --dump-outputs files; with the .npy headers the dump stays under 64 MB


def dump_members(M: int) -> np.ndarray:
    """The fixed, seeded sample of a rank's members whose NEE / GPP columns --dump-outputs keeps."""
    return np.sort(np.random.default_rng(20261020).choice(M, size=min(M, DUMP_MEMBERS), replace=False))


def dump_steps(T: int, values_per_step: int) -> np.ndarray:
    """The steps --dump-outputs keeps: all T of them, or as many evenly spaced ones (first and last included) as fit
    DUMP_BYTES when the run is too long for all."""
    n = min(T, DUMP_BYTES // (8 * values_per_step))
    return np.linspace(0, T - 1, n).round().astype(np.int64)


def dump_outputs(path: str, ens, M: int, T: int) -> None:
    """--dump-outputs: the team summaries of the last pass as its caller receives them, and the NEE / GPP columns of
    dump_members(M), at the steps dump_steps() keeps."""
    os.makedirs(path, exist_ok=True)
    arrays = {"mean": ens.mean(), "variance": ens.variance(), "quantiles": ens.quantiles()}
    pick = dump_members(M)
    steps = dump_steps(T, sum(a.size for a in arrays.values()) // T + 2 * pick.size)
    arrays = {name: a[..., steps] for name, a in arrays.items()}
    arrays["member_nee_gpp"] = kept_columns(ens, M, T)[:, :, pick.tolist()][:, steps.tolist()].cpu().numpy()
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_BYTES
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def oracle_spot_check(site, params, ens):
    """A seeded sample of the bench ensemble's members against the oracle (CPU restatement, pinned to the reference),
    bit for bit: the kept summary columns of the big run, and all 32 columns through a small full-output handle."""
    from oracle.pyoracle import Oracle
    from sipnet_b200 import _abi as A, api, synth
    import torch
    rng = np.random.default_rng(20261017)
    pick = sorted(int(x) for x in rng.choice(params.shape[1], size=3, replace=False))
    T = site.nsteps
    M = params.shape[1]
    kept = kept_columns(ens, M, T)[:, :, pick].cpu().numpy()  # [2][T][3]: NEE, GPP of the picked members
    orc = Oracle()
    with api.Ensemble([site], np.ascontiguousarray(params[:, pick]), None, dict(synth.SYNTH_FLAGS), outputs=A.OUT_FULL,
                      math=A.MATH_FAST, device=torch.cuda.current_device()) as small:
        small.run()
        full = small.output()
    ok = True
    for j, m in enumerate(pick):
        rc, done, o_out, _, _ = orc.run(synth.SYNTH_FLAGS, params[:, m], site, want_debug=False)
        ok &= rc == 0 and done == T
        ok &= bool(np.array_equal(full[:, :, j].T, o_out, equal_nan=True))
        ok &= bool(np.array_equal(kept[0, :, j], o_out[:, A.O["nee"]]) and np.array_equal(kept[1, :, j], o_out[:, A.O["gpp"]]))
    if not ok:
        raise SystemExit(f"bench.py: members {pick} of the bench ensemble differ from the oracle")
    return {"members": pick, "columns": 32, "steps": T, "bit_identical_to_oracle": True}


def section_c5(args, D: Dist, site):
    """C5 share: draws scored by the on-device NEE log-likelihood, gathered over all ranks through the C ABI."""
    from sipnet_b200 import _abi as A, api, synth
    M = C5_DRAWS_PER_GPU
    T = site.nsteps
    rng = np.random.default_rng(7)
    site.nee_obs = np.where(rng.uniform(size=T) < 0.2, np.nan, rng.normal(0, 1.5, T))
    params = synth.synth_params(M, stream=200 + D.rank)
    ens = api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), math=A.MATH_FAST, device=D.local,
                       outputs=A.OUT_LOGLIK, nee_sigma=0.5)
    ens.join_team(D.world, D.rank, D.comm_id(api))
    ll = np.empty(M * D.world)

    def one_pass():
        ens.reset()
        ens.run(0, T)
        ens.team_loglik(ll)

    one_pass()
    D.barrier()
    n = 3
    t0 = time.perf_counter()
    kern = []
    for _ in range(n):
        one_pass()
        kern.append(ens.last_run_ms())
    ms = D.max(1e3 * (time.perf_counter() - t0) / n)
    D.barrier()
    assert np.isfinite(ll).all()
    site.nee_obs = None
    ens.close()
    return {"workload": f"C5 (weak scaling): {M} parameter draws per GPU x {T} steps, on-device NEE log-likelihood, "
                        "all-gather of the scores over NCCL (sipnet_gpu_comm_gather_loglik) into host memory",
            "value": D.world * M * T / (ms * 1e-3), "unit": UNIT, "ms_per_pass": ms, "kernel_ms": float(np.mean(kern)),
            "comm_nranks": D.world, "timing": "wall clock around the pass (includes the gather to host), max over ranks"}


def section_c2(args, D: Dist, lib, site):
    """C2 (BASELINE.json configs[1]): 4096 members, FULL per-step output; device-resident and host-delivered.
    With N ranks every GPU runs its own C2 (replicas: the full-output mode has no exchange step); the host-delivered
    figure is the aggregate over the ranks, and a plain device->pinned-host copy of the same bytes, issued by all
    ranks at once, is timed beside it as the box's ceiling for this mode."""
    from sipnet_b200 import _abi as A, api, synth
    torch = D.torch
    M, T = 4096, site.nsteps
    params = synth.synth_params(M, stream=D.rank)
    ens = api.Ensemble([site], params, None, dict(synth.SYNTH_FLAGS), outputs=A.OUT_FULL, math=A.MATH_FAST, device=D.local)
    for _ in range(2):
        ens.reset()
        ens.run(0, T)
    ens.sync()
    D.barrier()
    ens.timer_start()
    for _ in range(5):
        ens.reset()
        ens.run(0, T)
    dev_ms = D.max(ens.timer_stop_ms() / 5)
    kern_ms = ens.last_run_ms()
    out_bytes = A.NOUT * T * M * 8
    par_bytes = A.NPARAMS * M * 8
    hout, hpar = pinned(lib, out_bytes), pinned(lib, par_bytes)
    C.memmove(hpar, params.ctypes.data, par_bytes)
    ens.set_params(hpar, M)
    ens.run_to_host(hout, 0, T, nbytes=out_bytes)
    D.barrier()
    ens.timer_start()
    for _ in range(3):
        ens.set_params(hpar, M)
        ens.run_to_host(hout, 0, T, nbytes=out_bytes)
    e2e_ms = D.max(ens.timer_stop_ms() / 3)
    # the ceiling: one plain copy of the same bytes, device -> the same pinned buffer, all ranks at once
    src = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")
    dst = torch.frombuffer((C.c_ubyte * out_bytes).from_address(hout), dtype=torch.uint8)
    dst.copy_(src)
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    probe_ms = D.max(e0.elapsed_time(e1) / 3)
    del src, dst
    lib.sipnet_gpu_host_free(hout)
    lib.sipnet_gpu_host_free(hpar)
    ens.close()
    W = D.world
    return {"workload": "C2: 1 site x 4096 members x 10 yr half-daily, full per-step output (32 doubles per member-step)"
                        + (f", one replica per GPU x {W}" if W > 1 else ""),
            "value": W * M * T / (dev_ms * 1e-3), "unit": UNIT, "ms_per_step": dev_ms, "kernel_ms": kern_ms,
            "e2e": {"value": W * M * T / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": par_bytes, "d2h_bytes_per_step": out_bytes,
                    "d2h_gb_s_all_ranks": W * out_bytes / (e2e_ms * 1e-3) / 1e9},
            "d2h_probe": {"gb_s_all_ranks": W * out_bytes / (probe_ms * 1e-3) / 1e9, "ms": probe_ms,
                          "what": "plain device -> pinned host copy of the same bytes, all ranks at once (the box's "
                                  "ceiling for host-delivered full output)"},
            "cpu_affinity": D.affinity,
            "note": "4096 members = 128 warps on 592 warp schedulers: latency-bound by construction (round-1 headline)"}


def host_writer_rate(T: int, members: int = 64) -> dict:
    """Rows/s of the drop-in driver's main-output writer (host/sip_output.c: printf-free byte-identical sipnet.out rows,
    member blocks on all host cores) on this box -- CPU only, beside the reference-with-text-output baseline: it is what
    a many-member launch with the main output on spends after the run."""
    lib = C.CDLL(os.path.join(ROOT, "sipnet_b200", "libsipnet_host.so"))
    lib.sip_write_state_files.restype = C.c_int
    lib.sip_write_state_files.argtypes = [C.c_char_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.POINTER(C.c_int32)),
                                          C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_double)), C.c_int64,
                                          C.POINTER(C.c_double), C.c_int, C.c_int]
    path_max = 256 + 32                                            # SIP_STATE_PATH_MAX
    nout = 32
    rng = np.random.default_rng(5)
    scale = 10.0 ** np.array([4, 2, 0, 4, 3, 2, 3, 1, 0, 1] + [0] * 10 + [-1, -1, 0, 2, 1, 0, -4, -3, -3, -2, -3, 2], float)
    buf = np.ascontiguousarray((rng.uniform(0, 1, (T, members, nout)) * scale).transpose(2, 0, 1))   # [col][T][M]
    year = np.full(T, 2015, np.int32)
    day = (np.arange(T) // 2 % 365 + 1).astype(np.int32)
    tm = np.where(np.arange(T) % 2 == 0, 0.0, 12.0)
    ns = np.full(members, T, np.int64)
    yp = (C.POINTER(C.c_int32) * members)(*[year.ctypes.data_as(C.POINTER(C.c_int32))] * members)
    dp = (C.POINTER(C.c_int32) * members)(*[day.ctypes.data_as(C.POINTER(C.c_int32))] * members)
    tp = (C.POINTER(C.c_double) * members)(*[tm.ctypes.data_as(C.POINTER(C.c_double))] * members)
    with tempfile.TemporaryDirectory() as td:
        paths = C.create_string_buffer(members * path_max)
        for m in range(members):
            name = os.path.join(td, f"w.out.{m}").encode()
            paths[m * path_max: m * path_max + len(name)] = name
        t0 = time.perf_counter()
        rc = lib.sip_write_state_files(paths, members, ns.ctypes.data_as(C.POINTER(C.c_int64)), yp, dp, tp, T,
                                       buf.ctypes.data_as(C.POINTER(C.c_double)), 1, 0)
        dt = time.perf_counter() - t0
        nbytes = sum(os.path.getsize(os.path.join(td, f"w.out.{m}")) for m in range(members))
    if rc != 0:
        raise RuntimeError(f"sip_write_state_files returned {rc}")
    return {"value": members * T / dt, "unit": "rows/s (one row = one member-timestep of sipnet.out text)",
            "text_gb_s": nbytes / dt / 1e9, "threads": min(os.cpu_count() or 1, 64, (members + 7) // 8),
            "sample": f"{members} members x {T} steps into {nbytes / 1e6:.0f} MB of text in a temporary directory",
            "what": "sip_write_state_files (host C, no GPU work): the writer behind the drop-in driver's per-member "
                    "main output; compare with cpu_baseline_text_output, the reference writing the same rows"}


def run_ours(args):
    from sipnet_b200 import _abi as A, api, synth
    D = Dist()
    lib = api.load_library()
    site = synth.synth_site(0, args.years, "half-daily")
    peak = C.c_double(0.0)
    lib.sipnet_gpu_measure_fp64_peak(D.local, C.byref(peak))
    fp64_peak_tflops = float(peak.value)

    r = section_c4(args, D, lib, site, fp64_peak_tflops)
    thr = None if args.no_extras else section_throughput_policy(args, D, site)
    c5 = None if args.no_extras else section_c5(args, D, site)
    c2 = None if args.no_extras else section_c2(args, D, lib, site)

    if D.rank == 0:
        M, T, world = r["M"], r["T"], D.world
        value = world * M * T / (r["ms_per_step"] * 1e-3)
        peaks, facts = {}, {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        try:
            facts = json.load(open(KERNEL_FACTS))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        rate_kernel = M * T / (r["kern_ms"] * 1e-3)              # member-steps/s of one GPU inside the step kernel
        # FP64 roofline of the step kernel.  Basis (DESIGN.md 4): the FP64-pipe instructions the kernel executes per
        # member-step (DFMA + DADD + DMUL + DSETP, from this round's ncu capture), each counted as one pipe slot = one
        # FMA = 2 flop, against the pipe's issue rate -- 16 lanes per SM sub-partition and clock at the SM clock sampled
        # during the timed region.  This is what ncu reports as sm__inst_executed_pipe_fp64 (% of peak).
        e = float(facts.get("fp64_pipe_inst_per_member_step") or FP64_INST_PER_MEMBER_STEP_FALLBACK)
        sm_hz = 1e6 * float(r["clocks"].get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0))
        pipe_rate = 148 * 4 * 16 * sm_hz                           # thread-level FP64 instructions per second
        fp64_ach = rate_kernel * e * 2.0 / 1e12
        fp64_peak = pipe_rate * 2.0 / 1e12
        roof = {"bound": "fp64", "kernel": "sip::k1::run_kernel", "kernel_ms": r["kern_ms"],
                "achieved": fp64_ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": fp64_ach / fp64_peak,
                "algorithmic": f"{e:.0f} FP64-pipe instructions/member-step (= {2 * e:.0f} FMA-equivalent flop) x {M * T} "
                               f"member-steps per launch",
                "peak_source": "FP64 pipe issue rate: 148 SMs x 4 sub-partitions x 16 lanes x 2 flop x the SM clock sampled "
                               "in the timed region (MEASURED_PEAKS.json holds no FP64 figure); a live DFMA probe is "
                               "reported beside it",
                "frac_executed": fp64_ach / fp64_peak,
                "probe": {"tflops": fp64_peak_tflops, "frac_vs_probe": fp64_ach / fp64_peak_tflops if fp64_peak_tflops > 0 else None,
                          "what": "sipnet_gpu_measure_fp64_peak: 8 independent DFMA chains per thread, this GPU, this run"},
                "executed": {"fp64_pipe_inst_per_member_step": e, "all_inst_per_member_step": facts.get("inst_per_member_step"),
                             "pipe_rate_inst_per_s": pipe_rate, "sm_mhz": sm_hz / 1e6,
                             "ncu_fp64_pipe_pct": facts.get("ncu_fp64_pipe_pct"), "ncu_issue_active_pct": facts.get("ncu_issue_active_pct"),
                             "source": facts.get("source")},
                # SURVEY 8(d)'s estimate, kept for continuity with round 1: it prices a pow at CUDA libm's 150-200
                # instructions; the glibc-exact restatement needs a quarter of that, so this basis is NOT a roofline
                "survey_basis": {"flop_per_member_step": FLOP_PER_MEMBER_STEP, "tflops": rate_kernel * FLOP_PER_MEMBER_STEP / 1e12,
                                 "note": "overstates the executed FP64 work about 2x; not used for frac"}}
        # summary columns written by the step kernel (2 x 8 B per member-step) against HBM
        hbm_ach = rate_kernel * 16.0 / 1e9
        roof["traffic"] = facts.get("dram_bytes_per_launch")
        roof["traffic_source"] = (facts.get("source") or "none") + " (a capture of this configuration, not of this run)"
        roof_alt = {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                    "peak_source": hbm_src, "algorithmic": f"16 B/member-step (two kept columns) x {M * T} member-steps"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": bench_config(args, T),
            "phases_ms": {"step_kernel": r["kern_ms"], "team_summaries": r["summ_ms"], "select_levels": r["levels"]},
            "comm_nranks": world, "replayed_members": r["replayed"],
            "roofline": roof, "roofline_alt": roof_alt, "clocks": r["clocks"], "gpu_launches": int(r["launches"]),
            "e2e": {"value": world * M * T / (r["e2e_ms"] * 1e-3), "unit": UNIT, "ms_per_step": r["e2e_ms"],
                    "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "path": "pinned host params -> sipnet_gpu_set_params -> run -> sipnet_gpu_comm_summaries -> gather of "
                            "mean/variance/quantiles into pinned host memory"},
        }
        line["e2e_cold"] = {"value": world * M * T / r["cold_s"], "unit": UNIT, "s": r["cold_s"], "init_s": r["init_s"],
                            "what": "sipnet_gpu_init (+ team) + first pass + summaries gathered to the host, wall clock"}
        if r["spot"]:
            line["oracle_spot_check"] = r["spot"]
        if thr:
            line["throughput_policy"] = thr
        if c5:
            line["c5"] = c5
        if c2:
            line["c2"] = c2
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            params = synth.synth_params(min(M, 96 * cores), stream=100)
            cpu = CpuReference(site, params, dict(synth.SYNTH_FLAGS), cores)
            cpu.sample(2)
            v, sample = cpu.sample(max(1, min(96, M // cores)))
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": cpu.kind, "sample": sample}
            if cpu.kind == "reference":   # SURVEY 8(d)'s second figure: the reference WITH its sipnet.out text output
                with tempfile.TemporaryDirectory() as td:
                    vt, st = cpu.sample(max(1, min(24, M // cores)), text_dir=td)
                line["cpu_baseline_text_output"] = {"value": vt, "unit": UNIT, "cores": cores, "kind": cpu.kind, "sample": st}
            cpu.close()
            try:   # informational, CPU only: never allowed to cost the bench line
                line["host_writer"] = host_writer_rate(T)
            except Exception as exc:
                line["host_writer"] = {"error": str(exc)[:200]}
        print(json.dumps(line), flush=True)
    D.close()


def run_c3(args):
    """BASELINE.json configs[2] (C3) as one extra line: 10k sites x 100 members with events, whole sites per rank,
    per-site NEE mean/variance on the device (no collective: sites are independent)."""
    from sipnet_b200 import _abi as A, api, synth
    D = Dist()
    nsites = args.sites or 10000 // D.world
    t0 = time.perf_counter()
    sites, params, ms, flags = synth.config_c3(nsites=nsites, members_per_site=100, nyears=args.years, site0=D.rank * nsites)
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    ens = api.Ensemble(sites, params, ms, flags, math=A.MATH_FAST, device=D.local, outputs=A.OUT_MOMENTS,
                       summary_cols=[A.O["nee"]], out_steps_capacity=256)
    t_init = time.perf_counter() - t0
    t_lib_init = ens.init_seconds
    T = ens.max_steps

    def one_pass():
        ens.reset()
        for a in range(0, T, 256):
            ens.run(a, min(T, a + 256))
            ens.device_ptr(A.GATHER_MEAN)                      # per-site moments of the segment stay on the device
        ens.sync()

    one_pass()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass()
    dt = D.max((time.perf_counter() - t0) / args.steps)
    ens.close()
    if D.rank == 0:
        print(json.dumps({"metric": METRIC, "workload": f"C3: {nsites * D.world} sites x 100 members, {args.years} yr half-daily, "
                          "events.in schedule, per-site NEE mean/variance", "value": D.world * nsites * 100 * T / dt, "unit": UNIT,
                          "n_gpus": D.world, "s_per_pass": dt, "input_build_s": t_build, "init_s": t_init, "sipnet_gpu_init_s": t_lib_init,
                          "dtype": "f64", "data": "synthetic"}), flush=True)
    D.close()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "c3":
        run_c3(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
