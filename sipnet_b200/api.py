"""Host-side Python view of the C ABI (include/sipnet_gpu.h).

Python is plumbing here: it builds `sipnet_gpu_config` from numpy arrays, calls
`sipnet_gpu_init / run / gather` through ctypes and hands numpy arrays back.
All compute happens in the CUDA library; there is no CPU fallback -- if
libsipnet_gpu.so is missing or no device is usable, these calls raise.

The names mirror the reference interface this path replaces
(`setupModel`/`updateState`/`outputState`, reference src/sipnet/sipnet.h:26-54).
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import _abi as A

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SIPNET_GPU_LIB") or os.path.join(_PKG_DIR, "libsipnet_gpu.so")


class SipnetGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"sipnet_gpu error {code}: {msg}")
        self.code = code


_lib = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libsipnet_gpu.so (built in-tree by __graft_entry__.build())."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(p, mode=C.RTLD_GLOBAL)
    lib.sipnet_gpu_init.restype = C.c_int
    lib.sipnet_gpu_init.argtypes = [C.POINTER(A.Config), C.POINTER(C.c_void_p)]
    lib.sipnet_gpu_run.restype = C.c_int
    lib.sipnet_gpu_run.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    lib.sipnet_gpu_gather.restype = C.c_int
    lib.sipnet_gpu_gather.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    lib.sipnet_gpu_run_to_host.restype = C.c_int
    lib.sipnet_gpu_run_to_host.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_size_t, C.c_int64]
    lib.sipnet_gpu_gather_bytes.restype = C.c_size_t
    lib.sipnet_gpu_gather_bytes.argtypes = [C.c_void_p, C.c_int]
    lib.sipnet_gpu_sync.restype = C.c_int
    lib.sipnet_gpu_sync.argtypes = [C.c_void_p]
    lib.sipnet_gpu_reset.restype = C.c_int
    lib.sipnet_gpu_reset.argtypes = [C.c_void_p]
    lib.sipnet_gpu_set_params.restype = C.c_int
    lib.sipnet_gpu_set_params.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.sipnet_gpu_set_state.restype = C.c_int
    lib.sipnet_gpu_set_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
    lib.sipnet_gpu_ring_slots.restype = C.c_int32
    lib.sipnet_gpu_ring_slots.argtypes = [C.c_void_p]
    lib.sipnet_gpu_timer_start.restype = C.c_int
    lib.sipnet_gpu_timer_start.argtypes = [C.c_void_p]
    lib.sipnet_gpu_timer_stop_ms.restype = C.c_int
    lib.sipnet_gpu_timer_stop_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.sipnet_gpu_destroy.restype = None
    lib.sipnet_gpu_destroy.argtypes = [C.c_void_p]
    lib.sipnet_gpu_last_run_ms.restype = C.c_int
    lib.sipnet_gpu_last_run_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.sipnet_gpu_launch_count.restype = C.c_int64
    lib.sipnet_gpu_launch_count.argtypes = [C.c_void_p]
    lib.sipnet_gpu_device_ptr.restype = C.c_void_p
    lib.sipnet_gpu_device_ptr.argtypes = [C.c_void_p, C.c_int]
    lib.sipnet_gpu_host_alloc.restype = C.c_void_p
    lib.sipnet_gpu_host_alloc.argtypes = [C.c_size_t]
    lib.sipnet_gpu_host_free.restype = None
    lib.sipnet_gpu_host_free.argtypes = [C.c_void_p]
    lib.sipnet_gpu_last_error.restype = C.c_char_p
    lib.sipnet_gpu_last_error.argtypes = []
    lib.sipnet_gpu_abi_version.restype = C.c_int
    lib.sipnet_gpu_abi_version.argtypes = []
    lib.sipnet_gpu_measure_fp64_peak.restype = C.c_int
    lib.sipnet_gpu_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    lib.sipnet_gpu_rows_summary.restype = C.c_int
    lib.sipnet_gpu_rows_summary.argtypes = [C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int32,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    # multi-GPU entry points
    lib.sipnet_gpu_comm_unique_id.restype = C.c_int
    lib.sipnet_gpu_comm_unique_id.argtypes = [C.c_void_p]
    lib.sipnet_gpu_comm_init_rank.restype = C.c_int
    lib.sipnet_gpu_comm_init_rank.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.sipnet_gpu_comm_destroy.restype = None
    lib.sipnet_gpu_comm_destroy.argtypes = [C.c_void_p]
    lib.sipnet_gpu_comm_nranks.restype = C.c_int32
    lib.sipnet_gpu_comm_nranks.argtypes = [C.c_void_p]
    lib.sipnet_gpu_comm_summaries.restype = C.c_int
    lib.sipnet_gpu_comm_summaries.argtypes = [C.c_void_p]
    lib.sipnet_gpu_comm_last_levels.restype = C.c_int32
    lib.sipnet_gpu_comm_last_levels.argtypes = [C.c_void_p]
    lib.sipnet_gpu_comm_gather_loglik.restype = C.c_int
    lib.sipnet_gpu_comm_gather_loglik.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.sipnet_gpu_comm_member_counts.restype = C.c_int
    lib.sipnet_gpu_comm_member_counts.argtypes = [C.c_void_p, C.c_void_p]
    lib.sipnet_gpu_multi_init.restype = C.c_int
    lib.sipnet_gpu_multi_init.argtypes = [C.POINTER(A.Config), C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.sipnet_gpu_multi_run.restype = C.c_int
    lib.sipnet_gpu_multi_run.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    lib.sipnet_gpu_multi_gather.restype = C.c_int
    lib.sipnet_gpu_multi_gather.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    lib.sipnet_gpu_multi_gather_bytes.restype = C.c_size_t
    lib.sipnet_gpu_multi_gather_bytes.argtypes = [C.c_void_p, C.c_int]
    lib.sipnet_gpu_multi_reset.restype = C.c_int
    lib.sipnet_gpu_multi_reset.argtypes = [C.c_void_p]
    lib.sipnet_gpu_multi_sync.restype = C.c_int
    lib.sipnet_gpu_multi_sync.argtypes = [C.c_void_p]
    lib.sipnet_gpu_multi_ndevices.restype = C.c_int32
    lib.sipnet_gpu_multi_ndevices.argtypes = [C.c_void_p]
    lib.sipnet_gpu_multi_handle.restype = C.c_void_p
    lib.sipnet_gpu_multi_handle.argtypes = [C.c_void_p, C.c_int32]
    lib.sipnet_gpu_multi_destroy.restype = None
    lib.sipnet_gpu_multi_destroy.argtypes = [C.c_void_p]
    lib.sipnet_gpu_assimilate.restype = C.c_int
    lib.sipnet_gpu_assimilate.argtypes = [C.c_void_p, C.POINTER(A.ObsSpec), C.c_void_p]
    lib.sipnet_gpu_comm_assimilate.restype = C.c_int
    lib.sipnet_gpu_comm_assimilate.argtypes = [C.c_void_p, C.POINTER(A.ObsSpec), C.c_void_p]
    lib.sipnet_gpu_multi_assimilate.restype = C.c_int
    lib.sipnet_gpu_multi_assimilate.argtypes = [C.c_void_p, C.POINTER(A.ObsSpec), C.c_void_p]
    for name in ("sipnet_gpu_assimilate_inflated", "sipnet_gpu_comm_assimilate_inflated",
                 "sipnet_gpu_multi_assimilate_inflated"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, C.POINTER(A.ObsSpec), C.POINTER(A.InflationSpec), C.c_void_p]
    for name in ("sipnet_gpu_resample", "sipnet_gpu_comm_resample", "sipnet_gpu_multi_resample"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    for name in ("sipnet_gpu_rejuvenate", "sipnet_gpu_comm_rejuvenate", "sipnet_gpu_multi_rejuvenate"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, C.POINTER(A.JitterSpec), C.c_void_p]
    lib.sipnet_gpu_eval_libm.restype = C.c_int
    lib.sipnet_gpu_eval_libm.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    if path is None:
        _lib = lib
    return lib


def _dp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


@dataclass
class SiteData:
    """One site's forcing (post-readClimData units, reference sipnet.c:205-238)
    and its events.in schedule (file order)."""
    year: np.ndarray
    day: np.ndarray
    clim: dict                      # name -> float64[T] for A.CLIM_COLS
    events: list = field(default_factory=list)  # (year, day, type, method, p0..p3)
    nee_obs: Optional[np.ndarray] = None

    def __post_init__(self):
        self.year = np.ascontiguousarray(self.year, dtype=np.int32)
        self.day = np.ascontiguousarray(self.day, dtype=np.int32)
        self.clim = {k: np.ascontiguousarray(self.clim[k], dtype=np.float64)
                     for k in A.CLIM_COLS}
        if self.nee_obs is not None:
            self.nee_obs = np.ascontiguousarray(self.nee_obs, dtype=np.float64)

    @property
    def nsteps(self) -> int:
        return int(self.year.shape[0])

    def event_array(self):
        n = len(self.events)
        arr = (A.Event * max(n, 1))()
        for i, ev in enumerate(self.events):
            y, d, typ, method, *p = ev
            arr[i].year, arr[i].day, arr[i].type, arr[i].method = int(y), int(d), int(typ), int(method)
            for k in range(4):
                arr[i].p[k] = float(p[k]) if k < len(p) else 0.0
        return arr, n

    def to_struct(self, keep: list) -> A.Site:
        s = A.Site()
        s.nsteps = self.nsteps
        s.year = _ip(self.year)
        s.day = _ip(self.day)
        for k in A.CLIM_COLS:
            setattr(s, k, _dp(self.clim[k]))
        arr, n = self.event_array()
        keep.append(arr)
        s.nevents = n
        s.events = C.cast(arr, C.POINTER(A.Event))
        if self.nee_obs is not None:
            s.nee_obs = _dp(self.nee_obs)
        return s


def flags_struct(flags: dict) -> A.Flags:
    f = A.Flags()
    merged = dict(A.DEFAULT_FLAGS)
    merged.update(flags or {})
    for n in A.FLAG_NAMES:
        setattr(f, n, int(merged[n]))
    return f


def flags_array(flags: dict) -> np.ndarray:
    merged = dict(A.DEFAULT_FLAGS)
    merged.update(flags or {})
    return np.array([int(merged[n]) for n in A.FLAG_NAMES], dtype=np.int32)


EVAL_FLAGGED = 0x7ff8bad0bad0bad0     # sipnet_gpu.h SIPNET_GPU_EVAL_FLAGGED
_EVAL_OPS = {"exp": 0, "pow": 1, "fast_exp": 2, "fast_pow": 3, "fast_powc": 4, "fast_div": 5, "thr_div": 6,
             "thr_divw": 7, "seed": 8}


def device_libm(op: str, x: np.ndarray, y: Optional[np.ndarray] = None, device: int = 0) -> np.ndarray:
    """Evaluate the DEVICE exp/pow (glibc-exact restatement) on arrays (validation hook).  The fast_* ops run the
    production kernel's optimistic policy; inputs outside its guards come back as the bit pattern EVAL_FLAGGED.
    thr_div / thr_divw are the throughput policy's divisions, seed the refined reciprocal of x (sip_num.cuh)."""
    lib = load_library()
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    yp = None
    if op not in ("exp", "fast_exp", "seed"):
        y = np.ascontiguousarray(y, dtype=np.float64)
        yp = y.ctypes.data
    rc = lib.sipnet_gpu_eval_libm(device, _EVAL_OPS[op], x.ctypes.data, yp, out.ctypes.data, x.size)
    if rc != 0:
        raise SipnetGpuError(rc, (lib.sipnet_gpu_last_error() or b"").decode())
    return out


class Ensemble:
    """A batched SIPNET run on one GPU (wraps a sipnet_gpu_handle)."""

    def __init__(self, sites: Sequence[SiteData], params: np.ndarray,
                 member_site: Optional[np.ndarray] = None, flags: Optional[dict] = None,
                 outputs: int = A.OUT_FULL, math: int = A.MATH_VALIDATION,
                 device: int = 0, out_steps_capacity: int = 0,
                 summary_cols: Sequence[int] = (), quantiles: Sequence[float] = (),
                 nee_sigma: float = 1.0, max_event_records: int = 0,
                 block_threads: int = 0, stream: int = 0, ring_slots: int = 0, lib: Optional[C.CDLL] = None):
        self.lib = lib or load_library()
        cfg = self._configure(sites, params, member_site, flags, outputs, math, device, out_steps_capacity, summary_cols,
                              quantiles, nee_sigma, max_event_records, block_threads, stream, ring_slots)
        self.handle = C.c_void_p()
        t0 = time.perf_counter()
        rc = self.lib.sipnet_gpu_init(C.byref(cfg), C.byref(self.handle))
        self.init_seconds = time.perf_counter() - t0           # the library call alone (not the ctypes marshalling)
        if rc != 0:
            self.handle = None
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (0, 0)

    def _configure(self, sites, params, member_site, flags, outputs, math, device, out_steps_capacity, summary_cols,
                   quantiles, nee_sigma, max_event_records, block_threads, stream, ring_slots) -> "A.Config":
        """sipnet_gpu_config from numpy inputs (the arrays it points into are kept alive in self._keep)."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.ndim != 2 or params.shape[0] != A.NPARAMS:
            raise ValueError("params must be float64 [80][M] (struct Parameters order)")
        self.nmembers = int(params.shape[1])
        self.sites = list(sites)
        self.nsites = len(self.sites)
        self._keep = [params]
        site_structs = (A.Site * self.nsites)()
        for i, s in enumerate(self.sites):
            site_structs[i] = s.to_struct(self._keep)
        self._keep.append(site_structs)
        cfg = A.Config()
        cfg.abi_version = A.ABI_VERSION
        cfg.device = device
        cfg.flags = flags_struct(flags)
        cfg.nsites = self.nsites
        cfg.sites = C.cast(site_structs, C.POINTER(A.Site))
        cfg.nmembers = self.nmembers
        if member_site is not None:
            ms = np.ascontiguousarray(member_site, dtype=np.int32)
            self._keep.append(ms)
            cfg.member_site = _ip(ms)
            self.member_site = ms
        else:
            self.member_site = np.zeros(self.nmembers, dtype=np.int32)
        cfg.params = _dp(params)
        cfg.params_ld = self.nmembers
        cfg.outputs = outputs
        cfg.math = math
        cfg.out_steps_capacity = out_steps_capacity
        sc = np.ascontiguousarray(summary_cols, dtype=np.int32)
        q = np.ascontiguousarray(quantiles, dtype=np.float64)
        self._keep += [sc, q]
        cfg.n_summary_cols = sc.size
        cfg.summary_cols = _ip(sc) if sc.size else None
        cfg.n_quantiles = q.size
        cfg.quantiles = _dp(q) if q.size else None
        cfg.nee_sigma = nee_sigma
        cfg.max_event_records = max_event_records
        cfg.block_threads = block_threads
        cfg.stream = stream or None
        cfg.ring_slots = ring_slots
        self.n_summary_cols = int(sc.size)
        self.n_quantiles = int(q.size)
        self.max_event_records = max_event_records
        self.max_steps = max(s.nsteps for s in self.sites)
        return cfg

    # -- reference: the while(climate) loop, sipnet.c:1969-1982
    def run(self, step_begin: int = 0, step_end: Optional[int] = None) -> None:
        if step_end is None:
            step_end = self.max_steps
        rc = self.lib.sipnet_gpu_run(self.handle, step_begin, step_end)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (step_begin, step_end)

    def run_to_host(self, dst, step_begin: int = 0, step_end: Optional[int] = None, chunk_steps: int = 0,
                    nbytes: Optional[int] = None) -> None:
        """Pipelined run + delivery of the full output into a host buffer [32][n][M]
        (numpy array, or a raw pointer with `nbytes`, ideally pinned)."""
        if step_end is None:
            step_end = self.max_steps
        if isinstance(dst, np.ndarray):
            ptr, nbytes = dst.ctypes.data, dst.nbytes
        else:
            ptr = int(dst)
        rc = self.lib.sipnet_gpu_run_to_host(self.handle, step_begin, step_end, C.c_void_p(ptr), nbytes, chunk_steps)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (step_end, step_end)

    def _gather(self, what: int, dtype, shape) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        self.gather_into(what, out)
        return out

    def gather_into(self, what: int, out: np.ndarray) -> None:
        rc = self.lib.sipnet_gpu_gather(self.handle, what, out.ctypes.data_as(C.c_void_p), out.nbytes)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())

    def gather_raw(self, what: int, ptr: int, nbytes: int) -> None:
        rc = self.lib.sipnet_gpu_gather(self.handle, what, C.c_void_p(ptr), nbytes)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())

    @property
    def nrun(self) -> int:
        return self.last_range[1] - self.last_range[0]

    def output(self) -> np.ndarray:
        """[32][n][M] -- outputState() columns for the last run range."""
        return self._gather(A.GATHER_FULL, np.float64, (A.NOUT, self.nrun, self.nmembers))

    def debug(self) -> np.ndarray:
        return self._gather(A.GATHER_DEBUG, np.float64, (A.NDEBUG, self.nrun, self.nmembers))

    def balance(self) -> np.ndarray:
        """[2][n][M]: deltaC, deltaN of the reference's mass-balance check (balance.c:129-148); needs OUT_DEBUG."""
        return self._gather(A.GATHER_BALANCE, np.float64, (A.NBALANCE, self.nrun, self.nmembers))

    def counters(self) -> np.ndarray:
        """[NCOUNTERS][members] uint32: how often the reference would have printed each informational message
        (CNT_* order) since init / reset; validation dump (OUT_DEBUG) only."""
        return self._gather(A.GATHER_COUNTERS, np.uint32, (A.NCOUNTERS, self.nmembers))

    def loglik(self) -> np.ndarray:
        return self._gather(A.GATHER_LOGLIK, np.float64, (self.nmembers,))

    def loglik_n(self) -> np.ndarray:
        return self._gather(A.GATHER_LOGLIK_N, np.float64, (self.nmembers,))

    def status(self) -> np.ndarray:
        return self._gather(A.GATHER_STATUS, np.uint32, (self.nmembers,))

    def state(self) -> np.ndarray:
        return self._gather(A.GATHER_STATE, np.float64, (A.NSTATE, self.nmembers))

    @property
    def ring_slots(self) -> int:
        return int(self.lib.sipnet_gpu_ring_slots(self.handle))

    def ring(self):
        """(values, weights), each [ring_slots][M]: the mean-NPP tracker's arrays (runmean.h)."""
        shape = (self.ring_slots, self.nmembers)
        return (self._gather(A.GATHER_RING_VALUES, np.float64, shape), self._gather(A.GATHER_RING_WEIGHTS, np.float64, shape))

    def set_state(self, state: np.ndarray, ring_values: Optional[np.ndarray] = None,
                  ring_weights: Optional[np.ndarray] = None, next_step: int = 0) -> None:
        """Overwrite the carried state (restartLoadCheckpoint semantics); the next run starts at next_step."""
        state = np.ascontiguousarray(state, dtype=np.float64)
        if state.shape != (A.NSTATE, self.nmembers):
            raise ValueError(f"state must be [{A.NSTATE}][{self.nmembers}]")
        rv = rw = None
        if ring_values is not None:
            rv = np.ascontiguousarray(ring_values, dtype=np.float64)
            rw = np.ascontiguousarray(ring_weights, dtype=np.float64)
            if rv.shape != (self.ring_slots, self.nmembers) or rw.shape != rv.shape:
                raise ValueError(f"rings must be [{self.ring_slots}][{self.nmembers}]")
        rc = self.lib.sipnet_gpu_set_state(self.handle, state.ctypes.data, self.nmembers,
                                           None if rv is None else rv.ctypes.data, None if rw is None else rw.ctypes.data,
                                           self.nmembers, next_step)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())

    def obs_spec(self, rows, op, value, variance):
        """(A.ObsSpec, the arrays it points into, n_obs) for sipnet_gpu_*_assimilate.  rows: pool rows (A.S indices
        0..11); op: [n_obs][n_rows]; value, variance: [nsites][n_obs] (NaN value = not observed)."""
        rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        op = np.ascontiguousarray(op, dtype=np.float64)
        value = np.ascontiguousarray(value, dtype=np.float64)
        variance = np.ascontiguousarray(variance, dtype=np.float64)
        if op.ndim != 2 or op.shape[1] != rows.size:
            raise ValueError(f"op must be [n_obs][{rows.size}]")
        nobs = op.shape[0]
        if value.shape != (self.nsites, nobs) or variance.shape != value.shape:
            raise ValueError(f"value and variance must be [{self.nsites}][{nobs}]")
        spec = A.ObsSpec(rows.size, _ip(rows), nobs, _dp(op), _dp(value), _dp(variance))
        return spec, (rows, op, value, variance), nobs

    def _assimilate(self, fn, target, rows, op, value, variance, *infl) -> np.ndarray:
        spec, _keep, nobs = self.obs_spec(rows, op, value, variance)
        diag = np.empty((self.nsites, nobs, 4), np.float64)
        self._check(fn(target, C.byref(spec), *infl, diag.ctypes.data))
        return diag

    def inflation_spec(self, lam, lam_sd=None, lambda_bounds=(1.0, 100.0), sd_min=0.0):
        """(A.InflationSpec, (lambda, lambda_sd)) for sipnet_gpu_*_assimilate_inflated: lam, lam_sd: [nsites] (lam NaN
        or 1: no inflation; lam_sd None: all fixed, 0: fixed at that site), copied -- the call updates the copies."""
        lam = np.array(np.broadcast_to(lam, (self.nsites,)), dtype=np.float64)
        sd = None if lam_sd is None else np.array(np.broadcast_to(lam_sd, (self.nsites,)), dtype=np.float64)
        lo, hi = lambda_bounds
        spec = A.InflationSpec(_dp(lam), None if sd is None else _dp(sd), float(lo), float(hi), float(sd_min))
        return spec, (lam, sd)

    def _assimilate_inflated(self, fn, target, rows, op, value, variance, lam, lam_sd, lambda_bounds, sd_min):
        spec, (lam, sd) = self.inflation_spec(lam, lam_sd, lambda_bounds, sd_min)
        diag = self._assimilate(fn, target, rows, op, value, variance, C.byref(spec))
        return diag, lam, sd

    def assimilate(self, rows, op, value, variance) -> np.ndarray:
        """Ensemble adjustment Kalman filter on the carried pools (sipnet_gpu_assimilate; see include/sipnet_gpu.h).
        Returns diag [nsites][n_obs][4] = (N, prior mean of y, its sample variance, analysis mean)."""
        return self._assimilate(self.lib.sipnet_gpu_assimilate, self.handle, rows, op, value, variance)

    def team_assimilate(self, rows, op, value, variance) -> np.ndarray:
        """Collective.  assimilate() over the members of every rank of the team (same arguments on every rank)."""
        return self._assimilate(self.lib.sipnet_gpu_comm_assimilate, self.comm, rows, op, value, variance)

    def assimilate_inflated(self, rows, op, value, variance, lam, lam_sd=None, lambda_bounds=(1.0, 100.0), sd_min=0.0):
        """assimilate() after a per-site prior inflation by lam, fixed or adaptive (sipnet_gpu_assimilate_inflated;
        see include/sipnet_gpu.h).  Returns (diag, the updated lam, the updated lam_sd or None); the inputs are not
        modified."""
        return self._assimilate_inflated(self.lib.sipnet_gpu_assimilate_inflated, self.handle, rows, op, value,
                                         variance, lam, lam_sd, lambda_bounds, sd_min)

    def team_assimilate_inflated(self, rows, op, value, variance, lam, lam_sd=None, lambda_bounds=(1.0, 100.0),
                                 sd_min=0.0):
        """Collective.  assimilate_inflated() over the members of every rank (same arguments on every rank)."""
        return self._assimilate_inflated(self.lib.sipnet_gpu_comm_assimilate_inflated, self.comm, rows, op, value,
                                         variance, lam, lam_sd, lambda_bounds, sd_min)

    def _resample(self, fn, target, nmembers, u, ess_fraction, log_weights):
        u = np.ascontiguousarray(u, dtype=np.float64).reshape(-1)
        if u.size != self.nsites:
            raise ValueError(f"u must hold one value per site ({self.nsites})")
        lw = None
        if log_weights is not None:
            lw = np.ascontiguousarray(log_weights, dtype=np.float64).reshape(-1)
            if lw.size != self.nmembers:
                raise ValueError(f"log_weights must hold one value per member ({self.nmembers})")
        ancestors = np.empty(nmembers, np.int64)
        diag = np.empty((self.nsites, 4), np.float64)
        self._check(fn(target, u.ctypes.data, float(ess_fraction), None if lw is None else lw.ctypes.data,
                       ancestors.ctypes.data, diag.ctypes.data))
        return ancestors, diag

    def resample(self, u, ess_fraction: float = math.inf, log_weights=None):
        """Per-site systematic resampling of the members (sipnet_gpu_resample; see include/sipnet_gpu.h).  u: one
        value in [0, 1) per site (NaN: leave the site alone); log_weights: [nmembers], or None for the handle's
        log-likelihood.  Returns (ancestors [nmembers], -1 where a site was not resampled; diag [nsites][4] =
        (N, ESS, incremental log-evidence, distinct ancestors))."""
        return self._resample(self.lib.sipnet_gpu_resample, self.handle, self.nmembers, u, ess_fraction, log_weights)

    def team_resample(self, u, ess_fraction: float = math.inf, log_weights=None):
        """Collective.  resample() over the members of every rank (same u and ess_fraction on every rank;
        log_weights: this rank's members).  ancestors cover the whole team, rank-major."""
        n = int(self.team_member_counts().sum())
        return self._resample(self.lib.sipnet_gpu_comm_resample, self.comm, n, u, ess_fraction, log_weights)

    def params(self) -> np.ndarray:
        """[80][M]: the device's parameter rows, in device units (after setupModel(); see GATHER_PARAMS)."""
        return self._gather(A.GATHER_PARAMS, np.float64, (A.NPARAMS, self.nmembers))

    def jitter_spec(self, rows, transform, shrink, z, lower=None, upper=None):
        """(A.JitterSpec, the arrays it points into) for sipnet_gpu_*_rejuvenate.  rows: A.P indices; transform:
        A.TF_* per row; shrink: [nsites] (NaN = leave the site alone); z: [n_rows][nmembers]; lower / upper: the
        bounds of LOGIT rows (other entries are not read)."""
        rows = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
        tf = np.ascontiguousarray(np.broadcast_to(transform, rows.shape), dtype=np.int32)
        shrink = np.ascontiguousarray(np.broadcast_to(shrink, (self.nsites,)), dtype=np.float64)
        z = np.ascontiguousarray(z, dtype=np.float64)
        if z.shape != (rows.size, self.nmembers):
            raise ValueError(f"z must be [{rows.size}][{self.nmembers}]")
        lo = None if lower is None else np.ascontiguousarray(np.broadcast_to(lower, rows.shape), dtype=np.float64)
        hi = None if upper is None else np.ascontiguousarray(np.broadcast_to(upper, rows.shape), dtype=np.float64)
        spec = A.JitterSpec(rows.size, _ip(rows), _ip(tf), None if lo is None else _dp(lo), None if hi is None else _dp(hi),
                            _dp(shrink), _dp(z))
        return spec, (rows, tf, lo, hi, shrink, z)

    def _rejuvenate(self, fn, target, rows, transform, shrink, z, lower, upper) -> np.ndarray:
        spec, _keep = self.jitter_spec(rows, transform, shrink, z, lower, upper)
        diag = np.empty((self.nsites, 4), np.float64)
        self._check(fn(target, C.byref(spec), diag.ctypes.data))
        return diag

    def rejuvenate(self, rows, transform, shrink, z, lower=None, upper=None) -> np.ndarray:
        """Liu-West kernel-shrinkage move of the listed parameter rows, per site (sipnet_gpu_rejuvenate; see
        include/sipnet_gpu.h).  Returns diag [nsites][4] = (N, rank (-1: site left alone), moved, kept)."""
        return self._rejuvenate(self.lib.sipnet_gpu_rejuvenate, self.handle, rows, transform, shrink, z, lower, upper)

    def team_rejuvenate(self, rows, transform, shrink, z, lower=None, upper=None) -> np.ndarray:
        """Collective.  rejuvenate() over the members of every rank (same arguments on every rank except z, which
        holds this rank's members)."""
        return self._rejuvenate(self.lib.sipnet_gpu_comm_rejuvenate, self.comm, rows, transform, shrink, z, lower, upper)

    def mean(self) -> np.ndarray:
        return self._gather(A.GATHER_MEAN, np.float64, (self.nsites, self.n_summary_cols, self.nrun))

    def variance(self) -> np.ndarray:
        return self._gather(A.GATHER_VARIANCE, np.float64, (self.nsites, self.n_summary_cols, self.nrun))

    def quantiles(self) -> np.ndarray:
        return self._gather(A.GATHER_QUANTILES, np.float64,
                            (self.nsites, self.n_summary_cols, self.n_quantiles, self.nrun))

    def event_counts(self) -> np.ndarray:
        return self._gather(A.GATHER_EVENT_COUNTS, np.int32, (self.nmembers,))

    def event_records(self):
        n = self.nmembers * self.max_event_records
        buf = (A.EventRecord * n)()
        rc = self.lib.sipnet_gpu_gather(self.handle, A.GATHER_EVENT_RECORDS, C.cast(buf, C.c_void_p),
                                        C.sizeof(buf))
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        counts = self.event_counts()
        return [[buf[m * self.max_event_records + i] for i in range(min(int(counts[m]), self.max_event_records))]
                for m in range(self.nmembers)]

    def sync(self) -> None:
        self.lib.sipnet_gpu_sync(self.handle)

    def reset(self) -> None:
        rc = self.lib.sipnet_gpu_reset(self.handle)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (0, 0)

    def set_params(self, params, ld: Optional[int] = None) -> None:
        """Upload a new [80][M] ensemble (numpy array or raw host pointer) and reset."""
        if isinstance(params, np.ndarray):
            params = np.ascontiguousarray(params, dtype=np.float64)
            ptr, ld = params.ctypes.data, params.shape[1]
        else:
            ptr = int(params)
        rc = self.lib.sipnet_gpu_set_params(self.handle, C.c_void_p(ptr), ld)
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (0, 0)

    def timer_start(self) -> None:
        self.lib.sipnet_gpu_timer_start(self.handle)

    def timer_stop_ms(self) -> float:
        ms = C.c_float()
        rc = self.lib.sipnet_gpu_timer_stop_ms(self.handle, C.byref(ms))
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        return float(ms.value)

    def last_run_ms(self) -> float:
        ms = C.c_float()
        self.lib.sipnet_gpu_last_run_ms(self.handle, C.byref(ms))
        return float(ms.value)

    def launch_count(self) -> int:
        return int(self.lib.sipnet_gpu_launch_count(self.handle))

    def device_ptr(self, what: int) -> int:
        return int(self.lib.sipnet_gpu_device_ptr(self.handle, what) or 0)

    # -- multi-GPU, one process per GPU (sipnet_gpu_comm_*): this handle holds ITS members of every site
    def _check(self, rc: int) -> None:
        if rc != 0:
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())

    def join_team(self, nranks: int = 1, rank: int = 0, comm_id: Optional[bytes] = None) -> None:
        """Collective.  comm_id: the 128 bytes of unique_comm_id() made on rank 0 and broadcast by the launcher."""
        self.comm = C.c_void_p()
        buf = C.create_string_buffer(comm_id, A.COMM_ID_BYTES) if comm_id is not None else None
        self._check(self.lib.sipnet_gpu_comm_init_rank(self.handle, nranks, rank, buf, C.byref(self.comm)))
        self.team_size = nranks

    def team_summaries(self) -> None:
        """Collective.  Afterwards mean() / variance() / quantiles() return the whole team's result."""
        self._check(self.lib.sipnet_gpu_comm_summaries(self.comm))

    def team_last_levels(self) -> int:
        return int(self.lib.sipnet_gpu_comm_last_levels(self.comm))

    def team_member_counts(self) -> np.ndarray:
        counts = np.zeros(self.team_size, np.int64)
        self._check(self.lib.sipnet_gpu_comm_member_counts(self.comm, counts.ctypes.data))
        return counts

    def team_loglik(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Collective.  Log-likelihoods of all ranks' members, rank-major."""
        if out is None:
            out = np.empty(int(self.team_member_counts().sum()), np.float64)
        self._check(self.lib.sipnet_gpu_comm_gather_loglik(self.comm, out.ctypes.data, out.nbytes))
        return out

    def close(self) -> None:
        if getattr(self, "comm", None):
            self.lib.sipnet_gpu_comm_destroy(self.comm)
            self.comm = None
        if self.handle:
            self.lib.sipnet_gpu_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def unique_comm_id(lib: Optional[C.CDLL] = None) -> bytes:
    """sipnet_gpu_comm_unique_id: made on rank 0, broadcast to the other ranks by the caller's launcher."""
    lib = lib or load_library()
    buf = C.create_string_buffer(A.COMM_ID_BYTES)
    rc = lib.sipnet_gpu_comm_unique_id(buf)
    if rc != 0:
        raise SipnetGpuError(rc, (lib.sipnet_gpu_last_error() or b"").decode())
    return buf.raw


class MultiEnsemble(Ensemble):
    """One process, several GPUs (sipnet_gpu_multi_*): the single-GPU configuration, partitioned by the library.
    gather-style accessors return exactly what one GPU would."""

    def __init__(self, sites: Sequence[SiteData], params: np.ndarray, member_site: Optional[np.ndarray] = None,
                 flags: Optional[dict] = None, outputs: int = A.OUT_FULL, math: int = A.MATH_VALIDATION,
                 devices: Optional[Sequence[int]] = None, out_steps_capacity: int = 0,
                 summary_cols: Sequence[int] = (), quantiles: Sequence[float] = (), nee_sigma: float = 1.0,
                 max_event_records: int = 0, block_threads: int = 0, ring_slots: int = 0, lib: Optional[C.CDLL] = None):
        self.lib = lib or load_library()
        self.handle = None
        cfg = self._configure(sites, params, member_site, flags, outputs, math, 0, out_steps_capacity, summary_cols,
                              quantiles, nee_sigma, max_event_records, block_threads, 0, ring_slots)
        devs = np.ascontiguousarray(devices if devices is not None else [], dtype=np.int32)
        self.multi = C.c_void_p()
        rc = self.lib.sipnet_gpu_multi_init(C.byref(cfg), int(devs.size), devs.ctypes.data if devs.size else None,
                                            C.byref(self.multi))
        if rc != 0:
            self.multi = None
            raise SipnetGpuError(rc, (self.lib.sipnet_gpu_last_error() or b"").decode())
        self.last_range = (0, 0)
        self._ring_slots = int(self.lib.sipnet_gpu_ring_slots(self.lib.sipnet_gpu_multi_handle(self.multi, 0)))

    @property
    def ndevices(self) -> int:
        return int(self.lib.sipnet_gpu_multi_ndevices(self.multi))

    @property
    def ring_slots(self) -> int:
        return self._ring_slots

    def run(self, step_begin: int = 0, step_end: Optional[int] = None) -> None:
        if step_end is None:
            step_end = self.max_steps
        self._check(self.lib.sipnet_gpu_multi_run(self.multi, step_begin, step_end))
        self.last_range = (step_begin, step_end)

    def gather_into(self, what: int, out: np.ndarray) -> None:
        self._check(self.lib.sipnet_gpu_multi_gather(self.multi, what, out.ctypes.data_as(C.c_void_p), out.nbytes))

    def event_records(self):
        n = self.nmembers * self.max_event_records
        buf = (A.EventRecord * n)()
        self._check(self.lib.sipnet_gpu_multi_gather(self.multi, A.GATHER_EVENT_RECORDS, C.cast(buf, C.c_void_p), C.sizeof(buf)))
        counts = self.event_counts()
        return [[buf[m * self.max_event_records + i] for i in range(min(int(counts[m]), self.max_event_records))]
                for m in range(self.nmembers)]

    def assimilate(self, rows, op, value, variance) -> np.ndarray:
        return self._assimilate(self.lib.sipnet_gpu_multi_assimilate, self.multi, rows, op, value, variance)

    def assimilate_inflated(self, rows, op, value, variance, lam, lam_sd=None, lambda_bounds=(1.0, 100.0), sd_min=0.0):
        return self._assimilate_inflated(self.lib.sipnet_gpu_multi_assimilate_inflated, self.multi, rows, op, value,
                                         variance, lam, lam_sd, lambda_bounds, sd_min)

    def resample(self, u, ess_fraction: float = math.inf, log_weights=None):
        return self._resample(self.lib.sipnet_gpu_multi_resample, self.multi, self.nmembers, u, ess_fraction, log_weights)

    def rejuvenate(self, rows, transform, shrink, z, lower=None, upper=None) -> np.ndarray:
        return self._rejuvenate(self.lib.sipnet_gpu_multi_rejuvenate, self.multi, rows, transform, shrink, z, lower, upper)

    def sync(self) -> None:
        self.lib.sipnet_gpu_multi_sync(self.multi)

    def reset(self) -> None:
        self._check(self.lib.sipnet_gpu_multi_reset(self.multi))
        self.last_range = (0, 0)

    def close(self) -> None:
        if getattr(self, "multi", None):
            self.lib.sipnet_gpu_multi_destroy(self.multi)
            self.multi = None
