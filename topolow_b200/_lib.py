"""ctypes binding of libtopolow_b200.so (the C ABI in include/topolow_b200.h).

There is no CPU fallback: if the shared library is missing this module raises at import of
the first symbol, and every compute entry point returns TOPOLOW_ERR_CUDA without a device.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TOPOLOW_B200_LIB") or os.path.join(_HERE, "lib", "libtopolow_b200.so")

OK, ERR_BAD_ARG, ERR_NONFINITE, ERR_CUDA, ERR_TOO_FEW_POINTS, ERR_INTERRUPTED = range(6)
MODE_COLOURED, MODE_REPLAY, MODE_ROWBLOCK = 0, 1, 2
PREC_F32, PREC_F64_EXACT = 0, 1

_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)


class Problem(C.Structure):
    _fields_ = [("n", C.c_int64), ("ndim", C.c_int32), ("n_edges", C.c_int64), ("edge_i", _i32p),
                ("edge_j", _i32p), ("edge_dist", _dp), ("edge_thresh", _i32p), ("degrees", _i32p),
                ("initial_positions", _dp), ("n_holdout", C.c_int64), ("holdout_i", _i32p), ("holdout_j", _i32p),
                ("holdout_truth", _dp)]


class Params(C.Structure):
    _fields_ = [("n_iter", C.c_int32), ("k0", C.c_double), ("cooling_rate", C.c_double),
                ("c_repulsion", C.c_double), ("relative_epsilon", C.c_double),
                ("convergence_window", C.c_int32), ("convergence_check_freq", C.c_int32),
                ("verbose", C.c_int32), ("mode", C.c_int32), ("precision", C.c_int32), ("seed", C.c_uint64),
                ("pair_order", _i32p), ("pairs_per_iter", C.c_int64), ("device", C.c_int32),
                ("max_ctas", C.c_int32), ("max_warps", C.c_int32), ("tile_points", C.c_int32),
                ("n_shards", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("positions", _dp), ("converged", C.c_int32), ("iterations", C.c_int32),
                ("final_mae", C.c_double), ("final_k", C.c_double), ("status", C.c_int32),
                ("fail_iter", C.c_int32), ("iterations_run", C.c_int32), ("pair_updates", C.c_int64),
                ("device_ms", C.c_double), ("trace_mae", _dp), ("holdout_sum_abs", C.c_double),
                ("holdout_count", C.c_int64), ("message", C.c_char * 256)]


INTERRUPT_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)

EXPORTS = [
    "topolow_fit", "topolow_fit_interruptible", "topolow_optimize_layout_exact", "topolow_fit_batch",
    "topolow_fit_batch_interruptible", "topolow_fit_batch_devices",
    "topolow_plan_create", "topolow_plan_run", "topolow_plan_result", "topolow_plan_info",
    "topolow_plan_destroy", "topolow_plan_enumerate", "topolow_schedule_enumerate", "topolow_plan_run_job",
    "topolow_plan_end_iteration", "topolow_plan_layout", "topolow_plan_positions", "topolow_plan_enumerate_job",
    "topolow_est_distances", "topolow_holdout_errors", "topolow_components", "topolow_microbench", "topolow_device_info",
    "topolow_version", "topolow_abi_sizes",
    "topolow_shard_create", "topolow_shard_handle_bytes", "topolow_shard_export", "topolow_shard_attach",
    "topolow_shard_attach_local", "topolow_shard_run", "topolow_shard_run_local", "topolow_shard_time_kernels",
    "topolow_shard_result", "topolow_shard_info", "topolow_shard_slot_order", "topolow_shard_destroy",
]

_lib = None


class TopolowLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load the CUDA library (built by __graft_entry__.build() / make -C topolow_b200/csrc)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TopolowLibraryMissing(
            f"{LIB_PATH} is missing: build it with `make -C topolow_b200/csrc` (nvcc, sm_100a). "
            "topolow_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.topolow_fit.restype = C.c_int
    L.topolow_fit.argtypes = [C.POINTER(Problem), C.POINTER(Params), C.POINTER(Result)]
    L.topolow_fit_interruptible.restype = C.c_int
    L.topolow_fit_interruptible.argtypes = [C.POINTER(Problem), C.POINTER(Params), C.POINTER(Result),
                                            INTERRUPT_FN, C.c_void_p]
    L.topolow_optimize_layout_exact.restype = C.c_int
    L.topolow_optimize_layout_exact.argtypes = [
        _dp, C.c_int32, C.c_int32, _dp, _i32p, _i32p, _i32p, _i32p, _dp, _i32p, C.c_int64, C.c_int32,
        C.c_double, C.c_double, C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_int32, _dp, _i32p, _i32p,
        _dp, _dp, C.c_char_p, C.c_int32]
    L.topolow_fit_batch.restype = C.c_int
    L.topolow_fit_batch.argtypes = [C.c_int32, C.POINTER(Problem), C.POINTER(Params), C.POINTER(Result), C.c_int32]
    L.topolow_fit_batch_interruptible.restype = C.c_int
    L.topolow_fit_batch_interruptible.argtypes = [C.c_int32, C.POINTER(Problem), C.POINTER(Params), C.POINTER(Result),
                                                  C.c_int32, INTERRUPT_FN, C.c_void_p]
    L.topolow_fit_batch_devices.restype = C.c_int
    L.topolow_fit_batch_devices.argtypes = [C.c_int32, C.POINTER(Problem), C.POINTER(Params), C.POINTER(Result), _i32p,
                                            C.c_int32, INTERRUPT_FN, C.c_void_p]
    L.topolow_plan_create.restype = C.c_int
    L.topolow_plan_create.argtypes = [C.POINTER(Problem), C.POINTER(Params), C.POINTER(C.c_void_p), C.c_char_p,
                                      C.c_int32]
    L.topolow_plan_run.restype = C.c_int
    L.topolow_plan_run.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, _dp]
    L.topolow_plan_result.restype = C.c_int
    L.topolow_plan_result.argtypes = [C.c_void_p, C.POINTER(Result)]
    L.topolow_plan_info.restype = C.c_int
    L.topolow_plan_info.argtypes = [C.c_void_p, _i64p, C.c_int32]
    L.topolow_plan_destroy.restype = None
    L.topolow_plan_destroy.argtypes = [C.c_void_p]
    L.topolow_plan_enumerate.restype = C.c_int64
    L.topolow_plan_enumerate.argtypes = [C.c_void_p, C.c_int32, _i32p, C.c_int64]
    L.topolow_schedule_enumerate.restype = C.c_int64
    L.topolow_schedule_enumerate.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                             C.c_int32, _i32p, C.c_int64, _i64p, C.c_int32]
    L.topolow_plan_run_job.restype = C.c_int
    L.topolow_plan_run_job.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.topolow_plan_end_iteration.restype = C.c_int
    L.topolow_plan_end_iteration.argtypes = [C.c_void_p, C.c_void_p]
    L.topolow_plan_layout.restype = C.c_int
    L.topolow_plan_layout.argtypes = [C.c_void_p, _i64p, C.c_int32]
    L.topolow_plan_positions.restype = C.c_void_p
    L.topolow_plan_positions.argtypes = [C.c_void_p]
    L.topolow_plan_enumerate_job.restype = C.c_int64
    L.topolow_plan_enumerate_job.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                             _i32p, C.c_int64]
    L.topolow_est_distances.restype = C.c_int
    L.topolow_est_distances.argtypes = [_dp, C.c_int64, C.c_int32, _dp, C.c_int32]
    L.topolow_components.restype = C.c_int
    L.topolow_components.argtypes = [C.c_int64, C.c_int64, _i32p, _i32p, C.c_int32, C.POINTER(C.c_uint8), _i64p, _i64p, _i64p,
                                     C.c_int32]
    L.topolow_holdout_errors.restype = C.c_int
    L.topolow_holdout_errors.argtypes = [_dp, C.c_int64, C.c_int32, C.c_int64, _i32p, _i32p, _dp, _dp, _i64p,
                                         C.c_int32]
    L.topolow_microbench.restype = C.c_int
    L.topolow_microbench.argtypes = [C.c_int32, C.c_int32, _dp]
    L.topolow_device_info.restype = C.c_int
    L.topolow_device_info.argtypes = [C.c_int32, _i32p, _i32p, _i32p, _i64p]
    L.topolow_version.restype = C.c_char_p
    L.topolow_version.argtypes = []
    L.topolow_abi_sizes.restype = None
    L.topolow_abi_sizes.argtypes = [C.POINTER(C.c_int64 * 3)]
    L.topolow_shard_create.restype = C.c_int
    L.topolow_shard_create.argtypes = [C.POINTER(Problem), C.POINTER(Params), C.c_int32, C.c_int32,
                                       C.POINTER(C.c_void_p), C.c_char_p, C.c_int32]
    L.topolow_shard_handle_bytes.restype = C.c_int64
    L.topolow_shard_handle_bytes.argtypes = []
    L.topolow_shard_export.restype = C.c_int
    L.topolow_shard_export.argtypes = [C.c_void_p, C.c_void_p]
    L.topolow_shard_attach.restype = C.c_int
    L.topolow_shard_attach.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_char_p, C.c_int32]
    L.topolow_shard_attach_local.restype = C.c_int
    L.topolow_shard_attach_local.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_char_p, C.c_int32]
    L.topolow_shard_run.restype = C.c_int
    L.topolow_shard_run.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, _dp]
    L.topolow_shard_run_local.restype = C.c_int
    L.topolow_shard_run_local.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, _dp]
    L.topolow_shard_time_kernels.restype = C.c_int
    L.topolow_shard_time_kernels.argtypes = [C.c_void_p, C.c_int32, _dp, C.c_int32]
    L.topolow_shard_result.restype = C.c_int
    L.topolow_shard_result.argtypes = [C.c_void_p, C.POINTER(Result)]
    L.topolow_shard_info.restype = C.c_int
    L.topolow_shard_info.argtypes = [C.c_void_p, _i64p, C.c_int32]
    L.topolow_shard_slot_order.restype = C.c_int
    L.topolow_shard_slot_order.argtypes = [C.c_int64, _i32p]
    L.topolow_shard_destroy.restype = None
    L.topolow_shard_destroy.argtypes = [C.c_void_p]
    sizes = (C.c_int64 * 3)()
    L.topolow_abi_sizes(C.byref(sizes))
    if list(sizes) != [C.sizeof(Problem), C.sizeof(Params), C.sizeof(Result)]:
        raise ImportError(f"libtopolow_b200 struct sizes {list(sizes)} differ from the ctypes declarations "
                          f"{[C.sizeof(Problem), C.sizeof(Params), C.sizeof(Result)]}: rebuild the library")
    _lib = L
    return L


class TopolowError(RuntimeError):
    """A non-zero status from the C ABI; `.status` is the TOPOLOW_* code."""

    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


class ProblemArrays:
    """Owns the numpy buffers a `Problem` struct points into."""

    def __init__(self, initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, holdout=None):
        init = np.asarray(initial_positions, dtype=np.float64)
        if init.ndim != 2:
            raise ValueError("initial_positions must be a matrix")
        self.n, self.ndim = init.shape
        self.init = np.asfortranarray(init)  # column-major like an R matrix
        self.degrees = np.ascontiguousarray(degrees, dtype=np.int32)
        self.edge_i = np.ascontiguousarray(edge_i, dtype=np.int32)
        self.edge_j = np.ascontiguousarray(edge_j, dtype=np.int32)
        self.edge_dist = np.ascontiguousarray(edge_dist, dtype=np.float64)
        self.edge_thresh = np.ascontiguousarray(edge_thresh, dtype=np.int32)
        if len(self.degrees) != self.n:
            raise ValueError("degrees must have one entry per point")
        if not (len(self.edge_i) == len(self.edge_j) == len(self.edge_dist) == len(self.edge_thresh)):
            raise ValueError("edge arrays must have equal length")
        self.struct = Problem(self.n, self.ndim, len(self.edge_i), self.edge_i.ctypes.data_as(_i32p),
                              self.edge_j.ctypes.data_as(_i32p), self.edge_dist.ctypes.data_as(_dp),
                              self.edge_thresh.ctypes.data_as(_i32p), self.degrees.ctypes.data_as(_i32p),
                              self.init.ctypes.data_as(_dp), 0, None, None, None)
        if holdout is not None:   # (cell_i, cell_j, truth): scored on the final positions inside the call
            self.hold_i = np.ascontiguousarray(holdout[0], dtype=np.int32)
            self.hold_j = np.ascontiguousarray(holdout[1], dtype=np.int32)
            self.hold_t = np.ascontiguousarray(holdout[2], dtype=np.float64)
            if not (len(self.hold_i) == len(self.hold_j) == len(self.hold_t)):
                raise ValueError("hold-out arrays must have equal length")
            self.struct.n_holdout = len(self.hold_i)
            self.struct.holdout_i = self.hold_i.ctypes.data_as(_i32p)
            self.struct.holdout_j = self.hold_j.ctypes.data_as(_i32p)
            self.struct.holdout_truth = self.hold_t.ctypes.data_as(_dp)


def make_params(n_iter, k0, cooling_rate, c_repulsion, relative_epsilon=1e-4, convergence_window=5,
                convergence_check_freq=3, verbose=False, mode=MODE_COLOURED, precision=PREC_F32, seed=0,
                pair_order=None, device=0, max_ctas=0, max_warps=0, tile_points=0, n_shards=0):
    p = Params()
    p.n_iter = int(n_iter)
    p.k0, p.cooling_rate, p.c_repulsion = float(k0), float(cooling_rate), float(c_repulsion)
    p.relative_epsilon = float(relative_epsilon)
    p.convergence_window, p.convergence_check_freq = int(convergence_window), int(convergence_check_freq)
    p.verbose, p.mode, p.precision = int(bool(verbose)), int(mode), int(precision)
    p.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    keep = None
    if pair_order is not None:
        keep = np.ascontiguousarray(pair_order, dtype=np.int32)
        if keep.ndim != 3 or keep.shape[2] != 2 or keep.shape[0] < n_iter:
            raise ValueError("pair_order must be [n_iter][pairs][2]")
        p.pair_order = keep.ctypes.data_as(_i32p)
        p.pairs_per_iter = keep.shape[1]
    p.device, p.max_ctas, p.max_warps = int(device), int(max_ctas), int(max_warps)
    p.tile_points = int(tile_points)
    p.n_shards = int(n_shards)
    return p, keep


def result_dict(res: Result, positions, trace=None):
    out = dict(converged=bool(res.converged),
               iterations=int(res.iterations), final_mae=float(res.final_mae), final_k=float(res.final_k),
               iterations_run=int(res.iterations_run), pair_updates=int(res.pair_updates),
               device_ms=float(res.device_ms), status=int(res.status),
               holdout_sum_abs=float(res.holdout_sum_abs), holdout_count=int(res.holdout_count))
    if positions is not None:
        out["positions"] = np.ascontiguousarray(positions)
    if trace is not None:
        out["trace_mae"] = trace
    return out


def fit(initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, n_iter, k0, cooling_rate,
        c_repulsion, relative_epsilon=1e-4, convergence_window=5, convergence_check_freq=3, *, verbose=False,
        mode=MODE_COLOURED, precision=PREC_F32, seed=0, pair_order=None, device=0, max_ctas=0, max_warps=0,
        tile_points=0, trace=False, interrupt=None, holdout=None):
    """One call of the native optimiser (the .Call boundary of R/core.R:439-456) on host buffers.
    holdout = (cell_i, cell_j, truth): also return sum |truth - distance| and the count over those cells."""
    L = lib()
    pa = ProblemArrays(initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, holdout)
    pr, _keep = make_params(n_iter, k0, cooling_rate, c_repulsion, relative_epsilon, convergence_window,
                            convergence_check_freq, verbose, mode, precision, seed, pair_order, device, max_ctas, max_warps,
                            tile_points)
    out = np.empty((pa.n, pa.ndim), dtype=np.float64, order="F")
    res = Result()
    res.positions = out.ctypes.data_as(_dp)
    tr = None
    if trace:
        tr = np.full(max(int(n_iter), 1), np.nan)
        res.trace_mae = tr.ctypes.data_as(_dp)
    if interrupt is None:
        rc = L.topolow_fit(C.byref(pa.struct), C.byref(pr), C.byref(res))
    else:
        cb = INTERRUPT_FN(lambda _u: int(bool(interrupt())))
        rc = L.topolow_fit_interruptible(C.byref(pa.struct), C.byref(pr), C.byref(res), cb, None)
    if rc != OK:
        raise TopolowError(rc, res.message.decode() or f"topolow_fit failed with status {rc}")
    return result_dict(res, out, tr)


def fit_batch(jobs, device=0, interrupt=None, keep_positions=True):
    """jobs: list of dicts with the keyword arguments of `fit`; `mode` is MODE_COLOURED (the default) or MODE_ROWBLOCK
    (large maps and ndim 17..32: each such job is exactly `fit(..., mode=MODE_ROWBLOCK)`), and `trace=True` adds
    'trace_mae'.  Returns a list of result dicts; a failed job yields {'status': code, 'message': ...} instead of raising
    (R/adaptive_sampling.R:2657-2666 turns fit errors into NA rows).

    keep_positions=False: the positions do not come back (a CV grid needs only the hold-out sums, which are the same
    either way) and the result dicts have no 'positions'.

    device: a CUDA ordinal, or a sequence of ordinals (topolow_fit_batch_devices): the jobs are dealt over the
    devices of the list, one host thread each, and every result is bit for bit what the batch returns on the first
    device of the list.  An ordinal may repeat.

    interrupt: a callable polled while the batch runs (topolow_fit_batch_interruptible); when it returns True the
    fits stop and TopolowError(ERR_INTERRUPTED) is raised with the per-job list attached as `.results`.  There a job
    that was stopped is a full result dict with status ERR_INTERRUPTED and a 'message' (its best state as of its last
    completed iteration); jobs that had already ended are what the uninterrupted call returns."""
    L = lib()
    devices = None
    if not isinstance(device, (int, np.integer)):
        devices = np.ascontiguousarray([int(d) for d in device], dtype=np.int32)
        device = int(devices[0]) if len(devices) else 0     # Params.device (ignored by the batch) stays an int
    n = len(jobs)
    probs, pars, ress = (Problem * n)(), (Params * n)(), (Result * n)()
    keep, outs, traces = [], [], []
    for j, job in enumerate(jobs):
        job = dict(job)
        pa = ProblemArrays(job.pop("initial_positions"), job.pop("degrees"), job.pop("edge_i"), job.pop("edge_j"),
                           job.pop("edge_dist"), job.pop("edge_thresh"), job.pop("holdout", None))
        tr = np.full(max(int(job["n_iter"]), 1), np.nan) if job.pop("trace", False) else None
        pr, k2 = make_params(job.pop("n_iter"), job.pop("k0"), job.pop("cooling_rate"), job.pop("c_repulsion"),
                             device=device, **job)
        out = np.empty((pa.n, pa.ndim), dtype=np.float64, order="F") if keep_positions else None
        probs[j], pars[j] = pa.struct, pr
        if out is not None:
            ress[j].positions = out.ctypes.data_as(_dp)
        if tr is not None:
            ress[j].trace_mae = tr.ctypes.data_as(_dp)
        keep.append((pa, k2))
        outs.append(out)
        traces.append(tr)
    cb = INTERRUPT_FN() if interrupt is None else INTERRUPT_FN(lambda _u: int(bool(interrupt())))   # (null: no poll)
    if devices is not None:
        rc = L.topolow_fit_batch_devices(n, probs, pars, ress, devices.ctypes.data_as(_i32p), len(devices), cb, None)
        if rc not in (OK, ERR_INTERRUPTED):
            why = ress[0].message.decode() if n else ""
            raise TopolowError(rc, why or f"topolow_fit_batch_devices failed with status {rc}")
    elif interrupt is None:
        rc = L.topolow_fit_batch(n, probs, pars, ress, device)
    else:
        rc = L.topolow_fit_batch_interruptible(n, probs, pars, ress, device, cb, None)
    if rc not in (OK, ERR_INTERRUPTED):
        raise TopolowError(rc, f"topolow_fit_batch failed with status {rc}")
    results = []
    for j in range(n):
        if ress[j].status == ERR_INTERRUPTED:
            results.append(dict(result_dict(ress[j], outs[j], traces[j]), message=ress[j].message.decode()))
        elif ress[j].status != OK:
            results.append(dict(status=int(ress[j].status), message=ress[j].message.decode()))
        else:
            results.append(result_dict(ress[j], outs[j], traces[j]))
    if rc == ERR_INTERRUPTED:
        err = TopolowError(rc, "interrupted")
        err.results = results
        raise err
    return results


class Plan:
    """Device-resident fit (topolow_plan_*): inputs live in HBM, iterations are stepped by the caller."""

    def __init__(self, initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, n_iter, k0,
                 cooling_rate, c_repulsion, relative_epsilon=1e-4, convergence_window=5,
                 convergence_check_freq=3, *, precision=PREC_F32, seed=0, device=0, max_ctas=0, max_warps=0,
                 tile_points=0, n_shards=0):
        self._L = lib()
        self._pa = ProblemArrays(initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh)
        pr, _ = make_params(n_iter, k0, cooling_rate, c_repulsion, relative_epsilon, convergence_window,
                            convergence_check_freq, False, MODE_COLOURED, precision, seed, None, device, max_ctas, max_warps,
                            tile_points, n_shards)
        self.n_iter = int(n_iter)
        self._h = C.c_void_p()
        msg = C.create_string_buffer(256)
        rc = self._L.topolow_plan_create(C.byref(self._pa.struct), C.byref(pr), C.byref(self._h), msg, 256)
        if rc != OK:
            raise TopolowError(rc, msg.value.decode() or f"topolow_plan_create failed with status {rc}")

    def run(self, n_iters, stream=None) -> float:
        ms = C.c_double(0)
        rc = self._L.topolow_plan_run(self._h, int(n_iters), C.c_void_p(stream) if stream else None, C.byref(ms))
        if rc != OK:
            raise TopolowError(rc, f"topolow_plan_run failed with status {rc}")
        return ms.value

    def result(self, trace=False):
        out = np.empty((self._pa.n, self._pa.ndim), dtype=np.float64, order="F")
        res = Result()
        res.positions = out.ctypes.data_as(_dp)
        tr = None
        if trace:
            tr = np.full(max(self.n_iter, 1), np.nan)
            res.trace_mae = tr.ctypes.data_as(_dp)
        rc = self._L.topolow_plan_result(self._h, C.byref(res))
        if rc != OK:
            raise TopolowError(rc, res.message.decode())
        return result_dict(res, out, tr)

    def info(self):
        v = (C.c_int64 * 13)()
        self._L.topolow_plan_info(self._h, v, 13)
        keys = ["tiles", "super_blocks", "warps_per_cta", "ctas", "tasks_per_cta", "rounds", "pairs_per_iter",
                "smem_bytes", "iters_per_launch", "launches", "tile_points", "iterations_done", "stopped"]
        return dict(zip(keys, [int(x) for x in v]))

    def enumerate(self, it):
        P = self._pa.n * (self._pa.n - 1) // 2
        out = np.empty((P, 2), dtype=np.int32)
        got = self._L.topolow_plan_enumerate(self._h, int(it), out.ctypes.data_as(_i32p), P)
        if got != P:
            raise TopolowError(ERR_BAD_ARG, f"schedule enumerated {got} pairs, expected {P}")
        return out

    # ---- job-by-job stepping of a map shared by several ranks (topolow_b200/sharded.py) ----
    def run_job(self, kind, t0, tc, y0=0, yc=0, stream=None):
        rc = self._L.topolow_plan_run_job(self._h, int(kind), int(t0), int(tc), int(y0), int(yc),
                                          C.c_void_p(stream) if stream else None)
        if rc != OK:
            raise TopolowError(rc, f"topolow_plan_run_job failed with status {rc}")

    def end_iteration(self, stream=None):
        rc = self._L.topolow_plan_end_iteration(self._h, C.c_void_p(stream) if stream else None)
        if rc != OK:
            raise TopolowError(rc, f"topolow_plan_end_iteration failed with status {rc}")

    def layout(self):
        v = (C.c_int64 * 6)()
        self._L.topolow_plan_layout(self._h, v, 6)
        keys = ["total_tiles", "tile_points", "ndim", "element_bytes", "n_shards", "total_slots"]
        return dict(zip(keys, [int(x) for x in v]))

    def positions_ptr(self):
        return int(self._L.topolow_plan_positions(self._h))

    def enumerate_job(self, it, kind, t0, tc, y0=0, yc=0):
        cap = self._pa.n * (self._pa.n - 1) // 2
        out = np.empty((cap, 2), dtype=np.int32)
        got = self._L.topolow_plan_enumerate_job(self._h, int(it), int(kind), int(t0), int(tc), int(y0), int(yc),
                                                 out.ctypes.data_as(_i32p), cap)
        if got < 0:
            raise TopolowError(ERR_BAD_ARG, f"topolow_plan_enumerate_job failed ({got})")
        return out[:got]

    def close(self):
        if self._h:
            self._L.topolow_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def schedule_enumerate(n, ndim, it, *, precision=PREC_F32, sm_count=148, max_ctas=0, seed=0, pairs=True,
                       tile_points=0):
    """Host-only walk of the coloured schedule: (pair order [P][2], geometry dict)."""
    L = lib()
    P = n * (n - 1) // 2
    geo = (C.c_int64 * 8)()
    out = np.empty((P, 2), dtype=np.int32) if pairs else None
    got = L.topolow_schedule_enumerate(n, ndim, precision, sm_count, max_ctas, int(seed) & 0xFFFFFFFFFFFFFFFF,
                                       int(it), out.ctypes.data_as(_i32p) if pairs else None, P, geo, int(tile_points))
    keys = ["tiles", "super_blocks", "warps_per_cta", "ctas", "tasks_per_cta", "rounds", "pairs_per_iter",
            "smem_bytes"]
    g = dict(zip(keys, [int(x) for x in geo]))
    if pairs and got != P:
        raise TopolowError(ERR_BAD_ARG, f"schedule enumerated {got} pairs, expected {P}")
    return out, g


def est_distances(positions, device=0):
    pos = np.asfortranarray(positions, dtype=np.float64)
    n, d = pos.shape
    out = np.empty((n, n), dtype=np.float64)
    rc = lib().topolow_est_distances(pos.ctypes.data_as(_dp), n, d, out.ctypes.data_as(_dp), device)
    if rc != OK:
        raise TopolowError(rc, f"topolow_est_distances failed with status {rc}")
    return out


def holdout_errors(positions, cell_i, cell_j, truth, device=0):
    pos = np.asfortranarray(positions, dtype=np.float64)
    n, d = pos.shape
    ci = np.ascontiguousarray(cell_i, dtype=np.int32)
    cj = np.ascontiguousarray(cell_j, dtype=np.int32)
    tr = np.ascontiguousarray(truth, dtype=np.float64)
    s, c = C.c_double(0), C.c_int64(0)
    rc = lib().topolow_holdout_errors(pos.ctypes.data_as(_dp), n, d, len(ci), ci.ctypes.data_as(_i32p),
                                      cj.ctypes.data_as(_i32p), tr.ctypes.data_as(_dp), C.byref(s), C.byref(c), device)
    if rc != OK:
        raise TopolowError(rc, f"topolow_holdout_errors failed with status {rc}")
    return s.value, c.value


def components(n, edge_i, edge_j, masks=None, device=0):
    """Connected components of the measurement graph for every candidate point subset in `masks` ([n_masks][n] bool;
    None = all points once).  -> (components, points, edges) int64 arrays of length n_masks."""
    ei = np.ascontiguousarray(edge_i, dtype=np.int32)
    ej = np.ascontiguousarray(edge_j, dtype=np.int32)
    mk, n_masks = None, 1
    if masks is not None:
        mk = np.ascontiguousarray(np.atleast_2d(masks), dtype=np.uint8)
        if mk.shape[1] != n:
            raise ValueError("masks must be [n_masks][n]")
        n_masks = mk.shape[0]
    comp, pts, edg = (np.zeros(n_masks, dtype=np.int64) for _ in range(3))
    rc = lib().topolow_components(int(n), len(ei), ei.ctypes.data_as(_i32p), ej.ctypes.data_as(_i32p), n_masks,
                                  None if mk is None else mk.ctypes.data_as(C.POINTER(C.c_uint8)), comp.ctypes.data_as(_i64p),
                                  pts.ctypes.data_as(_i64p), edg.ctypes.data_as(_i64p), device)
    if rc != OK:
        raise TopolowError(rc, f"topolow_components failed with status {rc}")
    return comp, pts, edg


def microbench(which, device=0) -> float:
    v = C.c_double(0)
    rc = lib().topolow_microbench(which, device, C.byref(v))
    if rc != OK:
        raise TopolowError(rc, f"topolow_microbench({which}) failed with status {rc}")
    return v.value


def device_info(device=0):
    sm, ma, mi, mem = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int64(0)
    rc = lib().topolow_device_info(device, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem))
    if rc != OK:
        raise TopolowError(rc, "no usable CUDA device")
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), global_mem=mem.value)
