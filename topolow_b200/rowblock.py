"""One large map, row-block sharded over the GPUs of a box (BASELINE.json configs[3], SURVEY section 8e).

Rank r owns a contiguous block of rows and a replica of all positions; per iteration it computes the
one-sided updates of its rows (src/optimization.cpp:199-282 seen from the row's endpoint: repulsion
from every other point, then its own springs one after another), stores the new rows straight into
every replica (NVLink peer stores from inside the spring kernel) and raises one flag per peer.  No
host code, no torch op and no NCCL call sits in the loop: torch.distributed only carries the CUDA-IPC
handles at set-up and the barrier before tear-down.  The result does not depend on the number of
ranks; one rank is `_lib.fit(..., mode=_lib.MODE_ROWBLOCK)`.

  Shard          one rank's part (topolow_shard_* of include/topolow_b200.h)
  RowBlockMap    what a torchrun rank uses: create, exchange handles, attach, step, result
  LocalShards    all ranks in ONE process: on one GPU they run in lock step (how a single GPU checks the
                 multi-GPU path bit for bit), on several GPUs concurrently
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import OK, TopolowError

INFO_KEYS = ["slots", "ndim", "stride", "n_ranks", "rank", "row0", "own_rows", "partner_chunks", "spring_records",
             "mae_records", "launches", "iterations_done", "stopped", "peer_store_bytes_per_iteration",
             "repulsion_items", "repulsion_ctas", "repulsion_form",
             "tensor_form_iterations", "walk_ring", "walk_ctas"]
KERNELS = ["repulse", "spring", "mae", "controller", "snapshot"]


class Shard:
    def __init__(self, initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, n_iter, k0, cooling_rate,
                 c_repulsion, relative_epsilon=1e-4, convergence_window=5, convergence_check_freq=3, *, rank=0,
                 n_ranks=1, device=0, seed=0, holdout=None):
        self._L = _lib.lib()
        self._pa = _lib.ProblemArrays(initial_positions, degrees, edge_i, edge_j, edge_dist, edge_thresh, holdout)
        pr, _ = _lib.make_params(n_iter, k0, cooling_rate, c_repulsion, relative_epsilon, convergence_window,
                                 convergence_check_freq, False, _lib.MODE_ROWBLOCK, _lib.PREC_F32, seed, None, device)
        self.n_iter, self.rank, self.n_ranks, self.device = int(n_iter), int(rank), int(n_ranks), int(device)
        self._h = C.c_void_p()
        msg = C.create_string_buffer(256)
        rc = self._L.topolow_shard_create(C.byref(self._pa.struct), C.byref(pr), self.rank, self.n_ranks,
                                          C.byref(self._h), msg, 256)
        if rc != OK:
            raise TopolowError(rc, msg.value.decode() or f"topolow_shard_create failed with status {rc}")

    def export(self) -> bytes:
        nb = int(self._L.topolow_shard_handle_bytes())
        buf = C.create_string_buffer(nb)
        rc = self._L.topolow_shard_export(self._h, buf)
        if rc != OK:
            raise TopolowError(rc, f"topolow_shard_export failed with status {rc}")
        return buf.raw

    def attach(self, handles):
        """handles: the `export()` of every rank, in rank order."""
        blob = b"".join(handles)
        msg = C.create_string_buffer(256)
        rc = self._L.topolow_shard_attach(self._h, blob, len(handles), msg, 256)
        if rc != OK:
            raise TopolowError(rc, msg.value.decode() or f"topolow_shard_attach failed with status {rc}")

    def run(self, n_iters, stream=None) -> float:
        ms = C.c_double(0)
        rc = self._L.topolow_shard_run(self._h, int(n_iters), C.c_void_p(stream) if stream else None, C.byref(ms))
        if rc != OK:
            raise TopolowError(rc, f"topolow_shard_run failed with status {rc}")
        return ms.value

    def time_kernels(self, n_iters):
        v = (C.c_double * 7)()
        rc = self._L.topolow_shard_time_kernels(self._h, int(n_iters), v, 7)
        if rc != OK:
            raise TopolowError(rc, f"topolow_shard_time_kernels failed with status {rc}")
        out = dict(zip(KERNELS, [float(x) for x in v[:5]]))
        out["mae_launches"] = int(v[5])
        out["combine"] = float(v[6])
        return out

    def result(self, trace=False):
        out = np.empty((self._pa.n, self._pa.ndim), dtype=np.float64, order="F")
        res = _lib.Result()
        res.positions = out.ctypes.data_as(_lib._dp)
        tr = None
        if trace:
            tr = np.full(max(self.n_iter, 1), np.nan)
            res.trace_mae = tr.ctypes.data_as(_lib._dp)
        rc = self._L.topolow_shard_result(self._h, C.byref(res))
        if rc != OK:
            raise TopolowError(rc, res.message.decode() or f"topolow_shard_result failed with status {rc}")
        return _lib.result_dict(res, out, tr)

    def info(self):
        v = (C.c_int64 * len(INFO_KEYS))()
        self._L.topolow_shard_info(self._h, v, len(INFO_KEYS))
        return dict(zip(INFO_KEYS, [int(x) for x in v]))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.topolow_shard_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def slot_order(n):
    """slot_of_point of the row-block layout."""
    out = np.empty(int(n), dtype=np.int32)
    rc = _lib.lib().topolow_shard_slot_order(int(n), out.ctypes.data_as(_lib._i32p))
    if rc != OK:
        raise TopolowError(rc, "topolow_shard_slot_order failed")
    return out


class LocalShards:
    """All ranks of a map in one process (`devices[r]` = CUDA ordinal of rank r; default: all on device 0)."""

    def __init__(self, *fit_args, n_ranks, devices=None, **kw):
        devices = list(devices) if devices is not None else [0] * int(n_ranks)
        self.shards = [Shard(*fit_args, rank=r, n_ranks=n_ranks, device=devices[r], **kw) for r in range(int(n_ranks))]
        self._L = _lib.lib()
        self._arr = (C.c_void_p * len(self.shards))(*[s._h for s in self.shards])
        msg = C.create_string_buffer(256)
        rc = self._L.topolow_shard_attach_local(self._arr, len(self.shards), msg, 256)
        if rc != OK:
            raise TopolowError(rc, msg.value.decode() or f"topolow_shard_attach_local failed with status {rc}")

    def run(self, n_iters) -> float:
        ms = C.c_double(0)
        rc = self._L.topolow_shard_run_local(self._arr, len(self.shards), int(n_iters), C.byref(ms))
        if rc != OK:
            raise TopolowError(rc, f"topolow_shard_run_local failed with status {rc}")
        return ms.value

    def result(self, rank=0, trace=False):
        return self.shards[rank].result(trace=trace)

    def close(self):
        for s in self.shards:
            s.close()


class RowBlockMap:
    """The part of one torchrun rank.  `group` = a torch.distributed process group (None = the default one);
    with world size 1 no process group is needed."""

    def __init__(self, *fit_args, rank=0, world_size=1, device=0, group=None, **kw):
        self.rank, self.world = int(rank), int(world_size)
        self.group = group
        self.shard = Shard(*fit_args, rank=self.rank, n_ranks=self.world, device=device, **kw)
        if self.world > 1:
            import torch.distributed as dist
            handles = [None] * self.world
            dist.all_gather_object(handles, self.shard.export(), group=group)   # host plumbing: 88 bytes per rank
            self.shard.attach(handles)
            dist.barrier(group=group)                                          # every rank has mapped every block

    def step(self, n_iters, stream=None) -> float:
        """Up to n_iters further iterations (all ranks call this with the same count); CUDA-event ms."""
        return self.shard.run(n_iters, stream)

    def result(self, trace=False):
        return self.shard.result(trace=trace)

    def info(self):
        return self.shard.info()

    def time_kernels(self, n_iters):
        return self.shard.time_kernels(n_iters)

    def close(self):
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.synchronize()
            dist.barrier(group=self.group)     # peers store into this rank's block until their last iteration ends
        self.shard.close()
