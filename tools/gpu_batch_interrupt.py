"""Cost and latency of stopping a batch (topolow_fit_batch_interruptible), measured on the GPU.

  python tools/gpu_batch_interrupt.py [out.json]      (prints the report; also writes it to out.json when given)

* overhead: the bench's CV-grid shape (64 samples x 4 folds = 256 fits of 5 000 points, 95 % missing, ndim 2..10,
  250 iterations, early stopping off, hold-out cells scored on the device) through _lib.fit_batch without and with a
  poll that never fires, alternated three times;
* latency: the time from the poll returning non-zero to the call returning, for that grid and for a batch of two
  40 000-point fits that run on many CTAs each, next to the device time of one iteration of the batch's longest fit.
The card's name and power limit are read in the same run."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from tools import synth  # noqa: E402
from topolow_b200 import _lib  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def grid_jobs():
    n, _d, missing = bench.WORKLOADS["cfg5"]
    prob, jobs, meta = bench.cfg5_jobs(n, missing, 64, 250, seed=0)
    held = {}
    for _s, f, h in meta:
        held.setdefault(f, (np.ascontiguousarray(prob["edge_i"][h]), np.ascontiguousarray(prob["edge_j"][h]),
                            np.ascontiguousarray(prob["edge_dist"][h])))
    return [dict(j, convergence_window=251, holdout=held[f]) for j, (_s, f, _h) in zip(jobs, meta)]


def multi_jobs():
    prob = synth.make_problem(40_000, 5, 0.99, seed=3, thresholds=False)
    a = synth.fit_args(prob)
    return [dict(initial_positions=a[0], degrees=a[1], edge_i=a[2], edge_j=a[3], edge_dist=a[4], edge_thresh=a[5], n_iter=400,
                 k0=5.0, cooling_rate=0.01, c_repulsion=0.02, convergence_window=401, seed=s) for s in range(2)]


def timed(jobs, interrupt=None):
    t0 = time.perf_counter()
    out = _lib.fit_batch(jobs, interrupt=interrupt)
    return time.perf_counter() - t0, out


def latency(jobs, after_s, reps=3):
    """Seconds from the poll's first non-zero answer to the call's return, and what the stopped fits had done."""
    res = []
    for _ in range(reps):
        t = {}

        def poll():
            now = time.perf_counter()
            t.setdefault("start", now)
            if now - t["start"] > after_s:
                t["fired"] = now
                return True
            return False
        try:
            _lib.fit_batch(jobs, interrupt=poll)
            raise RuntimeError("the batch was not interrupted")
        except _lib.TopolowError as e:
            back = time.perf_counter()
            if e.status != _lib.ERR_INTERRUPTED:
                raise
            rs = e.results
        res.append(dict(latency_ms=(back - t["fired"]) * 1e3,
                        stopped=sum(r["status"] == _lib.ERR_INTERRUPTED for r in rs),
                        iterations_run=sorted({r.get("iterations_run", -1) for r in rs})[:8]))
    return res


def per_iteration_ms(out):
    """Device time of one iteration of the longest fit (a group's launch time over its fits' iterations)."""
    longest = max(out, key=lambda r: r["device_ms"])
    return longest["device_ms"] / max(longest["iterations_run"], 1), longest["iterations_run"]


def main():
    dev = card()
    grid = grid_jobs()
    _lib.fit_batch([dict(j, n_iter=2) for j in grid])              # kernels loaded, pools grown
    _lib.fit_batch([dict(j, n_iter=2) for j in grid], interrupt=lambda: False)
    plain, polled = [], []
    ref = None
    for _ in range(3):
        t, out = timed(grid)
        plain.append(t)
        ref = ref or out
        calls = []
        t, out2 = timed(grid, interrupt=lambda: calls.append(1) and False)
        polled.append(t)
        assert all(np.array_equal(a["positions"], b["positions"]) and a["final_mae"] == b["final_mae"] for a, b in zip(out, out2))
    it_ms, it_n = per_iteration_ms(ref)
    lat_grid = latency(grid, 0.5)

    multi = multi_jobs()
    _lib.fit_batch([dict(j, n_iter=2) for j in multi])
    t_multi, mout = timed(multi)
    m_it_ms = max(r["device_ms"] / max(r["iterations_run"], 1) for r in mout)
    lat_multi = latency(multi, 0.5)

    rep = {
        "device": dev,
        "grid": {"shape": "256 fits (64 samples x 4 folds) of 5000 points, 95% missing, ndim 2..10, 250 iterations, "
                          "early stopping off, hold-out scored on the device",
                 "wall_s_plain": plain, "wall_s_polled_never_firing": polled,
                 "polls_per_call": len(calls),
                 "longest_fit_ms_per_iteration": it_ms, "longest_fit_iterations": it_n,
                 "interrupt_after_0.5s": lat_grid},
        "multi_cta": {"shape": "2 fits of 40000 points, ndim 5, 99% missing, 400 iterations, early stopping off, "
                               "convergence_check_freq 3 (one fit at a time on the whole chip)",
                      "wall_s_plain": t_multi, "ms_per_iteration": m_it_ms,
                      "interrupt_after_0.5s": lat_multi},
    }
    print(json.dumps(rep, indent=1))
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
