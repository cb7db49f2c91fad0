"""Row-block jobs in fit batches, measured on the GPU: a cross-validation step of a large map and an ndim-24 grid.

  python tools/gpu_batch_rowblock.py [--out profiles/batch_rowblock.json]

1. Large-map CV step.  The bench's cfg4 map (100 000 points, ndim 16, 99 % missing, tools/synth.make_problem), 4 folds
   (each holds out a random eighth of the exact cells, degrees recomputed) x 2 parameter samples = 8 row-block fits with
   hold-out cells, mapping_max_iter 1000 with early stopping on (the package defaults).  One _lib.fit_batch call with
   keep_positions=False against the same 8 fits as separate _lib.fit calls: wall seconds per fold fit, device seconds
   (CUDA-event time of the fits) and host seconds (wall minus device: record build, uploads, read-back), and whether
   every job's hold-out sum and count, MAE, iterations and pair count are equal.
2. ndim-24 grid.  16 parameter samples x 4 folds = 64 row-block fits of 5 000 points (95 % missing, the cfg5 map size),
   mapping_max_iter 250, early stopping on, one fit_batch call on device [0] and on [0, 0, 0, 0] (four shares on one GPU:
   four row-block fits at once).
   CV embeddings per minute; the [0, 0, 0, 0] results are checked against [0].
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools import synth  # noqa: E402
from topolow_b200 import _lib  # noqa: E402

KEYS = ("holdout_sum_abs", "holdout_count", "final_mae", "iterations", "iterations_run", "pair_updates", "status")
HYPER = dict(cooling_rate=0.01, c_repulsion=0.02, relative_epsilon=1e-4, convergence_window=5, convergence_check_freq=3)


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def folds_of(prob, n, folds, seed):
    """Training arrays and hold-out cells of each fold: a random eighth of the exact cells per fold, disjoint."""
    ei, ej, ed, et = prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"]
    which = np.random.default_rng(seed).integers(0, 2 * folds, len(ei))
    out = []
    for f in range(folds):
        held = (which == f) & (et == 0)
        tr = ~held
        deg = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
        train = dict(degrees=deg, edge_i=np.ascontiguousarray(ei[tr]), edge_j=np.ascontiguousarray(ej[tr]),
                     edge_dist=np.ascontiguousarray(ed[tr]), edge_thresh=np.ascontiguousarray(et[tr]))
        out.append((train, (np.ascontiguousarray(ei[held]), np.ascontiguousarray(ej[held]), np.ascontiguousarray(ed[held]))))
    return out


def grid_jobs(prob, n, folds, samples, n_iter, seed):
    fj = folds_of(prob, n, folds, seed)
    rng = np.random.default_rng(seed + 1)
    jobs = []
    for s in range(samples):
        k0 = float(rng.uniform(2.0, 8.0))
        for f, (train, held) in enumerate(fj):
            jobs.append(dict(initial_positions=prob["initial_positions"], n_iter=n_iter, k0=k0, holdout=held,
                             mode=_lib.MODE_ROWBLOCK, seed=1000 * s + f, **train, **HYPER))
    return jobs


def single(job):
    j = dict(job)
    args = [j.pop(k) for k in ("initial_positions", "degrees", "edge_i", "edge_j", "edge_dist", "edge_thresh", "n_iter", "k0",
                               "cooling_rate", "c_repulsion", "relative_epsilon", "convergence_window",
                               "convergence_check_freq")]
    return _lib.fit(*args, **j)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def large_map_step():
    n, d, missing = 100_000, 16, 0.99
    t0 = time.perf_counter()
    prob = synth.make_problem(n, d, missing, seed=0)
    gen_s = time.perf_counter() - t0
    jobs = grid_jobs(prob, n, 4, 2, 1000, seed=3)
    single(dict(jobs[0], n_iter=2))                                          # loads the kernels, grows the pools
    batch, wall_b = timed(lambda: _lib.fit_batch(jobs, keep_positions=False))
    alone = []
    wall_s = 0.0
    for j in jobs:
        r, w = timed(lambda: single(j))
        alone.append(r)
        wall_s += w
    dev_b = sum(r["device_ms"] for r in batch) * 1e-3
    dev_s = sum(r["device_ms"] for r in alone) * 1e-3
    diff = [k for k, (x, y) in enumerate(zip(batch, alone)) if any(x[key] != y[key] for key in KEYS)]
    return {"map": {"n_points": n, "ndim": d, "missing": missing, "edges": int(len(prob["edge_i"])), "generate_s": gen_s},
            "jobs": len(jobs), "folds": 4, "parameter_samples": 2, "mapping_max_iter": 1000,
            "iterations_run": [r["iterations_run"] for r in batch],
            "heldout_mae": [r["holdout_sum_abs"] / max(r["holdout_count"], 1) for r in batch],
            "batch": {"wall_s": wall_b, "device_s": dev_b, "host_s": wall_b - dev_b, "wall_s_per_fit": wall_b / len(jobs),
                      "host_s_per_fit": (wall_b - dev_b) / len(jobs)},
            "separate_fits": {"wall_s": wall_s, "device_s": dev_s, "host_s": wall_s - dev_s, "wall_s_per_fit": wall_s / len(jobs),
                              "host_s_per_fit": (wall_s - dev_s) / len(jobs)},
            "equal_to_separate_fits": not diff, "unequal_jobs": diff}


def ndim24_grid():
    n, d, missing = 5000, 24, 0.95
    prob = synth.make_problem(n, d, missing, seed=1)
    jobs = grid_jobs(prob, n, 4, 16, 250, seed=5)
    _lib.fit_batch([dict(j, n_iter=2) for j in jobs[:2]])
    rows, base = [], None
    for devices in ([0], [0, 0, 0, 0]):
        walls, out = [], None
        for _ in range(2):
            out, w = timed(lambda: _lib.fit_batch(jobs, device=devices, keep_positions=False))
            walls.append(w)
        wall = float(np.median(walls))
        row = {"devices": devices, "fits": len(jobs), "wall_s": walls, "cv_embeddings_per_min": len(jobs) / wall * 60.0,
               "mean_iterations_run": float(np.mean([r["iterations_run"] for r in out])),
               "device_s_sum": sum(r["device_ms"] for r in out) * 1e-3}
        if base is None:
            base = out
        else:
            row["equal_to_one_share"] = all(all(x[k] == y[k] for k in KEYS) for x, y in zip(out, base))
        rows.append(row)
    return {"map": {"n_points": n, "ndim": d, "missing": missing, "edges": int(len(prob["edge_i"]))}, "mapping_max_iter": 250,
            "runs": rows}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batch_rowblock.json"))
    args = ap.parse_args()
    if torch.cuda.device_count() < 1:
        sys.exit("no CUDA device: this measurement runs on the GPU only")
    report = {"tool": "tools/gpu_batch_rowblock.py", "cards": cards(), "device_count": torch.cuda.device_count()}
    report["large_map_cv_step"] = large_map_step()
    print(json.dumps({k: v for k, v in report["large_map_cv_step"].items() if k not in ("heldout_mae",)}), flush=True)
    report["ndim24_grid"] = ndim24_grid()
    print(json.dumps(report["ndim24_grid"]), flush=True)
    report["two_to_eight_gpus"] = f"not measured ({torch.cuda.device_count()} GPU on the box)"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps({"cards": report["cards"], "out": args.out}))
    ok = report["large_map_cv_step"]["equal_to_separate_fits"] and all(
        r.get("equal_to_one_share", True) for r in report["ndim24_grid"]["runs"])
    if not ok:
        sys.exit("batch results differ from the separate fits")


if __name__ == "__main__":
    main()
