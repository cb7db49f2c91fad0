"""Scaling of one CV-grid call over the GPUs of a box (topolow_fit_batch_devices), measured on the GPU.

  python tools/gpu_batch_devices.py [--out profiles/batch_devices_cfg5.json] [--steps 2]

Workload: the bench's cfg5 grid step (bench.cfg5_jobs: 64 parameter samples x 4 folds = 256 fits of 5 000 points per
device, 95 % missing, ndim 2..10, mapping_max_iter 250, early stopping on, hold-out cells scored on the device), k x 256
fits in ONE _lib.fit_batch call with device = [0 .. k-1], for k = 1, 2, 4, 8 (as many as the box has).  On a box with
one GPU the list [0, 0] is run as well: two shares on one device, which measures the host side of the multi-device path.

Per configuration and step: CV embeddings/min, wall seconds, device seconds (the longest CUDA-event span of a fit group
on any device, from the first launch to the end of its last fit) and host seconds (wall minus device: validation, edge
records, uploads, result read-back, release).  Every configuration with more than one list entry is checked against
the plain batch of the same jobs on the first device of its list: per-job hold-out sums and counts, MAE, iterations
and pair counts must be equal bit for bit.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from topolow_b200 import _lib  # noqa: E402

SAMPLES_PER_DEVICE, FIT_ITERS = 64, 250
KEYS = ("holdout_sum_abs", "holdout_count", "final_mae", "iterations", "iterations_run", "pair_updates", "status")


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q or ["unknown"]


def grid(k):
    n, _d, missing = bench.WORKLOADS["cfg5"]
    prob, jobs, meta = bench.cfg5_jobs(n, missing, SAMPLES_PER_DEVICE * k, FIT_ITERS, seed=0)
    held = {}
    for (_s, f, h) in meta:
        if f not in held:
            held[f] = (np.ascontiguousarray(prob["edge_i"][h]), np.ascontiguousarray(prob["edge_j"][h]),
                       np.ascontiguousarray(prob["edge_dist"][h]))
    return [dict(j, holdout=held[f]) for j, (_s, f, _h) in zip(jobs, meta)]


def measure(devices, steps):
    import torch
    jobs = grid(len(devices))
    _lib.fit_batch([dict(j, n_iter=2) for j in jobs], device=devices)   # loads every kernel, grows every pool
    walls, dev_s, out = [], [], None
    for _ in range(steps):
        for d in set(devices):
            torch.cuda.synchronize(d)
        t0 = time.perf_counter()
        out = _lib.fit_batch(jobs, device=devices)
        walls.append(time.perf_counter() - t0)
        dev_s.append(max(r["device_ms"] for r in out) * 1e-3)
    wall, dev = float(np.median(walls)), float(np.median(dev_s))
    row = {"devices": list(devices), "fits_per_step": len(jobs), "steps": steps, "wall_s": walls, "device_s": dev_s,
           "host_s": [w - d for w, d in zip(walls, dev_s)], "cv_embeddings_per_min": len(jobs) / wall * 60.0,
           "median_wall_s": wall, "median_device_s": dev, "median_host_s": wall - dev,
           "mean_iterations_run": float(np.mean([r["iterations_run"] for r in out]))}
    if len(devices) > 1:
        want = _lib.fit_batch(jobs, device=devices[0])
        diff = [j for j, (x, y) in enumerate(zip(out, want)) if any(x[k] != y[k] for k in KEYS)]
        row["equal_to_one_device"] = not diff
        row["unequal_jobs"] = diff[:20]
    return row


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batch_devices_cfg5.json"))
    ap.add_argument("--steps", type=int, default=2)
    args = ap.parse_args()
    count = torch.cuda.device_count()
    if count < 1:
        sys.exit("no CUDA device: this measurement runs on the GPU only")
    lists = [list(range(k)) for k in (1, 2, 4, 8) if k <= count]
    if count == 1:
        lists.append([0, 0])
    rows = []
    for devices in lists:
        rows.append(measure(devices, args.steps))
        print(json.dumps({k: v for k, v in rows[-1].items() if not isinstance(v, list) or k == "devices"}), flush=True)
    base = rows[0]["cv_embeddings_per_min"]
    for r in rows:
        r["speedup_vs_one_device"] = r["cv_embeddings_per_min"] / base
    report = {"tool": "tools/gpu_batch_devices.py", "cards": cards(), "device_count": count,
              "workload": f"cfg5 grid step: {SAMPLES_PER_DEVICE} samples x 4 folds = {4 * SAMPLES_PER_DEVICE} fits of "
                          f"{bench.WORKLOADS['cfg5'][0]} points per device, mapping_max_iter {FIT_ITERS}, early stopping on, "
                          "hold-out cells scored on the device; one fit_batch call per step",
              "runs": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps({"cards": report["cards"], "summary": [(r["devices"], round(r["cv_embeddings_per_min"]),
                                                             r.get("equal_to_one_device")) for r in rows]}))
    if not all(r.get("equal_to_one_device", True) for r in rows):
        sys.exit("multi-device results differ from the one-device batch")


if __name__ == "__main__":
    main()
