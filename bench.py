#!/usr/bin/env python
"""bench.py - pair-updates/s of the force-directed embedding loop on B200.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg4|cfg3|cfg2|small]

A step is ONE iteration of the reference's loop (src/optimization.cpp:193-366): all N(N-1)/2 pair
updates, cooling, and - every convergence_check_freq iterations - the edge MAE + controller.  The
default workload is BASELINE.json configs[3]: synthetic, 100 000 points, 99 % missing, ndim = 16
(tools/synth.py, seed 0), early stopping disabled so that exactly K iterations run
(convergence_counter = n_iter + 1, SURVEY.md section 8d).

  value      whole-job pair-updates/s with the problem resident in HBM (topolow_plan_run), CUDA events
             on the launching stream, max over ranks.
  e2e        the same metric through the reference-facing call with HOST buffers (topolow_fit: upload,
             device set-up, K iterations, download), wall clock around the call.
  roofline   the persistent tile kernel is FP32-FMA bound (no tensor-core work exists on this path):
             achieved = algorithmic flop per iteration / kernel time, peak = FFMA rate measured live by
             topolow_microbench on the same GPU.  `hbm` gives the edge stream against MEASURED_PEAKS.
  cpu_baseline / --impl reference: oracle/ (the CPU restatement of src/optimization.cpp) on the host.

  --dump-outputs DIR   after the timed steps, what the resident leg hands its caller as float64 DIR/<name>.npy:
                       the best-iteration positions (the snapshot topolow_shard_result / topolow_plan_result
                       return, as in the reference), the MAE at each check iteration and the controller scalars;
                       the inputs are seeded, so two builds run with the same arguments can be compared output
                       for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n, ndim, missing fraction)
    "cfg4": (100_000, 16, 0.99),
    "cfg3": (10_000, 10, 0.95),
    "small": (2_000, 5, 0.90),
    "cfg5": (5_000, 5, 0.95),     # Euclidify grid: parameter samples x 4 folds, independent fits
}
HYPER = dict(k0=5.0, cooling_rate=0.01, c_repulsion=0.02, relative_epsilon=1e-4, convergence_check_freq=3)


def flop_per_iter(n, d, n_edges):
    """SURVEY.md section 8d: 7d+8 per unmeasured pair update, 7d+12 per spring pair update."""
    pairs = n * (n - 1) // 2
    return (pairs - n_edges) * (7 * d + 8) + n_edges * (7 * d + 12)


def edge_bytes_per_iter(n, d, n_edges):
    """Edge stream: 16-byte record per measured pair + every FP32 position read and written once."""
    return n_edges * 16 + 2 * n * d * 4


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._idx = gpu_index
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self._idx), f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=3)

    def summary(self):
        if not self.samples:
            return None
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def cpu_sample(prob, n, d, sample_pairs, kind="O2", seed=0):
    """Time the oracle's pair loop on the same workload.  n <= 12000: one full iteration exactly as the
    reference runs it (dense lookup, std::shuffle of all pairs).  Larger n (the reference cannot run
    these: int overflow and dense n x n inputs, src/optimization.cpp:143-150): a bounded sample of
    uniformly random pairs in explicit order with the sparse lookup; set-up (hash build, final MAE) is
    measured by a zero-pair call and subtracted.  Returns (pair-updates/s, seconds, description)."""
    from oracle import cpu_oracle
    from tools import synth
    fa = synth.fit_args(prob)
    hp = (HYPER["k0"], HYPER["cooling_rate"], HYPER["c_repulsion"], HYPER["relative_epsilon"], 3, 7)
    if n <= 12000:
        t0 = time.perf_counter()
        cpu_oracle.optimize_layout_exact(*fa, 0, *hp, seed=seed, dense=True, kind=kind)
        setup = time.perf_counter() - t0          # dense matrices + all_pairs construction
        t0 = time.perf_counter()
        res = cpu_oracle.optimize_layout_exact(*fa, 2, *hp, seed=seed, dense=True, kind=kind)
        dt = max(time.perf_counter() - t0 - setup, 1e-9)
        return res["visited"] / dt, dt, ("two full iterations, dense lookup + std::shuffle of all pairs (the reference's own "
                                         "scheme); set-up time subtracted")
    rng = np.random.default_rng(seed)
    i = rng.integers(0, n, size=sample_pairs, dtype=np.int32)
    j = rng.integers(0, n - 1, size=sample_pairs, dtype=np.int32)
    j = np.where(j >= i, j + 1, j).astype(np.int32)
    order = np.stack([i, j], axis=1)[None]
    empty = np.full((1, 1, 2), -1, dtype=np.int32)
    t0 = time.perf_counter()
    cpu_oracle.optimize_layout_exact(*fa, 1, *hp, pair_order=empty, dense=False, kind=kind)
    setup = time.perf_counter() - t0
    t0 = time.perf_counter()
    res = cpu_oracle.optimize_layout_exact(*fa, 1, *hp, pair_order=order, dense=False, kind=kind)
    dt = max(time.perf_counter() - t0 - setup, 1e-9)
    return res["visited"] / dt, dt, (f"{sample_pairs} uniformly random pair visits in explicit order, sparse (hash) lookup; "
                                     "set-up time subtracted")


def map_config(workload, n, d, missing, E, early_stop=None):
    """The workload, named the same way by both arms (ours and --impl reference)."""
    pairs = n * (n - 1) // 2
    return {"workload": workload,
            "description": f"synthetic low-rank dissimilarities (tools/synth.py, seed 0): {n} points, {missing:.0%} missing, ndim={d}, "
                           "5 % '>' and 5 % '<' thresholds; k0=5, cooling_rate=0.01, c_repulsion=0.02, check every 3 iterations",
            "n_points": n, "ndim": d, "missing": missing, "n_edges": int(E), "pairs_per_iteration": pairs,
            "early_stop": early_stop or "disabled (convergence_counter = n_iter + 1): every step is one full iteration",
            "l2": "inputs larger than L2: the edge records streamed every iteration (%.0f MB over all ranks) exceed the 126 MB L2; "
                  "the %.1f MB position replica is the resident working set, as in production" % (E * 16 / 1e6, n * d * 4 / 1e6)}


DUMP_SCALARS = ("final_mae", "final_k", "iterations", "iterations_run", "converged", "pair_updates")


def dump_outputs(out_dir, res):
    """Write the result dict of the timed leg (positions are n x ndim: 12.8 MB at cfg4) as float64 .npy files.
    The MAE trace is NaN at iterations without a check (and past the last one run): only the checked entries are
    written, with their iteration numbers."""
    tr = np.asarray(res["trace_mae"])
    checked = np.flatnonzero(~np.isnan(tr))
    arrays = {"positions": res["positions"], "trace_iteration": checked, "trace_mae": tr[checked]}
    arrays.update({k: np.array([res[k]]) for k in DUMP_SCALARS})
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    bad = [name for name, a in arrays.items() if not np.all(np.isfinite(a))]
    if bad:
        raise SystemExit(f"--dump-outputs: non-finite values in {', '.join(bad)}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, n, d, missing):
    """--impl reference: the CPU implementation of the path on this box's host cores."""
    from tools import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    prob = synth.make_problem(n, d, missing, seed=0)
    pairs = n * (n - 1) // 2
    sample = int(min(pairs, 4e7, 3e8 / max(args.steps, 1)))   # bounded: the whole run stays within a few minutes
    from oracle import cpu_oracle
    cpu_oracle.build(ref=False)
    for w in range(args.warmup):
        cpu_sample(prob, n, d, max(sample // 8, 1000), seed=100 + w)
    visited, busy, desc = 0.0, 0.0, ""
    for k in range(args.steps):
        rate, dt, desc = cpu_sample(prob, n, d, sample, seed=k)
        visited += rate * dt
        busy += dt
    wall = busy
    value = visited / wall
    sample = int(round(visited / args.steps))
    line = {
        "impl": "reference", "metric": "pair-updates/s", "value": value, "unit": "pair-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3 * (pairs / sample),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": map_config(args.workload, n, d, missing, len(prob["edge_i"])),
        "cpu_baseline": {"value": value, "unit": "pair-updates/s", "cores": 1, "kind": "port",
                         "sample": f"per step: {desc} (oracle = CPU restatement of src/optimization.cpp, g++ -O2, "
                                   "1 thread: a fit is single-threaded in the reference); ms_per_step is scaled to a full iteration"},
        "e2e": {"value": value, "unit": "pair-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cfg5_jobs(n, missing, samples, fit_iters, seed):
    """`samples` parameter draws x 4 CV folds on one synthetic matrix: the unit of work of
    initial_parameter_optimization (R/adaptive_sampling.R:419-425,516-528)."""
    from tools import synth
    rng = np.random.default_rng(seed)
    prob = synth.make_problem(n, 5, missing, seed=0, thresholds=False)
    ei, ej, ed = prob["edge_i"], prob["edge_j"], prob["edge_dist"]
    E = len(ei)
    folds = []
    perm = rng.permutation(E)
    hold = E // 8            # floor(num_non_NA / (2 * folds)) cells = E/8 pairs in each of the 4 folds... per fold
    for f in range(4):
        mask = np.ones(E, dtype=bool)
        mask[perm[f * hold:(f + 1) * hold]] = False
        deg = (np.bincount(ei[mask], minlength=n) + np.bincount(ej[mask], minlength=n) + 1).astype(np.int32)
        # one training edge list per fold, shared by every parameter sample (topolow_fit_batch then builds
        # its device records once per fold; cv.likelihood_batch hands over its folds the same way)
        train = dict(edge_i=np.ascontiguousarray(ei[mask], dtype=np.int32), edge_j=np.ascontiguousarray(ej[mask], dtype=np.int32),
                     edge_dist=np.ascontiguousarray(ed[mask], dtype=np.float64),
                     edge_thresh=np.ascontiguousarray(prob["edge_thresh"][mask], dtype=np.int32))
        folds.append((train, deg, perm[f * hold:(f + 1) * hold]))
    jobs, meta = [], []
    for s_ in range(samples):
        ndim = int(rng.integers(2, 11))
        k0, cr, c = float(rng.uniform(1, 15)), float(10 ** rng.uniform(-3, -1.3)), float(10 ** rng.uniform(-3, -1.3))
        for f, (train, deg, held) in enumerate(folds):
            init = np.vstack([np.zeros((1, ndim)), np.cumsum(rng.uniform(0, 2 * ed.max() / n, size=(n - 1, ndim)), axis=0)])
            jobs.append(dict(initial_positions=init, degrees=deg, **train, n_iter=fit_iters, k0=k0, cooling_rate=cr, c_repulsion=c,
                             relative_epsilon=1e-4, convergence_window=5, seed=1000 * s_ + f))
            meta.append((s_, f, held))
    return prob, jobs, meta


def _cpu_fit_iters(job, iters):
    """Worker of the CV-grid CPU baseline: `iters` iterations of one fold fit on one core; returns seconds."""
    from oracle import cpu_oracle
    t0 = time.perf_counter()
    cpu_oracle.optimize_layout_exact(job["initial_positions"], job["degrees"], job["edge_i"], job["edge_j"], job["edge_dist"],
                                     job["edge_thresh"], iters, job["k0"], job["cooling_rate"], job["c_repulsion"], 1e-4,
                                     iters + 1, 3, seed=0, dense=True)
    return time.perf_counter() - t0


def cv_grid_cpu_baseline(jobs, mean_iters_run, fit_iters):
    """The host-core baseline of the CV grid, like for like: one fold fit per core on ALL cores at once (what
    parallel::mclapply does, R/adaptive_sampling.R:645-672), each timed for 0 and for 2 iterations (the difference
    is the per-iteration cost under full-socket contention), scaled to the MEAN NUMBER OF ITERATIONS THE GPU
    ARM'S FITS ACTUALLY RAN (same early-stopping rule, same work)."""
    import multiprocessing as mp
    from oracle import cpu_oracle
    cpu_oracle.build(ref=False)
    cores = os.cpu_count() or 1
    pick = [jobs[(i * 7) % len(jobs)] for i in range(cores)]          # a stratified handful: different ndim / folds
    pick = [{k: v for k, v in j.items() if k != "holdout"} for j in pick]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        setup = pool.starmap(_cpu_fit_iters, [(j, 0) for j in pick])
        two = pool.starmap(_cpu_fit_iters, [(j, 2) for j in pick])
        busy = time.perf_counter() - t0
    per_iter = max(float(np.mean([b - a for a, b in zip(setup, two)])) / 2.0, 1e-9)
    per_fit = per_iter * mean_iters_run + float(np.mean(setup))
    return {"value": 60.0 / per_fit * cores, "unit": "CV embeddings/min", "cores": cores, "kind": "port",
            "sample": f"{cores} fold fits at once, one per core (oracle, g++ -O2): {per_iter:.2f} s per iteration and "
                      f"{np.mean(setup):.2f} s set-up per fit under full-socket load; scaled to the {mean_iters_run:.1f} iterations the "
                      f"GPU arm's fits ran on average (mapping_max_iter={fit_iters}, same early stopping); {busy:.0f} s of wall time"}


def cv_grid_measure(local, rank, world, samples, fit_iters, steps, warmup, n, missing, with_cpu):
    """BASELINE.json configs[4]: `samples` parameter draws x 4 folds of independent fits PER GPU and step, through
    topolow_fit_batch on host buffers (set-up, upload, fits, hold-out residuals, download: the path IS end to
    end).  Weak scaling: every rank runs its own share, no collective on the data path."""
    import torch
    import torch.distributed as dist
    from topolow_b200 import _lib

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    prob, jobs, meta = cfg5_jobs(n, missing, samples, fit_iters, seed=rank)
    warm = [dict(j, n_iter=2) for j in jobs]   # loads every ndim variant of the kernel, grows every pool the steps use
    for _ in range(max(warmup, 1)):
        _lib.fit_batch(warm, device=local)
    held_cells = {}   # the hold-out cells of a fold (fixed for the whole grid), scored on the device inside the batch
    for (_s, f, held) in meta:
        if f not in held_cells:
            held_cells[f] = (np.ascontiguousarray(prob["edge_i"][held]), np.ascontiguousarray(prob["edge_j"][held]),
                             np.ascontiguousarray(prob["edge_dist"][held]))
    jobs = [dict(j, holdout=held_cells[f]) for j, (_s, f, _h) in zip(jobs, meta)]
    barrier()
    t0 = time.perf_counter()
    done, pair_updates, iters_run, flop, held_mae = 0, 0, 0, 0.0, []
    with ClockSampler(local) as clk:
        for _ in range(steps):
            out = _lib.fit_batch(jobs, device=local)
            held_mae.extend(r["holdout_sum_abs"] / max(r["holdout_count"], 1) for r in out)
            done += len(out)
            pair_updates += sum(r["pair_updates"] for r in out)
            iters_run += sum(r["iterations_run"] for r in out)
            flop += sum(r["pair_updates"] * (7.0 * j["initial_positions"].shape[1] + 8.0) for r, j in zip(out, jobs))
            kernel_ms = max(r["device_ms"] for r in out)
        barrier()
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], dtype=torch.float64, device="cuda")
    tot = torch.tensor([done, pair_updates, iters_run, flop], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank != 0:
        return None
    wall = float(t[0])
    fits, mean_iters = float(tot[0]), float(tot[2]) / max(float(tot[0]), 1.0)
    ffma_peak = _lib.microbench(0, local)
    ach = float(tot[3]) / wall / world          # algorithmic flop/s per GPU over the whole end-to-end step
    res = {"metric": "CV embeddings/min", "value": fits / wall * 60.0, "unit": "CV embeddings/min", "scaling": "weak",
           "fits_per_gpu_per_step": len(jobs), "steps": steps, "ms_per_step": wall / steps * 1e3,
           "workload": f"cfg5: Euclidify grid, 512 parameter samples x 4 folds = 2048 fits on 8 GPUs, i.e. {samples} samples x 4 folds "
                       f"= {len(jobs)} independent fits per GPU and step; {n}-point synthetic matrix ({missing:.0%} missing), ndim sampled "
                       f"in 2..10, mapping_max_iter={fit_iters}, early stopping on; hold-out residuals scored on the device",
           "mean_iterations_run": mean_iters, "pair_updates_per_s": float(tot[1]) / wall,
           "mean_holdout_mae": float(np.mean(held_mae)), "clocks": clk.summary(),
           "h2d_bytes_per_step": int(sum(j["initial_positions"].nbytes + len(j["edge_i"]) * 20 + n * 4 for j in jobs)),
           "d2h_bytes_per_step": int(sum(j["initial_positions"].nbytes for j in jobs)),
           # per step: one tile_batch_kernel launch per ndim group (one CTA per fit) + one hold-out kernel per fit
           "gpu_launches": int(steps * (len({j["initial_positions"].shape[1] for j in jobs}) + len(jobs))),
           "roofline": {"bound": "fp32", "kernel": "tile_batch_kernel<D,FastF32> (one CTA per fit)", "achieved": ach / 1e12,
                        "peak": ffma_peak / 1e12, "unit": "TFLOP/s", "frac": ach / ffma_peak,
                        "note": "algorithmic flop (7 ndim + 8 per executed pair update, summed over the fits) / END-TO-END wall time "
                                "of the step per GPU (set-up, upload and hold-out scoring included); peak = FFMA rate measured live"},
           "cpu_baseline": cv_grid_cpu_baseline(jobs, mean_iters, fit_iters) if with_cpu else None}
    if res["cpu_baseline"]:
        res["speedup_vs_host_cores"] = res["value"] / res["cpu_baseline"]["value"]
    return res


def main_cfg5(args, n, missing):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = cv_grid_measure(local, rank, world, args.samples, args.fit_iters, args.steps, args.warmup, n, missing, not args.no_cpu)
    if rank == 0:
        line = {"metric": res["metric"], "value": res["value"], "unit": res["unit"], "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": res["workload"]},
                "clocks": res["clocks"],
                "e2e": {"value": res["value"], "unit": res["unit"], "h2d_bytes_per_step": res["h2d_bytes_per_step"],
                        "d2h_bytes_per_step": res["d2h_bytes_per_step"],
                        "note": "the measured path IS end to end: topolow_fit_batch on host buffers"},
                "gpu_launches": res["gpu_launches"], "roofline": res["roofline"], "cpu_baseline": res["cpu_baseline"],
                "cv_grid": res}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="rowblock", choices=["rowblock", "exact"],
                    help="rowblock: owner-computes row blocks (one map over all GPUs, the mode that scales); exact: the coloured "
                         "schedule with the reference's sequential semantics (1 GPU; with --gpus > 1 independent replicas)")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cv", action="store_true", help="skip the cv_grid block (Metric 2) of the default line")
    ap.add_argument("--no-exact", action="store_true", help="skip the short exact-mode comparison run at 1 GPU")
    ap.add_argument("--samples", type=int, default=64, help="CV grid: parameter samples per GPU per step (x 4 folds); 64 = 512 / 8")
    ap.add_argument("--fit-iters", type=int, default=250, help="CV grid: mapping_max_iter of every fit (R/core.R:945)")
    ap.add_argument("--cv-steps", type=int, default=2)
    ap.add_argument("--converge", action="store_true",
                    help="the north-star target run instead of the throughput bench: the map fitted to convergence "
                         "(mapping_max_iter 1000, early stopping on) with 10 %% of the exact cells held out; prints held-out MAE, "
                         "iterations and wall time, and the same fit against the CPU reference loop at --oracle-n points")
    ap.add_argument("--oracle-n", type=int, default=4000, help="--converge: size of the CPU comparison (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result they leave (best-iteration positions as "
                         "topolow_shard_result / topolow_plan_result return them, MAE trace, controller scalars) as "
                         "float64 DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload == "cfg5" or args.impl == "reference" or args.converge):
        ap.error("--dump-outputs applies to the map throughput run (--impl ours, workloads cfg4 / cfg3 / small)")
    n, d, missing = WORKLOADS[args.workload]
    if args.workload == "cfg5":
        return main_cfg5(args, n, missing)
    if args.impl == "reference":
        run_reference(args, n, d, missing)
        return
    if args.converge:
        return main_converge(args, n, d, missing)
    main_map(args, n, d, missing)


def heldout_split(prob, n, frac, seed):
    """Hold `frac` of the exact (non-threshold) cells out of the fit: training arrays with recomputed degrees
    (R/adaptive_sampling.R:2605-2616 masks the cells to NA before euclidean_embedding counts them) + the held cells."""
    ei, ej, ed, et = prob["edge_i"], prob["edge_j"], prob["edge_dist"], prob["edge_thresh"]
    held = (np.random.default_rng(seed).random(len(ei)) < frac) & (et == 0)
    tr = ~held
    deg = (np.bincount(ei[tr], minlength=n) + np.bincount(ej[tr], minlength=n) + 1).astype(np.int32)
    train = (prob["initial_positions"], deg, np.ascontiguousarray(ei[tr]), np.ascontiguousarray(ej[tr]),
             np.ascontiguousarray(ed[tr]), np.ascontiguousarray(et[tr]))
    return train, (np.ascontiguousarray(ei[held]), np.ascontiguousarray(ej[held]), np.ascontiguousarray(ed[held]))


def main_converge(args, n, d, missing):
    """BASELINE.json north_star target: the cfg4 map converged to the reference's held-out MAE.  The held-out MAE is
    the pooled |truth - distance| over cells the fit never saw (R/adaptive_sampling.R:2639-2656)."""
    import torch
    import torch.distributed as dist
    from tools import synth
    from topolow_b200 import _lib
    from topolow_b200.rowblock import RowBlockMap

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    hp = (HYPER["k0"], HYPER["cooling_rate"], HYPER["c_repulsion"], HYPER["relative_epsilon"], 5, HYPER["convergence_check_freq"])
    max_iter = 1000

    def fit_map(nn, dd, miss, seed):
        prob = synth.make_problem(nn, dd, miss, seed=seed)
        train, held = heldout_split(prob, nn, 0.10, seed + 1)
        barrier()
        t0 = time.perf_counter()
        m = RowBlockMap(*train, max_iter, *hp, rank=rank, world_size=world, device=local, seed=0, holdout=held)
        ms = m.step(max_iter)
        res = m.result(trace=True)
        barrier()
        wall = time.perf_counter() - t0
        m.close()
        out = {"n_points": nn, "ndim": dd, "missing": miss, "train_edges": int(len(train[2])), "heldout_cells": int(len(held[0])),
               "mapping_max_iter": max_iter, "iterations_run": res["iterations_run"], "best_iteration": res["iterations"],
               "converged": res["converged"], "edge_mae_train": res["final_mae"],
               "heldout_mae": res["holdout_sum_abs"] / max(res["holdout_count"], 1), "wall_s": wall, "device_s": ms * 1e-3,
               "ms_per_iteration": ms / max(res["iterations_run"], 1)}
        tr = res["trace_mae"]
        out["mae_trace_every_30"] = [round(float(x), 4) for x in tr[~np.isnan(tr)][::10]]
        return out, train, held

    big, _, _ = fit_map(n, d, missing, 0)
    small, cpu = None, None
    if args.oracle_n > 0:
        # the same generator, hyper-parameters and hold-out rule at a size the dense CPU loop finishes in minutes
        on, omiss = args.oracle_n, 0.90
        if world == 1 or on >= 256 * world:
            small, train, held = fit_map(on, d, omiss, 7)
        if rank == 0 and small is not None:
            from oracle import cpu_oracle
            cpu_oracle.build(ref=False)
            t0 = time.perf_counter()
            c = cpu_oracle.optimize_layout_exact(*train, max_iter, *hp, seed=0)
            dist_h = np.linalg.norm(c["positions"][held[0]] - c["positions"][held[1]], axis=1)
            cpu = {"iterations": c["iterations"], "converged": c["converged"], "edge_mae_train": c["final_mae"],
                   "heldout_mae": float(np.abs(held[2] - dist_h).mean()), "wall_s": time.perf_counter() - t0,
                   "what": "oracle/topolow_oracle.cpp = the reference's sequential std::shuffle loop (src/optimization.cpp:108-382), 1 core"}
    if rank == 0:
        line = {"metric": "held-out MAE of the converged map", "n_gpus": world, "mode": "rowblock", "target": big,
                "comparison": {"gpu": small, "cpu_reference_loop": cpu,
                               "heldout_mae_ratio_gpu_over_cpu": (small["heldout_mae"] / cpu["heldout_mae"]) if (small and cpu) else None},
                "config": map_config(args.workload, n, d, missing, big["train_edges"] + big["heldout_cells"],
                                     early_stop="on: relative_epsilon 1e-4, convergence_counter 5, checked every 3 iterations "
                                                "(the package defaults, R/core.R:184-199)")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main_map(args, n, d, missing):
    import torch
    import torch.distributed as dist
    from tools import synth
    from topolow_b200 import _lib
    from topolow_b200.rowblock import RowBlockMap

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: topolow_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    prec = {"f32": _lib.PREC_F32, "f64": _lib.PREC_F64_EXACT}[args.precision]
    prob = synth.make_problem(n, d, missing, seed=0)
    fa = synth.fit_args(prob)
    E = int(len(prob["edge_i"]))
    pairs = n * (n - 1) // 2
    warm = max(args.warmup, 3) if args.warmup else 0
    probe_iters = 6                                       # per-kernel event timing after the timed region
    total_iters = warm + args.steps + probe_iters         # every iteration run is inside n_iter
    nw = total_iters + 1                                  # convergence window > n_iter: no early stop
    hp = (HYPER["k0"], HYPER["cooling_rate"], HYPER["c_repulsion"], HYPER["relative_epsilon"])
    freq = HYPER["convergence_check_freq"]
    rowblock = args.mode == "rowblock"
    one_map = rowblock or world == 1

    # ---- device-resident leg -------------------------------------------------------------------
    kt = None
    if rowblock:
        m = RowBlockMap(*fa, total_iters, *hp, nw, freq, rank=rank, world_size=world, device=local, seed=0)
        info0 = m.info()
        m.step(warm)
        launches_before = m.info()["launches"]
        barrier()
        with ClockSampler(local) as clk:
            t0 = time.perf_counter()
            ms = m.step(args.steps)                       # CUDA events on the launching stream around the K iterations
            barrier()
            wall_ms = (time.perf_counter() - t0) * 1e3
        launches = m.info()["launches"] - launches_before
        timed = m.result(trace=True) if args.dump_outputs else None   # before the probe iterations move the map on
        kt = m.time_kernels(probe_iters)                  # events around every launch (all ranks step together)
        res = m.result()
        info0["tensor_form_iterations"] = m.info().get("tensor_form_iterations", -1)   # read back by result(): of all iterations run
        m.close()
    else:
        plan = _lib.Plan(*fa, total_iters, *hp, nw, freq, precision=prec, seed=0, device=local)
        info0 = plan.info()
        plan.run(warm)
        launches_before = plan.info()["launches"]
        barrier()
        with ClockSampler(local) as clk:
            t0 = time.perf_counter()
            ms = plan.run(args.steps)
            barrier()
            wall_ms = (time.perf_counter() - t0) * 1e3
        launches = plan.info()["launches"] - launches_before
        res = timed = plan.result(trace=bool(args.dump_outputs))
        plan.close()
    if args.dump_outputs and rank == 0:
        assert timed["iterations_run"] == warm + args.steps, (timed["iterations_run"], warm, args.steps)
        dump_outputs(args.dump_outputs, timed)
    ms_max, wall_max = max_over_ranks(ms, wall_ms)
    # one map: every unordered pair once per iteration whatever the rank count (strong scaling);
    # exact mode on several GPUs: `world` independent maps (weak scaling)
    maps = 1 if one_map else world
    value = maps * pairs * args.steps / (ms_max * 1e-3)

    # ---- end-to-end leg: host buffers through the public call -----------------------------------
    e2e = None
    if not args.no_e2e:
        def one_call(arrays):
            barrier()
            t0 = time.perf_counter()
            if rowblock and world > 1:
                mm = RowBlockMap(*arrays, args.steps, *hp, args.steps + 1, freq, rank=rank, world_size=world, device=local, seed=0)
                mm.step(args.steps)
                r2 = mm.result()
                mm.close()
            else:
                r2 = _lib.fit(*arrays, args.steps, *hp, args.steps + 1, freq, precision=prec, seed=0, device=local,
                              mode=_lib.MODE_ROWBLOCK if rowblock else _lib.MODE_COLOURED)
            barrier()
            return max_over_ranks(time.perf_counter() - t0)[0], r2
        # the step's inputs wait in pinned host memory (page-locked views handed to the C ABI as plain pointers) ...
        keep_pinned = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in fa[1:]]
        wall_pin, r2 = one_call((fa[0],) + tuple(t.numpy() for t in keep_pinned))
        # ... and, as an R caller would hand them over, in ordinary pageable memory
        wall_page, _ = one_call(fa)
        h2d = n * d * 8 + n * 4 + E * (4 + 4 + 8 + 4)
        d2h = n * d * 8
        e2e = {"value": maps * pairs * r2["iterations_run"] / wall_pin, "unit": "pair-updates/s",
               "h2d_bytes_per_step": h2d // max(args.steps, 1), "d2h_bytes_per_step": d2h // max(args.steps, 1),
               "note": "one fit of K iterations from pinned host buffers through the C ABI (topolow_fit; per rank topolow_shard_* "
                       "when sharded: every rank uploads the edge list and keeps its rows): upload, record build, K iterations, "
                       "download; bytes are the call's totals (per rank) divided by K",
               "wall_s": wall_pin, "kernel_ms": r2["device_ms"],
               "pageable": {"value": maps * pairs * r2["iterations_run"] / wall_page, "wall_s": wall_page,
                            "note": "the same call with the caller's arrays in pageable memory (what R hands over)"}}

    # ---- the exact (coloured) mode beside it, 1 GPU: the reference's sequential semantics -----------
    exact = None
    if rowblock and world == 1 and not args.no_exact and prec == _lib.PREC_F32:
        ex_iters = 9
        plan = _lib.Plan(*fa, ex_iters, *hp, ex_iters + 1, freq, precision=prec, seed=0, device=local)
        plan.run(3)
        ex_ms = plan.run(6)
        plan.close()
        exact = {"ms_per_step": ex_ms / 6, "value": pairs * 6 / (ex_ms * 1e-3), "unit": "pair-updates/s",
                 "note": "mode=coloured (tile_kernel): matchings of commuting pair updates, one sequential order of the reference's "
                         "loop per iteration; 6 iterations after 3 warm-up"}

    # ---- Metric 2 in the same line ---------------------------------------------------------------------
    cv = None
    if not args.no_cv:
        cn, _cd, cmiss = WORKLOADS["cfg5"]
        cv = cv_grid_measure(local, rank, world, args.samples, args.fit_iters, args.cv_steps, 1, cn, cmiss, not args.no_cpu)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline ---------------------------------------------------------------------------------
    def tracked_ncu(kernel):
        """Pipe utilisation of `kernel` from the tracked ncu capture (profiles/traffic.json), else None."""
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                e = json.load(f).get("%s/%d/%s" % (args.workload, world, kernel))
            return e.get("ncu") if e else None
        except (OSError, ValueError, KeyError):
            return None

    def tracked_traffic(kernel):
        """DRAM bytes per launch of `kernel` from a tracked ncu capture of this workload at this GPU count, else None."""
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                e = json.load(f).get("%s/%d/%s" % (args.workload, world, kernel))
            return e["bytes"] if e else None
        except (OSError, ValueError, KeyError):
            return None

    peaks, peak_src = measured_peaks()
    ffma_peak = _lib.microbench(0, local)      # flop/s, measured now on this GPU
    flop = flop_per_iter(n, d, E)
    if rowblock:
        # the dominant kernel: repulse_kernel, one launch per iteration and rank, rows/world x (n - 1) one-sided
        # interactions = that many HALF pair updates of SURVEY 8d's 7d + 8 flop
        rep_flop = (7 * d + 8) * pairs / world
        rep_s = kt["repulse"] * 1e-3
        edge_b = edge_bytes_per_iter(n, d, E) / world
        form = info0.get("repulsion_form", 5)
        rep_names = {11: "image_tc_kernel + image_t2_kernel + repulse_tc2_kernel<ndim/2> (tcgen05: pair distances as a 3-pass TF32 GEMM into "
                         "TMEM, weights computed in place by the FP32 / special-function pipes, sum w x_j and sum w as an A-from-TMEM GEMM)",
                     10: "image_tc_kernel + repulse_tc_kernel<ndim/2> (pair distances as a 3-pass TF32 GEMM on tcgen05 with TMEM "
                         "accumulators; weights and accumulation on the FP32 pipes)"}
        rep_kernel = {11: "repulse_tc2_kernel", 10: "repulse_tc_kernel"}.get(form, "repulse_kernel")
        one_sided = pairs * 2.0 / world                       # interactions one launch evaluates (every pair from both sides)
        mufu_peak = _lib.microbench(4, local) * 32.0          # MUFU lane-operations / s, measured now on this GPU
        mufu_per = 1.0 if form == 11 else 3.0                 # form 11 in a spread-out map: one rsqrt (the weight's series form); forms 5 / 10: sqrt, lg2, ex2
        roofline = {"bound": "fp32", "kernel": rep_names.get(form, "repulse_kernel<ndim/2, 2 rows per thread>") + " (one launch per iteration and rank)",
                    "repulsion_form": form,
                    "achieved": rep_flop / rep_s / 1e12, "peak": ffma_peak / 1e12, "unit": "TFLOP/s",
                    "frac": rep_flop / rep_s / ffma_peak,
                    "peak_source": "topolow_microbench FFMA, measured live on this GPU (FP32 is not in MEASURED_PEAKS.json)",
                    "algorithmic_flop_per_launch": rep_flop, "launch_ms": kt["repulse"],
                    "note": "algorithmic = (7 ndim + 8) flop per unordered pair (SURVEY 8d) against the FP32 FFMA peak, the denominator the "
                            "north-star names; the kernel visits every pair from both sides (one-sided updates). In form 11 both "
                            "contractions (the 5 ndim flop of the distance and the accumulation) run on the tensor cores, so the fraction "
                            "exceeds what the FP32 pipes alone could reach. What is left on the FP32 side is one rsqrt + a cubic per "
                            "interaction (7.6 instructions); ncu (`tracked_ncu`, profiles/r2_ncu_rowblock_cfg4.md): 75 % of the issue slots, "
                            "FMA pipe 40 %, special-function unit 45 %, tensor-core unit 40 % - the pass is bound by instruction issue. The "
                            "FP32 difference form (ndim < 5, and iterations 0-1 of the reference's start, chosen on the device) ran at 0.51",
                    "special_function_unit": {"ops_per_launch": mufu_per * one_sided, "achieved": mufu_per * one_sided / rep_s / 1e12,
                                              "peak": mufu_peak / 1e12, "unit": "T lane-ops/s",
                                              "frac": mufu_per * one_sided / rep_s / mufu_peak,
                                              "peak_source": "topolow_microbench MUFU.RSQ, measured live on this GPU"},
                    "tensor": {"executed_flop_per_launch": (2.0 * 56 + 2.0 * 32) * one_sided if form == 11 else
                                                           (2.0 * 56 * one_sided if form == 10 else 0.0),
                               "achieved_tflops": ((2.0 * 56 + 2.0 * 32) if form == 11 else (2.0 * 56 if form == 10 else 0.0)) * one_sided / rep_s / 1e12,
                               "peak_tflops": 0.5 * float(peaks.get("bf16_tflops", 0.0)),
                               "frac": (((2.0 * 56 + 2.0 * 32) if form == 11 else (2.0 * 56 if form == 10 else 0.0)) * one_sided / rep_s / 1e12
                                        / (0.5 * float(peaks["bf16_tflops"]))) if peaks.get("bf16_tflops") else None,
                               "peak_source": "half of the dense bf16 figure of MEASURED_PEAKS.json (%s): TF32 runs at half the bf16 rate" % peak_src,
                               "note": "executed TF32 flop: GEMM 1 K = 24 + 16 + 16 (hi x hi, hi x lo, lo x hi with the half norms in K), "
                                       "GEMM 2 K = 32 partners x N = 32 columns (17 used); TF32 dense peak is half of the bf16 figure in "
                                       "MEASURED_PEAKS.json - the tensor pipe is not the bound"},
                    "traffic": tracked_traffic(rep_kernel),
                    "tracked_ncu": tracked_ncu(rep_kernel),
                    "kernels_ms": kt,
                    "edge_pass": {"bound": "hbm", "kernel": "mae_kernel (edge MAE on check iterations)",
                                  "achieved": edge_b / (kt["mae"] * 1e-3) / 1e9 if kt["mae"] > 0 else None, "peak": peaks["hbm_gbs"],
                                  "unit": "GB/s", "frac": edge_b / (kt["mae"] * 1e-3) / 1e9 / peaks["hbm_gbs"] if kt["mae"] > 0 else None,
                                  "peak_source": peak_src, "algorithmic_bytes_per_launch": edge_b, "launch_ms": kt["mae"],
                                  "traffic": tracked_traffic("mae_kernel"),
                                  "gather_bytes_per_launch": info0["mae_records"] * (8 + 4 * ((d + 3) // 4 * 4)),
                                  "note": "SURVEY 8d: 16 bytes per measured pair + every FP32 position read and written once, per rank. "
                                          "The kernel streams 8-byte records (DRAM) and gathers one partner row per record from the "
                                          "L2-resident replica (gather_bytes_per_launch): ncu shows it bound by the L1TEX gather path "
                                          "(66 % of peak; L2 25 %, DRAM 8 %), not by HBM"},
                    "spring_pass": {"launch_ms": kt["spring"],
                                    "achieved_gbs": (2 * E * 8 / world + 2 * n * d * 4 / world) / (kt["spring"] * 1e-3) / 1e9,
                                    "note": "walks both directions of every measured pair (8-byte records) and gathers one 64-byte "
                                            "partner row per record from the L2-resident replica"}}
    else:
        kernel_s = ms_max * 1e-3 / args.steps        # device time of one iteration (all of it is tile_kernel launches)
        ach = flop / kernel_s
        roofline = {"bound": "fp32", "kernel": "tile_kernel<D,%s>" % ("FastF32" if prec == 0 else "ExactF64"),
                    "achieved": ach / 1e12, "peak": ffma_peak / 1e12, "unit": "TFLOP/s", "frac": ach / ffma_peak,
                    "peak_source": "topolow_microbench FFMA, measured live on this GPU (not in MEASURED_PEAKS.json)",
                    "flop_per_iteration": flop, "traffic": None}

    cpu = None
    if not args.no_cpu:
        from oracle import cpu_oracle
        cpu_oracle.build(ref=False)
        sample = int(min(pairs, 1e8))
        rate, dt, desc = cpu_sample(prob, n, d, sample)
        rate3, dt3, _ = cpu_sample(prob, n, d, sample, kind="fast")
        cpu = {"value": rate, "unit": "pair-updates/s", "cores": 1, "kind": "port",
               "sample": f"{desc}; {dt:.1f} s of CPU work (oracle = CPU restatement of src/optimization.cpp, g++ -O2 = R's package "
                         "default, 1 thread: a fit is single-threaded in the reference)",
               "value_O3": rate3, "O3_note": f"the same sample built with g++ -O3 -march=x86-64-v3 ({dt3:.1f} s)"}

    if rowblock:
        par = ("1 GPU, row-block mode" if world == 1 else
               f"one map, {world} row blocks (one per GPU): every rank computes the one-sided updates of its rows against a replica of all "
               f"positions and stores its new rows into every replica over NVLink inside the spring kernel ({info0['peer_store_bytes_per_iteration']} "
               "bytes per rank and iteration), one flag per peer and iteration; no host code, NCCL call or torch op in the loop")
    else:
        par = "1 GPU, exact coloured mode" if world == 1 else f"{world} independent replicas of the exact mode (no collective)"
    line = {
        "metric": "pair-updates/s", "value": value, "unit": "pair-updates/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "strong" if one_map else "weak", "vs_baseline": None,
        "dtype": "f32" if prec == 0 else "f64", "data": "synthetic",
        "config": map_config(args.workload, n, d, missing, E),
        "mode": args.mode, "parallelism": par, "layout": info0,
        "wall_ms_per_step": wall_max / args.steps,
        "final_mae": res["final_mae"],
        "clocks": clk.summary(),
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "exact_mode": exact,
        "cv_grid": cv,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
