"""Does the spring walk run under the repulsion pass?  torch.profiler (CUDA activities) over a few row-block iterations
of a bench workload on one GPU; prints, per iteration, the device intervals of repulse_tc2_kernel and spring_kernel and
how much of the walk lies inside the pass.

    python tools/gpu_overlap_trace.py [--workload cfg4] [--iters 6] [--out DIR]

--out keeps the Chrome trace (DIR/overlap_trace.json) and writes the summary as DIR/overlap_summary.json."""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload table and hyper-parameters the bench uses)
from tools import synth  # noqa: E402


def kernel_intervals(trace_path):
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    out = {"repulse_tc2_kernel": [], "spring_kernel": []}
    for e in events:
        if e.get("cat") != "kernel":
            continue
        for k in out:
            if k in e.get("name", ""):
                out[k].append((float(e["ts"]), float(e["ts"]) + float(e["dur"])))
    return {k: sorted(v) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4", choices=["cfg4", "cfg3", "small"])
    ap.add_argument("--iters", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=4, help="iterations before the trace (the first ones run the FP32 form)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from topolow_b200.rowblock import RowBlockMap

    n, d, missing = bench.WORKLOADS[args.workload]
    fa = synth.fit_args(synth.make_problem(n, d, missing, seed=0))
    hp = (bench.HYPER["k0"], bench.HYPER["cooling_rate"], bench.HYPER["c_repulsion"], bench.HYPER["relative_epsilon"])
    total = args.warmup + args.iters
    m = RowBlockMap(*fa, total, *hp, total + 1, bench.HYPER["convergence_check_freq"], rank=0, world_size=1, device=0, seed=0)
    m.step(args.warmup)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.step(args.iters)
        torch.cuda.synchronize()
    m.close()

    out_dir = args.out or tempfile.mkdtemp()
    os.makedirs(out_dir, exist_ok=True)
    trace = os.path.join(out_dir, "overlap_trace.json")
    prof.export_chrome_trace(trace)
    iv = kernel_intervals(trace)
    rows = []
    for (r0, r1), (s0, s1) in zip(iv["repulse_tc2_kernel"], iv["spring_kernel"]):   # one of each per iteration
        inside = max(0.0, min(s1, r1) - max(s0, r0))
        rows.append({"repulse_us": [0.0, round(r1 - r0, 1)], "spring_us": [round(s0 - r0, 1), round(s1 - r0, 1)],
                     "spring_inside_fraction": round(inside / max(s1 - s0, 1e-9), 3)})
    summary = {"workload": args.workload, "device": torch.cuda.get_device_name(0), "iterations": rows,
               "all_inside": bool(rows) and all(r["spring_inside_fraction"] >= 0.999 for r in rows)}
    print(json.dumps(summary, indent=1))
    if args.out:
        with open(os.path.join(out_dir, "overlap_summary.json"), "w") as f:
            json.dump(summary, f, indent=1)
    else:
        os.remove(trace)


if __name__ == "__main__":
    main()
