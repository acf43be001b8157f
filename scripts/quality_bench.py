"""Cost of gicpEvaluate (registration quality at device transforms) against the registration it follows.  Needs a CUDA
device; writes one JSON file.
    python scripts/quality_bench.py --out quality_bench.json [--pairs 1024] [--reps 7]
Three workloads, each registered once and then timed by CUDA events on the current stream (median of --reps, set-up
excluded, every shape warmed up first):
- batch:  the config-4 batch (synthetic.patches3d_batch_device, 32768 points per cloud), --pairs pairs, f32 storage;
- pair:   one such pair (the first of the batch's generator);
- scan:   one 360-ray scan pair of the robot demo (tests/demo_inputs.lidar_sequence), f64, the demo's parameters.
For each: register ms, evaluate ms (at register().T, no synchronisation in between), and their ratio."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def time_ms(torch, fn, reps):
    fn()                                                  # warm-up of this shape
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def measure(torch, eng, reps, what):
    r = eng.register(history=False)
    T = r.T
    reg = time_ms(torch, lambda: eng.register(history=False), reps)
    ev = time_ms(torch, lambda: eng.evaluate(T), reps)
    q = eng.evaluate(T)
    torch.cuda.synchronize()
    row = dict(workload=what, register_ms_median=float(np.median(reg)), evaluate_ms_median=float(np.median(ev)),
               evaluate_over_register=float(np.median(ev) / np.median(reg)), register_ms_all=reg, evaluate_ms_all=ev,
               mean_outer_iterations=float(r.n_outer.float().mean()), mean_fitness=float(q.fitness.mean()),
               mean_inlier_rmse=float(q.inlier_rmse.mean()))
    print(what, row["register_ms_median"], row["evaluate_ms_median"], row["evaluate_over_register"], flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file the results are written to")
    ap.add_argument("--pairs", type=int, default=1024)
    ap.add_argument("--points", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("quality_bench.py needs a CUDA device")
    import demo_inputs
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine

    rows = []
    for n_pairs, what in ((args.pairs, f"config4 batch of {args.pairs} pairs"), (1, "config4 single pair")):
        src, tgt, off, _ = synthetic.patches3d_batch_device(n_pairs, n=args.points, seed=0)
        eng = GicpEngine(3, "f32")
        eng.set_params(**synthetic.CONFIG4_PARAMS)
        eng.set_target(tgt, off.cpu().numpy())
        eng.set_source(src, off.cpu().numpy())
        rows.append(measure(torch, eng, args.reps, what))
        eng.close()
        del src, tgt
        torch.cuda.empty_cache()
    scans, _ = demo_inputs.lidar_sequence(seed=3, num_rays=360, n_scans=2)
    eng = GicpEngine(2, "f64")
    eng.set_params(max_distance_nearest_neighbors=200.0, tolerance=1.0)
    eng.set_target(np.asarray(scans[1], np.float64))
    eng.set_source(np.asarray(scans[0], np.float64))
    rows.append(measure(torch, eng, max(args.reps, 50), "360-ray scan pair"))
    res = dict(card=card(), points_per_cloud=args.points, reps=args.reps, rows=rows)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
