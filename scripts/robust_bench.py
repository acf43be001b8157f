"""Robust kernels (gicpSetRobustKernel) on the GPU: cost on the bench workload, accuracy on inputs with structured
outliers, and the odometry drive with and without a kernel.  Needs a CUDA device; writes one JSON file.
    python scripts/robust_bench.py --out robust_bench.json [--pairs 1024]
- bench: the config-4 batch (32768 points per cloud) registered with no kernel and with each kind; register time by CUDA
  events (median of --reps, set-up excluded), pairs/s, mean outer iterations, and the accumulate stage (K3b) from
  gicpProfile in a separate profiled run.
- moved_patch: the moved-object pairs of tests/test_gpu_robust.py (one patch of eight shifted 1 m along its normal,
  inside the 2 m gate), seeds 0..15, error against the generating motion for each kind at a few scales.
- odometry: scripts/odometry_eval.py (360 rays, 36 scans) without and with each kind."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KINDS = [None, "huber", "cauchy", "tukey"]
BENCH_SCALES = {None: None, "huber": 0.1, "cauchy": 0.1, "tukey": 0.3}    # metres; the clouds carry 2 cm noise
MOVED_SCALES = {"huber": [0.1, 0.2, 0.5], "cauchy": [0.05, 0.1, 0.2], "tukey": [0.3, 0.5, 1.0]}
ODO_SCALES = {"huber": 4.0, "cauchy": 4.0, "tukey": 12.0}                # pixels; the ranges carry +-2 px noise


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def motion_error(T, Tg):
    dR = T[:3, :3] @ Tg[:3, :3].T
    return float(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))), float(np.linalg.norm(T[:3, 3] - Tg[:3, 3]))


def bench(args, torch):
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    src, tgt, off, Tg = synthetic.patches3d_batch_device(args.pairs, n=args.points, seed=0)
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    eng.set_target(tgt, off.cpu().numpy())
    eng.set_source(src, off.cpu().numpy())
    Tg = Tg.cpu().numpy()
    out = {}
    for kind in KINDS:
        eng.set_robust_kernel(kind, BENCH_SCALES[kind])
        eng.register(history=False)                       # warm-up
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = eng.register(history=False)
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        n_outer = r.n_outer.cpu().numpy()
        errs = np.array([motion_error(T, g) for T, g in zip(r.T.cpu().numpy(), Tg)])
        eng.profile(True)
        eng.register(history=False)
        prof = eng.profile_read()
        eng.profile(False)
        ms = float(np.median(times))
        out[str(kind)] = dict(scale_m=BENCH_SCALES[kind], register_ms_median=ms, register_ms_all=times,
                              pairs_per_s=args.pairs / (ms / 1e3), mean_outer_iterations=float(n_outer.mean()),
                              max_outer_iterations=int(n_outer.max()),
                              accumulate_ms_profiled=prof["accumulate"][0], accumulate_launches=prof["accumulate"][1],
                              correspond_ms_profiled=prof["correspond"][0],
                              rot_err_median_rad=float(np.median(errs[:, 0])), trans_err_median_m=float(np.median(errs[:, 1])))
        print(kind, out[str(kind)]["register_ms_median"], out[str(kind)]["mean_outer_iterations"], flush=True)
    return out


def moved_patch(torch):
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    srcs, tgts, Tgs = [], [], []
    for seed in range(16):
        s, t, T = synthetic.patches3d_pair(n=3000, n_patches=8, cube=30.0, patch=20.0, seed=seed, moved_patches=1,
                                           moved_offset=1.0)
        srcs.append(s)
        tgts.append(t)
        Tgs.append(T)
    off = np.arange(17, dtype=np.int64) * 3000
    eng = GicpEngine(3, "f64")
    eng.set_params(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0)
    eng.set_target(torch.as_tensor(np.concatenate(tgts), device="cuda").double(), off)
    eng.set_source(torch.as_tensor(np.concatenate(srcs), device="cuda").double(), off)
    rows = []
    for kind in KINDS:
        for c in ([None] if kind is None else MOVED_SCALES[kind]):
            eng.set_robust_kernel(kind, c)
            r = eng.register(history=False)
            torch.cuda.synchronize()
            e = np.array([motion_error(T, g) for T, g in zip(r.T.cpu().numpy(), Tgs)])
            rows.append(dict(kind=str(kind), scale_m=c, rot_err_median_rad=float(np.median(e[:, 0])),
                             rot_err_max_rad=float(e[:, 0].max()), trans_err_median_m=float(np.median(e[:, 1])),
                             trans_err_max_m=float(e[:, 1].max()), mean_outer_iterations=float(r.n_outer.float().mean())))
            print(rows[-1], flush=True)
    return rows


def odometry():
    rows = []
    for kind in KINDS:
        cmd = [sys.executable, os.path.join(ROOT, "scripts", "odometry_eval.py"), "360", "36"]
        if kind is not None:
            cmd += ["--robust", f"{kind}:{ODO_SCALES[kind]}"]
        out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
        rows.append(json.loads(out))
        print(rows[-1], flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file the results are written to")
    ap.add_argument("--pairs", type=int, default=1024)
    ap.add_argument("--points", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("robust_bench.py needs a CUDA device")
    res = {"card (name, power limit, max SM clock)": card(), "pairs": args.pairs, "points_per_cloud": args.points}
    res["bench_config4"] = bench(args, torch)
    res["moved_patch"] = moved_patch(torch)
    res["odometry_360rays_36scans"] = odometry()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
