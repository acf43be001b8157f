"""Voxel distributions (gicpSetVoxelized) against raw GICP and downsample + GICP on the GPU, on the inputs of
scripts/voxel_bench.py.  Needs a CUDA device; writes one JSON file.
    python scripts/voxel_gicp_bench.py --out profiles/voxel_gicp_bench.json [--pairs 4096] [--pairs-dense 1024]
1. the bench batch (CONFIG4, CONFIG4_PARAMS): set-up + register time of every arm, and its per-stage split
   (profile_read, a separate run with per-stage timing on);
2. the 4x-density config-4 pairs: the same arms plus rotation / translation error against the generating motion;
3. one 100k-point pair (CONFIG3) and one 360-ray scan pair: latency of the voxelized set-up of both sides.
Times are a host clock around work that ends in a device synchronise; every arm runs once to warm up, then the
median of --reps runs is reported."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file the results are written to")
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--points", type=int, default=32768)
    ap.add_argument("--pairs-dense", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("voxel_gicp_bench.py needs a CUDA device")
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    res = {"card (name, power limit, max SM clock)": card()}
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)

    def setup(arm, src, tgt, off):
        if arm == "raw":
            eng.set_pair(tgt, src, off, off)
            return None
        # "<kind>_<leaf>m" or "<kind>_<leaf>m_min<m>"
        parts = arm.split("_")
        mp = int(parts[-1][3:]) if parts[-1].startswith("min") else 1
        leaf = float((parts[-2] if parts[-1].startswith("min") else parts[-1])[:-1])
        if arm.startswith("downsample"):
            ds, so = eng.voxel_downsample(src, off, voxel_size=leaf, min_points=mp)
            dt, to = eng.voxel_downsample(tgt, off, voxel_size=leaf, min_points=mp)
            eng.set_pair(dt, ds, to, so)
        else:
            _, to = eng.set_target_voxelized(tgt, off, voxel_size=leaf, min_points=mp)
            _, so = eng.set_source_voxelized(src, off, voxel_size=leaf, min_points=mp)
        return float(np.median(np.diff(so))), float(np.median(np.diff(to)))

    def run(arm, src, tgt, off, Tt=None):
        ts, tset = [], []
        for _ in range(args.reps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sizes = setup(arm, src, tgt, off)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            r = eng.register(history=False)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            ts.append(t2 - t0)
            tset.append(t1 - t0)
        P = len(off) - 1
        s = float(np.median(ts[1:]))
        info = dict(setup_plus_register_ms=1e3 * s, setup_ms=1e3 * float(np.median(tset[1:])), pairs_per_s=P / s,
                    converged=int((r.converged_at >= 0).sum()), n_outer_median=float(r.n_outer.float().median()))
        if sizes:
            info["points_per_cloud_median (source, target)"] = sizes
        if Tt is not None:
            T = r.T.cpu().numpy()
            dR = np.einsum("pji,pjk->pik", T[:, :3, :3], Tt[:, :3, :3])
            ang = np.arccos(np.clip((np.trace(dR, axis1=1, axis2=2) - 1) / 2, -1, 1))
            tr = np.linalg.norm(T[:, :3, 3] - Tt[:, :3, 3], axis=1)
            info.update(rot_median_rad=float(np.median(ang)), rot_max_rad=float(ang.max()),
                        trans_median_m=float(np.median(tr)), trans_max_m=float(tr.max()))
        # per-stage split: one more run with per-stage timing on (it disables the fused loop; not the timed run)
        eng.profile(True)
        setup(arm, src, tgt, off)
        eng.register(history=False)
        info["stages_ms"] = {k: v[0] for k, v in eng.profile_read().items()}
        eng.profile(False)
        print(arm, json.dumps(info), flush=True)
        return info

    arms = ("raw", "downsample_1.0m", "voxel_distributions_1.0m", "voxel_distributions_0.5m")

    # ---- 1. the bench batch ----
    src, tgt, off_t, _ = synthetic.patches3d_batch_device(args.pairs, n=args.points, seed=0, **cfg)
    off = off_t.cpu().numpy()
    res["bench_batch"] = dict(pairs=args.pairs, points_per_cloud=args.points,
                              **{a: run(a, src, tgt, off) for a in arms})
    del src, tgt
    torch.cuda.empty_cache()

    # ---- 2. 4x-density config-4 pairs ----
    src, tgt, off_t, T_true = synthetic.patches3d_batch_device(args.pairs_dense, n=4 * args.points, seed=8, **cfg)
    off = off_t.cpu().numpy()
    Tt = T_true.cpu().numpy()
    res["dense_config4"] = dict(pairs=args.pairs_dense, points_per_cloud=4 * args.points,
                                **{a: run(a, src, tgt, off, Tt) for a in arms[:3] + ("voxel_distributions_1.0m_min3",)})
    del src, tgt
    torch.cuda.empty_cache()

    # ---- 3. latency of the voxelized set-up of both sides ----
    lat = {}

    def latency(e, s, t, leaf, reps=30):
        ts = []
        for _ in range(reps + 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e.set_target_voxelized(t, voxel_size=leaf)
            e.set_source_voxelized(s, voxel_size=leaf)
            torch.cuda.synchronize()
            ts.append(1e3 * (time.perf_counter() - t0))
        return float(np.median(ts[3:]))

    s, t, _ = synthetic.patches3d_pair(**synthetic.CONFIG3, seed=1)
    e3 = GicpEngine(3, "f32")
    e3.set_params(**synthetic.CONFIG3_PARAMS)
    S, T = torch.as_tensor(s, device="cuda"), torch.as_tensor(t, device="cuda")
    lat["3d_100k_pair_leaf_0.5m_both_sides_ms"] = latency(e3, S, T, 0.5)
    import demo_inputs
    scans, _ = demo_inputs.lidar_sequence(seed=3, num_rays=360, n_scans=2)
    e2 = GicpEngine(2, "f64")
    e2.set_params(max_distance_nearest_neighbors=200.0)
    S2 = torch.as_tensor(np.asarray(scans[0], dtype=np.float64), device="cuda")
    T2 = torch.as_tensor(np.asarray(scans[1], dtype=np.float64), device="cuda")
    lat["2d_360_ray_pair_leaf_1_both_sides_ms"] = latency(e2, S2, T2, 1.0)
    res["latency"] = lat
    print(json.dumps(lat), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
