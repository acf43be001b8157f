"""Voxel-grid downsampling (gicpVoxelDownsample) on the GPU: throughput on the bench batch, latency of single clouds,
and the 4x-density config-4 batch registered raw and after downsampling.  Needs a CUDA device; writes one JSON file.
    python scripts/voxel_bench.py --out voxel_bench.json [--pairs-dense 1024]
Times are CUDA events around each call (the call synchronises its stream), medians of the repeats."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("voxel_bench.py needs a CUDA device")
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    res = {"card (name, power limit, max SM clock)": card()}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        peaks = {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    res["hbm_peak_gbs"] = peak
    res["hbm_peak_source"] = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    i64p = C.POINTER(C.c_int64)

    def timed(eng, pts, off, leaf, out, oo, vox, cnt, reps, min_points=1):
        """median ms of gicpVoxelDownsample with preallocated outputs (CUDA events; the call synchronises)"""
        st = torch.cuda.current_stream()
        offa = np.ascontiguousarray(off, dtype=np.int64)
        ts = []
        for _ in range(reps + 1):   # the first call warms up this shape
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            rc = eng.lib.gicpVoxelDownsample(eng._h, C.c_void_p(pts.data_ptr()), offa.ctypes.data_as(i64p),
                                             len(offa) - 1, float(leaf), min_points, C.c_void_p(out.data_ptr()),
                                             oo.ctypes.data_as(i64p), C.c_void_p(vox.data_ptr()),
                                             C.c_void_p(cnt.data_ptr()), C.c_void_p(st.cuda_stream))
            b.record(st)
            b.synchronize()
            assert rc == 0, eng.lib.gicpGetLastError()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts[1:]))

    def host_latency(eng, pts, off, leaf, out, oo, vox, cnt, reps):
        offa = np.ascontiguousarray(off, dtype=np.int64)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        ts = []
        for _ in range(reps + 3):
            t0 = time.perf_counter()
            eng.lib.gicpVoxelDownsample(eng._h, C.c_void_p(pts.data_ptr()), offa.ctypes.data_as(i64p), len(offa) - 1,
                                        float(leaf), 1, C.c_void_p(out.data_ptr()), oo.ctypes.data_as(i64p),
                                        C.c_void_p(vox.data_ptr()), C.c_void_p(cnt.data_ptr()), st)
            ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts[3:]))

    # ---- 1. the bench batch's source side ----
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    src, tgt, off_t, T_true = synthetic.patches3d_batch_device(args.pairs, n=args.points, seed=0, **cfg)
    off = off_t.cpu().numpy()
    n = src.shape[0]
    del tgt
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    out = torch.empty_like(src)
    vox = torch.empty((n,), dtype=torch.int32, device="cuda")
    cnt = torch.empty((n,), dtype=torch.int32, device="cuda")
    oo = np.zeros(len(off), dtype=np.int64)
    eng.profile(True)
    grid_ms = []
    for _ in range(args.reps + 1):
        eng.set_source(src, off)
        grid_ms.append(eng.profile_read()["grid_build"][0])
    eng.profile(False)
    res["bench_batch"] = dict(clouds=args.pairs, points=n, grid_build_one_side_ms=float(np.median(grid_ms[1:])))
    rows = []
    for leaf in (0.25, 0.5, 1.0):
        ms = timed(eng, src, off, leaf, out, oo, vox, cnt, args.reps)
        m = int(oo[-1])
        algo = 12.0 * n + 4.0 * n + 16.0 * m     # read the point, write voxel_of, write the output row + its count
        gbs = algo / (ms * 1e-3) / 1e9
        rows.append(dict(leaf_m=leaf, ms=ms, output_points=m, mean_points_per_voxel=n / max(m, 1),
                         points_per_s=n / (ms * 1e-3), algorithmic_GBps=gbs, share_of_hbm_peak=gbs / peak,
                         vs_grid_build=ms / res["bench_batch"]["grid_build_one_side_ms"]))
        print(json.dumps(rows[-1]), flush=True)
    res["bench_batch"]["downsample"] = rows
    del out, vox, cnt, src
    torch.cuda.empty_cache()

    # ---- 2. latency of single clouds ----
    lat = {}
    rng = np.random.default_rng(0)
    e2 = GicpEngine(2, "f64")
    p = torch.as_tensor(rng.uniform(-200, 200, size=(360, 2)), device="cuda")
    bufs = (torch.empty_like(p), np.zeros(2, dtype=np.int64), torch.empty(360, dtype=torch.int32, device="cuda"),
            torch.empty(360, dtype=torch.int32, device="cuda"))
    lat["2d_360_points_leaf_1m"] = dict(device_ms=timed(e2, p, [0, 360], 1.0, *bufs, 50),
                                        host_ms=host_latency(e2, p, [0, 360], 1.0, *bufs, 50))
    s, _, _ = synthetic.patches3d_pair(**synthetic.CONFIG3, seed=1)
    for name, pts, leaf in (("3d_100k_points_leaf_0.5m", s, 0.5),
                            ("3d_100k_points_all_in_one_voxel", rng.uniform(0.01, 0.99, size=(100000, 3)).astype(np.float32), 1.0)):
        p = torch.as_tensor(pts, device="cuda")
        bufs = (torch.empty_like(p), np.zeros(2, dtype=np.int64), torch.empty(len(p), dtype=torch.int32, device="cuda"),
                torch.empty(len(p), dtype=torch.int32, device="cuda"))
        lat[name] = dict(device_ms=timed(eng, p, [0, len(p)], leaf, *bufs, 50),
                         host_ms=host_latency(eng, p, [0, len(p)], leaf, *bufs, 50), output_points=int(bufs[1][-1]))
    # the bench batch with every cloud in one voxel each
    big = torch.rand((args.pairs * args.points, 3), device="cuda") * 0.98 + 0.01
    bufs = (torch.empty_like(big), np.zeros(len(off), dtype=np.int64),
            torch.empty(len(big), dtype=torch.int32, device="cuda"), torch.empty(len(big), dtype=torch.int32, device="cuda"))
    lat["bench_batch_every_cloud_one_voxel"] = dict(device_ms=timed(eng, big, off, 1.0, *bufs, args.reps))
    del big, bufs
    res["latency"] = lat
    print(json.dumps(lat), flush=True)
    torch.cuda.empty_cache()

    # ---- 3. 4x-density config-4 pairs: raw vs downsampled (1 m) registration ----
    P = args.pairs_dense
    src, tgt, off_t, T_true = synthetic.patches3d_batch_device(P, n=4 * args.points, seed=8, **cfg)
    off = off_t.cpu().numpy()
    Tt = T_true.cpu().numpy()

    def errors(T):
        dR = np.einsum("pji,pjk->pik", T[:, :3, :3], Tt[:, :3, :3])
        ang = np.arccos(np.clip((np.trace(dR, axis1=1, axis2=2) - 1) / 2, -1, 1))
        tr = np.linalg.norm(T[:, :3, 3] - Tt[:, :3, 3], axis=1)
        return dict(rot_max_rad=float(ang.max()), rot_median_rad=float(np.median(ang)), trans_max_m=float(tr.max()),
                    trans_median_m=float(np.median(tr)))

    def run(downsample):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if downsample:
            ds, so = eng.voxel_downsample(src, off, voxel_size=1.0)
            dt, to = eng.voxel_downsample(tgt, off, voxel_size=1.0)
            eng.set_pair(dt, ds, to, so)
        else:
            eng.set_pair(tgt, src, off, off)
        r = eng.register(history=False)
        torch.cuda.synchronize()
        dtm = time.perf_counter() - t0
        info = dict(s=dtm, pairs_per_s=P / dtm, converged=int((r.converged_at >= 0).sum()), **errors(r.T.cpu().numpy()))
        if downsample:
            info["points_per_cloud_median"] = float(np.median(np.diff(so)))
        return info

    dense = {}
    for mode in ("raw", "downsampled_1m", "raw", "downsampled_1m"):   # second round after warm-up is reported
        dense[mode] = run(mode != "raw")
    dense["pairs"] = P
    dense["points_per_cloud_raw"] = 4 * args.points
    res["dense_config4"] = dense
    print(json.dumps(dense), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
