"""Pair lists against the one-to-one batch (gicpSetPairList, include/gicp_b200.h) on a multi-frame odometry graph.

    python scripts/pair_list_bench.py --out FILE [--clouds 1024] [--points 32768] [--span 3] [--runs 5] [--warmup 2]

N config-4 sequence clouds (synthetic.patches3d_sequence: one patch scene, config-4 density and noise, known poses),
with an edge from every cloud to each of the next `span` clouds.  Two ways to register every edge, alternated in one
process, each timed on the host clock from the first call to a device synchronise:
  - pair list: the N clouds set up once as a target set, gicpSetPairList(source_set = GICP_TARGET), gicpRegister;
  - one-to-one: the edges' clouds concatenated beforehand on the device (not timed), gicpSetTarget + gicpSetSource
    of the E clouds per side, gicpRegister.
The outputs (T, n_outer, converged_at) are compared bit for bit.  The gather of gicpSetPairList is also timed on its
own with CUDA events (median of repeats), with the bandwidth its bytes imply.  Accuracy: median rotation and
translation error of the pair-list results against the generated relative poses."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power)
    except Exception as e:   # the card name still comes from torch
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--clouds", type=int, default=1024)
    ap.add_argument("--points", type=int, default=32768)
    ap.add_argument("--span", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pair_list_bench needs a CUDA device")
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import TARGET, GicpEngine

    t0 = time.perf_counter()
    clouds, poses = synthetic.patches3d_sequence(a.clouds, n=a.points, seed=a.seed)
    gen_s = time.perf_counter() - t0
    n, N = a.points, a.clouds
    edges = np.array([(k, k + d) for d in range(1, a.span + 1) for k in range(N - d)], dtype=np.int64)
    E = len(edges)
    dev = torch.device("cuda", 0)
    pts = torch.as_tensor(np.concatenate(clouds), device=dev)
    del clouds
    off = np.arange(N + 1, dtype=np.int64) * n
    rows = torch.arange(n, device=dev)
    e_dev = torch.as_tensor(edges, device=dev)
    src_cat = pts[(e_dev[:, 0, None] * n + rows).reshape(-1)]
    tgt_cat = pts[(e_dev[:, 1, None] * n + rows).reshape(-1)]
    e_off = np.arange(E + 1, dtype=np.int64) * n
    prm = dict(synthetic.CONFIG4_PARAMS)

    pl = GicpEngine(3, "f32")
    pl.set_params(**prm)
    ref = GicpEngine(3, "f32")
    ref.set_params(**prm)

    def run_pairs():
        t = time.perf_counter()
        pl.set_target(pts, off)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        pl.set_pair_list(edges[:, 0], edges[:, 1], TARGET)
        r = pl.register(history=False)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return r, t2 - t, t1 - t

    def run_ref():
        t = time.perf_counter()
        ref.set_target(tgt_cat, e_off)
        ref.set_source(src_cat, e_off)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        r = ref.register(history=False)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return r, t2 - t, t1 - t

    for _ in range(a.warmup):
        run_pairs()
        run_ref()
    tp, tr, sp, sr = [], [], [], []
    for _ in range(a.runs):
        rp, x, s = run_pairs()
        tp.append(x)
        sp.append(s)
        rr, x, s = run_ref()
        tr.append(x)
        sr.append(s)
    same = {f: bool(np.array_equal(getattr(rp, f).cpu().numpy().view(np.uint8), getattr(rr, f).cpu().numpy().view(np.uint8)))
            for f in ("T", "n_outer", "converged_at")}

    # the gather alone: gicpSetPairList on the set-up target set, CUDA events, median of repeats
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
    torch.cuda.synchronize()
    for b, e in ev:
        b.record()
        pl.set_pair_list(edges[:, 0], edges[:, 1], TARGET)
        e.record()
    torch.cuda.synchronize()
    g_ms = float(np.median([b.elapsed_time(e) for b, e in ev]))
    n_rows = E * n
    g_bytes = 2 * n_rows * (16 + 6 * 4)          # records (16 B) + covariances (6 floats), read and written
    T = rp.T.cpu().numpy()
    rot_err, tr_err = [], []
    for p, (i, j) in enumerate(edges):
        G = synthetic.relative_pose(poses, int(i), int(j))
        dR = T[p, :3, :3] @ G[:3, :3].T
        rot_err.append(np.degrees(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))))
        tr_err.append(np.linalg.norm(T[p, :3, 3] - G[:3, 3]))
    conv = rp.converged_at.cpu().numpy()
    res = dict(
        card=card(), clouds=N, points=n, span=a.span, edges=E, runs=a.runs, warmup=a.warmup, params=prm,
        storage="f32", generate_s=round(gen_s, 1),
        pair_list=dict(total_ms_median=1e3 * float(np.median(tp)), setup_ms_median=1e3 * float(np.median(sp)),
                       list_and_register_ms_median=1e3 * float(np.median(np.array(tp) - np.array(sp))),
                       total_ms_all=[1e3 * x for x in tp]),
        one_to_one=dict(total_ms_median=1e3 * float(np.median(tr)), setup_ms_median=1e3 * float(np.median(sr)),
                        register_ms_median=1e3 * float(np.median(np.array(tr) - np.array(sr))),
                        total_ms_all=[1e3 * x for x in tr]),
        speedup_median=float(np.median(tr) / np.median(tp)),
        bitwise_equal=same,
        gather=dict(ms_median=g_ms, rows=n_rows, bytes=g_bytes, GB_per_s=g_bytes / (g_ms * 1e-3) / 1e9,
                    note="records 16 B + covariances 24 B per row, read and written; plus the list upload"),
        accuracy=dict(rot_err_deg_median=float(np.median(rot_err)), trans_err_m_median=float(np.median(tr_err)),
                      rot_err_deg_p95=float(np.percentile(rot_err, 95)),
                      trans_err_m_p95=float(np.percentile(tr_err, 95)),
                      not_converged=int((conv < 0).sum())),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
