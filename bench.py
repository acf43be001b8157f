#!/usr/bin/env python
"""bench.py - registered point-correspondences/s (and scan pairs/s) of the GICP hot path.

Workload (BASELINE.json configs[3], the one the metric is quoted on at 1/2/4/8 GPUs): a batch of
4096 independent synthetic 3-D scan pairs, 32768 points per side, k = 20 covariance
neighbourhoods, partitioned over the ranks by pairs (generalized_icp_b200.sharding.pair_range: 4096 pairs in
TOTAL, strong scaling, as configs[3] words it; --scaling weak gives every rank --pairs pairs of its own) with no
data-path collective.  A "step" is one complete
registration of the whole batch: grid build + covariances of both sides + the outer loop to
convergence.  correspondences = sum over pairs of N_src * outer iterations executed.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this engine
    python bench.py --impl reference [...]                          # the CPU arm (oracle port)
    python bench.py --dump-outputs DIR [...]                        # + the last timed step's results as DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "registered_point_correspondences_per_sec"
UNIT = "correspondences/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=4096, help="scan pairs of the job (strong scaling) / per GPU (--scaling weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --pairs in total, partitioned over the ranks (BASELINE configs[3]); weak: --pairs per rank")
    ap.add_argument("--points", type=int, default=32768, help="points per cloud")
    ap.add_argument("--cpu-pairs", type=int, default=0, help="pairs in the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--workload", default="config4", choices=["config4", "config5"],
                    help="config4 (default): the batch of independent pairs the metric is quoted on; config5: ONE 3-D pair of "
                         "16.7 M points per side, source sharded over the ranks with an NCCL all-reduce per outer iteration")
    ap.add_argument("--config5-points", type=int, default=0, help="points per side of the config5 pair (0 = 16 777 216)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's results (T, n_outer, converged_at of "
                         "every pair) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    return args


def workload_config(args):
    from generalized_icp_b200 import synthetic
    cfg = dict(synthetic.CONFIG4)
    cfg["n"] = args.points
    prm = dict(synthetic.CONFIG4_PARAMS)
    return cfg, prm


def config_json(args, cfg, prm, n_gpus):
    total = args.pairs if args.scaling == "strong" else args.pairs * n_gpus
    return {"workload": f"batch of {total} independent 3-D scan pairs, {args.points} points per side "
                        f"(BASELINE configs[3]), {cfg['n_patches']} planar {cfg['patch']:.0f} m patches in a "
                        f"{cfg['cube']:.0f} m cube, sigma {cfg['sigma']} m, motion <= {cfg['max_rot_deg']} deg / "
                        f"{cfg['max_trans']} m",
            "pairs_total": total, "pairs_per_gpu": total / n_gpus, "points_per_cloud": args.points, "k": prm["k"],
            "knn_radius": prm["max_distance_nearest_neighbors"], "d_max": prm["max_distance_correspondence"],
            "tolerance": prm["tolerance"], "max_iterations": 100, "storage": "f32",
            "partitioning": f"{total} pairs partitioned over {n_gpus} rank(s) by sharding.pair_range ({args.scaling} scaling), "
                            "no collective on the data path",
            "l2": "inputs (>= 3 GB per rank) exceed the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's vectorised float64 restatement on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_one(job):
    import numpy as np  # noqa: F401
    from generalized_icp_b200 import synthetic
    from oracle import gicp_oracle as O
    cfg, prm, seed = job
    src, tgt, _ = synthetic.patches3d_pair(**cfg, seed=seed)
    t0 = time.perf_counter()
    out = O.gicp_oracle(src, tgt, inner="newton", recompute_src_cov=False, record=False, **prm)
    return len(src) * out["n_outer"], out["n_outer"], time.perf_counter() - t0


def cpu_arm(args, cfg, prm, steps, warmup):
    """Registers a bounded sample of the workload's pairs with the CPU oracle, one pair per worker
    process, all host cores busy.  Returns (correspondences/s, pairs/s, details)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    n_pairs = args.cpu_pairs or procs
    procs = min(procs, n_pairs)
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    ctx = mp.get_context("spawn")
    times, corr, iters = [], 0, []
    with ctx.Pool(procs) as pool:
        for s in range(warmup + steps):
            jobs = [(cfg, prm, args.seed * 7919 + 100000 * s + i) for i in range(n_pairs)]
            t0 = time.perf_counter()
            res = pool.map(_cpu_one, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if s >= warmup:
                times.append(dt)
                corr += sum(r[0] for r in res)
                iters += [r[1] for r in res]
    total = sum(times)
    return corr / total, n_pairs * len(times) / total, dict(
        cores=procs, pairs_per_step=n_pairs, ms_per_step=1e3 * total / len(times),
        mean_outer_iterations=sum(iters) / max(1, len(iters)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, prm = workload_config(args)
    steps, warmup = max(1, args.steps), max(0, min(args.warmup, 1))
    cps, pps, d = cpu_arm(args, cfg, prm, steps, warmup)
    sample = (f"{d['pairs_per_step']} pairs of the workload per step (of {args.pairs}), one pair per process on "
              f"{d['cores']} host processes, oracle/gicp_oracle.py float64 (cKDTree + numpy, converged Newton inner "
              f"solve, R C R^T shortcut)")
    line = {"impl": "reference", "metric": METRIC, "value": cps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": d["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "pairs_per_sec": pps, "mean_outer_iterations": d["mean_outer_iterations"],
            "config": config_json(args, cfg, prm, args.gpus),
            "cpu_baseline": {"value": cps, "unit": UNIT, "cores": d["cores"], "kind": "port", "sample": sample},
            "e2e": {"value": cps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, f"/tmp/gicp_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from generalized_icp_b200 import sharding, synthetic
    from generalized_icp_b200.engine import GicpEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    cfg, prm = workload_config(args)
    # the batch is partitioned by pairs, no collective on the data path.  strong (default, BASELINE configs[3]):
    # rank r registers pairs sharding.pair_range(--pairs, r, world) of ONE job; weak: every rank has --pairs of its own
    if args.scaling == "strong":
        p0, p1 = sharding.pair_range(args.pairs, rank, world)
    else:
        p0, p1 = rank * args.pairs, (rank + 1) * args.pairs
    my_pairs = p1 - p0
    gen_cfg = {k: v for k, v in cfg.items() if k != "n"}
    src, tgt, off, T_true = synthetic.patches3d_batch_device(my_pairs, n=args.points, seed=args.seed, device=dev,
                                                             first_pair=p0, **gen_cfg)
    off_h = off.cpu().numpy()
    eng = GicpEngine(3, "f32", device=local)
    eng.set_params(**prm)

    def step():
        eng.set_target(tgt, off_h)
        eng.set_source(src, off_h)
        return eng.register(history=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        res = step()
    torch.cuda.synchronize()
    n_outer = res.n_outer.cpu().numpy().astype(np.int64)
    corr_per_step = int(n_outer.sum()) * args.points

    # ---- value: inputs resident in HBM, device-timed, max over ranks ----
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, world, gather=True)
    launches = eng.launch_count - l0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(corr_per_step), float(my_pairs), float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_total = float(ms.item())
    corr_all, pairs_all, launches_all = (float(x) for x in tot.tolist())
    value = corr_all * args.steps / (ms_total * 1e-3)
    pairs_per_s = pairs_all * args.steps / (ms_total * 1e-3)

    # ---- per-kernel timing for the roofline (separate pass: events around every launch) ----
    eng.profile(True)
    step()
    prof = eng.profile_read()
    eng.profile(False)
    pts_rank = 2 * my_pairs * args.points
    iters_sum = int(n_outer.sum())
    stage_bytes = {   # ALGORITHMIC bytes per step on this rank (SURVEY 8d / DESIGN.md)
        "grid_build": 36.0 * 2 * pts_rank,                 # two grids per cloud (k-NN order, 1-NN order)
        "knn_cov": 40.0 * pts_rank,
        "correspond": 36.0 * iters_sum * args.points,      # source point + match index + matched target point
        "accumulate": 80.0 * iters_sum * args.points,      # both points + both covariances
        "solve": 640.0 * iters_sum,
    }
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    kernels = {}
    for st, (ms_st, cnt) in prof.items():
        gbs = stage_bytes[st] / (ms_st * 1e-3) / 1e9 if ms_st > 0 else 0.0
        kernels[st] = {"ms_per_step": ms_st, "launches": cnt, "algorithmic_gb": stage_bytes[st] / 1e9,
                       "achieved_gbs": gbs, "frac": gbs / peak}
    dom = max(("knn_cov", "correspond", "accumulate", "grid_build"), key=lambda s: kernels[s]["ms_per_step"])
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (a smaller batch of the
    # same workload), scaled per point to this launch
    traffic, traffic_note = None, None
    try:
        cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.startswith("traffic_"))
        tj = json.load(open(os.path.join(ROOT, "profiles", cands[-1])))
        kname = {"knn_cov": "knn_hist_kernel", "correspond": "correspond_kernel", "accumulate": "accumulate_kernel"}[dom]
        per_pt = sum(tj["launches"][kname]) / len(tj["launches"][kname]) / tj["points_per_launch"]
        units = kernels[dom]["launches"]
        pts_per_launch = (pts_rank / 2) if dom == "knn_cov" else iters_sum * args.points / max(1, units)
        traffic = per_pt * pts_per_launch
        traffic_note = f"{cands[-1]}: {per_pt:.1f} B/point measured on a 64-pair batch, scaled to this launch"
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "avg_launch_ms": kernels[dom]["ms_per_step"] / max(1, kernels[dom]["launches"]),
                "kernels": kernels}

    # ---- e2e: host buffers in, host results out, through the public engine API ----
    e2e = None
    if not args.no_e2e:
        h_src = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
        h_tgt = torch.empty(tgt.shape, dtype=tgt.dtype, pin_memory=True)
        h_src.copy_(src)
        h_tgt.copy_(tgt)
        # <= 2048 pairs per chunk (measured: 512 / 1024 / 2048 -> 93.1 / 96.4 / 97.5 % of the device-resident rate) and at least two full chunks, so that a small first chunk (1/8) exists whose
        # upload is the only exposed one (register_host_batch)
        chunk_pairs = max(1, min(int(os.environ.get("GICP_E2E_CHUNK", "2048")), (my_pairs + 1) // 2))

        def e2e_step():
            # host buffers in, host results out; the H2D copy of chunk i+1 overlaps the registration of chunk i
            T_h, n_h, _ = eng.register_host_batch(h_src, h_tgt, off_h, chunk_pairs=chunk_pairs)
            return int(n_h.sum().item())

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        c = 0
        for _ in range(args.steps):
            c += e2e_step() * args.points
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        cc = torch.tensor([float(c)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dist.all_reduce(cc, op=dist.ReduceOp.SUM)
        e2e = {"value": float(cc.item()) / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(h_src.numel() * 4 + h_tgt.numel() * 4) * world,
               "d2h_bytes_per_step": int(my_pairs * (16 * 8 + 4 + 4)) * world,
               "pairs_per_sec": pairs_all * args.steps / float(dt.item()),
               "api": "GicpEngine.register_host_batch (chunks of <= 2048 pairs, first chunk 1/8; set_target/set_source/register over ctypes -> "
                      "libgicp_b200.so), pinned host buffers, H2D of the next chunk overlapped with compute"}
        del h_src, h_tgt

    # ---- accuracy sanity on this rank (not timed): error against the generating motion ----
    Tg = res.T
    dR = Tg[:, :3, :3].transpose(1, 2) @ T_true[:, :3, :3]
    ang = torch.arccos(torch.clamp((dR.diagonal(dim1=1, dim2=2).sum(1) - 1) / 2, -1, 1))
    terr = (Tg[:, :3, 3] - T_true[:, :3, 3]).norm(dim=1)
    acc = {"median_rot_err_rad": float(ang.median()), "median_trans_err_m": float(terr.median()),
           "converged_frac": float((res.converged_at >= 0).double().mean()),
           "mean_outer_iterations": float(n_outer.mean())}

    free_b, total_b = torch.cuda.mem_get_info(dev)
    hbm_used = torch.tensor([float(total_b - free_b)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(hbm_used, op=dist.ReduceOp.MAX)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU oracle, in a separate process (no fork after CUDA init), on a bounded sample
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
               "--pairs", str(args.pairs), "--points", str(args.points)]
        if args.cpu_pairs:
            cmd += ["--cpu-pairs", str(args.cpu_pairs)]
        try:
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, check=True).stdout.strip().splitlines()
            cpu = json.loads(out[-1])["cpu_baseline"]
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32 storage and per-thread accumulators; f64 neighbour ranking, per-point algebra and cross-warp sums",
                "data": "synthetic", "pairs_per_sec": pairs_per_s, "config": config_json(args, cfg, prm, n_gpus),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_all), "roofline": roofline,
                "cpu_baseline": cpu, "accuracy": acc,
                "hbm_used_gb_max_rank": float(hbm_used.item()) / 1e9}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_config5(args):
    """BASELINE configs[4]: one 3-D pair, 16.7 M points per side.  Every rank holds both clouds; the covariance
    stage (K2) and the per-iteration stages (K3) run on the rank's slice, the covariances are all-gathered once and
    the 80-double reduced form is all-reduced every outer iteration (ncclAllReduce inside libgicp_b200.so)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = dict(synthetic.CONFIG5)
    if args.config5_points:
        # same density and patch size at another size: the patch count follows the point count, the cube the patch count
        f = args.config5_points / cfg["n"]
        cfg.update(n=args.config5_points, n_patches=max(4, int(round(cfg["n_patches"] * f))),
                   cube=cfg["cube"] * max(f, 4 / cfg["n_patches"]) ** (1 / 3))
    prm = dict(synthetic.CONFIG5_PARAMS)
    n = cfg["n"]
    src, tgt, _, T_true = synthetic.patches3d_batch_device(1, seed=args.seed + 5, device=dev, chunk=1, **cfg)
    eng = GicpEngine(3, "f32", device=local)
    if world > 1:
        uid = [GicpEngine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(world, rank, uid[0])
    eng.set_params(**prm)

    def step():
        eng.set_target(tgt)
        eng.set_source(src)
        return eng.register(history=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        res = step()
    barrier()
    n_outer = int(res.n_outer[0])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = step()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, world, gather=False)   # every rank solves the same pair
    launches = eng.launch_count - l0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = float(n) * n_outer * args.steps / (ms_total * 1e-3)

    eng.profile(True)
    step()
    prof = eng.profile_read()
    eng.profile(False)
    stage_ms = torch.tensor([prof[s][0] for s in GicpEngine.STAGES], dtype=torch.float64, device=dev)
    stage_all = [torch.zeros_like(stage_ms) for _ in range(world)]
    if world > 1:
        dist.all_gather(stage_all, stage_ms)
    else:
        stage_all = [stage_ms]
    # ALGORITHMIC bytes on this rank: both grids are built by every rank; K2/K3 work on the rank's slice
    stage_bytes = {"grid_build": 36.0 * 2 * n, "knn_cov": 40.0 * 2 * n / world, "correspond": 36.0 * n_outer * n / world,
                   "accumulate": 80.0 * n_outer * n / world, "solve": 640.0 * n_outer}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    kernels = {}
    for st_name in GicpEngine.STAGES:
        ms_st, cnt = prof[st_name]
        gbs = stage_bytes[st_name] / (ms_st * 1e-3) / 1e9 if ms_st > 0 else 0.0
        kernels[st_name] = {"ms_per_step": ms_st, "launches": cnt, "algorithmic_gb": stage_bytes[st_name] / 1e9,
                            "achieved_gbs": gbs, "frac": gbs / peak}
    dom = max(("knn_cov", "correspond", "accumulate", "grid_build"), key=lambda s_: kernels[s_]["ms_per_step"])
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "kernels": kernels,
                "stage_ms_per_rank": {s_: [float(t[i]) for t in stage_all] for i, s_ in enumerate(GicpEngine.STAGES)}}

    # e2e: host clouds in (pinned), host transform out
    e2e = None
    if not args.no_e2e:
        h_src, h_tgt = src.cpu().pin_memory(), tgt.cpu().pin_memory()
        d_src, d_tgt = torch.empty_like(src), torch.empty_like(tgt)

        def e2e_step():
            d_tgt.copy_(h_tgt, non_blocking=True)
            eng.set_target(d_tgt)
            d_src.copy_(h_src, non_blocking=True)
            eng.set_source(d_src)
            r = eng.register(history=False)
            return r.T.cpu(), int(r.n_outer.cpu()[0])

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        c = 0
        for _ in range(args.steps):
            c += e2e_step()[1] * n
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": float(c) / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": int(2 * n * 12) * world,
               "d2h_bytes_per_step": (16 * 8 + 4) * world,
               "api": "GicpEngine.set_target/set_source/register over ctypes -> libgicp_b200.so, pinned host clouds copied to "
                      "every rank inside the timed region"}
        del h_src, h_tgt, d_src, d_tgt
    Tg = res.T[0].cpu().numpy()
    Tt = T_true[0].cpu().numpy()
    ang = float(np.arccos(np.clip((np.trace(Tg[:3, :3].T @ Tt[:3, :3]) - 1) / 2, -1, 1)))
    free_b, total_b = torch.cuda.mem_get_info(dev)
    if rank == 0:
        emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
              "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None,
              "dtype": "f32 storage and per-thread accumulators; f64 neighbour ranking, per-point algebra and cross-warp sums",
              "data": "synthetic", "pairs_per_sec": args.steps / (ms_total * 1e-3),
              "config": {"workload": f"ONE 3-D scan pair, {n} points per side (BASELINE configs[4]), {cfg['n_patches']} planar "
                                     f"{cfg['patch']:.0f} m patches in a {cfg['cube']:.0f} m cube; both clouds on every rank, K2 and "
                                     f"K3 on the rank's slice, NCCL all-gather of the covariances once + all-reduce of 80 f64 per "
                                     f"outer iteration over {world} rank(s)",
                         "points_per_cloud": n, "k": prm["k"], "knn_radius": prm["max_distance_nearest_neighbors"],
                         "d_max": prm["max_distance_correspondence"], "tolerance": prm["tolerance"], "storage": "f32",
                         "outer_iterations": n_outer, "l2": "inputs (>= 400 MB) exceed the 126 MB L2; no explicit flush"},
              "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": None,
              "accuracy": {"rot_err_rad": ang, "trans_err_m": float(np.linalg.norm(Tg[:3, 3] - Tt[:3, 3]))},
              "hbm_used_gb_rank0": float(total_b - free_b) / 1e9})
    if world > 1:
        eng.comm_destroy()
        dist.destroy_process_group()


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly one JSON line: whatever a library prints to fd 1 (NCCL's version banner)
    is sent to stderr, the line itself is written to the descriptor stdout had at start-up."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


DUMP_MAX_BYTES = 60 * 10**6     # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(out_dir, res, world, gather):
    """Writes what register() returned in the last timed step: T (P, 4, 4) f64, n_outer (P,) and converged_at (P,)
    as f64, pairs in job order (gather: the ranks' shares are concatenated on rank 0).  Beyond DUMP_MAX_BYTES a fixed
    seeded sample of pairs is written, with the sampled pair indices in pair_index.npy."""
    import numpy as np
    import torch.distributed as dist
    part = {"T": res.T.cpu().numpy(), "n_outer": res.n_outer.cpu().numpy().astype(np.float64),
            "converged_at": res.converged_at.cpu().numpy().astype(np.float64)}
    parts = [part]
    if gather and world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, part)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    out = {k: np.concatenate([p[k] for p in parts]) for k in part}
    n_pairs = len(out["T"])
    per_pair = sum(v[0].nbytes for v in out.values())
    if n_pairs * per_pair > DUMP_MAX_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n_pairs, DUMP_MAX_BYTES // (per_pair + 8), replace=False))
        out = {k: v[keep] for k, v in out.items()}
        out["pair_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "config5":
        run_config5(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
