"""The adaptive robust scale (gicpSetRobustKernelAdaptive) on the GPU: its cost on both loop paths, accuracy on the
moved-patch pairs and the odometry drive.  Needs a CUDA device; writes one JSON file.
    python scripts/adaptive_bench.py --out adaptive_bench.json [--pairs 1024]
- bench_config4 (multi-launch loop): the config-4 batch (32768 points per cloud) with no kernel, each fixed scale of
  scripts/robust_bench.py and each kind with an adaptive scale; register time by CUDA events (median of --reps, set-up
  excluded), mean outer iterations, K3b and the select (one section of 8 launches per iteration) from gicpProfile and,
  from torch.profiler in a separate run, the time per launch of accumulate_kernel and scale_select_kernel.
- select_cost: the cost of the select per outer iteration on both paths.  An adaptive scale with kappa = 1e-300 is
  the fixed kernel at c = min_scale bit for bit (same iterations, same work), so the time difference over the outer
  iterations is the select alone.  Multi-launch: the config-4 batch and one config-4 pair alone (where the 8 launches
  per iteration are latency); fused: batches of ray-cast drive pairs (90 and 360 rays, one block per pair).
- moved_patch: the 16 moved-object pairs of scripts/robust_bench.py with each adaptive kind.
- odometry: scripts/odometry_eval.py (360 rays, 36 scans) plain, with each fixed scale and with each adaptive kind."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from robust_bench import BENCH_SCALES, ODO_SCALES, card, motion_error  # noqa: E402

KINDS = ["huber", "cauchy", "tukey"]
BENCH_KAPPA, BENCH_MIN = 3.0, 0.02     # metres; the config-4 clouds carry 2 cm noise
MOVED_KAPPA, MOVED_MIN = {"huber": 0.5, "cauchy": 0.5, "tukey": 1.0}, 0.02
ODO_KAPPA, ODO_MIN = {"huber": [3.0, 4.5], "cauchy": [3.0, 4.5], "tukey": [3.0, 4.5]}, 1.0   # pixels


def _timed(eng, torch, reps):
    eng.register(history=False)                           # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = eng.register(history=False)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), times, r


def _kernel_times(eng, torch):
    """{kernel family: (total ms, launches)} of one registration, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.register(history=False)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for fam in ("scale_select_kernel", "accumulate_kernel", "correspond_kernel"):
            if fam in ev.key:
                ms, n = out.get(fam, (0.0, 0))
                out[fam] = (ms + ev.device_time_total / 1e3, n + ev.count)
    return {k: dict(ms=v[0], launches=v[1], us_per_launch=1e3 * v[0] / max(v[1], 1)) for k, v in out.items()}


def single_pair_select_cost(args, torch):
    """One config-4 pair in the multi-launch loop: fixed Huber vs adaptive with kappa 1e-300 (the same iterations)."""
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    src, tgt, off, _ = synthetic.patches3d_batch_device(1, n=args.points, seed=0)
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    eng.set_target(tgt, off.cpu().numpy())
    eng.set_source(src, off.cpu().numpy())
    res = {}
    for name, kw in (("fixed", dict(scale=BENCH_SCALES["huber"])),
                     ("adaptive", dict(adaptive=1e-300, min_scale=BENCH_SCALES["huber"]))):
        eng.set_robust_kernel("huber", **kw)
        ms, times, r = _timed(eng, torch, max(args.reps, 5))
        res[name] = dict(register_ms_median=ms, register_ms_all=times, n_outer=int(r.n_outer[0]))
    res["select_us_per_iteration"] = 1e3 * (res["adaptive"]["register_ms_median"] -
                                            res["fixed"]["register_ms_median"]) / res["fixed"]["n_outer"]
    print("single pair", res, flush=True)
    return res


def bench(args, torch):
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    src, tgt, off, Tg = synthetic.patches3d_batch_device(args.pairs, n=args.points, seed=0)
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    eng.set_target(tgt, off.cpu().numpy())
    eng.set_source(src, off.cpu().numpy())
    Tg = Tg.cpu().numpy()
    settings = [("none", None, {})] + [(f"{k} fixed", k, dict(scale=BENCH_SCALES[k])) for k in KINDS]
    settings += [(f"{k} adaptive", k, dict(adaptive=BENCH_KAPPA, min_scale=BENCH_MIN)) for k in KINDS]
    settings += [("huber adaptive, kappa 1e-300 (= huber fixed)", "huber",
                  dict(adaptive=1e-300, min_scale=BENCH_SCALES["huber"]))]
    out = {}
    for name, kind, kw in settings:
        eng.set_robust_kernel(kind, **kw)
        ms, times, r = _timed(eng, torch, args.reps)
        n_outer = r.n_outer.cpu().numpy()
        errs = np.array([motion_error(T, g) for T, g in zip(r.T.cpu().numpy(), Tg)])
        eng.profile(True)
        eng.register(history=False)
        prof = eng.profile_read(scale_select=True)
        eng.profile(False)
        out[name] = dict(kw, register_ms_median=ms, register_ms_all=times, mean_outer_iterations=float(n_outer.mean()),
                         max_outer_iterations=int(n_outer.max()),
                         accumulate_ms_profiled=prof["accumulate"][0], accumulate_launches=prof["accumulate"][1],
                         select_ms_profiled=prof["scale_select"][0], select_sections=prof["scale_select"][1],
                         select_ms_per_section=prof["scale_select"][0] / max(prof["scale_select"][1], 1),
                         accumulate_ms_per_launch=prof["accumulate"][0] / max(prof["accumulate"][1], 1),
                         kernels=_kernel_times(eng, torch),
                         rot_err_median_rad=float(np.median(errs[:, 0])), trans_err_median_m=float(np.median(errs[:, 1])))
        print(name, ms, out[name]["max_outer_iterations"], out[name]["kernels"], flush=True)
    a, f = out["huber adaptive, kappa 1e-300 (= huber fixed)"], out["huber fixed"]
    launches = a["max_outer_iterations"]                  # the host loop launches every pair's stages this often
    out["select_ms_per_iteration"] = (a["register_ms_median"] - f["register_ms_median"]) / launches
    return out


def fused_select_cost(torch, reps):
    """Batches of one drive pair repeated (every block the same work): fixed Huber vs adaptive with kappa 1e-300."""
    from generalized_icp_b200.engine import GicpEngine, ray_cast
    rows = []
    for num_rays in (90, 360):
        poses = np.array([[60.0, 400.0, 0.0], [69.9, 401.0, 10.0]])
        noise = np.random.default_rng(7).uniform(-2, 2, size=(2, num_rays))
        rel, hit = ray_cast(poses, num_rays=num_rays, noise=noise)
        torch.cuda.synchronize()
        s, t = rel[0][hit[0]], rel[1][hit[1]]
        for n_pairs in (1, 512):
            eng = GicpEngine(2, "f64")
            eng.set_params(max_distance_nearest_neighbors=200.0, tolerance=1.0)
            off = np.arange(n_pairs + 1, dtype=np.int64)
            eng.set_target(t.repeat(n_pairs, 1), off * len(t))
            eng.set_source(s.repeat(n_pairs, 1), off * len(s))
            res = {}
            for name, kw in (("fixed", dict(scale=4.0)), ("adaptive", dict(adaptive=1e-300, min_scale=4.0))):
                eng.set_robust_kernel("huber", **kw)
                ms, times, r = _timed(eng, torch, reps)
                res[name] = dict(register_ms_median=ms, register_ms_all=times, n_outer=int(r.n_outer[0]))
            rows.append(dict(num_rays=num_rays, points=int(len(s)), pairs=n_pairs, **res,
                             select_us_per_iteration=1e3 * (res["adaptive"]["register_ms_median"] -
                                                            res["fixed"]["register_ms_median"]) / res["fixed"]["n_outer"]))
            print(rows[-1], flush=True)
    return rows


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
    for kind in [None] + KINDS:
        kw = {} if kind is None else dict(adaptive=MOVED_KAPPA[kind], min_scale=MOVED_MIN)
        eng.set_robust_kernel(kind, **kw)
        r = eng.register(history=False)
        torch.cuda.synchronize()
        e = np.array([motion_error(T, g) for T, g in zip(r.T.cpu().numpy(), Tgs)])
        rows.append(dict(kind=str(kind), **kw, rot_err_median_rad=float(np.median(e[:, 0])),
                         trans_err_median_m=float(np.median(e[:, 1])), trans_err_max_m=float(e[:, 1].max()),
                         mean_outer_iterations=float(r.n_outer.float().mean())))
        print(rows[-1], flush=True)
    return rows


def odometry():
    specs = [None] + [f"{k}:{ODO_SCALES[k]}" for k in KINDS]
    specs += [f"{k}:adaptive:{kappa}:{ODO_MIN}" for k in KINDS for kappa in ODO_KAPPA[k]]
    rows = []
    for spec in specs:
        cmd = [sys.executable, os.path.join(ROOT, "scripts", "odometry_eval.py"), "360", "36"]
        if spec is not None:
            cmd += ["--robust", spec]
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
        raise SystemExit("adaptive_bench.py needs a CUDA device")
    res = {"card (name, power limit, max SM clock)": card(), "pairs": args.pairs, "points_per_cloud": args.points}
    res["bench_config4"] = bench(args, torch)
    res["single_pair_select_cost"] = single_pair_select_cost(args, torch)
    res["fused_select_cost"] = fused_select_cost(torch, max(args.reps, 5))
    res["moved_patch"] = moved_patch(torch)
    res["odometry_360rays_36scans"] = odometry()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
