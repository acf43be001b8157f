"""8f rows 1-3 together: scripted drive -> GPU ray caster -> streaming GICP odometry -> the slide deck's
metrics (position / orientation error, RMSE / MAX, alignment-time series; presentation/main.typ:729-749).
    python scripts/odometry_eval.py [num_rays] [n_scans] [--robust KIND:SCALE | --robust KIND:adaptive:KAPPA:MIN]
--robust registers every pair with a robust kernel (huber, cauchy or tukey; scale in px), or with the adaptive scale
max(MIN, KAPPA * median distance) of every outer iteration, and adds it to the output."""
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from generalized_icp_b200.engine import ray_cast  # noqa: E402
from generalized_icp_b200.odometry import ScanOdometry, trajectory_errors  # noqa: E402

args = sys.argv[1:]
robust_kernel = robust_scale = robust_adaptive = robust_min_scale = None
if "--robust" in args:
    i = args.index("--robust")
    spec = args[i + 1].split(":")
    robust_kernel = spec[0]
    if len(spec) == 4 and spec[1] == "adaptive":
        robust_adaptive, robust_min_scale = float(spec[2]), float(spec[3])
    elif len(spec) == 2:
        robust_scale = float(spec[1])
    else:
        sys.exit(f"--robust takes KIND:SCALE or KIND:adaptive:KAPPA:MIN, not {args[i + 1]!r}")
    del args[i:i + 2]
num_rays = int(args[0]) if len(args) > 0 else 360
n_scans = int(args[1]) if len(args) > 1 else 120

# scripted drive with the demo's kinematics (robot-visualization.py:210-220): 5 ticks per scan
x, y, yaw = 50.0, 400.0, 0
poses = []
for s in range(n_scans):
    block = (s // 6) % 3
    for _ in range(5):
        if block == 1:
            yaw += 2
        if block == 2:
            yaw -= 2
        x += 2 * math.cos(math.radians(yaw))
        y += 2 * math.sin(math.radians(yaw))
    poses.append((x, y, yaw))
rng = np.random.default_rng(0)
noise = rng.uniform(-2, 2, size=(n_scans, num_rays))                 # NOISE = 2 (robot-visualization.py:26,74)
rel, hit = ray_cast(np.asarray(poses), num_rays=num_rays, noise=noise)
torch.cuda.synchronize()
scans = [rel[i][hit[i]] for i in range(n_scans)]

odo = ScanOdometry(start_pose=(0.0, 0.0, 0.0), robust_kernel=robust_kernel, robust_scale=robust_scale,
                   robust_adaptive=robust_adaptive, robust_min_scale=robust_min_scale)
times = []
for sc in scans:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    odo.push(sc.cpu().numpy())
    torch.cuda.synchronize()
    times.append(time.perf_counter() - t0)
est = np.asarray(odo.poses)
tru = np.asarray(poses)
# both trajectories relative to the first scan's pose and heading
c, s_ = math.cos(math.radians(tru[0, 2])), math.sin(math.radians(tru[0, 2]))
d = tru[:, :2] - tru[0, :2]
tru_rel = np.column_stack([c * d[:, 0] + s_ * d[:, 1], -s_ * d[:, 0] + c * d[:, 1], tru[:, 2] - tru[0, 2]])
err = trajectory_errors(est, tru_rel)
extra = {}
if robust_kernel is not None:
    extra["robust"] = (f"{robust_kernel}:{robust_scale:g}" if robust_adaptive is None
                       else f"{robust_kernel}:adaptive:{robust_adaptive:g}:{robust_min_scale:g}")
print(json.dumps({**extra, "num_rays": num_rays, "scans": n_scans, "points_per_scan_mean": float(np.mean([len(s) for s in scans])),
                  "alignment_ms_median": 1e3 * float(np.median(times[1:])), "alignment_ms_p95": 1e3 * float(np.percentile(times[1:], 95)),
                  "mean_outer_iterations": float(np.mean(odo.iterations)),
                  "position_rmse_px": err["position_rmse"], "position_max_px": err["position_max"],
                  "orientation_rmse_rad": err["orientation_rmse"], "orientation_max_rad": err["orientation_max"],
                  "path_length_px": float(np.sum(np.hypot(*np.diff(tru[:, :2], axis=0).T)))}))
