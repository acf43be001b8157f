"""Streaming scan-sequence odometry: the loop around the path in the reference's robot demo
(robot-visualization.py:151-166, 246-265), headless.

Consecutive scans are registered source = previous scan, target = current scan
(robot-visualization.py:250-251) with the demo's parameters (max_distance_nearest_neighbors=200,
tolerance=1, robot-visualization.py:160-161).  Unlike the reference, which rebuilds the KD-tree and
all covariances of both scans on every call (gicp.py:104,111), the target of pair k is promoted to the
source of pair k+1 on the device, so each scan is indexed and analysed once.  Poses are integrated
exactly as the demo does (robot-visualization.py:258-265).
"""
from __future__ import annotations

import math

import numpy as np


def integrate_pose(pose, T):
    """robot-visualization.py:258-265: pose = (x, y, yaw_rad) of the estimate; T = 3x3 result of gicp()."""
    x, y, yaw = pose
    dx, dy = -T[0, 2], -T[1, 2]
    dyaw = -math.atan2(T[1, 0], T[0, 0])
    return (x + dx * math.cos(yaw) - dy * math.sin(yaw), y + dx * math.sin(yaw) + dy * math.cos(yaw), yaw + dyaw)


class ScanOdometry:
    """Feed scans one at a time; every scan after the first yields the 3x3 transform of the pair
    (previous -> current) and the integrated pose."""

    def __init__(self, start_pose=(50.0, 400.0, 0.0), storage="f64", robust_kernel=None, robust_scale=None,
                 robust_adaptive=None, robust_min_scale=None, evaluate=False, **params):
        """``robust_kernel`` / ``robust_scale``, or ``robust_adaptive`` (kappa) / ``robust_min_scale``: see
        GicpEngine.set_robust_kernel (scales in pixels).  With ``evaluate`` every step's quality at its transform
        (dict(n_inliers, fitness, inlier_rmse, loss, H, b), GicpEngine.evaluate) is appended to ``self.quality``; it
        comes back with the transform in one copy."""
        from .engine import GicpEngine
        self.eng = GicpEngine(2, storage)
        p = dict(max_distance_nearest_neighbors=200.0, tolerance=1.0)   # robot-visualization.py:160-161
        p.update(params)
        self.eng.set_params(**p)
        self.eng.set_robust_kernel(robust_kernel, robust_scale, adaptive=robust_adaptive, min_scale=robust_min_scale)
        self.pose = tuple(start_pose)
        self.poses = [self.pose]
        self.transforms = []
        self.iterations = []
        self.evaluate = bool(evaluate)
        self.quality = []
        self._have = False

    def push(self, scan):
        r = self.eng.register_next_scan_host(np.asarray(scan, dtype=np.float64), self._have, evaluate=self.evaluate)
        if not self._have:
            self._have = True
            return None
        T = r["T"]
        self.transforms.append(T)
        self.iterations.append(r["n_outer"])
        if self.evaluate:
            self.quality.append(r["quality"])
        self.pose = integrate_pose(self.pose, T)
        self.poses.append(self.pose)
        return T


def trajectory_errors(estimated, truth):
    """Slide-deck metrics (presentation/main.typ:729-749): per-step position error, orientation error,
    RMSE and maximum.  estimated: [(x, y, yaw_rad)], truth: [(x, y, yaw_deg)] as LidarSim reports them."""
    est = np.asarray(estimated, dtype=np.float64)
    tru = np.asarray(truth, dtype=np.float64)
    n = min(len(est), len(tru))
    pos = np.hypot(est[:n, 0] - tru[:n, 0], est[:n, 1] - tru[:n, 1])
    dyaw = est[:n, 2] - np.deg2rad(tru[:n, 2])
    ori = np.abs((dyaw + np.pi) % (2 * np.pi) - np.pi)
    return dict(position_error=pos, orientation_error=ori, position_rmse=float(np.sqrt(np.mean(pos ** 2))),
                position_max=float(pos.max()), orientation_rmse=float(np.sqrt(np.mean(ori ** 2))),
                orientation_max=float(ori.max()))
