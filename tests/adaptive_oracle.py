"""Float64 restatement of the adaptive robust scale of the registration loop (include/gicp_b200.h,
gicpSetRobustKernelAdaptive).  TEST INFRASTRUCTURE ONLY: the package does not import it.

:func:`adaptive_scale` and :func:`lower_median` are the scale, written as the header writes it, so that
``tests/host_harness/adaptive_host.cu`` can compare the device helper with it bit for bit.  :func:`gicp_oracle` is the
loop of ``robust_oracle.gicp_oracle`` with the scale recomputed at every T_k from that iteration's gated-in distances;
every trace entry records it as ``c``.  It reuses the oracle's and robust_oracle's functions."""
from __future__ import annotations

import math

import numpy as np

import robust_oracle as RO
from oracle import gicp_oracle as O


def lower_median(d):
    """The element of rank floor((n-1)/2) of d in ascending order (ties included); 0.0 for an empty d."""
    d = np.asarray(d, dtype=np.float64)
    if d.size == 0:
        return 0.0
    return float(np.partition(d, (d.size - 1) // 2)[(d.size - 1) // 2])


def adaptive_scale(kappa, m, min_scale):
    """max(min_scale, kappa * m): the product rounded once, min_scale on ties; elementwise."""
    c = np.asarray(kappa, dtype=np.float64) * np.asarray(m, dtype=np.float64)
    return np.where(c > min_scale, c, np.asarray(min_scale, dtype=np.float64))


def scale_at(kappa, min_scale, idx, dist):
    """The scale of one pair from its correspondences (idx >= 0: gated in)."""
    return float(adaptive_scale(kappa, lower_median(dist[idx >= 0]), min_scale))


def gicp_oracle(source_points, target_points, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
                max_distance_nearest_neighbors=50, k=O.K_DEFAULT, lam_t=O.LAMBDA_TANGENT, lam_n=O.LAMBDA_NORMAL,
                knn="kdtree", record=True, covariance_model=0, adaptive=None):
    """The robust loop (robust_oracle.gicp_oracle) with ``adaptive`` = (kind, kappa, min_scale): at every T_k the
    scale is c_k = max(min_scale, kappa * lower median of the gated-in distances), and the weights are
    robust_weight(kind, d_i, c_k).  Returns what robust_oracle.gicp_oracle returns; every trace entry also holds c."""
    kind, kappa, min_scale = adaptive
    if kind not in ("huber", "cauchy", "tukey"):
        raise ValueError(f"an adaptive scale needs huber, cauchy or tukey, not {kind!r}")
    src = np.asarray(source_points, dtype=np.float64)
    tgt = np.asarray(target_points, dtype=np.float64)
    dim = src.shape[1]
    tgt_cov, _ = O.compute_covariances(tgt, max_distance_nearest_neighbors, k, lam_t, lam_n, knn)
    src_cov0, _ = O.compute_covariances(src, max_distance_nearest_neighbors, k, lam_t, lam_n, knn)
    if covariance_model in (1, 2):
        src_cov0 = np.zeros_like(src_cov0)
        if covariance_model == 1:
            tgt_cov = np.broadcast_to(np.eye(dim), tgt_cov.shape).copy()
    T = np.eye(dim + 1)
    all_T = [T]
    offset = np.zeros(3 if dim == 2 else 6)
    last = np.inf
    hw_src, hw_tgt, trace = [], [], []
    converged_at = None
    n_outer = 0
    for it in range(max_iterations):
        moved = O.apply_transformation(src, T)
        Rk = T[:dim, :dim]
        src_cov = Rk @ src_cov0 @ Rk.T
        n_outer += 1
        idx, dist = O.correspond(moved, tgt, max_distance_correspondence, knn)
        q = O.corresponding_points(tgt, idx)
        W = O.weights(src_cov, tgt_cov, idx)
        c = scale_at(kappa, min_scale, idx, dist)
        w = np.where(idx >= 0, RO.robust_weight(kind, dist, c), 1.0)
        Ww = w[:, None, None] * W
        x, fopt, warn, calls = O.inner_newton(offset, src, q, Ww)
        offset = x
        delta = abs(last - fopt)
        if record:
            trace.append(dict(T=T.copy(), idx=idx, dist=dist, W=W, w=w, c=c, q=q, offset=np.array(x), min_loss=fopt))
        if delta < tolerance:
            converged_at = it
            break
        last = fopt
        T = O.offset_to_matrix(offset, dim)
        all_T.append(T)
        order = np.argsort(np.linalg.det(Ww))[-5:]
        hw_src.append(moved[order])
        hw_tgt.append(q[order])
    return dict(T=T, all_T=all_T, src_cov0=src_cov0, tgt_cov=tgt_cov, hw_src=hw_src, hw_tgt=hw_tgt,
                converged_at=converged_at, n_outer=n_outer, trace=trace)


def drive_pairs(seed=0, num_rays=90, n_scans=12):
    """The scan pairs of demo_inputs.lidar_sequence and, for each, the motion that maps the earlier scan onto the
    later one (robot-relative points, yaw in degrees)."""
    import demo_inputs
    scans, poses = demo_inputs.lidar_sequence(seed=seed, num_rays=num_rays, n_scans=n_scans)

    def rot(a):
        a = math.radians(a)
        return np.array([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]])
    pairs = []
    for i in range(n_scans - 1):
        (x0, y0, a0), (x1, y1, a1) = poses[i], poses[i + 1]
        T = np.eye(3)
        T[:2, :2] = rot(a1).T @ rot(a0)
        T[:2, 2] = rot(a1).T @ np.array([x0 - x1, y0 - y1])
        pairs.append((np.asarray(scans[i], np.float64), np.asarray(scans[i + 1], np.float64), T))
    return pairs
