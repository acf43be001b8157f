"""Float64 restatement of the robust kernels of the registration loop (include/gicp_b200.h, "robust kernels").
TEST INFRASTRUCTURE ONLY: the package does not import it.

:func:`robust_weight` is the weight formula, written as the header writes it (every product and sum rounded on its
own), so that ``tests/host_harness/robust_host.cu`` can compare the device helper with it bit for bit.
:func:`gicp_oracle` is the outer loop of ``oracle.gicp_oracle.gicp_oracle`` with iteratively reweighted least squares:
at every T_k the weights w_i of the gated-in correspondences come from the 1-NN distance ``correspond`` returns, the
inner Newton solve minimises sum w_i r_i^T W_i r_i, and min_loss is that weighted minimum.  With ``robust=None`` it is
the plain loop, line for line."""
from __future__ import annotations

import numpy as np

from oracle import gicp_oracle as O

KINDS = {None: 0, "huber": 1, "cauchy": 2, "tukey": 3}


def robust_weight(kind, d, c):
    """w(d) of kind None / "huber" / "cauchy" / "tukey" at scale c, float64, elementwise (u = d / c)."""
    d = np.asarray(d, dtype=np.float64)
    c = np.asarray(c, dtype=np.float64)
    u = d / c
    if kind is None:
        return np.ones(np.broadcast(d, c).shape)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if kind == "huber":
            return np.where(d <= c, 1.0, c / d)
        if kind == "cauchy":
            return 1.0 / (1.0 + u * u)
        if kind == "tukey":
            a = 1.0 - u * u
            return np.where(u < 1.0, a * a, 0.0)
    raise ValueError(f"unknown robust kernel {kind!r}")


def gicp_oracle(source_points, target_points, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
                max_distance_nearest_neighbors=50, k=O.K_DEFAULT, lam_t=O.LAMBDA_TANGENT, lam_n=O.LAMBDA_NORMAL,
                knn="kdtree", record=True, covariance_model=0, robust=None):
    """The registration loop of the engine (R_k C_0 R_k^T source covariances, converged Newton inner solve) with the
    robust kernel ``robust`` = (kind, c) or None.  Returns what oracle.gicp_oracle.gicp_oracle returns; every trace
    entry also holds the weights ``w`` (1 for gated rows, whose W is 0 anyway)."""
    src = np.asarray(source_points, dtype=np.float64)
    tgt = np.asarray(target_points, dtype=np.float64)
    dim = src.shape[1]
    kind, c = robust if robust is not None else (None, 1.0)
    if kind not in KINDS:
        raise ValueError(f"unknown robust kernel {kind!r}")
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
        w = np.where(idx >= 0, robust_weight(kind, dist, c), 1.0)
        Ww = w[:, None, None] * W
        x, fopt, warn, calls = O.inner_newton(offset, src, q, Ww)
        offset = x
        delta = abs(last - fopt)
        if record:
            trace.append(dict(T=T.copy(), idx=idx, dist=dist, W=W, w=w, q=q, offset=np.array(x), min_loss=fopt))
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


def motion_error(T, T_true):
    """(rotation error in rad, translation error) of an estimate against the generating motion."""
    dim = T.shape[0] - 1
    dR = T[:dim, :dim] @ T_true[:dim, :dim].T
    if dim == 2:
        rot = abs(np.arctan2(dR[1, 0], dR[0, 0]))
    else:
        rot = float(np.arccos(np.clip((np.trace(dR) - 1.0) / 2.0, -1.0, 1.0)))
    return float(rot), float(np.linalg.norm(T[:dim, dim] - T_true[:dim, dim]))
