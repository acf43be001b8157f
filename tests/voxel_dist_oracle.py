"""float64 restatement of voxel distributions (gicpSetVoxelized, include/gicp_b200.h) that the tests compare the
device against, and a float64 registration loop fed with given covariances.  Test infrastructure only: nothing in
the package imports it."""
import numpy as np

import voxel_oracle
from oracle import gicp_oracle as O


def voxel_distributions(points, offsets, leaf, min_points=1, lam_t=O.LAMBDA_TANGENT, lam_n=O.LAMBDA_NORMAL):
    """The voxel means of ``voxel_oracle.voxel_downsample`` and, for every mean, the reference's covariance
    estimator (``O.covariances_from_neighbors``) with the voxel's member rows as the neighbour list.
    Returns (means (M, d) f64, out_offsets (P+1,) i64, covs (M, d, d) f64, counts (M,))."""
    P = np.asarray(points, dtype=np.float64)
    off = np.asarray(offsets, dtype=np.int64)
    d = P.shape[1]
    means, out_off, voxel_of, counts = voxel_oracle.voxel_downsample(P, off, leaf, min_points)
    covs = [np.zeros((0, d, d))]
    for c in range(len(off) - 1):
        m = int(out_off[c + 1] - out_off[c])
        if m == 0:
            continue
        Q = P[off[c]:off[c + 1]].copy()
        Q[~np.isfinite(Q).all(axis=1)] = 0.0        # never a member; keeps the estimator's masked products finite
        vo = voxel_of[off[c]:off[c + 1]]
        rows = np.nonzero(vo >= 0)[0]
        rows = rows[np.argsort(vo[rows], kind="stable")]          # members grouped by output row, ascending rows
        cnt = np.bincount(vo[rows], minlength=m)
        starts = np.concatenate([[0], np.cumsum(cnt)[:-1]])
        # the estimator takes one neighbour list per row of Q (m <= len(Q)); rows past m have no neighbours
        idx = np.full((len(Q), int(cnt.max())), len(Q), dtype=np.int64)
        idx[vo[rows], np.arange(len(rows)) - starts[vo[rows]]] = rows
        covs.append(O.covariances_from_neighbors(Q, idx, lam_t, lam_n)[:m])
    return means, out_off, np.concatenate(covs), counts


def gicp_given_cov(src, tgt, src_cov0, tgt_cov, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
                   covariance_model=0):
    """The engine's registration loop in float64 (R_k C_0 R_k^T source covariances, converged Newton inner solve,
    ``oracle.gicp_oracle.gicp_oracle`` with recompute_src_cov=False) with the covariances given instead of estimated;
    covariance_model 1 / 2 replace them as the engine does (C_src = 0; model 1 also C_tgt = I).
    Returns dict(T, n_outer, converged_at, min_loss per iteration)."""
    src = np.asarray(src, dtype=np.float64)
    tgt = np.asarray(tgt, dtype=np.float64)
    dim = src.shape[1]
    src_cov0 = np.asarray(src_cov0, dtype=np.float64)
    tgt_cov = np.asarray(tgt_cov, dtype=np.float64)
    if covariance_model in (1, 2):
        src_cov0 = np.zeros_like(src_cov0)
        if covariance_model == 1:
            tgt_cov = np.broadcast_to(np.eye(dim), tgt_cov.shape).copy()
    T = np.eye(dim + 1)
    offset = np.zeros(3 if dim == 2 else 6)
    last = np.inf
    converged_at, n_outer, losses = None, 0, []
    for it in range(max_iterations):
        moved = O.apply_transformation(src, T)
        Rk = T[:dim, :dim]
        n_outer += 1
        idx, _ = O.correspond(moved, tgt, max_distance_correspondence, "kdtree")
        q = O.corresponding_points(tgt, idx)
        W = O.weights(Rk @ src_cov0 @ Rk.T, tgt_cov, idx)
        x, fopt, _, _ = O.inner_newton(offset, src, q, W)
        offset = x
        losses.append(fopt)
        if abs(last - fopt) < tolerance:
            converged_at = it
            break
        last = fopt
        T = O.offset_to_matrix(offset, dim)
    return dict(T=T, n_outer=n_outer, converged_at=converged_at, min_loss=np.asarray(losses))
