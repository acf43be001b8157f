"""Drop-in for the reference module ``python-implementation/gicp.py``.

``gicp(source_points, target_points, max_iterations=100, tolerance=1e-6,
max_distance_correspondence=150, max_distance_nearest_neighbors=50)`` has the
signature and defaults of gicp.py:78 and returns the 7-tuple of gicp.py:174 as
host float64 numpy arrays (picklable: the robot demo sends them through a
multiprocessing.Queue, robot-visualization.py:166).  All computation runs on
the GPU through libgicp_b200.so; the engine is created lazily inside the call
so a forked worker can be the first to touch CUDA.  ``apply_transformation``
(gicp.py:176-177) stays pure numpy because the demos call it in the UI process.
"""
from __future__ import annotations

import os

import numpy as np

_ENGINES = {}


def apply_transformation(cloud, T):
    """gicp.py:176-177: ``cloud[:, :d] @ T[:d, :d].T + T[:d, d]`` (d = 2 for the reference's 3x3 T)."""
    d = T.shape[0] - 1
    return np.dot(cloud[:, :d], T[:d, :d].T) + T[:d, d]


def _engine(dim, storage, tag="main"):
    key = (os.getpid(), dim, storage, tag)
    eng = _ENGINES.get(key)
    if eng is None:
        from .engine import GicpEngine
        eng = GicpEngine(dim, storage)
        _ENGINES[key] = eng
    return eng


def _downsample(eng, cloud, voxel_size, min_points):
    pts, _ = eng.voxel_downsample(np.ascontiguousarray(cloud), voxel_size=voxel_size, min_points=min_points)
    return pts.cpu().numpy().astype(np.float64)


def voxel_downsample(cloud, voxel_size, min_points=1):
    """PCL-style voxel-grid filter of one (N, 2) or (N, 3) cloud on the GPU: the centroid of every voxel of edge
    ``voxel_size`` holding >= ``min_points`` finite points, in the order of each voxel's lowest row (semantics in
    include/gicp_b200.h).  float64 numpy in and out."""
    cloud = np.asarray(cloud, dtype=np.float64)
    if cloud.ndim != 2 or cloud.shape[1] not in (2, 3):
        raise ValueError(f"expected an (N, 2) or (N, 3) cloud, got {cloud.shape}")
    return _downsample(_engine(int(cloud.shape[1]), "f64"), cloud, voxel_size, min_points)


def gicp_extended(source_points, target_points, max_iterations=100, tolerance=1e-6,
                  max_distance_correspondence=150, max_distance_nearest_neighbors=50, k=6,
                  lambda_tangent=100.0, lambda_normal=10.0, storage="f64", full_history=True, covariance_model=0,
                  voxel_size=None, robust_kernel=None, robust_scale=None, robust_adaptive=None, robust_min_scale=None,
                  evaluate=False, voxel_distributions=False, voxel_min_points=1, **engine_params):
    """The registration with everything the engine knows (SURVEY.md discrepancy 3: the reference
    computes ``min_loss`` and drops it; here the loss history, inlier counts and the fitness-like
    final loss are returned as well).  Returns a dict.  With ``voxel_size`` both clouds are first
    voxel-grid downsampled on the GPU (in ``storage``); the dict then holds them as ``source_points`` /
    ``target_points`` (float64) and every per-point output refers to them.  ``robust_kernel`` (None, "huber",
    "cauchy" or "tukey") with ``robust_scale`` weights every correspondence by a robust kernel of its distance
    (GicpEngine.set_robust_kernel); ``hw_src`` / ``hw_tgt`` then rank the weighted matrices w W.  ``robust_adaptive``
    (kappa) with ``robust_min_scale`` replaces ``robust_scale`` by the adaptive scale of every outer iteration.
    With ``evaluate`` the dict also holds the registration's quality at the returned T (GicpEngine.evaluate):
    ``n_inliers``, ``fitness``, ``inlier_rmse``, ``information`` (H, rotation first) and ``gradient`` (-2 b, the
    gradient of the objective under a left perturbation of T).  With ``voxel_distributions`` (and ``voxel_size``) both
    sides are instead set up as voxel distributions (GicpEngine.set_source_voxelized / set_target_voxelized: the
    voxels with >= ``voxel_min_points`` points, each carrying the covariance of its own points, no k-NN search);
    ``source_points`` / ``target_points``, ``src_cov0`` / ``tgt_cov`` and every per-point output then refer to the
    voxels."""
    import torch

    src = np.asarray(source_points)
    tgt = np.asarray(target_points)
    if src.ndim != 2 or tgt.ndim != 2:
        raise ValueError("point clouds must be (N, d) arrays")
    dim = int(src.shape[1])
    if dim not in (2, 3) or tgt.shape[1] != dim:
        raise ValueError(f"expected (N, 2) or (N, 3) clouds of equal dimension, got {src.shape} and {tgt.shape}")
    eng = _engine(dim, storage)
    if voxel_distributions and voxel_size is None:
        raise ValueError("voxel_distributions needs voxel_size")
    raw_src, raw_tgt = src, tgt
    if voxel_size is not None and not voxel_distributions:
        src = _downsample(eng, src[:, :dim], voxel_size, 1)
        tgt = _downsample(eng, tgt[:, :dim], voxel_size, 1)
    eng.set_params(k=k, max_iterations=int(max_iterations), tolerance=float(tolerance),
                   max_distance_correspondence=float(max_distance_correspondence),
                   max_distance_nearest_neighbors=float(max_distance_nearest_neighbors),
                   lambda_tangent=float(lambda_tangent), lambda_normal=float(lambda_normal),
                   covariance_model=int(covariance_model), **engine_params)
    eng.set_robust_kernel(robust_kernel, robust_scale, adaptive=robust_adaptive, min_scale=robust_min_scale)
    if voxel_distributions:
        r = _register_voxelized(eng, raw_src[:, :dim], raw_tgt[:, :dim], voxel_size, voxel_min_points)
        src, tgt = r["source_points"], r["target_points"]
    else:
        r = eng.register_pair_host(src[:, :dim], tgt[:, :dim])  # gicp.py:104, 111, 116-167 in one staged round trip
    n_outer, conv = r["n_outer"], r["converged_at"]
    n_T = n_outer if conv >= 0 else n_outer + 1             # appendix A rule 12
    T_hist = r["T_hist"][:n_T]
    out = dict(T=T_hist[-1].copy(), all_T=[T_hist[i].copy() for i in range(n_T)], n_outer=n_outer,
               converged_at=conv, loss_hist=r["loss_hist"].copy(), inliers=r["inliers"].copy(), dim=dim,
               tgt_cov=r["tgt_cov"], src_cov0=r["src_cov0"])
    if voxel_size is not None:
        out["source_points"], out["target_points"] = src, tgt
    if evaluate:
        q = eng.evaluate(out["T"].reshape(1, dim + 1, dim + 1))
        out["n_inliers"] = int(q.n_inliers[0])
        out["fitness"], out["inlier_rmse"] = float(q.fitness[0]), float(q.inlier_rmse[0])
        out["information"], out["gradient"] = q.H[0].cpu().numpy(), (-2.0 * q.b[0]).cpu().numpy()
    if full_history:
        covs = eng.source_covariances_at(T_hist[:n_outer].reshape(n_outer, 1, dim + 1, dim + 1)).cpu().numpy()
        out["all_src_cov"] = [covs[i] for i in range(n_outer)]
        hw_s, hw_t = [], []
        src64 = np.asarray(src[:, :dim], dtype=np.float64)
        tgt64 = np.asarray(tgt[:, :dim], dtype=np.float64)
        reps = n_T - 1
        per_it = []
        if 0 < reps and reps * max(len(src64), len(tgt64)) <= (1 << 22) and os.environ.get("GICP_COMPAT_BATCH_HISTORY", "1") != "0":
            # gicp.py:170-172 (visualisation only): the correspondences and weights of EVERY outer iteration in one
            # batched call - the pair replicated once per iteration on a second handle, T_k as the k-th pair's
            # transform - instead of one host round trip per iteration (a batch equals its pairs bit for bit)
            np_dt = np.float64 if storage == "f64" else np.float32
            eh = _engine(dim, storage, "history")
            eh.set_params(k=k, max_iterations=int(max_iterations), tolerance=float(tolerance),
                          max_distance_correspondence=float(max_distance_correspondence),
                          max_distance_nearest_neighbors=float(max_distance_nearest_neighbors),
                          lambda_tangent=float(lambda_tangent), lambda_normal=float(lambda_normal),
                          covariance_model=int(covariance_model), **engine_params)
            eh.set_robust_kernel(robust_kernel, robust_scale, adaptive=robust_adaptive, min_scale=robust_min_scale)
            n_s, n_t = len(src64), len(tgt64)
            if voxel_distributions:      # the raw clouds replicated, every copy voxelized as the pair's own sides were
                for setv, cloud in ((eh.set_target_voxelized, raw_tgt), (eh.set_source_voxelized, raw_src)):
                    setv(torch.as_tensor(np.tile(np.ascontiguousarray(cloud[:, :dim], dtype=np_dt), (reps, 1)),
                                         device=eh.device), np.arange(reps + 1, dtype=np.int64) * len(cloud),
                         voxel_size=voxel_size, min_points=voxel_min_points)
            else:
                eh.set_target(torch.as_tensor(np.tile(np.ascontiguousarray(tgt[:, :dim], dtype=np_dt), (reps, 1)), device=eh.device),
                              np.arange(reps + 1, dtype=np.int64) * n_t)
                eh.set_source(torch.as_tensor(np.tile(np.ascontiguousarray(src[:, :dim], dtype=np_dt), (reps, 1)), device=eh.device),
                              np.arange(reps + 1, dtype=np.int64) * n_s)
            idx_all, _, W_all = eh.correspond(T_hist[:reps])
            idx_all = idx_all.cpu().numpy().reshape(reps, n_s)
            W_all = W_all.cpu().numpy().reshape(reps, n_s, dim, dim)
            per_it = [(idx_all[it], W_all[it]) for it in range(reps)]
        else:
            for it in range(reps):                          # very large clouds: one call per iteration
                idx, _, W = eng.correspond(T_hist[it])
                per_it.append((idx.cpu().numpy(), W.cpu().numpy()))
        for it, (idx, W) in enumerate(per_it):
            order = np.argsort(np.linalg.det(W))[-5:]
            q = np.zeros_like(src64)
            m = idx >= 0
            q[m] = tgt64[idx[m]]
            hw_s.append(apply_transformation(src64, T_hist[it])[order])
            hw_t.append(q[order])
        out["hw_src"], out["hw_tgt"] = hw_s, hw_t
    return out


def _register_voxelized(eng, src, tgt, voxel_size, min_points):
    """Both sides of one pair set up as voxel distributions, registered; the host arrays register_pair_host returns,
    plus the voxel means as ``source_points`` / ``target_points`` (float64)."""
    from .engine import SOURCE, TARGET
    np_dt = np.float64 if eng.storage == "f64" else np.float32
    tm, _ = eng.set_target_voxelized(np.ascontiguousarray(tgt, dtype=np_dt), voxel_size=voxel_size, min_points=min_points)
    sm, _ = eng.set_source_voxelized(np.ascontiguousarray(src, dtype=np_dt), voxel_size=voxel_size, min_points=min_points)
    res = eng.register(history=True)
    n_outer, conv = int(res.n_outer[0]), int(res.converged_at[0])
    T_hist = res.T_hist[0].cpu().numpy()
    T_hist[(n_outer if conv >= 0 else n_outer + 1):] = np.nan   # rows the loop wrote: SURVEY appendix A rule 12
    return dict(T=res.T[0].cpu().numpy(), T_hist=T_hist,
                loss_hist=res.loss_hist[0].cpu().numpy()[:n_outer], inliers=res.inliers[0].cpu().numpy()[:n_outer],
                src_cov0=eng.covariances(SOURCE).cpu().numpy(), tgt_cov=eng.covariances(TARGET).cpu().numpy(),
                n_outer=n_outer, converged_at=conv, source_points=sm.cpu().numpy().astype(np.float64),
                target_points=tm.cpu().numpy().astype(np.float64))


def register_pairs(clouds, pairs, T0=None, *, storage="f64", evaluate=True, **params):
    """Register every ``(source, target)`` pair of cloud indices over one set-up of ``clouds`` (a list of (N_i, d)
    arrays): each cloud's grids and covariances are built once, as a target set, and every pair registers its source
    cloud onto its target cloud (GicpEngine.set_pair_list with source_set=TARGET).  ``params`` are gicpParams fields
    (k, max_iterations, max_distance_correspondence, ...) over the library's defaults; ``T0`` (E, d+1, d+1) optional
    initial transforms.  Returns a dict of per-pair numpy arrays, the inputs of a pose graph: ``T`` (E, d+1, d+1),
    which maps the source cloud's points onto the target cloud's, ``n_outer`` and ``converged_at``, and with
    ``evaluate`` the quality at T: ``n_inliers``, ``fitness``, ``inlier_rmse`` and ``information`` (H, rotation
    first; include/gicp_b200.h, gicpEvaluate)."""
    import ctypes

    import torch
    from ._lib import GicpParams
    from .engine import TARGET

    if len(clouds) == 0:
        raise ValueError("no clouds")
    dim = int(np.asarray(clouds[0]).shape[1])
    if dim not in (2, 3):
        raise ValueError(f"expected (N, 2) or (N, 3) clouds, got {np.asarray(clouds[0]).shape}")
    pr = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    eng = _engine(dim, storage, "pairs")
    defaults = GicpParams()
    eng.lib.gicpDefaultParams(ctypes.byref(defaults))
    eng.set_params(**{**{f: getattr(defaults, f) for f, _ in GicpParams._fields_}, **params})
    eng.set_robust_kernel(None)
    np_dt = np.float64 if storage == "f64" else np.float32
    arrs = [np.asarray(c, dtype=np_dt).reshape(-1, dim) for c in clouds]
    off = np.zeros(len(arrs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(a) for a in arrs])
    eng.set_target(torch.as_tensor(np.concatenate(arrs, axis=0), device=eng.device), off)
    eng.set_pair_list(pr[:, 0], pr[:, 1], source_set=TARGET)
    r = eng.register(T0, history=False)
    out = dict(T=r.T.cpu().numpy(), n_outer=r.n_outer.cpu().numpy(), converged_at=r.converged_at.cpu().numpy())
    if evaluate:
        q = eng.evaluate(r.T)
        out.update(n_inliers=q.n_inliers.cpu().numpy(), fitness=q.fitness.cpu().numpy(),
                   inlier_rmse=q.inlier_rmse.cpu().numpy(), information=q.H.cpu().numpy())
    return out


def gicp(source_points, target_points, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
         max_distance_nearest_neighbors=50):
    """Same call, same 7-tuple as the reference (gicp.py:78,174):
    (transformation_matrix, all_transformations, initial_source_cov_matrices, target_cov_matrices,
     highest_weight_points_source, highest_weight_points_target, all_source_cov_matrices)."""
    r = gicp_extended(source_points, target_points, max_iterations, tolerance, max_distance_correspondence,
                      max_distance_nearest_neighbors)
    if r["converged_at"] >= 0:
        print("Converged at iteration", r["converged_at"])   # gicp.py:161 (observable behaviour)
    return (r["T"], r["all_T"], r["src_cov0"], r["tgt_cov"], r["hw_src"], r["hw_tgt"], r["all_src_cov"])
