"""The registration parameters beyond k, the distances, the iteration count, the tolerance and the covariance model,
away from their defaults, on the device:

A. the covariance regularisation (lambda_tangent, lambda_normal) through every K2 path (brute force, the general
   latency kernel, the histogram fast path with its hand-over, the general path at k = 32 and at f64 storage with
   k = 20): k-NN lists, covariances, W and whole registrations against the float64 oracle, and the metamorphic
   identity lambda_t = lambda_n = 0.5 -> W = I -> the point-to-point registration;
B. gicpSetParams' validation of the lambdas: refused, handle and engine unchanged;
C. inner_max_iterations: 0 means 50; with the inner solve capped at 1 or 3 LM iterations the loop's bookkeeping
   (inliers, loss_hist, T_hist) still describes what it did, iteration by iteration, and in 2-D the step is exactly
   that of the host build of the 2-D solver;
D. the cell edges and the cell budget (knn_cell, nn_cell, max_cells_per_cloud) as a fixed table (CELL_ROWS, whose
   plans tests/test_plan_host.py checks on the host): every row against exact references and the default-knob run.

All inputs are float32-representable, so f32 and f64 storage see the same coordinates."""
import numpy as np
import pytest

import robust_oracle as RO
from oracle import gicp_oracle as O
from test_gpu_search_exactness import (Batch, _offset, _pair2d, _rot_about, _same_bits, _walls2d,  # noqa: F401
                                       check_loop, env, exact_nn)
from test_host import solve_host  # noqa: F401  (fixture: csrc/solve.cuh compiled for the host)

pytestmark = pytest.mark.gpu

# (lambda_tangent, lambda_normal): the defaults as the control, the regularisation of fast_gicp / small_gicp, equal
# lambdas, an inverted pair and a ratio of 1e-7 (below what an f32-stored covariance resolves, include/gicp_b200.h)
LAMBDAS = [(100.0, 10.0), (1.0, 1e-3), (1.0, 1.0), (10.0, 100.0), (1e4, 1e-3)]
F32_UNRESOLVED = (1e4, 1e-3)
# f32 storage on the scan pair at (1, 1e-3): the loss is about 1e3 times the default one and its float32 reduced form
# (2e-5 relative, check_loop) no longer settles the stop rule's absolute 1e-6, so the loop stops later than the oracle
# (observed 53 outer iterations against 10) at the same transform
F32_STOP_UNSETTLED = {("scan_360", (1.0, 1e-3))}

# ------------------------------------------------------------------------------------------------
# D's table: every input of part D has max_distance_nearest_neighbors r = 4 and max_distance_correspondence
# d_max = 2, so a row means the same grids for all of them.  (name, knobs, knn cell, nn cell, shared, budget or None
# for the automatic one, single-block build for a cloud of <= 2048 points)
# ------------------------------------------------------------------------------------------------
CELL_R, CELL_DMAX = 4.0, 2.0
CELL_ROWS = [
    ("default", {}, 1.0, 1.0, 1, None, 1),
    ("knn_cell 0.01 -> r/8", dict(knn_cell=0.01), 0.5, 1.0, 1, None, 1),
    ("knn_cell r/2, nn_cell 0.01 -> d_max/8", dict(knn_cell=2.0, nn_cell=0.01), 2.0, 0.25, 0, None, 1),
    ("knn_cell 2r, nn_cell d_max", dict(knn_cell=8.0, nn_cell=2.0), 8.0, 2.0, 0, None, 1),
    ("nn_cell 4 d_max", dict(nn_cell=8.0), 1.0, 8.0, 1, None, 1),
    ("knn_cell r/2, nn_cell d_max", dict(knn_cell=2.0, nn_cell=2.0), 2.0, 2.0, 1, None, 1),
    ("budget 64", dict(max_cells_per_cloud=64), 1.0, 1.0, 1, 64, 1),
    ("budget 4096", dict(max_cells_per_cloud=4096), 1.0, 1.0, 1, 4096, 1),
    ("budget 2^20", dict(max_cells_per_cloud=1 << 20), 1.0, 1.0, 1, 1 << 20, 1),
    ("budget 2^20 + 1", dict(max_cells_per_cloud=(1 << 20) + 1), 1.0, 1.0, 1, (1 << 20) + 1, 0),
]
CELL_UNSHARED, CELL_BUDGET_LIMITED = "knn_cell 2r, nn_cell d_max", "budget 64"
# sizes of the inputs of part D (source / target clouds)
CELL_SIZES = {"3d_f32": ([2000], [2000]), "2d_f64": ([1500], [1500]), "batch": ([1200, 2500, 4000], [1250, 2400, 4100])}


def _f32(a):
    return np.asarray(a, dtype=np.float64).astype(np.float32).astype(np.float64)


def _motion_2d(deg, shift, c):
    th = np.deg2rad(deg)
    T = np.eye(3)
    T[:2, :2] = [[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]
    T[:2, 2] = np.asarray(c) - T[:2, :2] @ np.asarray(c) + np.asarray(shift)
    return T


def _pair_2d(n, seed, deg=3.0, shift=(0.6, -0.4)):
    """Scan-like 2-D pair (points on line segments in a 100 m box) and the motion mapping source onto target."""
    rng = np.random.default_rng(seed)
    s, t = _pair2d(rng, n, deg, shift)
    return _f32(s), _f32(t), _motion_2d(deg, shift, (50.0, 50.0))


def _pair_3d(n, seed, n_patches=6):
    from generalized_icp_b200 import synthetic
    s, t, Tg = synthetic.patches3d_pair(n=n, n_patches=n_patches, cube=30.0, patch=20.0, seed=seed)
    return s.astype(np.float64), t.astype(np.float64), Tg


def _scans():
    import demo_inputs
    scans, _ = demo_inputs.lidar_sequence(seed=3, num_rays=360, n_scans=2)
    return _f32(scans[0]), _f32(scans[1])


# ------------------------------------------------------------------------------------------------
# A. covariance regularisation
# ------------------------------------------------------------------------------------------------
# (path, n, k per dim, storages): brute <= 128 points; the general latency kernel 129-2048; the histogram fast path
# (k + 8 within the list: 32 f32 / 21 f64 entries) with the general path taking over overflowed warps; the general
# path at k = 32; f64 storage at k = 20 (beyond the f64 list)
K2_PATHS = [("brute", 100, {2: 6, 3: 20}, ("f32", "f64")),
            ("general_latency", 1500, {2: 6, 3: 20}, ("f32", "f64")),
            ("hist", 6000, {2: 6, 3: 12}, ("f32", "f64")),
            ("general_k32", 6000, {2: 32, 3: 32}, ("f32", "f64")),
            ("general_f64_k20", 6000, {2: 20, 3: 20}, ("f64",))]
K2_RADIUS = {2: 3.0, 3: 4.0}


def _k2_cloud(dim, n):
    """About 20 neighbours within the radius per point at every size."""
    small = n <= 128
    if dim == 3:
        from generalized_icp_b200 import synthetic
        patch = 10.0 if small else 20.0
        s, _, _ = synthetic.patches3d_pair(n=n, n_patches=2 if small else 4, cube=patch + 10.0, patch=patch, seed=n)
        return s.astype(np.float64)
    return _f32(_walls2d(np.random.default_rng(n), n, box=10.0 if small else 100.0))


def _knn_exact(cloud, k, r):
    """The oracle's k-NN rule (float64 key, then lower index, exclusive radius) from cKDTree candidates re-ranked by
    that key; (idx with -1 for missing, dist)."""
    from scipy.spatial import cKDTree
    n = len(cloud)
    kk = min(k + 4, n)
    _, cand = cKDTree(cloud).query(cloud, k=kk, distance_upper_bound=r * (1 + 1e-9), workers=-1)
    cand = cand.reshape(n, kk)
    safe = np.where(cand < n, cand, 0)
    d = cloud[safe] - cloud[:, None, :]
    key = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
    if cloud.shape[1] == 3:
        key = key + d[..., 2] * d[..., 2]
    key = np.where(cand < n, key, np.inf)
    order = np.lexsort((cand, key), axis=-1)
    cand, key = np.take_along_axis(cand, order, 1), np.take_along_axis(key, order, 1)
    # the candidates beyond the k-th must not tie with it (the tree's own order would then decide)
    if kk > k:
        assert not np.any(np.isfinite(key[:, k - 1]) & (key[:, k] == key[:, k - 1]))
    dist = np.sqrt(key[:, :k])
    ok = dist < r
    return np.where(ok, cand[:, :k], -1), np.where(ok, dist, np.inf)


def _neighbour_scatter(cloud, want):
    """Count, scatter eigenvalues (ascending) of every row's k-NN set (want: -1 = missing)."""
    nb = np.where(want < 0, 0, want)
    w = (want >= 0)[..., None].astype(np.float64)
    cnt = (want >= 0).sum(1)
    mean = (cloud[nb] * w).sum(1) / np.maximum(cnt, 1)[:, None]
    dev = (cloud[nb] - mean[:, None, :]) * w
    return cnt, np.linalg.eigvalsh(np.einsum("nki,nkj->nij", dev, dev))


def _check_covariances(cov, cloud, want, lam_t, lam_n, storage):
    dim = cloud.shape[1]
    cnt, ev = _neighbour_scatter(cloud, want)
    ref = O.covariances_from_neighbors(cloud, np.where(want < 0, len(cloud), want), lam_t, lam_n)
    lone = cnt <= 1
    assert np.array_equal(cov[lone], np.broadcast_to(np.eye(dim), (int(lone.sum()), dim, dim)))
    if lam_t == lam_n:
        assert np.array_equal(cov[~lone], np.broadcast_to(lam_t * np.eye(dim), (int((~lone).sum()), dim, dim)))
        return
    # the normal (3-D) / the main direction (2-D) is defined where the scatter's eigen-gap is healthy; the error of
    # the eigenvector grows as 1 / gap (the rule of test_host.py::test_covariance_tail_host)
    gap = (ev[:, 1] - ev[:, 0]) / np.maximum(ev[:, -1], 1e-300)
    healthy = (cnt > dim) & (gap > 1e-2)
    assert healthy.mean() > 0.5, healthy.mean()
    lam = max(lam_t, lam_n)
    tol = np.maximum(1e-9 * lam * 10 / np.maximum(gap, 1e-12), 1e-9 * lam)[:, None, None]
    if storage == "f32":
        tol = tol + 2.0 ** -24 * np.abs(ref)        # one float32 rounding of every entry
    err = np.abs(cov - ref)
    bad = healthy[:, None, None] & (err > tol)
    assert not bad.any(), (np.argwhere(bad)[:5], err[bad][:5])


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("path,n,ks,storages", K2_PATHS, ids=[p[0] for p in K2_PATHS])
def test_regularisation_on_every_k2_path(path, n, ks, storages, dim):
    """k-NN lists bit-exact (the lambdas do not change them), covariances against the oracle's with the same lambdas,
    and gicpCorrespond's W against inv(R C_A R^T + C_B) built from the device's own covariances."""
    k, r = ks[dim], K2_RADIUS[dim]
    cloud = _k2_cloud(dim, n)
    want, wd = _knn_exact(cloud, k, r)
    c = cloud.mean(0)
    T = _motion_2d(2.0, (0.3, -0.2), c) if dim == 2 else _rot_about(c, 2.0, seed=n)
    T[:dim, dim] += 0.1
    for storage in storages:
        b = Batch(dim, storage, [cloud], [cloud], k=k, max_distance_nearest_neighbors=r,
                  max_distance_correspondence=3.0)
        for lam_t, lam_n in LAMBDAS:
            b.eng.set_params(lambda_tangent=lam_t, lambda_normal=lam_n)
            b.setup()
            for which in (0, 1):
                idx, dist = b.eng.knn(which)
                assert np.array_equal(idx.cpu().numpy(), want), (storage, lam_t, lam_n, which)
                m = want >= 0
                assert np.all(np.abs(dist.cpu().numpy()[m] - wd[m]) <= 1e-12 * wd[m])
            cs = b.eng.covariances(0).cpu().numpy()
            ct = b.eng.covariances(1).cpu().numpy()
            assert np.array_equal(cs, ct)
            _check_covariances(ct, cloud, want, lam_t, lam_n, storage)
            gi, _, W = b.eng.correspond(T)
            gi, W = gi.cpu().numpy(), W.cpu().numpy()
            R = T[:dim, :dim]
            Wref = O.weights(R @ cs @ R.T, ct, gi)
            g = gi >= 0
            assert g.mean() > 0.5
            # inversion in float64: error up to ~cond * eps relative to the matrix
            M = R @ cs[g] @ R.T + ct[gi[g]]
            cond = np.linalg.cond(M)
            scale = np.abs(Wref[g]).max(axis=(1, 2))
            tol = np.maximum(1e-9, 64 * np.finfo(np.float64).eps * cond) * scale
            assert np.all(np.abs(W[g] - Wref[g]).max(axis=(1, 2)) <= tol), (storage, lam_t, lam_n)
            assert np.all(W[~g] == 0.0)


def _e2e_inputs(name):
    if name == "3d_patch":
        s, t, _ = _pair_3d(1500, seed=1)
        return 3, s, t, dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0), 30.0
    s, t = _scans()
    return 2, s, t, dict(max_distance_nearest_neighbors=200.0), 400.0


@pytest.mark.parametrize("name", ["3d_patch", "scan_360"])
@pytest.mark.parametrize("lam", LAMBDAS, ids=[f"{a:g}-{b:g}" for a, b in LAMBDAS])
def test_regularisation_end_to_end(name, lam, env):
    """Both storages, fused loop and multi-launch loop, against the float64 oracle with the reference's covariance
    recomputation every outer iteration: same iteration count and convergence flag, <= 1e-5 rad, <= 1e-5 extent.
    At lambda_n / lambda_t = 1e-7 with f32 storage the rounded covariances no longer resolve lambda_n: there the
    registration must stay finite and stop."""
    dim, s, t, params, extent = _e2e_inputs(name)
    lam_t, lam_n = lam
    ref = O.gicp_oracle(s, t, lam_t=lam_t, lam_n=lam_n, inner="newton", recompute_src_cov=True, record=False,
                        **params)
    conv_ref = -1 if ref["converged_at"] is None else ref["converged_at"]
    assert len(s) <= 2048                                     # the fused loop is the default
    for storage in ("f32", "f64"):
        b = Batch(dim, storage, [s], [t], lambda_tangent=lam_t, lambda_normal=lam_n, **params)
        for fused in ("1", "0"):
            r = env(b.register, GICP_FUSED_LOOP=fused)
            n_out = int(r.n_outer[0])
            what = (storage, fused, n_out, ref["n_outer"])
            rot, trans = RO.motion_error(r.T[0].cpu().numpy(), ref["T"])
            if storage == "f32" and (name, lam) in F32_STOP_UNSETTLED:
                # the final T agrees; the iteration at which |last - min_loss| first drops below 1e-6 does not
                assert np.isfinite(r.loss_hist.cpu().numpy()[0, :n_out]).all(), what
                assert rot <= 1e-5 and trans <= 1e-5 * extent, (what, rot, trans)
                continue
            if storage == "f32" and lam == F32_UNRESOLVED:
                assert 1 <= n_out <= b.eng.params.max_iterations, what
                assert np.isfinite(r.T.cpu().numpy()).all(), what
                assert np.isfinite(r.loss_hist.cpu().numpy()[0, :n_out]).all(), what
                print(f"{name} f32 lambda {lam} fused={fused}: n_outer {n_out} (oracle {ref['n_outer']}), "
                      f"error vs oracle {rot:.3g} rad, {trans:.3g}")
                continue
            assert n_out == ref["n_outer"], what
            assert int(r.converged_at[0]) == conv_ref, what
            assert rot <= 1e-5 and trans <= 1e-5 * extent, (what, rot, trans)


@pytest.mark.parametrize("dim,storage", [(2, "f64"), (3, "f32"), (3, "f64")])
def test_equal_half_lambdas_are_point_to_point(dim, storage, env):
    """lambda_t = lambda_n = 0.5 on clouds where every point has >= 2 neighbours: every C is 0.5 I, so
    W = inv(0.5 R R^T + 0.5 I) = I, which is the point-to-point model (C_A = 0, C_B = I).  The two registrations agree:
    same iteration count, convergence flag and inliers, T history to 1e-9."""
    if dim == 3:
        s, t, Tg = _pair_3d(1500, seed=4)
        params = dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0)
        T = _rot_about(np.full(3, 15.0), 2.0, seed=2) @ Tg
    else:
        s, t = _scans()
        params = dict(max_distance_nearest_neighbors=200.0)
        T = _motion_2d(1.0, (2.0, -1.0), (0.0, 0.0))
    for cloud in (s, t):
        nb, _ = O.knn_kdtree(cloud, 2, params["max_distance_nearest_neighbors"])
        assert (nb[:, 1] < len(cloud)).all()
    half = Batch(dim, storage, [s], [t], lambda_tangent=0.5, lambda_normal=0.5, **params)
    gi, _, W = half.eng.correspond(T)
    g = gi.cpu().numpy() >= 0
    assert g.mean() > 0.5
    assert np.abs(W.cpu().numpy()[g] - np.eye(dim)).max() <= 1e-12
    p2p = Batch(dim, storage, [s], [t], covariance_model=1, **params)
    for fused in ("1", "0"):
        a = env(half.register, GICP_FUSED_LOOP=fused)
        c = env(p2p.register, GICP_FUSED_LOOP=fused)
        for f in ("n_outer", "converged_at", "inliers"):
            assert np.array_equal(getattr(a, f).cpu().numpy(), getattr(c, f).cpu().numpy()), (fused, f)
        n = int(a.n_outer[0])
        assert n >= 3
        dh = np.abs(a.T_hist.cpu().numpy()[0, :n] - c.T_hist.cpu().numpy()[0, :n])
        assert np.nanmax(dh) <= 1e-9, (fused, np.nanmax(dh))


# ------------------------------------------------------------------------------------------------
# B. validation
# ------------------------------------------------------------------------------------------------
BAD_LAMBDAS = [0.0, -1.0, -0.0, float("nan"), float("inf"), float("-inf")]


def test_invalid_lambdas_are_refused_and_nothing_changes():
    """gicpSetParams refuses a lambda that is not finite and > 0, naming the field; the engine keeps its parameters
    and its set-up clouds, and a later valid set gives bit-identical results to a fresh engine."""
    from generalized_icp_b200 import compat
    s, t = _scans()
    params = dict(max_distance_nearest_neighbors=200.0, lambda_tangent=1.0, lambda_normal=1e-3)
    compat_before = compat.gicp_extended(s, t, max_distance_nearest_neighbors=200.0, full_history=False)
    b = Batch(2, "f64", [s], [t], **params)
    ref = b.register()
    before = bytes(b.eng.params)
    for field in ("lambda_tangent", "lambda_normal"):
        for v in BAD_LAMBDAS:
            with pytest.raises(RuntimeError, match=f"{field} must be finite and > 0"):
                b.eng.set_params(**{field: v})
            assert bytes(b.eng.params) == before
            with pytest.raises(RuntimeError, match=f"{field} must be finite and > 0"):
                compat.gicp_extended(s, t, max_distance_nearest_neighbors=200.0, full_history=False, **{field: v})
    _same_bits(ref, b.register(), "set-up clouds kept")
    b.eng.set_params(lambda_tangent=100.0, lambda_normal=10.0)
    b.setup()
    fresh = Batch(2, "f64", [s], [t], max_distance_nearest_neighbors=200.0)
    _same_bits(fresh.register(), b.register(), "after refusals")
    got = compat.gicp_extended(s, t, max_distance_nearest_neighbors=200.0, full_history=False)
    for f in ("T", "loss_hist", "inliers", "n_outer", "converged_at"):
        assert np.array_equal(got[f], compat_before[f]), f


# ------------------------------------------------------------------------------------------------
# C. inner_max_iterations
# ------------------------------------------------------------------------------------------------
def _capped_case(dim):
    if dim == 2:
        s, t, Tg = _pair_2d(1500, seed=5, deg=4.0, shift=(1.0, -0.5))
        return 2, "f64", s, t, dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=5.0,
                                    max_iterations=25), None
    from generalized_icp_b200 import synthetic
    s, t, Tg = synthetic.patches3d_pair(n=1800, n_patches=4, cube=20.0, patch=15.0, seed=3)
    s, t = s.astype(np.float64), t.astype(np.float64)
    T0 = (_rot_about(np.full(3, 10.0), 6.0, seed=9) @ Tg)[None]
    return 3, "f32", s, t, dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0,
                                max_iterations=25), T0


def _check_capped(b, r, T0=None):
    """Every executed iteration k of every pair, with the inner solve stopped early: the inlier count is the exact
    gated count; loss_hist[k] is the frozen objective of the exact matches at T_hist[k + 1] (when T was updated), not
    above that objective at T_k and not below its minimum (the oracle's Newton solver)."""
    d, d1 = b.dim, b.dim + 1
    d_max = float(b.params["max_distance_correspondence"])
    rel = 2e-5 if b.storage == "f32" else 1e-9
    cs, ct = b.eng.covariances(0).cpu().numpy(), b.eng.covariances(1).cpu().numpy()
    T_hist, loss = r.T_hist.cpu().numpy(), r.loss_hist.cpu().numpy()
    inl, n_out, conv = r.inliers.cpu().numpy(), r.n_outer.cpu().numpy(), r.converged_at.cpu().numpy()
    if T0 is not None:
        assert np.array_equal(T_hist[:, 0], np.asarray(T0).reshape(-1, d1, d1))
    for k in range(int(n_out.max())):
        Tk_all = np.where(np.isnan(T_hist[:, k]), np.eye(d1), T_hist[:, k])
        idx_dev, _, _ = b.eng.correspond(Tk_all, with_W=False)
        idx_dev = idx_dev.cpu().numpy()
        for p in range(b.n_pairs):
            if n_out[p] <= k:
                continue
            s, t, Tk = b.srcs[p], b.tgts[p], T_hist[p, k]
            pp = s @ Tk[:d, :d].T + Tk[:d, d]
            idx, key, key2 = exact_nn(t, pp)
            dist = np.sqrt(key)
            want = np.where(dist > d_max, -1, idx)
            gi = idx_dev[b.off_s[p]:b.off_s[p + 1]]
            dp = 8 * np.finfo(np.float64).eps * np.abs(pp).max(1)
            ok = ~(key2 - key <= 1e-9 * key + 4 * dist * dp) & ~(np.abs(dist - d_max) <= 1e-9 * d_max + dp)
            assert np.array_equal(gi[ok], want[ok]), (p, k)
            m = np.where(ok, want, gi)
            g = m >= 0
            assert inl[p, k] == g.sum(), (p, k, inl[p, k], g.sum())
            Rk = Tk[:d, :d]
            q = t[m[g]]
            W = np.linalg.inv(Rk @ cs[b.off_s[p]:b.off_s[p + 1]][g] @ Rk.T + ct[b.off_t[p]:b.off_t[p + 1]][m[g]])
            e = q - pp[g]
            f_k = float(np.einsum("ni,nij,nj->", e, W, e))
            _, f_min, _, _ = O.inner_newton(_offset(Tk, d), s[g], q, W)
            scale = max(abs(f_k), abs(f_min))
            tol = rel * scale + 1e-12
            assert loss[p, k] <= f_k + tol, (p, k, loss[p, k], f_k)
            assert loss[p, k] >= f_min - tol, (p, k, loss[p, k], f_min)
            if conv[p] != k:
                dT = T_hist[p, k + 1] @ np.linalg.inv(Tk)
                res = q - (pp[g] @ dT[:d, :d].T + dT[:d, d])
                f_next = float(np.einsum("ni,nij,nj->", res, W, res))
                assert abs(loss[p, k] - f_next) <= rel * (scale if b.storage == "f32" else abs(f_next)) + 1e-12, \
                    (p, k, loss[p, k], f_next)
    for p in range(b.n_pairs):
        assert np.isnan(loss[p, n_out[p]:]).all() and (inl[p, n_out[p]:] == 0).all()


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_inner_iteration_cap(dim, fused, env, solve_host):
    import ctypes
    dim, storage, s, t, params, T0 = _capped_case(dim)
    assert len(s) <= 2048
    b = Batch(dim, storage, [s], [t], **params)
    full = env(lambda: b.register(T0), GICP_FUSED_LOOP=fused)
    runs = {}
    for cap in (0, 1, 3):
        b.eng.set_params(inner_max_iterations=cap)
        b.setup()
        runs[cap] = env(lambda: b.register(T0), GICP_FUSED_LOOP=fused)
    _same_bits(full, runs[0], "inner_max_iterations 0 = 50")
    assert not np.array_equal(runs[1].T_hist.cpu().numpy(), full.T_hist.cpu().numpy(), equal_nan=True)
    for cap in (1, 3):
        b.eng.set_params(inner_max_iterations=cap)
        b.setup()
        _check_capped(b, runs[cap], T0)
    if dim == 2:
        # one LM iteration of the host build of inner_solve_2d on the stage's reduced form at T_hist[k], un-centred
        # and composed as the loop does, is the loop's T_hist[k + 1] (the sums run in another order: 1e-9)
        b.eng.set_params(inner_max_iterations=1)
        b.setup()
        r = runs[1]
        dp = ctypes.POINTER(ctypes.c_double)
        T_hist, n_out, conv = r.T_hist.cpu().numpy()[0], int(r.n_outer[0]), int(r.converged_at[0])
        for k in range(n_out):
            if k == conv:
                continue
            T = T_hist[k]
            red = np.ascontiguousarray(b.eng.normal_equations(T)[0])
            out = np.zeros(8)
            assert solve_host.gicp_test_solve2d(red.ctypes.data_as(dp), 1, out.ctypes.data_as(dp)) == 0
            dtc, dR, mu = out[:2], out[4:].reshape(2, 2), red[26:28]
            Tn = np.eye(3)
            Tn[:2, :2] = dR @ T[:2, :2]
            Tn[:2, 2] = dR @ T[:2, 2] + dtc - (dR - np.eye(2)) @ mu
            assert np.abs(Tn - T_hist[k + 1]).max() <= 1e-9 * max(1.0, np.abs(T).max()), (k, Tn, T_hist[k + 1])


# ------------------------------------------------------------------------------------------------
# D. cell edges and cell budget
# ------------------------------------------------------------------------------------------------
def _cell_input(name):
    """(dim, storage, srcs, tgts, generating motions): sizes CELL_SIZES[name]."""
    ns, nt = CELL_SIZES[name]
    if name == "2d_f64":
        s, t, Tg = _pair_2d(ns[0], seed=8)
        return 2, "f64", [s], [t], [Tg]
    srcs, tgts, Ts = [], [], []
    for i, (a, c) in enumerate(zip(ns, nt)):
        s, _, Tg = _pair_3d(a, seed=60 + i)
        _, t, _ = _pair_3d(c, seed=60 + i)           # same patches and motion, another sample of the target
        srcs.append(s)
        tgts.append(t)
        Ts.append(Tg)
    return 3, ("f32" if name == "3d_f32" else "f64"), srcs, tgts, Ts


def _elongated(n=20000, seed=12):
    """A 3 km x 4 m x 4 m tunnel (wavy floor, two walls): at the default k-NN cell (r / 4 = 1 m) its long axis needs
    12 Morton bits, so choose_grid enlarges the cells to stay within 10."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.0, 3000.0, n)
    side = rng.integers(0, 3, n)
    u = rng.uniform(0.0, 4.0, n)
    floor = 0.5 * np.sin(x / 7.0)
    y = np.where(side == 0, u, np.where(side == 1, 0.0, 4.0))
    z = np.where(side == 0, floor, floor + u)
    src = np.stack([x, y, z], 1) + rng.normal(0, 0.01, (n, 3))
    T = _rot_about(np.array([1500.0, 2.0, 2.0]), 0.003, seed=seed)
    T[:3, 3] += (0.2, 0.1, 0.05)
    tgt = src @ T[:3, :3].T + T[:3, 3] + rng.normal(0, 0.01, (n, 3))
    return _f32(src), _f32(tgt), T


def _check_correspond(b, T_all):
    """gicpCorrespond at T against the exact 1-NN with the gate, near-ties and gate ties excluded as check_loop does."""
    d = b.dim
    d_max = float(b.params["max_distance_correspondence"])
    gi, _, _ = b.eng.correspond(np.stack(T_all), with_W=False)
    gi = gi.cpu().numpy()
    for p in range(b.n_pairs):
        T = T_all[p]
        pp = b.srcs[p] @ T[:d, :d].T + T[:d, d]
        idx, key, key2 = exact_nn(b.tgts[p], pp)
        dist = np.sqrt(key)
        dp = 8 * np.finfo(np.float64).eps * np.abs(pp).max(1)
        ok = ~(key2 - key <= 1e-9 * key + 4 * dist * dp) & ~(np.abs(dist - d_max) <= 1e-9 * d_max + dp)
        assert ok.mean() > 0.99
        assert np.array_equal(gi[b.off_s[p]:b.off_s[p + 1]][ok], np.where(dist > d_max, -1, idx)[ok]), p


def _same_run(a, c, what, storage):
    """A different grid reorders the fixed-order sums: counts identical, histories to 1e-9 relative.  With f32
    storage the covariances may also differ by their last bit (one f32 ulp, 6e-8 relative) and the reduced form is
    accumulated in float32: T history 1e-6, loss history 2e-5 (check_loop's f32 bound)."""
    tol = {"T_hist": 1e-6, "loss_hist": 2e-5} if storage == "f32" else {"T_hist": 1e-9, "loss_hist": 1e-9}
    for f in ("n_outer", "converged_at", "inliers"):
        assert np.array_equal(getattr(a, f).cpu().numpy(), getattr(c, f).cpu().numpy()), (what, f)
    for p in range(a.n_outer.shape[0]):
        n = int(a.n_outer[p])
        for f, rows in (("T_hist", n + 1 if int(a.converged_at[p]) < 0 else n), ("loss_hist", n)):
            x, y = getattr(a, f)[p, :rows].cpu().numpy(), getattr(c, f)[p, :rows].cpu().numpy()
            assert np.all(np.abs(x - y) <= tol[f] * np.maximum(np.abs(y), 1.0)), (what, f, p, np.abs(x - y).max())


def _cell_rows_on(dim, storage, srcs, tgts, Ts, params, rows, loop_rows):
    """Every row of `rows` on one input, the first being the default knobs; check_loop on the rows in `loop_rows`."""
    want = [_knn_exact(c, params["k"], params["max_distance_nearest_neighbors"])[0] for c in srcs + tgts]
    T_starts = [np.eye(dim + 1) for _ in srcs]
    ref = None
    for name, knobs, *_ in rows:
        b = Batch(dim, storage, srcs, tgts, **params, **knobs)
        for which, side in ((0, srcs), (1, tgts)):
            idx, _ = b.eng.knn(which)
            idx = idx.cpu().numpy()
            off = np.concatenate([[0], np.cumsum([len(c) for c in side])])
            for i in range(len(side)):
                wi = want[i] if which == 0 else want[len(srcs) + i]
                assert np.array_equal(idx[off[i]:off[i + 1]], wi), (name, which, i)
        cov = (b.eng.covariances(0).cpu().numpy(), b.eng.covariances(1).cpu().numpy())
        _check_correspond(b, T_starts)
        _check_correspond(b, Ts)
        r = b.register()
        assert (r.n_outer.cpu().numpy() >= 2).all()
        if ref is None:
            ref, ref_cov = r, cov
        else:
            for c, c0 in zip(cov, ref_cov):
                if storage == "f64":
                    assert np.abs(c - c0).max() <= 1e-12 * params.get("lambda_tangent", 100.0), name
                else:
                    ulp = np.spacing(np.abs(c0).astype(np.float32)).astype(np.float64)
                    assert np.all(np.abs(c - c0) <= ulp), name
            _same_run(r, ref, name, storage)
        if name in loop_rows:
            check_loop(b, r)


@pytest.mark.parametrize("case", list(CELL_SIZES))
def test_cell_table(case):
    """Every row of CELL_ROWS (shared and unshared grids, enlarged and raised cell edges, a budget that forces coarse
    cells, the single-block build's largest budget and one above it) on a 3-D f32 pair, a 2-D f64 pair and a 3-pair
    3-D f64 batch: k-NN lists bit-exact, covariances equal to the default-knob run's (f64 1e-12 of lambda_t, f32 one
    ulp), 1-NN at T = I and at the generating motion exact, the registration equal to the default-knob run (counts
    identical, histories 1e-9), and every loop iteration exact on the unshared and the budget-limited rows."""
    dim, storage, srcs, tgts, Ts = _cell_input(case)
    params = dict(k=6 if dim == 2 else 20, max_distance_nearest_neighbors=CELL_R,
                  max_distance_correspondence=CELL_DMAX, max_iterations=30)
    _cell_rows_on(dim, storage, srcs, tgts, Ts, params, CELL_ROWS, (CELL_UNSHARED, CELL_BUDGET_LIMITED))


def test_elongated_cloud_beyond_the_morton_axis_cap():
    """The tunnel at the default cells (the 10-bit axis cap enlarges them) and at 3 m cells (within the cap, no
    enlargement): the same checks as the table."""
    s, t, T = _elongated()
    params = dict(k=20, max_distance_nearest_neighbors=CELL_R, max_distance_correspondence=CELL_DMAX,
                  max_iterations=30)
    rows = [("default: enlarged cells", {}), ("3 m cells", dict(knn_cell=3.0, nn_cell=3.0))]
    _cell_rows_on(3, "f32", [s], [t], [T], params, rows, ("default: enlarged cells",))
