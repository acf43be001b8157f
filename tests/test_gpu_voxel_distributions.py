"""Voxel distributions (gicpSetVoxelized, include/gicp_b200.h) on the device: the set-up against the float64 oracle
(tests/voxel_dist_oracle.py) and bit for bit against gicpVoxelDownsample, batches against their clouds one at a time,
the registration loop iteration by iteration against exact references on every voxelized / raw combination, end to
end against the float64 loop fed with the oracle's voxel means and covariances, an exact equivalence with raw sides,
composition with the other entry points, and refusals that leave the set-up sides alone."""
import numpy as np
import pytest

import voxel_dist_oracle as VD
from test_gpu_search_exactness import Batch, _rot_about, _same_bits, check_loop, env  # noqa: F401 (env: fixture)

pytestmark = pytest.mark.gpu

SOURCE, TARGET = 0, 1
P3 = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0, max_iterations=40)


def _np_dt(storage):
    return np.float32 if storage == "f32" else np.float64


def _clustered(dim, per_vox, n_vox, leaf, seed):
    """n_vox distinct voxels (negative and positive indices) with per_vox points each, spread anisotropically inside
    the voxel (a healthy eigen-gap), in shuffled row order."""
    rng = np.random.default_rng(seed)
    cells = set()
    while len(cells) < n_vox:
        cells.add(tuple(rng.integers(-40, 40, size=dim)))
    cells = np.array(sorted(cells), dtype=np.float64)
    pts = []
    for c in cells:
        Q, _ = np.linalg.qr(rng.normal(size=(dim, dim)))
        z = rng.normal(size=(per_vox, dim)) * np.array([0.15, 0.08, 0.01][:dim]) @ Q.T
        pts.append((c + 0.5 + np.clip(z, -0.45, 0.45)) * leaf)
    P = np.concatenate(pts)
    return P[rng.permutation(len(P))]


def _engine(dim, storage, **prm):
    from generalized_icp_b200.engine import GicpEngine
    eng = GicpEngine(dim, storage)
    if prm:
        eng.set_params(**prm)
    return eng


def _check_covs(cov, pts64, off, leaf, min_points, storage, lam_t=100.0, lam_n=10.0):
    """Device covariances against the oracle's: one-point voxels exactly I, the rest within the eigen-gap-scaled bound
    of test_gpu_params.py where the voxel scatter's eigen-gap is healthy."""
    dim = pts64.shape[1]
    means, oo, ref, counts = VD.voxel_distributions(pts64, off, leaf, min_points, lam_t, lam_n)
    assert cov.shape == ref.shape
    lone = counts == 1
    assert np.array_equal(cov[lone], np.broadcast_to(np.eye(dim), (int(lone.sum()), dim, dim)))
    # eigenvalues of every voxel's scatter, from the oracle's own grouping
    from voxel_oracle import voxel_downsample
    _, oo2, voxel_of, _ = voxel_downsample(pts64, off, leaf, min_points)
    ev = np.zeros((len(ref), dim))
    for c in range(len(off) - 1):
        vo_c = voxel_of[off[c]:off[c + 1]]
        X = pts64[off[c]:off[c + 1]]
        for j in range(int(oo2[c + 1] - oo2[c])):
            Y = X[vo_c == j]
            if len(Y) > 1:
                D = Y - Y.mean(0)
                ev[oo2[c] + j] = np.linalg.eigvalsh(D.T @ D)
    gap = (ev[:, 1] - ev[:, 0]) / np.maximum(ev[:, -1], 1e-300)
    healthy = (counts > dim) & (gap > 1e-2)
    lam = max(lam_t, lam_n)
    tol = np.maximum(1e-9 * lam * 10 / np.maximum(gap, 1e-12), 1e-9 * lam)[:, None, None]
    if storage == "f32":
        tol = tol + 2.0 ** -24 * np.abs(ref)
    err = np.abs(cov - ref)
    bad = healthy[:, None, None] & (err > tol)
    assert not bad.any(), (np.argwhere(bad)[:5], err[bad][:5])
    return healthy


# ------------------------------------------------------------------------------------------------
# set-up against the oracle and against gicpVoxelDownsample
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("per_vox,min_points", [(1, 1), (5, 1), (5, 3), (100, 1), (100, 3)])
def test_setup_vs_oracle(dim, storage, per_vox, min_points):
    import torch
    leaf = 0.5
    n_vox = 300 if per_vox < 100 else 60
    a = _clustered(dim, per_vox, n_vox, leaf, seed=per_vox + dim)
    b = _clustered(dim, max(1, per_vox // 2), n_vox // 2, leaf, seed=7 + per_vox)     # a second cloud, 2-point voxels
    P = np.concatenate([a, b]).astype(_np_dt(storage))
    P[3] = np.nan                                                                     # a dropped row
    off = np.array([0, len(a), len(a), len(P)], dtype=np.int64)                       # an empty middle cloud
    pts = torch.as_tensor(P, device="cuda")
    eng = _engine(dim, storage)
    means, oo = eng.set_target_voxelized(pts, off, voxel_size=leaf, min_points=min_points)
    ds, do = eng.voxel_downsample(pts, off, voxel_size=leaf, min_points=min_points)
    assert np.array_equal(oo, do)
    assert torch.equal(means.view(torch.int32 if storage == "f32" else torch.int64),
                       ds.view(torch.int32 if storage == "f32" else torch.int64))
    assert eng._n[TARGET] == (int(oo[-1]), 3)
    cov = eng.covariances(TARGET).cpu().numpy()
    healthy = _check_covs(cov, P.astype(np.float64), off, leaf, min_points, storage)
    if per_vox >= 5:
        assert healthy.mean() > 0.5, healthy.mean()
    # the source side gives the same bits (covariance_model 0)
    sm, so = eng.set_source_voxelized(pts, off, voxel_size=leaf, min_points=min_points)
    assert np.array_equal(so, oo) and torch.equal(sm, means)
    assert torch.equal(eng.covariances(SOURCE), eng.covariances(TARGET))


# ------------------------------------------------------------------------------------------------
# batches, reproducibility
# ------------------------------------------------------------------------------------------------
def _pairs(n_pairs, n=8000, seed=0):
    from generalized_icp_b200 import synthetic
    out = []
    for i in range(n_pairs):
        s, t, Tg = synthetic.patches3d_pair(n=n + 313 * i, n_patches=4, cube=20.0, patch=10.0, seed=seed + i)
        out.append((s, t, Tg))
    return out


def test_batch_equals_clouds_one_at_a_time_and_reproducible():
    import torch
    pairs = _pairs(3)
    eng = _engine(3, "f32", **P3)
    leaf = 1.0
    singles = []
    for s, t, _ in pairs:
        tm, _ = eng.set_target_voxelized(torch.as_tensor(t, device="cuda"), voxel_size=leaf)
        sm, _ = eng.set_source_voxelized(torch.as_tensor(s, device="cuda"), voxel_size=leaf)
        r = eng.register()
        torch.cuda.synchronize()
        singles.append((tm.clone(), sm.clone(), eng.covariances(TARGET), eng.covariances(SOURCE), r))
    off_s = np.concatenate([[0], np.cumsum([len(p[0]) for p in pairs])])
    off_t = np.concatenate([[0], np.cumsum([len(p[1]) for p in pairs])])
    S = torch.as_tensor(np.concatenate([p[0] for p in pairs]), device="cuda")
    T = torch.as_tensor(np.concatenate([p[1] for p in pairs]), device="cuda")

    def batch():
        tm, to = eng.set_target_voxelized(T, off_t, voxel_size=leaf)
        sm, so = eng.set_source_voxelized(S, off_s, voxel_size=leaf)
        r = eng.register()
        torch.cuda.synchronize()
        return tm.clone(), to, sm.clone(), so, eng.covariances(TARGET), eng.covariances(SOURCE), r

    tm, to, sm, so, ct, cs, r = batch()
    for i, (tm1, sm1, ct1, cs1, r1) in enumerate(singles):
        assert torch.equal(tm[to[i]:to[i + 1]], tm1) and torch.equal(sm[so[i]:so[i + 1]], sm1)
        assert torch.equal(ct[to[i]:to[i + 1]], ct1) and torch.equal(cs[so[i]:so[i + 1]], cs1)
        for f in ("T", "n_outer", "converged_at", "T_hist", "loss_hist", "inliers"):
            a, b = getattr(r, f)[i], getattr(r1, f)[0]
            assert torch.equal(a.view(torch.int64) if a.dtype == torch.float64 else a,
                               b.view(torch.int64) if b.dtype == torch.float64 else b), (i, f)
    again = batch()
    assert torch.equal(again[0], tm) and torch.equal(again[4], ct) and torch.equal(again[5], cs)
    _same_bits(r, again[6], "run to run")


# ------------------------------------------------------------------------------------------------
# per-iteration exactness of the loop on voxelized sides
# ------------------------------------------------------------------------------------------------
class VoxBatch(Batch):
    """Batch whose set-up voxelizes the chosen sides; srcs / tgts / offsets become what the engine then holds."""

    def __init__(self, dim, storage, srcs, tgts, leaf, vox_src, vox_tgt, **params):
        self.leaf, self.vox_src, self.vox_tgt = leaf, vox_src, vox_tgt
        super().__init__(dim, storage, srcs, tgts, **params)

    def setup(self):
        if not hasattr(self, "_raw"):
            self._raw = (self.srcs, self.tgts, self.off_s, self.off_t)
        srcs, tgts, off_s, off_t = self._raw
        if self.vox_tgt:
            m, off_t = self.eng.set_target_voxelized(self.T, off_t, voxel_size=self.leaf)
            m = m.cpu().numpy().astype(np.float64)
            tgts = [m[off_t[i]:off_t[i + 1]] for i in range(len(off_t) - 1)]
        else:
            self.eng.set_target(self.T, off_t)
        if self.vox_src:
            m, off_s = self.eng.set_source_voxelized(self.S, off_s, voxel_size=self.leaf)
            m = m.cpu().numpy().astype(np.float64)
            srcs = [m[off_s[i]:off_s[i + 1]] for i in range(len(off_s) - 1)]
        else:
            self.eng.set_source(self.S, off_s)
        self.srcs, self.tgts, self.off_s, self.off_t = srcs, tgts, np.asarray(off_s), np.asarray(off_t)


def _vox_case(storage="f32"):
    pairs = _pairs(2, n=6000, seed=20)
    T0 = np.stack([_rot_about(np.full(3, 10.0), 4.0 + 2 * i, seed=i) @ p[2] for i, p in enumerate(pairs)])
    return [p[0] for p in pairs], [p[1] for p in pairs], T0


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "multi_launch"])
@pytest.mark.parametrize("vox_src,vox_tgt", [(True, True), (False, True), (True, False), (False, False)])
def test_loop_exact_every_iteration(vox_src, vox_tgt, fused, env):
    srcs, tgts, T0 = _vox_case()
    b = VoxBatch(3, "f32", srcs, tgts, 1.0, vox_src, vox_tgt, **P3)
    if vox_src:
        assert max(np.diff(b.off_s)) <= 2048      # the fused loop's source size
    loop = {} if fused else {"GICP_FUSED_LOOP": 0}
    r = env(lambda: b.register(T0), **loop)
    assert (r.n_outer.cpu().numpy() >= 3).all()
    check_loop(b, r, T0)
    _same_bits(r, env(lambda: b.register(T0), GICP_NO_SKIP=1, **loop), "no skip")


@pytest.mark.parametrize("kernel", ["huber_fixed", "tukey_adaptive"])
def test_loop_exact_every_iteration_robust(kernel):
    from robust_oracle import robust_weight
    srcs, tgts, T0 = _vox_case()
    b = VoxBatch(3, "f32", srcs, tgts, 1.0, True, True, **P3)
    if kernel == "huber_fixed":
        b.eng.set_robust_kernel("huber", 0.3)
        r = b.register(T0)
        check_loop(b, r, T0, weight=lambda p, k, d: robust_weight("huber", d, 0.3))
    else:
        b.eng.set_robust_kernel("tukey", adaptive=4.0, min_scale=0.2)
        r = b.register(T0)
        T_hist = r.T_hist.cpu().numpy()
        d1 = 4
        scales = {}

        def weight(p, k, d):
            if k not in scales:
                Tk = np.where(np.isnan(T_hist[:, k]), np.eye(d1), T_hist[:, k])
                scales[k] = b.eng.robust_scales(Tk)   # the scale the loop took at T_k (include/gicp_b200.h)
            return robust_weight("tukey", d, scales[k][p])

        check_loop(b, r, T0, nonconvex=range(b.n_pairs), weight=weight)


# ------------------------------------------------------------------------------------------------
# end to end against the float64 loop with the oracle's voxel means and covariances.  min_points 3: the normal of a
# 3-D voxel of two points (a rank-1 scatter) is any unit vector orthogonal to them, so device and oracle may pick
# different ones; from three points on the scatter has a unique smallest eigenvector.
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("model", [0, 1, 2])
def test_end_to_end_vs_oracle(storage, model):
    from generalized_icp_b200 import compat
    s, t, _ = _pairs(1, n=8000, seed=31)[0]
    leaf = 1.0
    dt = _np_dt(storage)
    s64, t64 = s.astype(dt).astype(np.float64), t.astype(dt).astype(np.float64)
    sm, _, sc, _ = VD.voxel_distributions(s64, [0, len(s64)], leaf, 3)
    tm, _, tc, _ = VD.voxel_distributions(t64, [0, len(t64)], leaf, 3)
    sm, tm = sm.astype(dt).astype(np.float64), tm.astype(dt).astype(np.float64)
    ref = VD.gicp_given_cov(sm, tm, sc, tc, max_iterations=P3["max_iterations"], tolerance=1e-6,
                            max_distance_correspondence=P3["max_distance_correspondence"], covariance_model=model)
    r = compat.gicp_extended(s, t, storage=storage, full_history=False, covariance_model=model, voxel_size=leaf,
                             voxel_distributions=True, voxel_min_points=3, tolerance=1e-6, **P3)
    assert np.array_equal(r["source_points"], sm) and np.array_equal(r["target_points"], tm)
    assert r["n_outer"] == ref["n_outer"], (r["n_outer"], ref["n_outer"])
    dR = r["T"][:3, :3].T @ ref["T"][:3, :3]
    ang = np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))
    assert ang <= 1e-5, ang
    assert np.linalg.norm(r["T"][:3, 3] - ref["T"][:3, 3]) <= 1e-5 * 20.0


def test_every_point_alone_equals_raw_point_to_point():
    """With a leaf so small that every point is alone in its voxel, the voxelized sides are the raw arrays bit for bit
    and have the raw side's search grid: point-to-point registration gives the raw sides' bits."""
    import torch
    s, t, Tg = _pairs(1, n=6000, seed=41)[0]
    S, T = torch.as_tensor(s, device="cuda"), torch.as_tensor(t, device="cuda")
    T0 = (_rot_about(np.full(3, 10.0), 5.0, seed=3) @ Tg)[None]
    for params in (P3, dict(P3, max_distance_nearest_neighbors=2.0)):      # shared and unshared raw plans
        eng = _engine(3, "f32", covariance_model=1, **params)
        eng.set_target(T)
        eng.set_source(S)
        raw = eng.register(T0)
        tm, to = eng.set_target_voxelized(T, voxel_size=1e-4)
        sm, so = eng.set_source_voxelized(S, voxel_size=1e-4)
        assert to[-1] == len(t) and so[-1] == len(s)
        assert torch.equal(tm, T) and torch.equal(sm, S)
        vox = eng.register(T0)
        _same_bits(raw, vox, "every point alone")


# ------------------------------------------------------------------------------------------------
# composition with the other entry points
# ------------------------------------------------------------------------------------------------
def test_composition():
    import torch
    import quality_oracle as QO
    from generalized_icp_b200 import compat
    s, t, Tg = _pairs(1, n=8000, seed=51)[0]
    S, T = torch.as_tensor(s, device="cuda"), torch.as_tensor(t, device="cuda")
    eng = _engine(3, "f32", **P3)
    tm, _ = eng.set_target_voxelized(T, voxel_size=1.0)
    sm, _ = eng.set_source_voxelized(S, voxel_size=1.0)
    r = eng.register()
    torch.cuda.synchronize()
    # a downsample between set-up and register leaves the result unchanged
    eng.voxel_downsample(S, voxel_size=0.3)
    _same_bits(r, eng.register(), "downsample in between")
    # evaluate() over the voxels against the quality oracle at the device's correspondences
    Tf = r.T.cpu().numpy()
    q = eng.evaluate(r.T)
    idx, dist, W = eng.correspond(Tf)
    idx, dist, W = idx.cpu().numpy(), dist.cpu().numpy(), W.cpu().numpy()
    sv, tv = sm.cpu().numpy().astype(np.float64), tm.cpu().numpy().astype(np.float64)
    g = idx >= 0
    pp = sv @ Tf[0, :3, :3].T + Tf[0, :3, 3]
    e = tv[idx[g]] - pp[g]
    row, H, bvec = QO.quality(pp[g], e, W[g], dist[g], len(sv), 3)
    assert int(q.n_inliers[0]) == int(row[0]) == int(g.sum())
    assert float(q.fitness[0]) == row[1]                         # counts voxels: n / number of source voxels
    assert abs(float(q.inlier_rmse[0]) - row[2]) <= 1e-9 * row[2]
    assert abs(float(q.loss[0]) - row[3]) <= 2e-5 * row[3]
    assert np.abs(q.H[0].cpu().numpy() - H).max() <= 2e-5 * np.abs(H).max()
    # gicpSourceCovariancesAt works on a voxelized source
    rc = eng.source_covariances_at(Tf[None]).cpu().numpy()[0]
    cs = eng.covariances(SOURCE).cpu().numpy()
    R = Tf[0, :3, :3]
    assert np.abs(rc - R @ cs @ R.T).max() <= 1e-9 * 100
    # promoting a voxelized target gives the bits of that cloud set up as a voxelized source
    e2 = _engine(3, "f32", **P3)
    e2.set_target_voxelized(S, voxel_size=1.0)
    e2.promote_target_to_source()
    e2.set_target_voxelized(T, voxel_size=1.0)
    _same_bits(r, e2.register(), "promoted")
    assert torch.equal(e2.covariances(SOURCE), eng.covariances(SOURCE))
    # gicp_extended(voxel_distributions=True) equals the engine calls
    c = compat.gicp_extended(s, t, storage="f32", voxel_size=1.0, voxel_distributions=True, full_history=True,
                             evaluate=True, tolerance=1e-6, **P3)
    assert np.array_equal(c["T"], Tf[0]) and c["n_outer"] == int(r.n_outer[0])
    assert np.array_equal(c["src_cov0"], cs) and np.array_equal(c["tgt_cov"], eng.covariances(TARGET).cpu().numpy())
    assert c["n_inliers"] == int(q.n_inliers[0])
    assert len(c["all_src_cov"]) == c["n_outer"] and len(c["hw_src"]) == len(c["all_T"]) - 1
    # the defaults keep today's behaviour: voxel_size alone downsamples and estimates k-NN covariances
    d = compat.gicp_extended(s, t, storage="f32", voxel_size=1.0, full_history=False, tolerance=1e-6, **P3)
    ds, _ = eng.voxel_downsample(S, voxel_size=1.0)
    assert np.array_equal(d["source_points"], ds.cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
def test_refusals_leave_the_sides_alone():
    import ctypes as C
    import torch
    from generalized_icp_b200 import _lib
    s, t, _ = _pairs(1, n=6000, seed=61)[0]
    S, T = torch.as_tensor(s, device="cuda"), torch.as_tensor(t, device="cuda")
    eng = _engine(3, "f32", **P3)
    eng.set_target_voxelized(T, voxel_size=1.0)
    eng.set_source_voxelized(S, voxel_size=1.0)
    want = eng.register()
    far = S.clone()
    far[0] = torch.tensor([-1e6, 0.0, 0.0])
    far[1] = torch.tensor([1e6, 0.0, 0.0])
    # bad voxel sizes, min_points 0, and a cloud spanning more than 2^21 voxels along x (the per-axis limit)
    bad = [(S, 0.0, 1), (S, -1.0, 1), (S, float("nan"), 1), (S, float("inf"), 1), (S, 1.0, 0), (far, 1e-3, 1)]
    for which in (SOURCE, TARGET):
        fn = eng.set_source_voxelized if which == SOURCE else eng.set_target_voxelized
        for pts, leaf, mp in bad:
            with pytest.raises(RuntimeError):
                fn(pts, voxel_size=leaf, min_points=mp)
            _same_bits(want, eng.register(), (which, leaf, mp))
    # a bad `which` through the C entry point
    out = torch.empty_like(S)
    oo = np.zeros(2, dtype=np.int64)
    i64p = C.POINTER(C.c_int64)
    rc = eng.lib.gicpSetVoxelized(eng._h, 2, C.c_void_p(S.data_ptr()), (C.c_int64 * 2)(0, len(s)), 1, 1.0, 1,
                                  C.c_void_p(out.data_ptr()), oo.ctypes.data_as(i64p),
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0 and b"which" in eng.lib.gicpGetLastError()
    _same_bits(want, eng.register(), "bad which")
    # knn() on a voxelized side
    for which in (SOURCE, TARGET):
        with pytest.raises(RuntimeError, match="no k-NN lists"):
            eng.knn(which)
    _same_bits(want, eng.register(), "knn refused")
    assert _lib.load().gicpVersion() == 106


def test_refused_on_a_handle_with_a_communicator():
    """A handle with a communicator (gicpCommInit) takes raw sides only; a one-rank communicator is enough to see the
    refusal.  Skipped where NCCL cannot be loaded."""
    import torch
    from generalized_icp_b200.engine import GicpEngine
    s, _, _ = _pairs(1, n=2000, seed=71)[0]
    eng = _engine(3, "f32", **P3)
    try:
        eng.comm_init(1, 0, GicpEngine.comm_unique_id())
    except RuntimeError as e:
        pytest.skip(f"no NCCL communicator: {e}")
    try:
        for setv in (eng.set_source_voxelized, eng.set_target_voxelized):
            with pytest.raises(RuntimeError, match="communicator"):
                setv(torch.as_tensor(s, device="cuda"), voxel_size=1.0)
    finally:
        eng.comm_destroy()


# ------------------------------------------------------------------------------------------------
# motion recovery on 4x-density config-4 pairs (recorded; only device-versus-oracle agreement is asserted)
# ------------------------------------------------------------------------------------------------
def test_motion_recovery_dense_config4(capsys):
    from generalized_icp_b200 import compat, synthetic
    from robust_oracle import motion_error
    cfg = dict(synthetic.CONFIG4, n=4 * synthetic.CONFIG4["n"])
    rows = []
    for seed in range(2):
        s, t, Tt = synthetic.patches3d_pair(seed=100 + seed, **cfg)
        r = compat.gicp_extended(s, t, storage="f32", voxel_size=1.0, voxel_distributions=True, voxel_min_points=3,
                                 full_history=False, **synthetic.CONFIG4_PARAMS)
        s64 = s.astype(np.float64)
        t64 = t.astype(np.float64)
        sm, _, sc, _ = VD.voxel_distributions(s64, [0, len(s64)], 1.0, 3)
        tm, _, tc, _ = VD.voxel_distributions(t64, [0, len(t64)], 1.0, 3)
        ref = VD.gicp_given_cov(sm.astype(np.float32).astype(np.float64), tm.astype(np.float32).astype(np.float64),
                                sc, tc, tolerance=synthetic.CONFIG4_PARAMS["tolerance"],
                                max_distance_correspondence=synthetic.CONFIG4_PARAMS["max_distance_correspondence"])
        dev_err, ref_err = motion_error(r["T"], Tt), motion_error(ref["T"], Tt)
        rows.append((seed, len(sm), r["n_outer"], dev_err, ref_err))
        dR = r["T"][:3, :3].T @ ref["T"][:3, :3]
        assert np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)) <= 1e-5
        assert np.linalg.norm(r["T"][:3, 3] - ref["T"][:3, 3]) <= 1e-5 * 40.0
    with capsys.disabled():
        for row in rows:
            print(f"\n[voxel distributions, 4x-density config 4] seed {row[0]}: {row[1]} source voxels, "
                  f"{row[2]} iterations, device (rot rad, trans m) {row[3]}, oracle {row[4]}")
