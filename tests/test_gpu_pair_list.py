"""Pair lists (gicpSetPairList, include/gicp_b200.h) on the device.  The reference throughout is the one-to-one batch
built by concatenating each pair's clouds and set up with gicpSetSource + gicpSetTarget: a pair list must reproduce it
bit for bit (T, n_outer, converged_at, loss_hist, T_hist, inliers and every stage entry point's rows), with the
sources taken from the source set or from the target set itself.  Every set-up here has the same cells per cloud
(max_cells_per_cloud, or clouds of one size), the condition of the bitwise contract."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SOURCE, TARGET = 0, 1
BUDGET = 1 << 16
P = {2: dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0, max_iterations=30,
             max_cells_per_cloud=BUDGET),
     3: dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=2.0, max_iterations=30,
             max_cells_per_cloud=BUDGET)}
FUSED_SIZES = [0, 1, 128, 129, 700, 2048]
MULTI_SIZES = [0, 1, 129, 2048, 3000, 1500]


def _clouds(dim, sizes, seed):
    """Clouds of one scene under small random motions: 3-D planar patches, 2-D line segments."""
    rng = np.random.default_rng(seed)
    if dim == 3:
        from generalized_icp_b200 import synthetic
        cl, _ = synthetic.patches3d_sequence(len(sizes), n=max(max(sizes), 1), cube=20.0, patch=12.0, max_rot_deg=1.0,
                                             max_trans=0.3, seed=seed)
        return [c[:n].astype(np.float64) for c, n in zip(cl, sizes)]
    segs = rng.uniform(0, 30, size=(12, 4))
    out = []
    for n in sizes:
        s = segs[rng.integers(0, len(segs), size=n)]
        u = rng.uniform(0, 1, size=(n, 1))
        p = s[:, :2] + u * (s[:, 2:] - s[:, :2]) + rng.normal(0, 0.02, size=(n, 2))
        th = rng.uniform(-0.02, 0.02)
        R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        out.append(p @ R.T + rng.uniform(-0.2, 0.2, size=2))
    return out


def _cat(eng, clouds):
    dt = np.float32 if eng.storage == "f32" else np.float64
    arr = np.concatenate([np.asarray(c, dtype=dt).reshape(-1, eng.dim) for c in clouds], axis=0)
    off = np.zeros(len(clouds) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    return torch.as_tensor(arr, device=eng.device), off


def _engine(dim, storage, robust=None, **prm):
    from generalized_icp_b200.engine import GicpEngine
    eng = GicpEngine(dim, storage)
    eng.set_params(**{**P[dim], **prm})
    if robust:
        eng.set_robust_kernel(*robust[0], **robust[1])
    return eng


def _bits(x):
    a = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return np.ascontiguousarray(a).view(np.uint8)


def _same(a, b, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(_bits(a), _bits(b)), what


def _same_result(r, q):
    for f in ("T", "n_outer", "converged_at", "loss_hist", "T_hist", "inliers"):
        _same(getattr(r, f), getattr(q, f), f)


def _T0(dim, n, seed):
    rng = np.random.default_rng(seed)
    T = np.tile(np.eye(dim + 1), (n, 1, 1))
    for p in range(n):
        th = rng.uniform(-0.02, 0.02)
        if dim == 2:
            T[p, :2, :2] = [[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]
        else:
            from generalized_icp_b200.synthetic import _rand_rotation
            T[p, :3, :3] = _rand_rotation(rng, 1.0)
        T[p, :dim, dim] = rng.uniform(-0.1, 0.1, size=dim)
    return T


def _pair_list(n, long, seed):
    """Self-pairs, repeats, (i, j) with (j, i); >= 64 pairs (the active list) when `long`."""
    rng = np.random.default_rng(seed)
    pairs = [(i, i) for i in range(n)] + [(0, 1), (1, 0), (2, n - 1), (n - 1, 2), (3, 4), (3, 4)]
    while long and len(pairs) < 70:
        pairs.append(tuple(int(v) for v in rng.integers(0, n, size=2)))
    return np.array(pairs)


def _setup_list(eng, src_set, tgt_set, pairs, source_set, vox=None):
    """The pair list's handle.  vox: (leaf, which sides are voxelized)."""
    sides = [(TARGET, tgt_set)] + ([(SOURCE, src_set)] if source_set == SOURCE else [])
    for which, cl in sides:
        pts, off = _cat(eng, cl)
        if vox and which in vox[1]:
            (eng.set_target_voxelized if which == TARGET else eng.set_source_voxelized)(pts, off, voxel_size=vox[0])
        else:
            (eng.set_target if which == TARGET else eng.set_source)(pts, off)
    return eng.set_pair_list(pairs[:, 0], pairs[:, 1], source_set)


def _setup_ref(eng, src_set, tgt_set, pairs, vox=None, src_vox=None):
    """The one-to-one batch of the same pairs: every pair's clouds concatenated, set up as target and source."""
    for which, cl in ((TARGET, [tgt_set[j] for j in pairs[:, 1]]), (SOURCE, [src_set[i] for i in pairs[:, 0]])):
        pts, off = _cat(eng, cl)
        if vox and ((which == TARGET and TARGET in vox[1]) or (which == SOURCE and src_vox)):
            (eng.set_target_voxelized if which == TARGET else eng.set_source_voxelized)(pts, off, voxel_size=vox[0])
        else:
            (eng.set_target if which == TARGET else eng.set_source)(pts, off)
    return eng


def _compare(dim, storage, src_set, tgt_set, pairs, source_set, T0=None, robust=None, vox=None, **prm):
    a = _engine(dim, storage, robust, **prm)
    off = _setup_list(a, src_set, tgt_set, pairs, source_set, vox)
    src_vox = vox is not None and (SOURCE in vox[1] if source_set == SOURCE else TARGET in vox[1])
    b = _setup_ref(_engine(dim, storage, robust, **prm), src_set, tgt_set, pairs, vox, src_vox)
    if not vox:
        assert off.tolist() == [0] + np.cumsum([len(src_set[i]) for i in pairs[:, 0]]).tolist()
    r, q = a.register(T0), b.register(T0)
    _same_result(r, q)
    torch.cuda.synchronize()
    return a, b, r


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
@pytest.mark.parametrize("sizes", ["fused", "multi"])
def test_register_bitwise(dim, storage, source_set, sizes):
    sz = FUSED_SIZES if sizes == "fused" else MULTI_SIZES
    tgt_set = _clouds(dim, sz, 1)
    src_set = _clouds(dim, sz[::-1], 2) if source_set == SOURCE else tgt_set
    for long in (False, True):
        pairs = _pair_list(len(sz), long, 3)
        for T0 in (None, _T0(dim, len(pairs), 4)):
            _, _, r = _compare(dim, storage, src_set, tgt_set, pairs, source_set, T0)
    assert int(r.n_outer.max()) > 1


@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
def test_register_large_acc_ppt(source_set):
    """80 pairs of 32768-point config-4 clouds: 2.6 M pair-source points, acc_ppt 17 (automatic budget, one size)."""
    from generalized_icp_b200 import synthetic
    cl, _ = synthetic.patches3d_sequence(8, seed=5)
    rng = np.random.default_rng(6)
    pairs = np.array([(k % 8, (k + 1 + k // 8) % 8) for k in range(80)])
    src_set = cl if source_set == TARGET else [c[rng.permutation(len(c))] for c in cl]
    prm = dict(synthetic.CONFIG4_PARAMS, max_cells_per_cloud=0, max_iterations=30)
    _compare(3, "f32", src_set, cl, pairs, source_set, **prm)


ROBUST = {"huber": (("huber", 0.5), {}), "tukey_adaptive": (("tukey",), dict(adaptive=3.0, min_scale=0.1))}


@pytest.mark.parametrize("robust", list(ROBUST))
@pytest.mark.parametrize("sizes", ["fused", "multi"])
@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
def test_robust_bitwise(robust, sizes, source_set):
    sz = FUSED_SIZES if sizes == "fused" else MULTI_SIZES
    tgt_set = _clouds(3, sz, 7)
    src_set = _clouds(3, sz, 8) if source_set == SOURCE else tgt_set
    _compare(3, "f64", src_set, tgt_set, _pair_list(len(sz), True, 9), source_set, robust=ROBUST[robust])


@pytest.mark.parametrize("model", [1, 2])
@pytest.mark.parametrize("sizes", ["fused", "multi"])
@pytest.mark.parametrize("dim", [2, 3])
def test_covariance_models_from_target_set(model, sizes, dim):
    """covariance_model 1 / 2 with the sources taken from a target set: C_src = 0, as a source set-up gives it."""
    sz = FUSED_SIZES if sizes == "fused" else MULTI_SIZES
    cl = _clouds(dim, sz, 10)
    a, b, _ = _compare(dim, "f32", cl, cl, _pair_list(len(sz), False, 11), TARGET, covariance_model=model)
    T = _T0(dim, 12, 12)[: a._loop_n()[1]]
    _same(a.source_covariances_at(T[None]), b.source_covariances_at(T[None]), "rotated source covariances")
    assert float(a.source_covariances_at(T[None]).abs().max()) == 0.0


@pytest.mark.parametrize("vox_sides,source_set", [((SOURCE,), SOURCE), ((TARGET,), SOURCE), ((SOURCE, TARGET), SOURCE),
                                                   ((TARGET,), TARGET)])
def test_voxelized_sets(vox_sides, source_set):
    tgt_set = _clouds(3, [900, 1500, 3000, 2000, 1], 13)
    src_set = _clouds(3, [2500, 700, 1200, 3000, 400], 14) if source_set == SOURCE else tgt_set
    _compare(3, "f32", src_set, tgt_set, _pair_list(5, True, 15), source_set, vox=(0.5, vox_sides))


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("sizes", ["fused", "multi"])
@pytest.mark.parametrize("source_set", [SOURCE, TARGET])
def test_stage_entry_points(storage, sizes, source_set):
    """gicpCorrespond, gicpNormalEquations, gicpRobustScales, gicpEvaluate (stream-ordered straight after gicpRegister)
    and gicpSourceCovariancesAt, row for row in the pair layout."""
    sz = FUSED_SIZES if sizes == "fused" else MULTI_SIZES
    tgt_set = _clouds(3, sz, 16)
    src_set = _clouds(3, sz, 17) if source_set == SOURCE else tgt_set
    pairs = _pair_list(len(sz), False, 18)
    robust = ROBUST["tukey_adaptive"]
    a = _engine(3, storage, robust)
    off = _setup_list(a, src_set, tgt_set, pairs, source_set)
    b = _setup_ref(_engine(3, storage, robust), src_set, tgt_set, pairs)
    ra, rb = a.register(history=False), b.register(history=False)
    qa, qb = a.evaluate(ra.T), b.evaluate(rb.T)           # stream-ordered, no synchronisation in between
    for f in ("n_inliers", "fitness", "inlier_rmse", "loss", "H", "b"):
        _same(getattr(qa, f), getattr(qb, f), f)
    T = _T0(3, len(pairs), 19)
    for x, y, what in zip(a.correspond(T), b.correspond(T), ("idx", "dist", "W")):
        _same(x, y, what)
    assert a.correspond(T)[0].shape[0] == off[-1]
    _same(a.normal_equations(T), b.normal_equations(T), "normal equations")
    _same(a.robust_scales(T), b.robust_scales(T), "robust scales")
    Ts = np.stack([T, _T0(3, len(pairs), 20)])
    _same(a.source_covariances_at(Ts), b.source_covariances_at(Ts), "source covariances at")
    # the stage rows of pair p are its source cloud's, in input order
    idx = a.correspond(T)[0].cpu().numpy()
    for p in range(len(pairs)):
        assert off[p + 1] - off[p] == len(src_set[pairs[p, 0]])
    assert len(idx) == off[-1]


def _raw_register_error(e, n_pairs):
    """gicpRegister straight through the library with outputs for n_pairs pairs (the list the handle had): its error
    message, or None when it ran.  Checks the library's own state, not the engine's bookkeeping."""
    import ctypes as C
    d1 = e.dim + 1
    T = torch.empty((n_pairs, d1, d1), dtype=torch.float64, device=e.device)
    n = torch.empty((2, n_pairs), dtype=torch.int32, device=e.device)
    rc = e.lib.gicpRegister(e._h, None, C.c_void_p(T.data_ptr()), C.c_void_p(n[0].data_ptr()),
                            C.c_void_p(n[1].data_ptr()), None, None, None, e._stream())
    torch.cuda.synchronize()
    return e.lib.gicpGetLastError().decode() if rc else None


def _fresh_one_to_one(dim, storage, src_set, tgt_set):
    e = _engine(dim, storage)
    e.set_target(*_cat(e, tgt_set))
    e.set_source(*_cat(e, src_set))
    return e.register()


def test_lifecycle_and_refusals():
    dim, storage = 3, "f64"
    tgt_set = _clouds(dim, [300, 900, 129, 2000], 21)
    src_set = _clouds(dim, [700, 128, 1000, 50], 22)
    pairs = np.array([(0, 1), (1, 0), (2, 2), (3, 1), (0, 1)])

    def with_list(source_set=SOURCE):
        e = _engine(dim, storage)
        _setup_list(e, src_set, tgt_set, pairs, source_set)
        return e

    ref_list = {s: with_list(s).register() for s in (SOURCE, TARGET)}
    fresh = _fresh_one_to_one(dim, storage, src_set, tgt_set)

    # every discarding call returns the handle to one-to-one, with a fresh handle's results
    def discard_by(name):
        e = with_list()
        if name == "set_source":
            e.set_source(*_cat(e, src_set))
        elif name == "set_target":
            e.set_target(*_cat(e, tgt_set))
        elif name == "set_pair":
            t, toff = _cat(e, tgt_set)
            s, soff = _cat(e, src_set)
            e.set_pair(t, s, toff, soff)
        elif name == "set_params":
            e.set_params(**P[dim])
            assert "set source and target first" in _raw_register_error(e, len(pairs))   # the library's list is gone
            e.set_target(*_cat(e, tgt_set))
            e.set_source(*_cat(e, src_set))
        elif name == "promote":
            e.set_target(*_cat(e, src_set))          # promoted below to the source
            e.set_pair_list([0], [0], SOURCE)
            e.promote_target_to_source()
            assert "set source and target first" in _raw_register_error(e, 1)   # no target, no list
            e.set_target(*_cat(e, tgt_set))
        return e

    for name in ("set_source", "set_target", "set_pair", "set_params", "promote"):
        e = discard_by(name)
        assert e._pairs is None
        _same_result(e.register(), fresh)
    # a voxelized side set up on a handle with a list
    e = with_list()
    e.set_source_voxelized(*_cat(e, src_set), voxel_size=0.5)
    f = _engine(dim, storage)
    f.set_target(*_cat(f, tgt_set))
    f.set_source_voxelized(*_cat(f, src_set), voxel_size=0.5)
    _same_result(e.register(), f.register())
    e = with_list()
    e.set_target_voxelized(*_cat(e, tgt_set), voxel_size=0.5)
    f = _engine(dim, storage)
    f.set_source(*_cat(f, src_set))
    f.set_target_voxelized(*_cat(f, tgt_set), voxel_size=0.5)
    _same_result(e.register(), f.register())
    # robust kernels keep the list
    e = with_list()
    e.set_robust_kernel("huber", 1e30)
    e.set_robust_kernel(None)
    _same_result(e.register(), ref_list[SOURCE])

    # every refusal leaves the previous list registering as before
    e = with_list()
    refusals = [
        ("n_pairs", lambda: e.set_pair_list([], [], SOURCE)),
        ("n_pairs", lambda: e.set_pair_list(np.zeros(65536, np.int64), np.zeros(65536, np.int64), SOURCE)),
        ("out of range", lambda: e.set_pair_list([4], [0], SOURCE)),
        ("out of range", lambda: e.set_pair_list([0], [4], TARGET)),
        ("out of range", lambda: e.set_pair_list([-1], [0], SOURCE)),
        ("source_set", lambda: e.set_pair_list([0], [0], 2)),
    ]
    for msg, call in refusals:
        with pytest.raises(RuntimeError, match=msg):
            call()
        _same_result(e.register(), ref_list[SOURCE])
    # a list over a set that is not set up
    g = _engine(dim, storage)
    g.set_target(*_cat(g, tgt_set))
    with pytest.raises(RuntimeError, match="set source and target first"):
        g.set_pair_list([0], [0], SOURCE)
    with pytest.raises(RuntimeError, match="set the target first"):
        _engine(dim, storage).set_pair_list([0], [0], TARGET)
    # a later list replaces the earlier one; a TARGET list needs no source set
    g.set_pair_list(pairs[:, 0], pairs[:, 1], TARGET)
    _same_result(g.register(), ref_list[TARGET])


def test_communicator_refuses():
    from generalized_icp_b200.engine import GicpEngine
    try:
        uid = GicpEngine.comm_unique_id()
    except RuntimeError as e:
        pytest.skip(f"no NCCL: {e}")
    cl = _clouds(3, [300, 400], 23)
    e = _engine(3, "f32")
    e.set_target(*_cat(e, cl))
    e.set_pair_list([0, 1], [1, 0], TARGET)
    e.comm_init(1, 0, uid)
    assert e._pairs is None
    try:
        assert "set source and target first" in _raw_register_error(e, 2)   # the library's list is gone
        e.set_target(*_cat(e, cl))
        e.set_source(*_cat(e, cl))
        with pytest.raises(RuntimeError, match="communicator"):
            e.set_pair_list([0, 1], [1, 0], TARGET)
    finally:
        e.comm_destroy()


def test_register_pairs_compat():
    """compat.register_pairs over a short sequence: every pair against the one-to-one batch, and near the truth."""
    from generalized_icp_b200 import compat, synthetic
    cl, poses = synthetic.patches3d_sequence(6, n=8192, seed=24)
    pairs = [(k, k + d) for d in (1, 2, 3) for k in range(6 - d)]
    prm = dict(synthetic.CONFIG4_PARAMS, max_iterations=50)
    out = compat.register_pairs(cl, pairs, storage="f32", **prm)
    b = _engine(3, "f32", max_cells_per_cloud=0, **prm)
    pr = np.array(pairs)
    _setup_ref(b, cl, cl, pr)
    rb = b.register(history=False)
    _same(out["T"], rb.T, "T")
    _same(out["n_outer"], rb.n_outer, "n_outer")
    qb = b.evaluate(rb.T)
    _same(out["information"], qb.H, "information")
    err = [np.abs(out["T"][p][:3, 3] - synthetic.relative_pose(poses, i, j)[:3, 3]).max()
           for p, (i, j) in enumerate(pairs)]
    assert np.median(err) < 0.05, err
    assert np.median(out["fitness"]) > 0.5


def test_k2_path_crossing_scan_odometry():
    """The second set-up choice of the bitwise contract: 100 2-D scans of 360 points (36000 points, K2's latency path),
    each against the next three (294 pairs), float64.  The list is bitwise equal to the one-to-one batch registered
    in two halves of 147 pairs (52920 points per side: the latency path too), and within the loop's tolerance of the
    same batch registered whole (105840 points per side: knn_hist_kernel, whose covariances round differently)."""
    dim, storage = 2, "f64"
    prm = dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0, max_iterations=50,
               max_cells_per_cloud=0)
    cl = _clouds(dim, [360] * 100, 25)
    pairs = np.array([(k, k + d) for d in (1, 2, 3) for k in range(100 - d)])
    a = _engine(dim, storage, **prm)
    _setup_list(a, cl, cl, pairs, TARGET)
    r = a.register()
    halves = []
    for part in (pairs[:147], pairs[147:]):
        b = _setup_ref(_engine(dim, storage, **prm), cl, cl, part)
        halves.append(b.register())
    for f in ("T", "n_outer", "converged_at", "loss_hist", "T_hist", "inliers"):
        _same(getattr(r, f), torch.cat([getattr(h, f) for h in halves]), f)
    w = _setup_ref(_engine(dim, storage, **prm), cl, cl, pairs)
    rw = w.register()
    # the whole batch's covariances: the same neighbours, another rounding
    cov_list = a.covariances(TARGET).cpu().numpy().reshape(100, 360, 2, 2)[pairs[:, 1]]
    cov_whole = w.covariances(TARGET).cpu().numpy().reshape(len(pairs), 360, 2, 2)
    rel = np.abs(cov_list - cov_whole).max() / np.abs(cov_list).max()
    dT = np.abs(r.T.cpu().numpy() - rw.T.cpu().numpy()).max(axis=(1, 2))
    same_it = (r.n_outer == rw.n_outer).cpu().numpy()
    print(f"covariance entries that differ: {int((cov_list != cov_whole).sum())} of {cov_list.size}, "
          f"max relative difference {rel:.3g}; pairs with equal n_outer {int(same_it.sum())} of {len(pairs)}; "
          f"max |dT| {dT.max():.3g} (equal n_outer: {dT[same_it].max() if same_it.any() else 0:.3g})")
    assert (cov_list != cov_whole).any()          # the two set-ups really took different K2 estimators
    assert rel < 1e-12
    assert same_it.mean() >= 0.95
    assert dT[same_it].max() < 1e-9
    assert dT.max() < 1e-4
