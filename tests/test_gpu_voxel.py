"""Voxel-grid downsampling on the device (gicpVoxelDownsample / GicpEngine.voxel_downsample) against the float64
oracle (tests/voxel_oracle.py): exact offsets, order, voxel_of and counts; centroids to 1e-12 relative
(f64) or one f32 ulp of the oracle's rounded value (f32).  Then the properties a registration pipeline relies on:
batch = clouds one at a time, both sort paths, identity at a tiny leaf, reproducibility, no interference with a
handle's registered sides, and the 4x-density bench pairs downsampled and registered without leaving the device."""
import numpy as np
import pytest

import voxel_oracle as VO
from oracle import gicp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engines():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from generalized_icp_b200.engine import GicpEngine
    cache = {}

    def get(dim, storage):
        if (dim, storage) not in cache:
            cache[(dim, storage)] = GicpEngine(dim, storage)
        return cache[(dim, storage)]

    return get


def _np_dtype(storage):
    return np.float32 if storage == "f32" else np.float64


def _gpu(eng, pts, off, leaf, min_points=1):
    out, oo, vox, cnt = eng.voxel_downsample(np.ascontiguousarray(pts), off, voxel_size=leaf, min_points=min_points,
                                             with_index=True)
    return out.cpu().numpy(), oo, vox.cpu().numpy(), cnt.cpu().numpy()


def _assert_matches_oracle(got, pts, off, leaf, min_points=1):
    out, oo, vox, cnt = got
    ref, roo, rvox, rcnt = VO.voxel_downsample(pts, off, leaf, min_points)
    assert np.array_equal(oo, roo)
    assert np.array_equal(vox, rvox)
    assert np.array_equal(cnt, rcnt)
    assert out.shape == ref.shape
    if out.dtype == np.float64:
        rel = np.abs(out - ref) / (np.abs(ref) + leaf)
        assert rel.size == 0 or float(rel.max()) <= 1e-12, float(rel.max())
    else:
        r32 = ref.astype(np.float32)
        diff = np.abs(out.astype(np.float64) - r32.astype(np.float64))
        assert np.all(diff <= np.spacing(np.abs(r32)).astype(np.float64))
    return ref


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _clouds(dim, seed):
    """A planar-patch cloud (30 m patches) and a uniform cloud, as one batch of two."""
    from generalized_icp_b200 import synthetic
    s, _, _ = synthetic.patches3d_pair(n=20000, n_patches=8, cube=30.0, patch=20.0, seed=seed)
    rng = np.random.default_rng(seed)
    u = rng.uniform(-15.0, 15.0, size=(15000, dim))
    pts = np.concatenate([s[:, :dim].astype(np.float64), u])
    return pts, np.array([0, 20000, 35000])


def _leaf_for(pts, off, per_voxel):
    """A leaf whose voxels hold about `per_voxel` points (bisection on the oracle's mean count)."""
    lo, hi = 1e-3, 50.0
    for _ in range(25):
        mid = (lo * hi) ** 0.5
        _, _, _, cnt = VO.voxel_downsample(pts, off, mid)
        if cnt.mean() < per_voxel:
            lo = mid
        else:
            hi = mid
    return float(f"{hi:.3g}")


# 1. ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("per_voxel", [1, 5, 100])
def test_against_oracle(engines, dim, storage, per_voxel):
    pts, off = _clouds(dim, seed=dim)
    pts = pts.astype(_np_dtype(storage))
    leaf = _leaf_for(pts, off, per_voxel) if per_voxel > 1 else 1e-4
    eng = engines(dim, storage)
    for mp in (1, 3):
        _assert_matches_oracle(_gpu(eng, pts, off, leaf, mp), pts, off, leaf, mp)


# 2. ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_lattices_on_voxel_faces(engines, dim, storage):
    eng = engines(dim, storage)
    rng = np.random.default_rng(7 + dim)
    dyadic = (rng.integers(-64, 65, size=(6000, dim)) / 8.0).astype(_np_dtype(storage))   # faces of every leaf below
    for leaf in (0.5, 1.0, 2.0, 0.1, 0.125):
        _assert_matches_oracle(_gpu(eng, dyadic, None, leaf), dyadic, [0, len(dyadic)], leaf)
    # L = 0.1 on multiples of 0.1 (neither is representable): floor of the IEEE quotient, not of a product
    tenths = (rng.integers(-300, 301, size=(6000, dim)) / 10.0).astype(_np_dtype(storage))
    _assert_matches_oracle(_gpu(eng, tenths, None, 0.1), tenths, [0, len(tenths)], 0.1)
    # far from the origin
    for far in (1e4, 1e5):
        p = (far + rng.uniform(0.0, 30.0, size=(8000, dim))).astype(_np_dtype(storage))
        p[:4000] *= -1.0                                  # a cloud on each side of the origin
        off = [0, 4000, 8000]
        _assert_matches_oracle(_gpu(eng, p, off, 0.05), p, off, 0.05)


@pytest.mark.parametrize("dim", [2, 3])
def test_per_axis_limit(engines, dim):
    import torch
    eng = engines(dim, "f64")
    bits = 21 if dim == 3 else 31
    rng = np.random.default_rng(11)
    for axis in range(dim):
        inside = rng.uniform(0.0, 2.0 ** bits - 1, size=(3000, dim))
        inside[0] = 0.0
        inside[1, axis] = 2.0 ** bits - 0.5                # floor(hi) - floor(lo) = 2^bits - 1
        _assert_matches_oracle(_gpu(eng, inside, None, 1.0), inside, [0, len(inside)], 1.0)
        outside = inside.copy()
        outside[1, axis] = 2.0 ** bits
        small = rng.uniform(0, 1, size=(10, dim))
        with pytest.raises(RuntimeError, match=rf"cloud 1 .* axis {'xyz'[axis]}, the limit is 2\^{bits}"):
            eng.voxel_downsample(np.concatenate([small, outside]), [0, 10, 10 + len(outside)], voxel_size=1.0)
        with pytest.raises(ValueError):
            VO.voxel_downsample(outside, [0, len(outside)], 1.0)
    with pytest.raises(RuntimeError, match="outside int64"):
        eng.voxel_downsample(np.full((4, dim), 1e300), voxel_size=1e-10)
    # the handle is still usable
    _assert_matches_oracle(_gpu(eng, inside, None, 1.0), inside, [0, len(inside)], 1.0)
    for bad in (dict(voxel_size=0.0), dict(voxel_size=float("nan")), dict(voxel_size=-1.0),
                dict(voxel_size=1.0, min_points=0)):
        with pytest.raises(RuntimeError):
            eng.voxel_downsample(inside, **bad)
    t = torch.as_tensor(inside, device=eng.device)
    import ctypes as C
    from generalized_icp_b200 import _lib
    oo = np.zeros(2, dtype=np.int64)
    rc = eng.lib.gicpVoxelDownsample(eng._h, C.c_void_p(t.data_ptr()), np.array([0, len(inside)], dtype=np.int64)
                                     .ctypes.data_as(C.POINTER(C.c_int64)), 1, 1.0, 1, C.c_void_p(t.data_ptr()),
                                     oo.ctypes.data_as(C.POINTER(C.c_int64)), None, None, eng._stream())
    assert rc != 0 and b"alias" in _lib.load().gicpGetLastError()


# 3. ----------------------------------------------------------------------------------------------------------------
def _mixed_batch(n_clouds, wide, seed=3):
    rng = np.random.default_rng(seed)
    parts = []
    for i in range(n_clouds):
        kind = i % 9
        if kind == 0:
            p = np.zeros((0, 3))
        elif kind == 1:
            p = rng.uniform(-5, 5, size=(1, 3))
        elif kind == 2:
            p = rng.uniform(0.01, 0.99, size=(int(rng.integers(40, 3000)), 3)) + rng.integers(-3, 3, size=3)  # one voxel
        elif kind == 3:
            p = np.full((int(rng.integers(1, 50)), 3), np.nan)
        else:
            p = rng.uniform(-5, 5, size=(int(rng.integers(2, 600)), 3))
            p[rng.random(len(p)) < 0.02, int(rng.integers(0, 3))] = np.inf
        parts.append(p)
    if wide:   # 2^21 - 1 voxels along every axis: 63 coordinate bits, so the batch sorts as segments
        w = rng.uniform(0, 2.0 ** 21 - 1, size=(2000, 3))
        w[0], w[1] = 0.0, 2.0 ** 21 - 0.5
        w[2:200] = w[2] + rng.uniform(0, 0.9, size=(198, 3))
        parts[len(parts) // 2] = w
    off = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)
    return np.concatenate(parts), off


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("wide", [False, True], ids=["radix", "segmented"])
def test_batch_equals_clouds_one_at_a_time(engines, storage, wide):
    eng = engines(3, storage)
    pts, off = _mixed_batch(1152, wide)
    pts = pts.astype(_np_dtype(storage))
    for mp in (1, 3):
        got = _gpu(eng, pts, off, 1.0, mp)
        _assert_matches_oracle(got, pts, off, 1.0, mp)
        out, oo, vox, cnt = got
        for c in range(len(off) - 1):
            one = _gpu(eng, pts[off[c]:off[c + 1]], None, 1.0, mp)
            assert _same_bits(one[0], out[oo[c]:oo[c + 1]])
            assert one[1][1] == oo[c + 1] - oo[c]
            assert np.array_equal(one[2], vox[off[c]:off[c + 1]])
            assert np.array_equal(one[3], cnt[oo[c]:oo[c + 1]])


# 4. ----------------------------------------------------------------------------------------------------------------
def test_tiny_leaf_is_the_identity_and_registers_identically(engines):
    import torch
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    src, tgt, off, _ = synthetic.patches3d_batch_device(8, n=8192, seed=2, device="cuda", **cfg)
    off = off.cpu().numpy()
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    leaf = 4e-5                                           # 40 m / 4e-5 = 1e6 voxels per axis, below 2^21
    ds, oo = eng.voxel_downsample(src, off, voxel_size=leaf)
    dt, _ = eng.voxel_downsample(tgt, off, voxel_size=leaf)
    assert np.array_equal(oo, off)
    assert torch.equal(ds.view(torch.int32), src.view(torch.int32))
    assert torch.equal(dt.view(torch.int32), tgt.view(torch.int32))
    eng.set_pair(tgt, src, off, off)
    raw = eng.register()
    eng.set_pair(dt, ds, off, off)
    again = eng.register()
    for a, b in ((raw.T, again.T), (raw.n_outer, again.n_outer), (raw.loss_hist, again.loss_hist),
                 (raw.T_hist, again.T_hist), (raw.inliers, again.inliers)):
        assert torch.equal(a.nan_to_num(), b.nan_to_num()) if a.is_floating_point() else torch.equal(a, b)
    # f64 with NaN rows: the output is the finite rows
    eng64 = engines(2, "f64")
    p = np.random.default_rng(4).uniform(-20, 20, size=(5000, 2))
    p[::97, 1] = np.nan
    out, oo, vox, cnt = _gpu(eng64, p, None, 1e-7)
    fin = np.isfinite(p).all(axis=1)
    assert _same_bits(out, p[fin]) and np.all(cnt == 1) and np.all(vox[~fin] == -1)


# 5. ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_reproducible_and_permutation_invariant(engines, storage):
    eng = engines(3, storage)
    pts, off = _clouds(3, seed=9)
    pts = pts.astype(_np_dtype(storage))
    a = _gpu(eng, pts, off, 0.7, 2)
    b = _gpu(eng, pts, off, 0.7, 2)
    assert all(_same_bits(x, y) for x, y in zip(a, b))
    rng = np.random.default_rng(1)
    perm = np.concatenate([off[c] + rng.permutation(off[c + 1] - off[c]) for c in range(len(off) - 1)])
    c = _gpu(eng, pts[perm], off, 0.7, 2)
    assert np.array_equal(a[1], c[1])
    # row r of the input sits at position inv[r] of the permuted input
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm))
    cloud = np.repeat(np.arange(len(off) - 1), np.diff(off))
    va, vc = a[2], c[2][inv]
    assert np.array_equal(va < 0, vc < 0)
    k = va >= 0
    ra, rc = a[1][cloud[k]] + va[k], c[1][cloud[k]] + vc[k]
    assert np.array_equal(a[3][ra], c[3][rc])
    ca, cc = a[0][ra].astype(np.float64), c[0][rc].astype(np.float64)
    tol = 1e-12 if storage == "f64" else 0.0
    if storage == "f64":
        assert float((np.abs(ca - cc) / (np.abs(ca) + 0.7)).max()) <= tol
    else:   # fp64 sums of a permutation round to f32 within one ulp
        assert np.all(np.abs(ca - cc) <= np.spacing(np.abs(a[0][ra])).astype(np.float64))


# 6. ----------------------------------------------------------------------------------------------------------------
def test_no_interference_with_registered_sides():
    import torch
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    src, tgt, off, _ = synthetic.patches3d_batch_device(16, n=32768, seed=6, device="cuda", **cfg)
    off = off.cpu().numpy()
    ref_eng = GicpEngine(3, "f32")
    ref_eng.set_params(**synthetic.CONFIG4_PARAMS)
    ref_eng.set_pair(tgt, src, off, off)
    ref = ref_eng.register()
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    eng.set_pair(tgt, src, off, off)
    eng.voxel_downsample(torch.cat([tgt, src]), np.concatenate([off, off[1:] + off[-1]]), voxel_size=0.3, min_points=2)
    got = eng.register()
    assert torch.equal(got.T, ref.T) and torch.equal(got.n_outer, ref.n_outer)
    assert torch.equal(got.T_hist.nan_to_num(), ref.T_hist.nan_to_num())
    # a downsampled tensor registered as a side survives later downsample calls
    ds, so = eng.voxel_downsample(src, off, voxel_size=0.5)
    dt, to = eng.voxel_downsample(tgt, off, voxel_size=0.5)
    keep_s, keep_t = ds.clone(), dt.clone()
    eng.set_pair(dt, ds, to, so)
    eng.voxel_downsample(src.flip(0).contiguous(), off, voxel_size=0.25)
    eng.voxel_downsample(tgt, off, voxel_size=2.0)
    r1 = eng.register()
    assert torch.equal(ds, keep_s) and torch.equal(dt, keep_t)
    ref_eng.set_pair(keep_t, keep_s, to, so)
    r2 = ref_eng.register()
    assert torch.equal(r1.T, r2.T) and torch.equal(r1.n_outer, r2.n_outer)


# 7. ----------------------------------------------------------------------------------------------------------------
def _angle(Ta, Tb):
    dR = Ta[:3, :3].T @ Tb[:3, :3]
    return float(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)))


def test_dense_pairs_downsampled_and_registered_on_device():
    """64 config-4 pairs at 4x density (131072 points per side) -> 1 m voxels on the device -> registration."""
    import torch
    from generalized_icp_b200 import synthetic
    from generalized_icp_b200.engine import GicpEngine
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    src, tgt, off, T_true = synthetic.patches3d_batch_device(64, n=4 * 32768, seed=8, device="cuda", **cfg)
    off = off.cpu().numpy()
    eng = GicpEngine(3, "f32")
    eng.set_params(**synthetic.CONFIG4_PARAMS)
    ds, soff = eng.voxel_downsample(src, off, voxel_size=1.0)
    dt, toff = eng.voxel_downsample(tgt, off, voxel_size=1.0)
    per_cloud = np.diff(np.concatenate([soff, toff[1:] + soff[-1]]))
    # sixteen 30 m x 30 m patches in 1 m voxels (a tilted plane crosses more voxels than its area in m^2)
    print(f"downsampled points per cloud: min {per_cloud.min()} median {np.median(per_cloud):.0f} max {per_cloud.max()}")
    assert 13000 <= per_cloud.min() and per_cloud.max() <= 18000     # measured on a B200: 14655 to 16535
    eng.set_pair(dt, ds, toff, soff)
    res = eng.register()
    torch.cuda.synchronize()
    assert bool((res.converged_at >= 0).all())
    T = res.T.cpu().numpy()
    Tt = T_true.cpu().numpy()
    ang = np.array([_angle(T[p], Tt[p]) for p in range(64)])
    terr = np.linalg.norm(T[:, :3, 3] - Tt[:, :3, 3], axis=1)
    print(f"vs generating motion: rotation max {ang.max():.2e} median {np.median(ang):.2e} rad, "
          f"translation max {terr.max():.2e} median {np.median(terr):.2e} m")
    # DESIGN section 7: the centroids sample each surface at other places than the raw points (a lattice fixed in
    # space, not moving with the surface), so the recovery is coarser than on the raw clouds (measured on a B200:
    # max 3.4e-3 rad / 0.18 m, median 1.5e-3 rad / 6.8 cm)
    assert ang.max() < 5e-3 and terr.max() < 0.25
    assert np.median(ang) < 2.5e-3 and np.median(terr) < 0.1
    for p in (0, 7, 23):
        s = ds[soff[p]:soff[p + 1]].cpu().numpy()
        t = dt[toff[p]:toff[p + 1]].cpu().numpy()
        ref = O.gicp_oracle(s, t, inner="newton", recompute_src_cov=True, record=False, **synthetic.CONFIG4_PARAMS)
        assert int(res.n_outer[p]) == ref["n_outer"], (p, int(res.n_outer[p]), ref["n_outer"])
        assert _angle(T[p], ref["T"]) <= 1e-5
        assert np.linalg.norm(T[p, :3, 3] - ref["T"][:3, 3]) <= 1e-5 * synthetic.CONFIG4["cube"]


# 8. ----------------------------------------------------------------------------------------------------------------
def test_gicp_extended_voxel_size():
    from generalized_icp_b200 import compat, synthetic
    s, t, _ = synthetic.patches3d_pair(n=12000, n_patches=5, cube=30.0, patch=20.0, seed=1)
    kw = dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0, full_history=False)
    got = compat.gicp_extended(s, t, voxel_size=0.4, **kw)
    ds, dt = compat.voxel_downsample(s, 0.4), compat.voxel_downsample(t, 0.4)
    assert _same_bits(got["source_points"], ds) and _same_bits(got["target_points"], dt)
    assert len(ds) < len(s) and got["tgt_cov"].shape == (len(dt), 3, 3) and got["src_cov0"].shape == (len(ds), 3, 3)
    direct = compat.gicp_extended(ds, dt, **kw)
    assert np.array_equal(got["T"], direct["T"]) and got["n_outer"] == direct["n_outer"]
    plain = compat.gicp_extended(s, t, **kw)
    assert "source_points" not in plain and plain["tgt_cov"].shape == (len(t), 3, 3)
