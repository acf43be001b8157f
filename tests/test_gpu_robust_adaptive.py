"""The adaptive robust scale (gicpSetRobustKernelAdaptive, semantics in include/gicp_b200.h) on the device: plumbing
(a tiny kappa is the fixed kernel at min_scale, bit for bit), the select's median against numpy at given transforms,
the fused loop's scale against the multi-launch loop's, end to end against the float64 oracle
(tests/adaptive_oracle.py), batches, the handle, and the accuracy the oracle shows.

Accuracy, as the CPU oracle gives it (error against the generating motion):
- MOVED (test_gpu_robust.py: one patch of eight shifted 1 m along its normal, inside the 2 m gate), min_scale 0.02 m:
  plain 2.76e-2 rad / 0.729 m; adaptive Huber kappa 0.5: 2.47e-2 / 0.633; Cauchy kappa 0.5: 1.73e-2 / 0.441; Tukey
  kappa 1: 7.4e-4 / 0.027.
- DRIVE: the 11 pairs of demo_inputs.lidar_sequence(seed=0, num_rays=90, n_scans=12), the demo's parameters, min_scale
  1 px: median translation error plain 2.71 px, adaptive Huber kappa 4.5 1.67 px.
"""
import numpy as np
import pytest

import adaptive_oracle as AO
from test_gpu_robust import P2, P3, _engine, _moved, _obstacle
from test_gpu_search_exactness import Batch, _big_batch, _same_bits, env  # noqa: F401  (env: fixture)

pytestmark = pytest.mark.gpu

DRIVE = dict(max_distance_nearest_neighbors=200.0, tolerance=1.0)
KAPPA3 = {"huber": 0.5, "cauchy": 0.5, "tukey": 1.0}
MIN3 = 0.02
# adaptive error / plain error on MOVED, as the CPU oracle showed them (0.90 / 0.63 / 0.04), with some room
GAIN3 = {"huber": 0.95, "cauchy": 0.75, "tukey": 0.1}
KAPPA2, MIN2 = 4.5, 1.0


def _run(eng, kind=None, scale=None, adaptive=None, min_scale=None, T0=None):
    import torch
    eng.set_robust_kernel(kind, scale, adaptive=adaptive, min_scale=min_scale)
    r = eng.register(T0=T0, history=True)
    torch.cuda.synchronize()
    return r


# ------------------------------------------------------------------------------------------------
# 1. plumbing: min_scale dominant is the fixed kernel at c = min_scale, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_tiny_kappa_is_the_fixed_kernel(dim, storage, fused, env):
    if dim == 3:
        src, tgt, _ = _moved(n=1500)
        params, kind, c = P3, "cauchy", 0.1
    else:
        src, tgt, _ = _obstacle()
        params, kind, c = P2, "tukey", 12.0
    eng = _engine(dim, storage, src, tgt, **params)
    fixed, ad = env(lambda: (_run(eng, kind, c), _run(eng, kind, adaptive=1e-300, min_scale=c)), GICP_FUSED_LOOP=fused)
    assert int(fixed.n_outer[0]) >= 3
    _same_bits(fixed, ad, (dim, storage, fused))


# ------------------------------------------------------------------------------------------------
# 2. the median at given transforms (teacher forced)
# ------------------------------------------------------------------------------------------------
def _check_scales(eng, T, kappa, min_scale, kind="huber"):
    """gicpRobustScales at T against numpy on gicpCorrespond's distances at T; d_W against w(d, c) * W."""
    eng.set_robust_kernel(None)
    idx, dist, W0 = (x.cpu().numpy() for x in eng.correspond(T))
    eng.set_robust_kernel(kind, adaptive=kappa, min_scale=min_scale)
    got = eng.robust_scales(T)
    idx1, dist1, W1 = (x.cpu().numpy() for x in eng.correspond(T))
    assert np.array_equal(idx, idx1) and np.array_equal(dist, dist1)
    off = eng._n_offsets
    want = np.array([AO.scale_at(kappa, min_scale, idx[a:b], dist[a:b]) for a, b in zip(off[:-1], off[1:])])
    assert np.array_equal(got.view(np.int64), want.view(np.int64)), (got, want)
    import robust_oracle as RO
    for p, (a, b) in enumerate(zip(off[:-1], off[1:])):
        g = idx[a:b] >= 0
        w = RO.robust_weight(kind, dist[a:b][g], got[p])
        ref = w[:, None, None] * W0[a:b][g]
        assert np.all(np.abs(W1[a:b][g] - ref) <= 1e-12 * np.abs(W0[a:b][g]).max(axis=(1, 2))[:, None, None])
    return got


def _batch_engine(dim, storage, srcs, tgts, **params):
    b = Batch(dim, storage, srcs, tgts, **params)
    b.eng._n_offsets = b.off_s
    return b


@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_scale_at_the_oracle_transforms(storage):
    src, tgt, _ = _moved()
    ref = AO.gicp_oracle(src, tgt, adaptive=("cauchy", KAPPA3["cauchy"], MIN3), **P3)
    b = _batch_engine(3, storage, [src], [tgt], **P3)
    for k in sorted({0, 1, ref["n_outer"] // 2, ref["n_outer"] - 1}):
        got = _check_scales(b.eng, ref["trace"][k]["T"][None], KAPPA3["cauchy"], MIN3, "cauchy")
        assert abs(got[0] - ref["trace"][k]["c"]) <= 1e-9 * ref["trace"][k]["c"]


@pytest.mark.parametrize("n", [20_000, 200_000])
def test_scale_of_large_pairs(n):
    """Pairs of many blocks: the multi-block select of the stage entry points."""
    from generalized_icp_b200 import synthetic
    src, tgt, Tg = synthetic.patches3d_pair(n=n, n_patches=32, cube=60.0, patch=25.0, seed=3, moved_patches=2,
                                            moved_offset=1.0)
    b = _batch_engine(3, "f32", [src], [tgt], k=20, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0)
    for T in (np.eye(4), Tg, np.linalg.inv(Tg)):
        _check_scales(b.eng, T[None], 3.0, 1e-3)


def _lattice(n, spacing=1.0):
    g = np.arange(n, dtype=np.float64) * spacing
    return np.stack(np.meshgrid(g, g, indexing="ij"), -1).reshape(-1, 2)


def _edge_case_clouds():
    """An all-gated-out pair, a single-inlier pair, even and odd inlier counts and a dyadic lattice full of ties."""
    rng = np.random.default_rng(4)
    lat = _lattice(12)
    srcs, tgts = [], []
    srcs.append(lat); tgts.append(lat + 100.0)                         # every point gated out: min_scale
    one = lat.copy(); one[1:] += 50.0                                  # a single gated-in point
    srcs.append(one); tgts.append(lat + np.array([0.25, 0.0]))
    for n in (64, 65):                                                 # even and odd inlier counts
        s = rng.uniform(0, 20, size=(n, 2))
        srcs.append(s); tgts.append(s + rng.normal(0, 0.05, size=s.shape))
    tie = lat + np.where(rng.random((len(lat), 1)) < 0.5, np.array([0.25, 0.0]), np.array([0.0, 0.5]))
    srcs.append(lat); tgts.append(tie)                                 # dyadic distances: 0.25 and 0.5, many ties
    return srcs, tgts


EDGE = dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0)


def test_scale_edge_cases_in_one_batch():
    srcs, tgts = _edge_case_clouds()
    b = _batch_engine(2, "f64", srcs, tgts, **EDGE)
    T = np.broadcast_to(np.eye(3), (len(srcs), 3, 3))
    for kappa, mn in ((2.0, 0.1), (1.0, 0.5), (3.0, 0.125)):
        got = _check_scales(b.eng, T, kappa, mn)
        assert got[0] == mn
    idx, _, _ = b.eng.correspond(T)
    idx = idx.cpu().numpy()
    assert (idx[b.off_s[0]:b.off_s[1]] < 0).all() and (idx[b.off_s[1]:b.off_s[2]] >= 0).sum() == 1


# ------------------------------------------------------------------------------------------------
# 3. the fused loop's scale: the same loop as the multi-launch path's
# ------------------------------------------------------------------------------------------------
def _same_loop_paths(eng, kind, kappa, mn, env):
    fused = env(lambda: _run(eng, kind, adaptive=kappa, min_scale=mn), GICP_FUSED_LOOP=1)
    multi = env(lambda: _run(eng, kind, adaptive=kappa, min_scale=mn), GICP_FUSED_LOOP=0)
    for f in ("n_outer", "converged_at", "inliers"):
        assert np.array_equal(getattr(fused, f).cpu().numpy(), getattr(multi, f).cpu().numpy()), f
    n = int(fused.n_outer[0])
    assert np.nanmax(np.abs(fused.T_hist.cpu().numpy()[0, :n] - multi.T_hist.cpu().numpy()[0, :n])) < 1e-9


@pytest.mark.parametrize("kind", ["huber", "cauchy", "tukey"])
def test_fused_equals_multi_launch_on_scans(kind, env):
    src, tgt, _ = _obstacle()
    _same_loop_paths(_engine(2, "f64", src, tgt, **P2), kind, 3.0, 1.0, env)


def test_fused_equals_multi_launch_on_the_edge_cases(env):
    """The edge-case batch registered by the fused loop (the in-block select: no gated-in match, one, even and odd
    counts, ties) and by the multi-launch loop (scale_select_kernel): the same loops."""
    srcs, tgts = _edge_case_clouds()
    b = Batch(2, "f64", srcs, tgts, **EDGE)
    for kappa, mn in ((2.0, 0.1), (1.0, 0.5), (3.0, 0.125)):
        b.eng.set_robust_kernel("cauchy", adaptive=kappa, min_scale=mn)
        fused = env(b.register, GICP_FUSED_LOOP=1)
        multi = env(b.register, GICP_FUSED_LOOP=0)
        for f in ("n_outer", "converged_at", "inliers"):
            assert np.array_equal(getattr(fused, f).cpu().numpy(), getattr(multi, f).cpu().numpy()), (kappa, f)
        lf, lm = fused.loss_hist.cpu().numpy(), multi.loss_hist.cpu().numpy()
        assert np.array_equal(np.isnan(lf), np.isnan(lm))
        ok = ~np.isnan(lf)
        assert np.all(np.abs(lf[ok] - lm[ok]) <= 1e-9 * np.abs(lm[ok]) + 1e-12), kappa
        hf, hm = fused.T_hist.cpu().numpy(), multi.T_hist.cpu().numpy()
        assert np.nanmax(np.abs(hf - hm)) < 1e-9, kappa
        assert int(fused.inliers[0, 0]) == 0 and int(fused.inliers[1, 0]) == 1


def test_fused_equals_multi_launch_on_the_drive(env):
    for s, t, _ in AO.drive_pairs()[:6]:
        _same_loop_paths(_engine(2, "f64", s, t, **DRIVE), "huber", KAPPA2, MIN2, env)


# ------------------------------------------------------------------------------------------------
# 4. end to end against the adaptive oracle
# ------------------------------------------------------------------------------------------------
def _check_vs_oracle(r, ref, extent):
    import robust_oracle as RO
    assert int(r.n_outer[0]) == ref["n_outer"], (int(r.n_outer[0]), ref["n_outer"])
    assert int(r.converged_at[0]) == (-1 if ref["converged_at"] is None else ref["converged_at"])
    rot, trans = RO.motion_error(r.T[0].cpu().numpy(), ref["T"])
    assert rot <= 1e-5 and trans <= 1e-5 * extent, (rot, trans)


@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_moved_patch_end_to_end_and_gain(storage):
    import robust_oracle as RO
    src, tgt, Tg = _moved()
    eng = _engine(3, storage, src, tgt, **P3)
    e_plain = RO.motion_error(_run(eng).T[0].cpu().numpy(), Tg)
    for kind, kappa in KAPPA3.items():
        r = _run(eng, kind, adaptive=kappa, min_scale=MIN3)
        _check_vs_oracle(r, AO.gicp_oracle(src, tgt, adaptive=(kind, kappa, MIN3), record=False, **P3), 30.0)
        e = RO.motion_error(r.T[0].cpu().numpy(), Tg)
        assert e[0] < GAIN3[kind] * e_plain[0] and e[1] < GAIN3[kind] * e_plain[1], (kind, e, e_plain)


def test_obstacle_scan_end_to_end():
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    for kind in ("huber", "cauchy", "tukey"):
        r = _run(eng, kind, adaptive=3.0, min_scale=1.0)
        _check_vs_oracle(r, AO.gicp_oracle(src, tgt, adaptive=(kind, 3.0, 1.0), record=False, **P2), 400.0)


@pytest.mark.parametrize("model", [1, 2])
def test_icp_variants_end_to_end(model):
    src, tgt, _ = _moved()
    eng = _engine(3, "f64", src, tgt, covariance_model=model, **P3)
    r = _run(eng, "cauchy", adaptive=0.5, min_scale=MIN3)
    ref = AO.gicp_oracle(src, tgt, adaptive=("cauchy", 0.5, MIN3), covariance_model=model, record=False, **P3)
    _check_vs_oracle(r, ref, 30.0)


def test_drive_end_to_end_and_gain():
    """Every drive pair against the oracle, and the accuracy claim: adaptive Huber beats plain GICP in median
    translation error."""
    import robust_oracle as RO
    plain, ad = [], []
    for s, t, Tg in AO.drive_pairs():
        eng = _engine(2, "f64", s, t, **DRIVE)
        plain.append(RO.motion_error(_run(eng).T[0].cpu().numpy(), Tg)[1])
        r = _run(eng, "huber", adaptive=KAPPA2, min_scale=MIN2)
        _check_vs_oracle(r, AO.gicp_oracle(s, t, adaptive=("huber", KAPPA2, MIN2), record=False, **DRIVE), 400.0)
        ad.append(RO.motion_error(r.T[0].cpu().numpy(), Tg)[1])
    assert np.median(ad) < np.median(plain), (np.median(ad), np.median(plain))


def test_compat_and_odometry_take_the_adaptive_scale():
    from generalized_icp_b200 import compat
    from generalized_icp_b200.odometry import ScanOdometry
    src, tgt, _ = _obstacle()
    got = compat.gicp_extended(src, tgt, robust_kernel="cauchy", robust_adaptive=3.0, robust_min_scale=1.0, **P2)
    ref = AO.gicp_oracle(src, tgt, adaptive=("cauchy", 3.0, 1.0), **P2)
    assert got["n_outer"] == ref["n_outer"]
    assert np.abs(got["T"] - ref["T"]).max() < 1e-6
    pairs = AO.drive_pairs()[:1]
    odo = ScanOdometry(robust_kernel="huber", robust_adaptive=KAPPA2, robust_min_scale=MIN2)
    odo.push(pairs[0][0])
    odo.push(pairs[0][1])
    want = AO.gicp_oracle(pairs[0][0], pairs[0][1], adaptive=("huber", KAPPA2, MIN2), record=False, **DRIVE)
    assert np.abs(odo.transforms[0] - want["T"]).max() < 1e-6


# ------------------------------------------------------------------------------------------------
# 5. batches
# ------------------------------------------------------------------------------------------------
def test_adaptive_batch_equals_its_pairs():
    from generalized_icp_b200 import synthetic
    srcs, tgts = [], []
    for seed in range(4):
        s, t, _ = synthetic.patches3d_pair(n=3000, n_patches=8, cube=30.0, patch=20.0, seed=seed, moved_patches=1,
                                           moved_offset=1.0)
        srcs.append(s)
        tgts.append(t)
    b = Batch(3, "f32", srcs, tgts, **P3)
    b.eng.set_robust_kernel("tukey", adaptive=1.0, min_scale=MIN3)
    rb = b.register()
    for p in range(4):
        one = Batch(3, "f32", [srcs[p]], [tgts[p]], **P3)
        one.eng.set_robust_kernel("tukey", adaptive=1.0, min_scale=MIN3)
        r1 = one.register()
        for f in ("T", "n_outer", "converged_at", "T_hist", "loss_hist", "inliers"):
            a, c = getattr(rb, f)[p:p + 1], getattr(r1, f)
            assert np.array_equal(a.cpu().numpy(), c.cpu().numpy(), equal_nan=True), (p, f)


def test_adaptive_big_batch_exact_alternatives(env):
    """1152 small 2-D pairs in the multi-launch loop (active list) with an adaptive Cauchy scale: the exact
    alternatives of the search and the full launches give the same bits as the default run."""
    srcs, tgts, params = _big_batch()
    b = Batch(2, "f64", srcs, tgts, **params)
    b.eng.set_robust_kernel("cauchy", adaptive=2.0, min_scale=0.1)
    ref = env(b.register, GICP_FUSED_LOOP=0)
    assert np.isfinite(ref.loss_hist.cpu().numpy()[:, 0]).all()
    for sw in ({"GICP_NO_SKIP": "1"}, {"GICP_TRACK_CELLS": "0"}, {"GICP_ACTIVE_LIST": "0"}):
        _same_bits(ref, env(b.register, GICP_FUSED_LOOP=0, **sw), sw)


# ------------------------------------------------------------------------------------------------
# 6. the handle
# ------------------------------------------------------------------------------------------------
def test_fixed_adaptive_none_adaptive_on_one_handle():
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    fixed = _run(eng, "huber", 4.0)
    ad = _run(eng, "huber", adaptive=3.0, min_scale=1.0)
    plain = _run(eng)
    _same_bits(ad, _run(eng, "huber", adaptive=3.0, min_scale=1.0))
    _same_bits(fixed, _run(eng, "huber", 4.0))
    _same_bits(plain, _run(eng))
    assert not np.array_equal(ad.T.cpu().numpy(), fixed.T.cpu().numpy())
    T = np.eye(3)[None]
    assert eng.robust_scales(T)[0] == 0.0
    eng.set_robust_kernel("huber", 4.0)
    assert eng.robust_scales(T)[0] == 4.0


def test_invalid_adaptive_arguments_are_rejected():
    from generalized_icp_b200 import _lib
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    ref = _run(eng, "cauchy", adaptive=3.0, min_scale=1.0)
    nan, inf = float("nan"), float("inf")
    for kind, kappa, mn, msg in ((0, 1.0, 1.0, "GICP_ROBUST_NONE"), (4, 1.0, 1.0, "must be GICP_ROBUST_HUBER"),
                                 (1, 0.0, 1.0, "kappa must be finite and > 0"), (1, nan, 1.0, "kappa"),
                                 (1, inf, 1.0, "kappa"), (2, 1.0, 0.0, "min_scale must be finite and > 0"),
                                 (3, 1.0, -1.0, "min_scale"), (3, 1.0, inf, "min_scale")):
        assert eng.lib.gicpSetRobustKernelAdaptive(eng._h, kind, kappa, mn) != 0
        assert msg in _lib.load().gicpGetLastError().decode()
    for kw in (dict(scale=1.0, adaptive=1.0, min_scale=1.0), dict(adaptive=1.0), dict(scale=1.0, min_scale=1.0), {}):
        with pytest.raises(ValueError):
            eng.set_robust_kernel("huber", **kw)
    with pytest.raises(ValueError):
        eng.set_robust_kernel(None, adaptive=1.0, min_scale=1.0)
    import torch
    r = eng.register(history=True)       # the rejected calls left the adaptive scale as it was
    torch.cuda.synchronize()
    _same_bits(ref, r)


def _sharded_worker(rank, world, port, src, tgt, prm, out):
    import os
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from generalized_icp_b200.engine import GicpEngine
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    uid = [GicpEngine.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    eng = GicpEngine(3, "f32", device=rank)
    eng.comm_init(world, rank, uid[0])
    eng.set_params(**prm)
    eng.set_target(torch.as_tensor(tgt, device=f"cuda:{rank}"))
    eng.set_source(torch.as_tensor(src, device=f"cuda:{rank}"))
    eng.set_robust_kernel("cauchy", adaptive=1.0, min_scale=0.02)
    try:
        eng.register()
        msg = ""
    except RuntimeError as e:
        msg = str(e)
    eng.set_robust_kernel("cauchy", 0.1)                  # the handle stays usable
    r = eng.register()
    torch.cuda.synchronize()
    out[rank] = (msg, int(r.n_outer[0]))
    eng.comm_destroy()
    dist.destroy_process_group()


def test_sharded_source_rejects_an_adaptive_scale():
    import socket
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from generalized_icp_b200 import synthetic
    src, tgt, _ = synthetic.patches3d_pair(n=20000, n_patches=8, cube=40.0, patch=25.0, seed=11)
    prm = dict(k=20, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_sharded_worker, args=(2, port, src, tgt, prm, out), nprocs=2, join=True)
    for r in range(2):
        msg, n = out[r]
        assert "adaptive robust scale" in msg and "sharded" in msg, msg
        assert n >= 1
