"""Robust kernels of the registration loop (gicpSetRobustKernel, semantics in include/gicp_b200.h) on the device:
plumbing (a huge scale is bit-identical to no kernel), the stage entry points at the oracle's T_k, end to end against
the robust float64 oracle (tests/robust_oracle.py), the accuracy gain on inputs with structured outliers, batch and
path consistency, edge cases and the sharded source.

Inputs with structured outliers, and what the CPU oracle gives on them (error against the generating motion):
- MOVED: ``synthetic.patches3d_pair(n=3000, n_patches=8, cube=30, patch=20, seed=1, moved_patches=1,
  moved_offset=1.0)`` - the target points of one patch of eight are shifted 1 m along its normal, inside the 2 m gate.
  Plain GICP 2.76e-2 rad / 0.729 m; Huber c = 0.2: 2.44e-2 rad / 0.625 m; Cauchy c = 0.1: 9.0e-3 rad / 0.228 m;
  Tukey c = 0.5: 7.3e-4 rad / 0.026 m.
- OBSTACLE: two 360-ray scans of the robot demo's world from (60, 400, 0 deg) and the pose five turning ticks later,
  range noise uniform in +-2 px (numpy seed 7); the target's world has an extra circle (150, 450, r = 25) that the
  source never sees.  Plain GICP 1.34e-2 rad / 2.30 px; Huber c = 4: 2.5e-3 rad / 0.46 px; Cauchy c = 4: 1.7e-3 rad /
  0.40 px; Tukey c = 12: 1.0e-3 rad / 0.31 px.
"""
import math
import os

import numpy as np
import pytest

import robust_oracle as RO
from oracle import gicp_oracle as O
from test_gpu_search_exactness import Batch, _big_batch, _same_bits, env  # noqa: F401  (env: fixture)

pytestmark = pytest.mark.gpu

P3 = dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0)
P2 = dict(max_distance_nearest_neighbors=200.0)
SCALES3 = {"huber": 0.2, "cauchy": 0.1, "tukey": 0.5}
SCALES2 = {"huber": 4.0, "cauchy": 4.0, "tukey": 12.0}
# robust error / plain error on the inputs above, as the CPU oracle showed them, with some room
GAIN3 = {"huber": 0.9, "cauchy": 0.4, "tukey": 0.1}
GAIN2 = {"huber": 0.3, "cauchy": 0.3, "tukey": 0.3}


def _moved(n=3000, seed=1):
    from generalized_icp_b200 import synthetic
    return synthetic.patches3d_pair(n=n, n_patches=8, cube=30.0, patch=20.0, seed=seed, moved_patches=1,
                                    moved_offset=1.0)


def _obstacle():
    """The two scans (device ray caster, two obstacle lists) and the motion mapping the first onto the second."""
    import torch
    from generalized_icp_b200.engine import ray_cast
    world = [(100, 250, 200, 50), (400, 450, 50, 200), (600, 300, 50), (200, 550, 75)]
    x, y, yaw = 60.0, 400.0, 0
    poses = [(x, y, yaw)]
    for _ in range(5):
        yaw += 2
        x += 2 * math.cos(math.radians(yaw))
        y += 2 * math.sin(math.radians(yaw))
    poses.append((x, y, yaw))
    noise = np.random.default_rng(7).uniform(-2, 2, size=(2, 360))
    scans = []
    for i, obs in enumerate((world, world + [(150, 450, 25)])):
        rel, hit = ray_cast(np.asarray(poses[i:i + 1], dtype=np.float64), num_rays=360, obstacles=obs, noise=noise[i:i + 1])
        torch.cuda.synchronize()
        scans.append(rel[0][hit[0]].cpu().numpy())

    def rot(a):
        a = math.radians(a)
        return np.array([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]])
    (x0, y0, a0), (x1, y1, a1) = poses
    T = np.eye(3)
    T[:2, :2] = rot(a1).T @ rot(a0)
    T[:2, 2] = rot(a1).T @ np.array([x0 - x1, y0 - y1])
    return scans[0], scans[1], T


def _engine(dim, storage, src, tgt, **params):
    import torch
    from generalized_icp_b200.engine import GicpEngine
    eng = GicpEngine(dim, storage)
    eng.set_params(**params)
    dt = torch.float32 if storage == "f32" else torch.float64
    eng.set_target(torch.as_tensor(np.asarray(tgt, np.float64), device="cuda").to(dt))
    eng.set_source(torch.as_tensor(np.asarray(src, np.float64), device="cuda").to(dt))
    return eng


def _run(eng, kind=None, scale=None, T0=None):
    import torch
    eng.set_robust_kernel(kind, scale)
    r = eng.register(T0=T0, history=True)
    torch.cuda.synchronize()
    return r


def _rot_trans_diff(Ta, Tb):
    return RO.motion_error(Ta, Tb)


# ------------------------------------------------------------------------------------------------
# 1. plumbing: a scale no distance reaches is the unweighted loop, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_huge_scale_is_bit_identical_to_no_kernel(dim, storage, fused, env):
    if dim == 3:
        src, tgt, _ = _moved(n=1500)
        params = P3
    else:
        src, tgt, _ = _obstacle()
        params = P2
    eng = _engine(dim, storage, src, tgt, **params)

    def runs():
        ref = _run(eng)
        return ref, [_run(eng, kind, 1e300) for kind in ("huber", "cauchy")], _run(eng)
    ref, huge, again = env(runs, GICP_FUSED_LOOP=fused)
    assert int(ref.n_outer[0]) >= 3
    for r in huge + [again]:
        _same_bits(ref, r, (dim, storage, fused))


# ------------------------------------------------------------------------------------------------
# 2. the stage entry points at the oracle's T_k
# ------------------------------------------------------------------------------------------------
def _numpy_reduced_form_loss(src, q, W, T_lin, T_eval):
    """sum_i r_i^T W_i r_i of the frozen matches at T_eval (what the reduced form evaluates)."""
    d = src.shape[1]
    r = q - (src @ T_eval[:d, :d].T + T_eval[:d, d])
    return float(np.einsum("ni,nij,nj->", r, W, r))


@pytest.mark.parametrize("kind", ["huber", "cauchy", "tukey"])
def test_stages_teacher_forced(kind):
    from generalized_icp_b200.engine import reduced_form_loss
    src, tgt, _ = _moved()
    c = SCALES3[kind]
    ref = RO.gicp_oracle(src, tgt, robust=(kind, c), **P3)
    eng = _engine(3, "f64", src, tgt, **P3)
    src64, tgt64 = np.asarray(src, np.float64), np.asarray(tgt, np.float64)
    for k in sorted({0, 1, 2, ref["n_outer"] // 2, ref["n_outer"] - 1}):
        Tk = ref["trace"][k]["T"]
        eng.set_robust_kernel(None)
        idx0, dist0, W0 = (x.cpu().numpy() for x in eng.correspond(Tk))
        eng.set_robust_kernel(kind, c)
        idx1, dist1, W1 = (x.cpu().numpy() for x in eng.correspond(Tk))
        assert np.array_equal(idx0, idx1) and np.array_equal(dist0, dist1)
        g = idx1 >= 0
        w = RO.robust_weight(kind, dist1[g], c)
        want = w[:, None, None] * W0[g]
        assert np.all(np.abs(W1[g] - want) <= 1e-12 * np.abs(W0[g]).max(axis=(1, 2))[:, None, None])
        assert np.all(W1[~g] == 0.0)
        # the weighted reduced form against numpy on the device's own matches, at T_k and at two nearby transforms
        red = eng.normal_equations(Tk)[0]
        assert int(red[73] + 0.5) == int(g.sum())               # gated-in count, whatever the weights
        q = tgt64[idx1[g]]
        for T_eval in (Tk, O.offset_to_matrix(ref["trace"][k]["offset"], 3),
                       O.offset_to_matrix(np.array([0.01, -0.02, 0.005, 1e-3, -2e-3, 5e-4]), 3) @ Tk):
            want_loss = _numpy_reduced_form_loss(src64[g], q, want, Tk, T_eval)
            got = reduced_form_loss(red, 3, Tk, T_eval)
            assert abs(got - want_loss) <= 1e-9 * abs(want_loss) + 1e-12, (k, got, want_loss)


# ------------------------------------------------------------------------------------------------
# 3 + 4. end to end against the robust oracle, and the accuracy claim against the generating motion
# ------------------------------------------------------------------------------------------------
def _check_vs_oracle(r, ref, extent):
    assert int(r.n_outer[0]) == ref["n_outer"], (int(r.n_outer[0]), ref["n_outer"])
    conv = int(r.converged_at[0])
    assert conv == (-1 if ref["converged_at"] is None else ref["converged_at"])
    rot, trans = _rot_trans_diff(r.T[0].cpu().numpy(), ref["T"])
    assert rot <= 1e-5 and trans <= 1e-5 * extent, (rot, trans)


@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_moved_patch_end_to_end_and_gain(storage):
    src, tgt, Tg = _moved()
    eng = _engine(3, storage, src, tgt, **P3)
    plain = _run(eng)
    plain_ref = RO.gicp_oracle(src, tgt, record=False, **P3)
    _check_vs_oracle(plain, plain_ref, 30.0)
    e_plain = RO.motion_error(plain.T[0].cpu().numpy(), Tg)
    for kind, c in SCALES3.items():
        r = _run(eng, kind, c)
        ref = RO.gicp_oracle(src, tgt, robust=(kind, c), record=False, **P3)
        _check_vs_oracle(r, ref, 30.0)
        e = RO.motion_error(r.T[0].cpu().numpy(), Tg)
        assert e[0] < GAIN3[kind] * e_plain[0] and e[1] < GAIN3[kind] * e_plain[1], (kind, e, e_plain)


def test_obstacle_scan_end_to_end_and_gain():
    src, tgt, Tg = _obstacle()
    assert max(len(src), len(tgt)) <= 2048                   # the fused loop
    eng = _engine(2, "f64", src, tgt, **P2)
    plain = _run(eng)
    _check_vs_oracle(plain, RO.gicp_oracle(src, tgt, record=False, **P2), 400.0)
    e_plain = RO.motion_error(plain.T[0].cpu().numpy(), Tg)
    for kind, c in SCALES2.items():
        r = _run(eng, kind, c)
        _check_vs_oracle(r, RO.gicp_oracle(src, tgt, robust=(kind, c), record=False, **P2), 400.0)
        e = RO.motion_error(r.T[0].cpu().numpy(), Tg)
        assert e[0] < GAIN2[kind] * e_plain[0] and e[1] < GAIN2[kind] * e_plain[1], (kind, e, e_plain)


@pytest.mark.parametrize("model", [1, 2])
def test_icp_variants_end_to_end(model):
    src, tgt, _ = _moved()
    eng = _engine(3, "f64", src, tgt, covariance_model=model, **P3)
    r = _run(eng, "cauchy", 0.2)
    ref = RO.gicp_oracle(src, tgt, robust=("cauchy", 0.2), covariance_model=model, record=False, **P3)
    _check_vs_oracle(r, ref, 30.0)


def test_compat_and_odometry_take_the_kernel():
    from generalized_icp_b200 import compat
    src, tgt, _ = _obstacle()
    got = compat.gicp_extended(src, tgt, robust_kernel="cauchy", robust_scale=4.0, **P2)
    ref = RO.gicp_oracle(src, tgt, robust=("cauchy", 4.0), **P2)
    assert got["n_outer"] == ref["n_outer"]
    assert np.abs(got["T"] - ref["T"]).max() < 1e-6
    # hw_src / hw_tgt rank the weighted matrices w W, as the oracle does (at T_0 = I both rank the same matrices)
    assert len(got["hw_tgt"]) == len(ref["hw_tgt"])
    assert np.abs(np.sort(got["hw_tgt"][0], axis=0) - np.sort(ref["hw_tgt"][0], axis=0)).max() < 1e-9
    # gicp() and a later call without a kernel are the plain registration again
    plain = compat.gicp_extended(src, tgt, **P2)
    assert plain["n_outer"] == RO.gicp_oracle(src, tgt, record=False, **P2)["n_outer"]


# ------------------------------------------------------------------------------------------------
# 5. batch and path consistency
# ------------------------------------------------------------------------------------------------
def test_robust_batch_equals_its_pairs():
    from generalized_icp_b200 import synthetic
    srcs, tgts = [], []
    for seed in range(4):
        s, t, _ = synthetic.patches3d_pair(n=3000, n_patches=8, cube=30.0, patch=20.0, seed=seed, moved_patches=1,
                                           moved_offset=1.0)
        srcs.append(s)
        tgts.append(t)
    b = Batch(3, "f32", srcs, tgts, **P3)
    b.eng.set_robust_kernel("tukey", 0.5)
    rb = b.register()
    for p in range(4):
        one = Batch(3, "f32", [srcs[p]], [tgts[p]], **P3)
        one.eng.set_robust_kernel("tukey", 0.5)
        r1 = one.register()
        # every cloud has 3000 points: the same grids in the batch and alone, so the same bits
        for f in ("T", "n_outer", "converged_at", "T_hist", "loss_hist", "inliers"):
            a, c = getattr(rb, f)[p:p + 1], getattr(r1, f)
            assert np.array_equal(a.cpu().numpy(), c.cpu().numpy(), equal_nan=True), (p, f)


def test_robust_big_batch_exact_alternatives(env):
    """1152 small 2-D pairs in the multi-launch loop (active list, two 1024-pair compaction chunks) with a Cauchy
    kernel: the exact alternatives of the search give the same bits as the default robust run."""
    srcs, tgts, params = _big_batch()
    b = Batch(2, "f64", srcs, tgts, **params)
    b.eng.set_robust_kernel("cauchy", 1.0)
    ref = env(b.register, GICP_FUSED_LOOP=0)
    assert np.isfinite(ref.loss_hist.cpu().numpy()[:, 0]).all()
    for sw in ({"GICP_NO_SKIP": "1"}, {"GICP_TRACK_CELLS": "0"}, {"GICP_ACTIVE_LIST": "0"}):
        _same_bits(ref, env(b.register, GICP_FUSED_LOOP=0, **sw), sw)


@pytest.mark.parametrize("kind", ["huber", "cauchy", "tukey"])
def test_fused_equals_multi_launch(kind, env):
    src, tgt, _ = _moved(n=1500)
    eng = _engine(3, "f64", src, tgt, **P3)
    fused = env(lambda: _run(eng, kind, SCALES3[kind]), GICP_FUSED_LOOP=1)
    multi = env(lambda: _run(eng, kind, SCALES3[kind]), GICP_FUSED_LOOP=0)
    assert np.array_equal(fused.n_outer.cpu().numpy(), multi.n_outer.cpu().numpy())
    assert np.array_equal(fused.converged_at.cpu().numpy(), multi.converged_at.cpu().numpy())
    assert np.array_equal(fused.inliers.cpu().numpy(), multi.inliers.cpu().numpy())
    n = int(fused.n_outer[0])
    dh = np.abs(fused.T_hist.cpu().numpy()[0, :n] - multi.T_hist.cpu().numpy()[0, :n])
    assert np.nanmax(dh) < 1e-9


# ------------------------------------------------------------------------------------------------
# 6. edge cases
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", ["1", "0"])
def test_tukey_beyond_every_distance_stops_like_an_all_gated_out_pair(fused, env):
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    r = env(lambda: _run(eng, "tukey", 1e-9), GICP_FUSED_LOOP=fused)
    assert int(r.n_outer[0]) == 2 and int(r.converged_at[0]) == 1
    assert np.array_equal(r.T[0].cpu().numpy(), np.eye(3))
    loss = r.loss_hist.cpu().numpy()[0, :2]
    assert np.array_equal(loss, [0.0, 0.0])
    assert (r.inliers.cpu().numpy()[0, :2] > 0).all()          # gated in, weighing nothing
    gated = _engine(2, "f64", src, tgt, max_distance_nearest_neighbors=200.0, max_distance_correspondence=1e-9)
    g = env(lambda: _run(gated), GICP_FUSED_LOOP=fused)
    assert int(g.n_outer[0]) == 2 and int(g.converged_at[0]) == 1
    assert np.array_equal(g.T[0].cpu().numpy(), r.T[0].cpu().numpy())
    assert np.array_equal(g.loss_hist.cpu().numpy()[0, :2], loss)


def test_set_clear_set_on_one_handle():
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    plain = _run(eng)
    a = _run(eng, "huber", 4.0)
    _same_bits(plain, _run(eng))
    _same_bits(a, _run(eng, "huber", 4.0))
    b = _run(eng, "tukey", 12.0)
    assert not np.array_equal(a.T.cpu().numpy(), b.T.cpu().numpy())
    _same_bits(plain, _run(eng, None))


def test_invalid_kernel_is_rejected_and_the_handle_stays_usable():
    from generalized_icp_b200 import _lib
    src, tgt, _ = _obstacle()
    eng = _engine(2, "f64", src, tgt, **P2)
    ref = _run(eng, "cauchy", 4.0)
    for kind, scale, msg in ((7, 1.0, "unknown robust kernel"), (-1, 1.0, "unknown robust kernel"),
                             (1, 0.0, "finite and > 0"), (2, -1.0, "finite and > 0"), (3, float("nan"), "finite and > 0"),
                             (1, float("inf"), "finite and > 0")):
        assert eng.lib.gicpSetRobustKernel(eng._h, kind, scale) != 0
        assert msg in _lib.load().gicpGetLastError().decode()
    with pytest.raises(ValueError):
        eng.set_robust_kernel("welsch", 1.0)
    with pytest.raises(ValueError):
        eng.set_robust_kernel("huber")
    # the rejected calls left the kernel as it was
    import torch
    r = eng.register(history=True)
    torch.cuda.synchronize()
    _same_bits(ref, r)
    assert eng.lib.gicpSetRobustKernel(eng._h, 0, float("nan")) == 0     # no kernel: the scale is not used


# ------------------------------------------------------------------------------------------------
# 7. sharded source
# ------------------------------------------------------------------------------------------------
def _sharded_worker(rank, world, port, src, tgt, prm, out):
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
    eng.set_robust_kernel("cauchy", 0.1)
    eng.set_target(torch.as_tensor(tgt, device=f"cuda:{rank}"))
    eng.set_source(torch.as_tensor(src, device=f"cuda:{rank}"))
    r = eng.register()
    torch.cuda.synchronize()
    out[rank] = (r.T[0].cpu().numpy(), int(r.n_outer[0]))
    eng.comm_destroy()
    dist.destroy_process_group()


def test_sharded_source_with_cauchy():
    import socket
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from generalized_icp_b200 import synthetic
    src, tgt, _ = synthetic.patches3d_pair(n=20000, n_patches=8, cube=40.0, patch=25.0, seed=11, moved_patches=1,
                                           moved_offset=1.0)
    prm = dict(k=20, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0)
    eng = _engine(3, "f32", src, tgt, **prm)
    ref = _run(eng, "cauchy", 0.1)
    T_ref, n_ref = ref.T[0].cpu().numpy(), int(ref.n_outer[0])
    del eng
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_sharded_worker, args=(2, port, src, tgt, prm, out), nprocs=2, join=True)
    for r in range(2):
        T, n = out[r]
        assert n == n_ref
        assert np.abs(T - T_ref).max() < 1e-7
