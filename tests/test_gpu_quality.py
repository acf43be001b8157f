"""gicpEvaluate / GicpEngine.evaluate (semantics in include/gicp_b200.h) on the device: teacher-forced against the
stage entry points and numpy (tests/quality_oracle.py), the perturbation convention against finite differences, the
loop's own inlier counts, device residency without a host synchronisation, no effect on later registrations, and what
the numbers tell a user (a degenerate corridor, a pair stopped in a wrong pose)."""
import numpy as np
import pytest

import quality_oracle as QO
from test_gpu_robust import P2, P3, _engine, _moved, _obstacle
from test_gpu_search_exactness import Batch, _same_bits, env  # noqa: F401  (env: fixture)
from test_quality_host import qmap  # noqa: F401  (fixture: the host build of the map)

pytestmark = pytest.mark.gpu

# H and b against numpy from the device's own W, per block: H relative to the block's norm, b relative to the norm of
# sum_i |J_i^T W_i e_i| (b vanishes where a registration converged).  f32 storage accumulates the reduced form in f32
# per thread; its bound is the measured worst case over the cases below with a margin (DESIGN §7).
HB_TOL = {"f64": 1e-9, "f32": 1e-6}
KERNELS = {"none": None, "huber": ("huber", dict(scale=0.3)), "tukey_adaptive": ("tukey", dict(adaptive=2.0,
                                                                                                min_scale=0.05))}
KERNELS2 = {"none": None, "huber": ("huber", dict(scale=4.0)), "tukey_adaptive": ("tukey", dict(adaptive=3.0,
                                                                                                 min_scale=1.0))}
NQ = {2: 24, 3: 72}


def _np(x):
    return x.detach().cpu().numpy()


def _set_kernel(eng, spec):
    if spec is None:
        eng.set_robust_kernel(None)
    else:
        eng.set_robust_kernel(spec[0], **spec[1])


def _reference(eng, srcs, tgts, T, dim):
    """Per pair (quality row, H, b) from gicpCorrespond's idx, dist and w W at T, in numpy."""
    idx, dist, W = (_np(x) for x in eng.correspond(T))
    out, a = [], 0
    for p, (s, t) in enumerate(zip(srcs, tgts)):
        b_ = a + len(s)
        g = idx[a:b_] >= 0
        R, tr = T[p, :dim, :dim], T[p, :dim, dim]
        pp = s[g] @ R.T + tr
        e = t[idx[a:b_][g]] - pp
        Wg = W[a:b_][g]
        out.append(QO.quality(pp, e, Wg, dist[a:b_][g], len(s), dim) + (QO.gradient_magnitude(pp, e, Wg),))
        a = b_
    return idx, out


def _check_teacher_forced(eng, srcs, tgts, T, dim, storage, qmap_fn, worst):
    T = np.ascontiguousarray(T, np.float64)
    q = eng.evaluate(T)
    qq, H, b = _np(q.n_inliers), _np(q.H), _np(q.b)
    fit, rmse, loss = _np(q.fitness), _np(q.inlier_rmse), _np(q.loss)
    red = eng.normal_equations(T)
    idx, ref = _reference(eng, srcs, tgts, T, dim)
    a = 0
    for p, (qr, Hr, br, bmag) in enumerate(ref):
        n = int((idx[a:a + len(srcs[p])] >= 0).sum())
        a += len(srcs[p])
        assert qq[p] == n == int(red[p, NQ[dim] + 1]), (p, qq[p], n, red[p, NQ[dim] + 1])
        assert loss[p].view(np.int64) == red[p, NQ[dim]].view(np.int64), (p, loss[p], red[p, NQ[dim]])
        assert fit[p] == (n / len(srcs[p]) if len(srcs[p]) else 0.0)
        assert abs(rmse[p] - qr[2]) <= 1e-12 * qr[2], (p, rmse[p], qr[2])
        if n == 0:
            assert not H[p].any() and not b[p].any() and rmse[p] == 0.0 and loss[p] == 0.0
            continue
        eh, eb = QO.block_rel_err(H[p], Hr, dim), QO.block_rel_err(b[p], br, dim, scale=bmag)
        worst[0] = max(worst[0], eh)
        worst[1] = max(worst[1], eb)
        assert eh < HB_TOL[storage] and eb < HB_TOL[storage], (p, storage, eh, eb)
    # the host build of the map on gicpNormalEquations' rows
    n_src = np.array([len(s) for s in srcs])
    _, Hh, bh = qmap_fn(dim, red, np.zeros(len(srcs)), n_src)
    for p in range(len(srcs)):
        assert QO.block_rel_err(H[p], Hh[p], dim) < 1e-12, p
        assert QO.block_rel_err(b[p], bh[p], dim, scale=ref[p][3]) < 1e-12, p
        assert np.array_equal(H[p], H[p].T)


def _perturb(T, dim, seed, deg=2.0, shift=0.3):
    rng = np.random.default_rng(seed)
    out = np.array(T, np.float64, copy=True)
    for p in range(len(out)):
        if dim == 3:
            ax = rng.normal(size=3)
            ax /= np.linalg.norm(ax)
            K = QO.skew(ax)
            a = np.deg2rad(deg)
            R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
        else:
            a = np.deg2rad(deg)
            R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        M = np.eye(dim + 1)
        M[:dim, :dim], M[:dim, dim] = R, shift * rng.normal(size=dim)
        out[p] = M @ out[p]
    return out


# ------------------------------------------------------------------------------------------------
# 1. teacher forced: every covariance model, kernel and storage, at the loop's transforms and perturbed ones
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("model", [0, 1, 2])
@pytest.mark.parametrize("kernel", list(KERNELS))
def test_teacher_forced(dim, storage, model, kernel, qmap):
    if dim == 3:
        src, tgt, _ = _moved(n=1500)
        params, spec = P3, KERNELS[kernel]
    else:
        src, tgt, _ = _obstacle()
        params, spec = P2, KERNELS2[kernel]
    eng = _engine(dim, storage, src, tgt, covariance_model=model, **params)
    _set_kernel(eng, spec)
    np_dt = np.float32 if storage == "f32" else np.float64
    s64 = np.asarray(src, np_dt).astype(np.float64)
    t64 = np.asarray(tgt, np_dt).astype(np.float64)
    r = eng.register(history=True)
    n_outer = int(r.n_outer[0])
    T_hist = _np(r.T_hist)[0]
    assert n_outer >= 2
    worst = [0.0, 0.0]
    for T in (T_hist[1], _np(r.T)[0], _perturb(_np(r.T), dim, 3)[0]):
        _check_teacher_forced(eng, [s64], [t64], T[None], dim, storage, qmap, worst)
    print(f"\n[quality] dim={dim} {storage} model={model} {kernel}: max block err H {worst[0]:.3e} b {worst[1]:.3e}")


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_teacher_forced_batch_edge_cases(dim, storage, qmap):
    """An empty source, an empty target, an all-gated-out pair, a pair 1e4 m from the origin, and a regular pair."""
    if dim == 3:
        s, t, Tg = _moved(n=1200)
        params, gate = P3, P3["max_distance_correspondence"]
    else:
        s, t, Tg = _obstacle()
        params, gate = P2, 150.0
    s, t = np.asarray(s, np.float64), np.asarray(t, np.float64)
    far = np.full(dim, 1e4)
    srcs = [s[:0], s, s, s + far, s]
    tgts = [t, t[:0], t + 10 * gate, t + far, t]
    b = Batch(dim, storage, srcs, tgts, **params)
    T = np.tile(np.eye(dim + 1), (5, 1, 1))
    T[3, :dim, dim] = far - Tg[:dim, :dim] @ far       # the far pair's truth, expressed about the origin
    T[3, :dim, :dim] = Tg[:dim, :dim]
    T[3, :dim, dim] += Tg[:dim, dim]
    T[4] = Tg
    worst = [0.0, 0.0]
    for TT in (T, _perturb(T, dim, 5, deg=0.5, shift=0.05)):
        _check_teacher_forced(b.eng, b.srcs, b.tgts, TT, dim, storage, qmap, worst)
    q = b.eng.evaluate(T)
    n = _np(q.n_inliers)
    assert n[0] == 0 and n[1] == 0 and n[2] == 0 and n[3] > 0 and n[4] > 0
    assert np.isfinite(_np(q.H)).all() and np.isfinite(_np(q.b)).all()
    print(f"\n[quality] edge batch dim={dim} {storage}: max block err H {worst[0]:.3e} b {worst[1]:.3e}")


# ------------------------------------------------------------------------------------------------
# 2. convention: b = -1/2 grad f, H_vv = 1/2 d2f/dv2, Open3D's information matrix
# ------------------------------------------------------------------------------------------------
def _frozen(eng, src, tgt, T, dim):
    idx, _, W = (_np(x) for x in eng.correspond(T[None]))
    g = idx >= 0
    p, q, W = src[g], tgt[idx[g]], W[g]

    def f(xi):
        if dim == 3:
            w = xi[:3]
            a = np.linalg.norm(w)
            K = QO.skew(w / a) if a > 0 else np.zeros((3, 3))
            R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
            v = xi[3:]
        else:
            R = np.array([[np.cos(xi[0]), -np.sin(xi[0])], [np.sin(xi[0]), np.cos(xi[0])]])
            v = xi[1:]
        pp = (p @ T[:dim, :dim].T + T[:dim, dim]) @ R.T + v
        e = q - pp
        return float(np.einsum("nk,nkl,nl->", e, W, e))
    return f, g.sum()


@pytest.mark.parametrize("dim", [2, 3])
def test_convention_against_finite_differences(dim):
    if dim == 3:
        src, tgt, _ = _moved(n=1500)
        params = P3
    else:
        src, tgt, _ = _obstacle()
        params = P2
    src, tgt = np.asarray(src, np.float64), np.asarray(tgt, np.float64)
    eng = _engine(dim, "f64", src, tgt, **params)
    eng.set_robust_kernel("cauchy", scale=0.5 if dim == 3 else 5.0)
    T = _perturb(_np(eng.register(history=False).T), dim, 9, deg=1.0, shift=0.2)[0]
    q = eng.evaluate(T[None])
    H, b = _np(q.H)[0], _np(q.b)[0]
    f, n = _frozen(eng, src, tgt, T, dim)
    assert n > 100
    k = QO.npar(dim)
    grad = np.zeros(k)
    for i in range(k):
        h = 1e-6 if i < k - dim else 1e-4
        e = np.zeros(k)
        e[i] = h
        grad[i] = (f(e) - f(-e)) / (2 * h)
    assert np.linalg.norm(b + 0.5 * grad) <= 1e-6 * np.linalg.norm(b), (b, -0.5 * grad)
    # translation enters linearly: f is quadratic in v, so the second difference is exact up to rounding
    hv = 1e-2
    for i in range(k - dim, k):
        for j in range(k - dim, k):
            ei, ej = np.zeros(k), np.zeros(k)
            ei[i], ej[j] = hv, hv
            d2 = (f(ei + ej) - f(ei - ej) - f(-ei + ej) + f(-ei - ej)) / (4 * hv * hv)
            assert abs(H[i, j] - 0.5 * d2) <= 1e-6 * np.abs(H[k - dim:, k - dim:]).max(), (i, j, H[i, j], 0.5 * d2)


def test_point_to_point_information_is_open3d_s():
    src, tgt, _ = _moved(n=1500)
    src, tgt = np.asarray(src, np.float64), np.asarray(tgt, np.float64)
    eng = _engine(3, "f64", src, tgt, covariance_model=1, **P3)
    T = _np(eng.register(history=False).T)[0]
    idx, _, _ = (_np(x) for x in eng.correspond(T[None]))
    pp = src[idx >= 0] @ T[:3, :3].T + T[:3, 3]
    H = _np(eng.evaluate(T[None]).H)[0]
    assert QO.block_rel_err(H, QO.open3d_information(pp), 3) < 1e-9


# ------------------------------------------------------------------------------------------------
# 3. consistency with the loop: n at T_hist[k] is the loop's inlier count of iteration k
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", ["1", "0"])
@pytest.mark.parametrize("dim", [2, 3])
def test_inliers_of_every_iteration(dim, fused, env):
    from generalized_icp_b200 import synthetic
    if dim == 3:
        pairs = [synthetic.patches3d_pair(n=1500, n_patches=8, cube=30.0, patch=20.0, seed=s) for s in range(3)]
        params = P3
    else:
        s0, t0, _ = _obstacle()
        pairs = [(s0, t0, None), (t0, s0, None)]
        params = P2
    b = Batch(dim, "f32", [p[0] for p in pairs], [p[1] for p in pairs], **params)
    r = env(b.register, GICP_FUSED_LOOP=fused)
    n_outer, inl, T_hist = _np(r.n_outer), _np(r.inliers), _np(r.T_hist)
    assert n_outer.min() >= 2
    for k in range(int(n_outer.max())):
        T = np.where(np.isnan(T_hist[:, k]), np.eye(dim + 1), T_hist[:, k])
        n = _np(env(lambda: b.eng.evaluate(np.ascontiguousarray(T)).n_inliers, GICP_FUSED_LOOP=fused))
        live = k < n_outer
        assert np.array_equal(n[live], inl[live, k]), (k, n, inl[:, k])


# ------------------------------------------------------------------------------------------------
# 4. device resident, non-intrusive, batches
# ------------------------------------------------------------------------------------------------
def _qbits(q):
    return [np.ascontiguousarray(_np(x)).view(np.uint8) for x in (q.n_inliers, q.fitness, q.inlier_rmse, q.loss, q.H, q.b)]


def _same_q(a, b, what=""):
    for x, y in zip(_qbits(a), _qbits(b)):
        assert np.array_equal(x, y), what


@pytest.mark.parametrize("fused", ["1", "0"])
def test_evaluate_reads_the_device_T_in_stream_order(fused, env):
    import torch
    src, tgt, _ = _moved(n=1500)
    eng = _engine(3, "f32", src, tgt, **P3)

    def run():
        r = eng.register(history=False)
        q_dev = eng.evaluate(r.T)              # no host synchronisation in between
        torch.cuda.synchronize()
        return r, q_dev
    r, q_dev = env(run, GICP_FUSED_LOOP=fused)
    _same_q(q_dev, eng.evaluate(_np(r.T)), fused)
    assert int(q_dev.n_inliers[0]) > 0


@pytest.mark.parametrize("fused", ["1", "0"])
def test_register_is_unchanged_by_evaluate(fused, env):
    import torch
    src, tgt, _ = _moved(n=1500)
    b = Batch(3, "f32", [src], [tgt], **P3)
    eng = b.eng
    eng.set_robust_kernel("tukey", adaptive=2.0, min_scale=0.05)

    def run():
        b.setup()
        r0 = b.register()
        eng.evaluate(_perturb(_np(r0.T), 3, 1))
        r1 = b.register()                      # register after evaluate
        b.setup()
        eng.evaluate(_np(r0.T))                # evaluate between the set-up and register
        r2 = b.register()
        torch.cuda.synchronize()
        return r0, r1, r2
    r0, r1, r2 = env(run, GICP_FUSED_LOOP=fused)
    _same_bits(r0, r1, "after evaluate")
    _same_bits(r0, r2, "evaluate after set-up")


@pytest.mark.parametrize("storage", ["f32", "f64"])
def test_batch_rows_equal_single_pairs(storage):
    from generalized_icp_b200 import synthetic
    srcs, tgts = [], []
    for seed in range(4):
        s, t, _ = synthetic.patches3d_pair(n=3000, n_patches=8, cube=30.0, patch=20.0, seed=seed, moved_patches=1,
                                           moved_offset=1.0)
        srcs.append(s)
        tgts.append(t)
    b = Batch(3, storage, srcs, tgts, **P3)
    T = _np(b.register().T)
    qb = b.eng.evaluate(T)
    for p in range(4):
        one = Batch(3, storage, [srcs[p]], [tgts[p]], **P3)
        q1 = one.eng.evaluate(T[p:p + 1])
        # every cloud has 3000 points: the same grids and block partition in the batch and alone, so the same bits
        for x, y in zip(_qbits(qb), _qbits(q1)):
            rows = len(x) // 4
            assert np.array_equal(x[p * rows:(p + 1) * rows], y), p


# ------------------------------------------------------------------------------------------------
# 5. does it tell the user something?
# ------------------------------------------------------------------------------------------------
def _sample_planes(rng, planes, density):
    pts = []
    for origin, u, v in planes:
        origin, u, v = (np.asarray(x, np.float64) for x in (origin, u, v))
        n = int(density * np.linalg.norm(u) * np.linalg.norm(v))
        ab = rng.uniform(0, 1, size=(n, 2))
        pts.append(origin + ab[:, :1] * u + ab[:, 1:] * v)
    return np.concatenate(pts) + rng.normal(0, 0.01, size=(sum(len(p) for p in pts), 3))


def _translation_block_eig(planes):
    rng = np.random.default_rng(0)
    src, tgt = _sample_planes(rng, planes, 20.0), _sample_planes(rng, planes, 20.0)
    eng = _engine(3, "f64", src, tgt, **P3)
    H = _np(eng.evaluate(np.eye(4)[None]).H)[0]
    lam, vec = np.linalg.eigh(H[3:, 3:])
    return lam, vec[:, 0]


def test_corridor_is_degenerate_along_its_axis_and_a_room_is_not():
    L, w, h = 40.0, 4.0, 3.0
    corridor = [((0, -w / 2, 0), (L, 0, 0), (0, w, 0)),                  # floor
                ((0, -w / 2, 0), (L, 0, 0), (0, 0, h)),                  # two walls along x
                ((0, w / 2, 0), (L, 0, 0), (0, 0, h))]
    lam_c, v_c = _translation_block_eig(corridor)
    angle = np.degrees(np.arccos(min(1.0, abs(v_c[0]))))
    assert angle < 3.0, (angle, v_c)
    room = [((0, -w / 2, 0), (w, 0, 0), (0, w, 0)),                     # a closed w x w x h room: floor, four walls
            ((0, -w / 2, 0), (w, 0, 0), (0, 0, h)), ((0, w / 2, 0), (w, 0, 0), (0, 0, h)),
            ((0, -w / 2, 0), (0, w, 0), (0, 0, h)), ((w, -w / 2, 0), (0, w, 0), (0, 0, h))]
    lam_r, _ = _translation_block_eig(room)
    cond_c, cond_r = lam_c[-1] / lam_c[0], lam_r[-1] / lam_r[0]
    print(f"\n[quality] translation-block condition: corridor {cond_c:.2f} (axis off by {angle:.2f} deg), room {cond_r:.2f}")
    assert cond_c > 3.0 * cond_r, (cond_c, cond_r)


def test_wrong_pose_has_lower_fitness_and_higher_rmse():
    src, tgt, _ = _moved(n=3000)
    eng = _engine(3, "f32", src, tgt, **P3)
    T = _np(eng.register(history=False).T)
    wrong = _perturb(T, 3, 2, deg=3.0, shift=0.0)
    wrong[0, :3, 3] += 1.0                      # 1 m along every axis and 3 degrees off
    good, bad = eng.evaluate(T), eng.evaluate(wrong)
    assert float(bad.fitness[0]) < float(good.fitness[0])
    assert float(bad.inlier_rmse[0]) > float(good.inlier_rmse[0])
    assert float(good.fitness[0]) > 0.5


# ------------------------------------------------------------------------------------------------
# 6. compat and odometry
# ------------------------------------------------------------------------------------------------
def test_compat_evaluate_reports_the_engine_values_and_keeps_the_default():
    import torch
    from generalized_icp_b200 import compat
    src, tgt, _ = _obstacle()
    kw = dict(max_distance_nearest_neighbors=200, tolerance=1)
    base = compat.gicp_extended(src, tgt, **kw)
    ext = compat.gicp_extended(src, tgt, evaluate=True, **kw)
    for k in ("T", "n_outer", "converged_at", "loss_hist", "inliers", "src_cov0", "tgt_cov"):
        assert np.array_equal(np.asarray(base[k]), np.asarray(ext[k])), k
    assert all(np.array_equal(a, b) for a, b in zip(base["all_T"], ext["all_T"]))
    assert "fitness" not in base
    eng = compat._engine(2, "f64")
    q = eng.evaluate(ext["T"][None])
    torch.cuda.synchronize()
    assert ext["n_inliers"] == int(q.n_inliers[0]) and ext["fitness"] == float(q.fitness[0])
    assert ext["inlier_rmse"] == float(q.inlier_rmse[0])
    assert np.array_equal(ext["information"], _np(q.H)[0]) and np.array_equal(ext["gradient"], -2.0 * _np(q.b)[0])


def test_odometry_evaluate_reports_the_engine_values_and_keeps_the_default():
    import sys
    import os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import demo_inputs
    from generalized_icp_b200.odometry import ScanOdometry
    scans, _ = demo_inputs.lidar_sequence(seed=0, num_rays=360, n_scans=5)
    plain, ev = ScanOdometry(), ScanOdometry(evaluate=True)
    for s in scans:
        a, b = plain.push(s), ev.push(s)
        if a is None:
            continue
        assert np.array_equal(a, b)
        q = ev.eng.evaluate(b[None])           # the pair just registered is still set up
        got = ev.quality[-1]
        assert got["n_inliers"] == int(q.n_inliers[0]) and got["fitness"] == float(q.fitness[0])
        assert got["inlier_rmse"] == float(q.inlier_rmse[0]) and got["loss"] == float(q.loss[0])
        assert np.array_equal(got["H"], _np(q.H)[0]) and np.array_equal(got["b"], _np(q.b)[0])
    assert plain.iterations == ev.iterations and len(ev.quality) == len(scans) - 1 and plain.quality == []
