"""The objective stages at the block shapes large batches run: 5 to 32 points per thread, against float64 references.

plan_loop (csrc/plan.h) sizes the accumulation from max_n * n_clouds: acc_ppt = clamp(max_n * n_clouds / (148 * 8 *
128), 1, 32), and the search split, the blocks per pair and the partial fold follow from it.  The stage entry points run
K3a and K3b at acc_ppt itself (up to 32 points per thread, unsplit at 17, 23, 31).  Every batch of more than 2.6 M
source points - the benchmark's 4096 x 32768 and the 2^24-point config-5 pair among them - runs at acc_ppt 17..32, where
the f32 accumulation sums up to 32 terms per thread and a 32-lane fp32 butterfly before anything is fp64.

Because the plan looks at max_n * n_clouds and not at the real point count, a few full-size pairs plus cheap filler
pairs reach any acc_ppt.  ROWS below does that: the p-rows share one set of full pairs (same tensors, same grids: the
cell budget depends only on max_n, which tests/test_plan_host.py checks together with every row's plan), the fillers
put pair ends on every kind of block edge.

Checks:
A. gicpNormalEquations slot by slot against float64 numpy on gicpCorrespond's matches at the same T and the device's
   own covariances, at the identity, the generating motion and a perturbed pose, within a bound derived from how K3b
   sums (see reference_form); count exact, loss to 1e-12, mu bit for bit (0 for an empty target).
B. The full pairs' matches bit-identical across p5 .. p32, their reduced forms within the two rows' bounds.
C. The loop (check_loop) on p8, p17, p23, p32 (f32, f64), fold32 and 2d32, and end to end against the float64 oracle.
D. Exact alternatives (search split, no skip, no active list) bit-identical at p17 and p32.
E. Robust kernels: the adaptive scale bit for bit, the weighted form within the bound, the weighted loop.
F. gicpEvaluate's count and loss against the reduced form at p32."""
import functools
import time

import numpy as np
import pytest

from test_gpu_inner_minimum import kernel_weights
from test_gpu_search_exactness import Batch, _pair2d, _rot_about, _same_bits, check_loop, env, exact_nn  # noqa: F401

pytestmark = pytest.mark.gpu

N_FULL = 32768
P3 = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=2.0, tolerance=1e-6, max_iterations=40)
P2 = dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=5.0, max_iterations=15)
N_2D = 2049                                 # > SMALL_GRID_MAX / the fused loop's 2048: the multi-launch 2-D loop


# ------------------------------------------------------------------------------------------------
# the row table (pure Python: tests/test_plan_host.py imports it without a GPU)
# ------------------------------------------------------------------------------------------------
def _fillers(ppt, bpp, max_n, n):
    """n filler pairs (n_src, n_tgt): empty source, empty target, 1, 127, 128, 129, ppt*128 - 1, ppt*128, ppt*128 + 1
    and bpp*ppt*128 - 1 points (those below max_n), then 64-point pairs."""
    edge = [ppt * 128 - 1, ppt * 128, ppt * 128 + 1, bpp * ppt * 128 - 1]
    sizes = [(0, 500), (500, 0)] + [(m, m) for m in [1, 127, 128, 129] + edge if m < max_n]
    sizes = list(dict.fromkeys(sizes))
    sizes += [(64, 64)] * (n - len(sizes))
    return sizes[:n]


# name: (dim, storage, full pairs, n_clouds, kernel, plan (acc_ppt, search_ppt, search_bpp, bpp, presum, bpp2,
# active_list)).  kernel: None, ("fixed", kind, c) or ("adaptive", kind, kappa, min_scale)
ROWS = {
    "p5": (3, "f32", 3, 24, None, (5, 5, 52, 52, 0, 1, 0)),
    "p8": (3, "f32", 3, 37, None, (8, 4, 64, 32, 0, 1, 0)),
    "p16": (3, "f32", 3, 74, None, (16, 8, 32, 16, 0, 1, 1)),
    "p17": (3, "f32", 3, 79, None, (17, 17, 16, 16, 0, 1, 1)),
    "p21": (3, "f32", 3, 98, None, (21, 7, 39, 13, 0, 1, 1)),
    "p23": (3, "f64", 3, 107, None, (23, 23, 12, 12, 0, 1, 1)),
    "p31": (3, "f32", 3, 144, ("fixed", "huber", 0.1), (31, 31, 9, 9, 0, 1, 1)),
    "p32": (3, "f32", 3, 148, None, (32, 8, 32, 8, 0, 1, 1)),
    "p32_f64": (3, "f64", 3, 148, None, (32, 8, 32, 8, 0, 1, 1)),
    "p32_tukey": (3, "f32", 3, 148, ("adaptive", "tukey", 4.0, 0.05), (32, 8, 32, 8, 0, 1, 1)),
    "p32_far": (3, "f32", 3, 148, None, (32, 8, 32, 8, 0, 1, 1)),
    "fold32": (3, "f32", 1, 9, None, (32, 8, 588, 147, 1, 3, 0)),
    "2d32_f32": (2, "f32", 3, 2367, None, (32, 8, 4, 1, 0, 1, 1)),
    "2d32_f64": (2, "f64", 3, 2367, None, (32, 8, 4, 1, 0, 1, 1)),
}
FOLD_N = 600_000
# p32_far: the p32 pairs FAR from the origin (then rounded to f32): pt = p' - mu must be formed in fp64 before it is
# rounded, else the rounding of p' (1 ms at 1e4 m) swamps the centred coordinates
FAR = np.array([1e4, -3e3, 500.0])
P_ROWS = [r for r in ROWS if r.startswith("p")]
# the batches bench.py times by default and the config-5 pair: sizes only, for the plan check
BENCH_PAIRS, CONFIG5_N = 4096, 1 << 24
BENCH_PLAN = (32, 8, 32, 8, 0, 1, 1)
CONFIG5_PLAN = (32, 8, 16384, 4096, 1, 64, 0)


def row_sizes(name):
    """[(n_src, n_tgt)] of every pair of the row, full pairs first."""
    dim, _, n_full, n_clouds, _, plan = ROWS[name]
    ppt, bpp = plan[0], plan[3]
    full_n = N_2D if dim == 2 else FOLD_N if name == "fold32" else N_FULL
    return [(full_n, full_n)] * n_full + _fillers(ppt, bpp, full_n, n_clouds - n_full)


def row_params(name):
    return P2 if ROWS[name][0] == 2 else P3


# ------------------------------------------------------------------------------------------------
# data
# ------------------------------------------------------------------------------------------------
def _rot2(deg, c):
    th = np.deg2rad(deg)
    T = np.eye(3)
    T[:2, :2] = [[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]
    T[:2, 2] = c - T[:2, :2] @ c
    return T


@functools.lru_cache(maxsize=None)
def _pair(dim, n_src, n_tgt, seed):
    """(src, tgt, T_gen): a 3-D CONFIG4 pair (32768 points: the bench's clouds), a denser small patch pair, the 600 k
    fold pair, or a 2-D wall pair; sliced to the sizes."""
    from generalized_icp_b200 import synthetic
    n = max(n_src, n_tgt, 1)
    if dim == 2:
        rng = np.random.default_rng(seed)
        deg, shift = rng.uniform(-3, 3), rng.uniform(-1, 1, 2)
        s, t = _pair2d(rng, n, deg, shift)
        Tg = _rot2(deg, np.full(2, 50.0))
        Tg[:2, 2] += shift
    elif n == N_FULL:
        s, t, Tg = synthetic.patches3d_pair(**dict(synthetic.CONFIG4, n=n), seed=seed)
    elif n == FOLD_N:
        s, t, Tg = synthetic.patches3d_pair(n=n, n_patches=64, cube=100.0, patch=30.0, seed=seed)
    else:
        s, t, Tg = synthetic.patches3d_pair(n=n, n_patches=3, cube=12.0, patch=10.0, seed=seed)
    return s[:n_src], t[:n_tgt], Tg


def _row_data(name):
    dim = ROWS[name][0]
    srcs, tgts, Tgs = [], [], []
    for i, (ns, nt) in enumerate(row_sizes(name)):
        # the full pairs are the same arrays in every row; fillers are seeded by their size
        s, t, Tg = _pair(dim, ns, nt, 100 + i if i < ROWS[name][2] else 1000 + ns + 7 * nt)
        srcs.append(s)
        tgts.append(t)
        Tgs.append(Tg)
    Tgs = np.stack(Tgs)
    if name == "p32_far":
        Tc = np.eye(4)
        Tc[:3, 3] = FAR
        srcs = [(np.asarray(x, np.float64) + FAR).astype(np.float32) for x in srcs]
        tgts = [(np.asarray(x, np.float64) + FAR).astype(np.float32) for x in tgts]
        Tgs = Tc @ Tgs @ np.linalg.inv(Tc)
    return srcs, tgts, Tgs


def _set_kernel(eng, kernel):
    if kernel is None:
        eng.set_robust_kernel(None)
    elif kernel[0] == "fixed":
        eng.set_robust_kernel(kernel[1], kernel[2])
    else:
        eng.set_robust_kernel(kernel[1], adaptive=kernel[2], min_scale=kernel[3])


@functools.lru_cache(maxsize=None)
def _batch(name):
    srcs, tgts, Tgs = _row_data(name)
    dim, storage = ROWS[name][:2]
    b = Batch(dim, storage, srcs, tgts, **row_params(name))
    _set_kernel(b.eng, ROWS[name][4])
    return b, Tgs


def _transforms(dim, Tgs, offset=0.0):
    """identity, the generating motion, a pose 1 degree (about the cube centre + offset) and 0.15 m off it."""
    n = len(Tgs)
    eye = np.broadcast_to(np.eye(dim + 1), (n, dim + 1, dim + 1)).copy()
    if dim == 3:
        P = _rot_about(np.full(3, 20.0) + offset, 1.0, seed=7)
        P[:3, 3] += [0.1, -0.05, 0.1]
    else:
        P = _rot2(1.0, np.full(2, 50.0))
        P[:2, 2] += [0.1, -0.1]
    return {"identity": eye, "generating": Tgs, "perturbed": P @ Tgs}


# ------------------------------------------------------------------------------------------------
# A: the reduced form against float64
# ------------------------------------------------------------------------------------------------
def _layout(dim):
    NP, NS = dim + 1, dim * (dim + 1) // 2
    NAB = NP * (NP + 1) // 2
    NH = NAB * NS
    return NP, NS, NAB, NH, NH + dim * NP


def _gamma(n, u):
    return n * u / (1 - n * u)


def reference_form(b, p, T, idx, dist, mu, acc_ppt, bpp, c=None, kind=None, chunk=1 << 20):
    """float64 reduced form of pair p at T from the device's matches (idx, dist: the pair's rows of gicpCorrespond) and
    covariances, and the per-slot bound of K3b's error.  Returns (slots (NQ,), bound (NQ,), loss, loss bound, count).

    f32 storage: every term t_i = pt_a pt_b W_cd (or v_c pt_i) takes 4 roundings (pt_a, pt_b, W, the product), then
    acc_ppt sequential fp32 adds and 5 butterfly levels before it is converted to fp64; the fp64 sums after that are
    negligible: |error| <= gamma_{acc_ppt + 9}(2^-24) sum_i |t_i|.  f64 storage: the same with u = 2^-53 and the fp64
    sums over the 4 warps and the bpp blocks added to n.  Both storages: the device forms M = R C_s R^T + C_t and W =
    inv(M) in fp64 in another order than numpy; R C_s R^T cancels in its off-diagonal entries, so the difference is
    absolute, |dM| ~ eps |M|, and to first order |dW_cd| <= 16 eps cond(M) |W|_2 for every entry (an entry that is 0 in
    exact arithmetic, as for the identity covariance of a one-point cloud under a rotation, is not 0 on either side).
    p' = R p + t is formed with FMA on the device, so it may lie 8 ulp of |p'| from numpy's (check_loop's delta).  The
    first-order effect of both on every term is added.  The loss slot is accumulated in fp64: 1e-12 relative plus the
    same p' effect."""
    import robust_oracle as RO
    d = b.dim
    NP, NS, NAB, NH, NQ = _layout(d)
    s0, s1, t0 = b.off_s[p], b.off_s[p + 1], b.off_t[p]
    cs, ct = b.cs, b.ct
    R, tt = T[:d, :d], T[:d, d]
    pairs = [(a, bb) for a in range(NP) for bb in range(a, NP)]
    cds = [(c_, dd) for c_ in range(d) for dd in range(c_, d)]
    f64 = b.storage == "f64"
    n_round = acc_ppt + 9 + ((4 + bpp) if f64 else 0)
    gam = _gamma(n_round, 2.0 ** -53 if f64 else 2.0 ** -24)
    eps = np.finfo(np.float64).eps
    want, absum, extra = np.zeros(NQ), np.zeros(NQ), np.zeros(NQ)
    loss, loss_abs, loss_extra, count = 0.0, 0.0, 0.0, 0
    for c0 in range(s0, s1, chunk):
        c1 = min(s1, c0 + chunk)
        g = idx[c0 - s0:c1 - s0] >= 0
        if not g.any():
            continue
        m = idx[c0 - s0:c1 - s0][g]
        s = b.srcs[p][c0 - s0:c1 - s0][g]
        q = b.tgts[p][m]
        pp = s @ R.T + tt
        M = R @ cs[c0:c1][g] @ R.T + ct[t0 + m]
        W = np.linalg.inv(M)
        ev = np.linalg.eigvalsh(M)
        w = np.ones(len(M)) if kind is None else RO.robust_weight(kind, dist[c0 - s0:c1 - s0][g], c)
        W = w[:, None, None] * W
        werr = 16 * eps * (ev[:, -1] / ev[:, 0]) * w / ev[:, 0]     # |dW_cd| bound: 16 eps cond(M) |W|_2
        e = q - pp
        v = np.einsum("nij,nj->ni", W, e)
        pt = np.concatenate([np.ones((len(pp), 1)), pp - mu], axis=1)
        delta = 8 * eps * np.abs(pp).max(1)                        # |p'_device - p'_numpy| per coordinate
        dpt = np.concatenate([np.zeros((len(pp), 1)), np.repeat(delta[:, None], d, 1)], axis=1)
        Wc = np.stack([W[:, c_, dd] for c_, dd in cds], 1)         # (n, NS)
        for ab, (a, bb) in enumerate(pairs):
            ptab = pt[:, a] * pt[:, bb]
            tv = ptab[:, None] * Wc
            want[ab * NS:(ab + 1) * NS] += tv.sum(0)
            absum[ab * NS:(ab + 1) * NS] += np.abs(tv).sum(0)
            dab = dpt[:, a] * np.abs(pt[:, bb]) + dpt[:, bb] * np.abs(pt[:, a]) + dpt[:, a] * dpt[:, bb]
            extra[ab * NS:(ab + 1) * NS] += (dab[:, None] * np.abs(Wc) + (np.abs(ptab) * werr)[:, None]).sum(0)
        dv = delta[:, None] * np.abs(W).sum(2) + (werr * np.abs(e).sum(1))[:, None]   # |W| |de| + |dW| |e|
        for c_ in range(d):
            tv = v[:, c_:c_ + 1] * pt
            want[NH + c_ * NP:NH + (c_ + 1) * NP] += tv.sum(0)
            absum[NH + c_ * NP:NH + (c_ + 1) * NP] += np.abs(tv).sum(0)
            extra[NH + c_ * NP:NH + (c_ + 1) * NP] += (dv[:, c_:c_ + 1] * np.abs(pt) + np.abs(v[:, c_:c_ + 1]) * dpt
                                                       ).sum(0)
        li = np.einsum("ni,ni->n", e, v)
        loss += li.sum()
        loss_abs += np.abs(li).sum()
        loss_extra += (2 * delta * np.abs(v).sum(1)).sum()
        count += int(g.sum())
    return want, gam * absum + extra, loss, 1e-12 * loss_abs + loss_extra, count


def _mu(tgt, dim):
    """init_state_kernel's centre: 0.5 * (min + max) of the target per axis.  choose_grid (grid.cuh) clamps an empty
    box to [0, 0] before the box is stored, so an empty target is centred at 0."""
    if len(tgt) == 0:
        return np.zeros(dim)
    return 0.5 * (tgt.min(0) + tgt.max(0))


def check_stage(b, T, acc_ppt, bpp, pairs, kernel=None, full=()):
    """Check A at the transforms T (all pairs) for the pairs listed: returns ({pair: (red slots, bound)}, worst
    error / bound ratio, idx, dist).  The pairs in `full` also have their matches checked against exact_nn."""
    d = b.dim
    NP, NS, NAB, NH, NQ = _layout(d)
    idx, dist, _ = b.eng.correspond(T, with_W=False)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    red = b.eng.normal_equations(T)
    scales = b.eng.robust_scales(T) if kernel is not None else None
    d_max = float(b.params["max_distance_correspondence"])
    worst, forms = 0.0, {}
    for p in pairs:
        a0, a1 = b.off_s[p], b.off_s[p + 1]
        pi, pdist = idx[a0:a1], dist[a0:a1]
        mu = _mu(b.tgts[p], d)
        got_mu = red[p, NQ + 2:NQ + 2 + d]
        assert np.array_equal(got_mu.view(np.int64), mu.view(np.int64)), (p, got_mu, mu)
        c = kind = None
        if kernel is not None:
            kind = kernel[1]
            if kernel[0] == "fixed":
                c = kernel[2]
                assert scales[p] == c
            else:
                import adaptive_oracle as AO
                c = AO.scale_at(kernel[2], kernel[3], pi, pdist)
                assert scales[p].view(np.int64) == np.float64(c).view(np.int64), (p, scales[p], c)
        if p in full:
            pp = b.srcs[p] @ T[p, :d, :d].T + T[p, :d, d]
            nn, key, key2 = exact_nn(b.tgts[p], pp)
            ed = np.sqrt(key)
            want_i = np.where(ed > d_max, -1, nn)
            dp = 8 * np.finfo(np.float64).eps * np.abs(pp).max(1)
            ok = ~(key2 - key <= 1e-9 * key + 4 * ed * dp) & ~(np.abs(ed - d_max) <= 1e-9 * d_max + dp)
            assert ok.mean() > 0.99, ok.mean()
            assert np.array_equal(pi[ok], want_i[ok]), (p, np.flatnonzero(pi[ok] != want_i[ok])[:5])
        want, bound, loss, loss_tol, count = reference_form(b, p, T[p], pi, pdist, got_mu, acc_ppt, bpp, c, kind)
        assert int(red[p, NQ + 1]) == count == int((pi >= 0).sum()), (p, red[p, NQ + 1], count)
        assert abs(red[p, NQ] - loss) <= loss_tol, (p, red[p, NQ], loss, loss_tol)
        err = np.abs(red[p, :NQ] - want)
        assert (err <= bound).all(), (p, np.flatnonzero(err > bound), err[err > bound], bound[err > bound])
        if count:
            worst = max(worst, float((err / np.maximum(bound, 1e-300)).max()))
        forms[p] = (red[p].copy(), bound)
    return forms, worst, idx, dist


def _host_copies(b):
    b.cs = b.eng.covariances(0).cpu().numpy()
    b.ct = b.eng.covariances(1).cpu().numpy()


@functools.lru_cache(maxsize=None)
def _stage_results(name):
    """Check A on every pair of the row at the three transforms.  {T name: (forms, worst ratio, full idx, full dist)}"""
    b, Tgs = _batch(name)
    _host_copies(b)
    plan = ROWS[name][5]
    n_full = ROWS[name][2]
    out = {}
    for tname, T in _transforms(b.dim, Tgs, FAR if name == "p32_far" else 0.0).items():
        forms, worst, idx, dist = check_stage(b, T, plan[0], plan[3], range(b.n_pairs), ROWS[name][4],
                                              full=range(n_full))
        n_f = b.off_s[n_full]
        out[tname] = (forms, worst, idx[:n_f].copy(), dist[:n_f].copy())
    return out


STAGE_ROWS = list(ROWS)


@pytest.mark.parametrize("name", STAGE_ROWS)
def test_reduced_form_against_float64(name):
    t0 = time.time()
    res = _stage_results(name)
    ratios = {t: f"{r[1]:.2e}" for t, r in res.items()}
    print(f"{name}: worst error / bound {ratios} ({time.time() - t0:.0f} s)")
    for t, r in res.items():
        assert r[1] > 0 or name.startswith("2d"), (name, t)      # something was compared


# ------------------------------------------------------------------------------------------------
# B: partition invariance of the full pairs
# ------------------------------------------------------------------------------------------------
def test_partition_invariance_of_the_full_pairs():
    """Same full pairs (same tensors, same grids) in p5 .. p32: the exact search's idx and dist bit-identical, the
    reduced forms within the sum of the two rows' bounds, counts equal."""
    rows = [r for r in P_ROWS if r != "p32_far"]
    ref = rows[0]
    base = _stage_results(ref)
    worst = 0.0
    for name in rows[1:]:
        res = _stage_results(name)
        for tname in base:
            f0, _, i0, d0 = base[tname]
            f1, _, i1, d1 = res[tname]
            assert np.array_equal(i0, i1) and np.array_equal(d0.view(np.int64), d1.view(np.int64)), (name, tname)
            if ROWS[name][4] is not None:
                continue                                            # a weighted form: another sum
            for p in range(ROWS[ref][2]):
                (r0, b0), (r1, b1) = f0[p], f1[p]
                NQ = _layout(3)[4]
                assert r0[NQ + 1] == r1[NQ + 1]
                err = np.abs(r0[:NQ] - r1[:NQ])
                assert (err <= b0 + b1).all(), (name, tname, p, np.flatnonzero(err > b0 + b1))
                worst = max(worst, float((err / (b0 + b1)).max()))
    print(f"full pairs across {rows}: worst difference / (sum of bounds) {worst:.2e}")


# ------------------------------------------------------------------------------------------------
# C: the loop
# ------------------------------------------------------------------------------------------------
def _nonconvex(b):
    # a target of one or two points: the frozen objective is not convex in the rotation (check_loop's escape)
    return {p for p in range(b.n_pairs) if 0 < len(b.tgts[p]) <= 2}


def _oracle_e2e(s, t, params, T_dev, n_out, conv, extent, kernel=None):
    import adaptive_oracle as AO
    import robust_oracle as RO
    from oracle import gicp_oracle as O
    s, t = np.asarray(s, np.float64), np.asarray(t, np.float64)
    if kernel is None:
        ref = O.gicp_oracle(s, t, inner="newton", recompute_src_cov=False, record=False, **params)
    else:
        ref = AO.gicp_oracle(s, t, adaptive=kernel[1:], record=False, **params)
    rot, trans = RO.motion_error(T_dev, ref["T"])
    assert n_out == ref["n_outer"], (n_out, ref["n_outer"])
    assert conv == (-1 if ref["converged_at"] is None else ref["converged_at"]), (conv, ref["converged_at"])
    assert rot <= 1e-5 and trans <= 1e-5 * extent, (rot, trans)
    return rot, trans / extent


LOOP_ROWS = ["p8", "p17", "p23", "p32", "p32_f64", "fold32", "2d32_f32", "2d32_f64"]


@functools.lru_cache(maxsize=None)
def _registered(name):
    b, Tgs = _batch(name)
    return b.register()


@pytest.mark.parametrize("name", LOOP_ROWS)
def test_loop_every_iteration(name):
    b, _ = _batch(name)
    r = _registered(name)
    n_out = r.n_outer.cpu().numpy()
    assert (n_out[:ROWS[name][2]] >= 3).all(), n_out[:ROWS[name][2]]
    check_loop(b, r, nonconvex=_nonconvex(b), weight=kernel_weights(b, r, ROWS[name][4]))
    if name in ("p32", "fold32"):
        for p in range(ROWS[name][2]):
            extent = float(np.linalg.norm(b.tgts[p].max(0) - b.tgts[p].min(0)))
            rot, trans = _oracle_e2e(b.srcs[p], b.tgts[p], b.params, r.T[p].cpu().numpy(), int(r.n_outer[p]),
                                     int(r.converged_at[p]), extent)
            print(f"{name} pair {p}: n_outer {int(r.n_outer[p])}, vs oracle {rot:.1e} rad {trans:.1e} extent")


def test_p32_full_pairs_alone():
    """The p32 full pairs registered as their own 3-pair batch (1 point per thread): same iteration counts and
    convergence, transforms within the north-star tolerance of their p32 results (the fp32 sums differ)."""
    import robust_oracle as RO
    b, _ = _batch("p32")
    r = _registered("p32")
    n = ROWS["p32"][2]
    one = Batch(3, "f32", b.srcs[:n], b.tgts[:n], **P3)
    ro = one.register()
    assert np.array_equal(ro.n_outer.cpu().numpy(), r.n_outer.cpu().numpy()[:n])
    assert np.array_equal(ro.converged_at.cpu().numpy(), r.converged_at.cpu().numpy()[:n])
    for p in range(n):
        rot, trans = RO.motion_error(ro.T[p].cpu().numpy(), r.T[p].cpu().numpy())
        print(f"p32 pair {p} alone vs in p32: {rot:.2e} rad, {trans:.2e} m")
        assert rot <= 1e-5 and trans <= 1e-5 * 40.0, (p, rot, trans)


# ------------------------------------------------------------------------------------------------
# D: exact alternatives
# ------------------------------------------------------------------------------------------------
# GICP_CORR_SPLIT values that do change the search block: 17 -> 1 point per thread at p17, 8 / 32 -> 4 / 1 at p32
ALTERNATIVES = {"p17": [{"GICP_CORR_SPLIT": "1"}, {"GICP_CORR_SPLIT": "4"}, {"GICP_CORR_SPLIT": "17"}],
                "p32": [{"GICP_CORR_SPLIT": "1"}, {"GICP_CORR_SPLIT": "4"}, {"GICP_CORR_SPLIT": "8"},
                        {"GICP_CORR_SPLIT": "32"}]}


@pytest.mark.parametrize("name", ["p17", "p32"])
def test_exact_alternatives(name, env):
    b, _ = _batch(name)
    ref = _registered(name)
    for sw in ALTERNATIVES[name] + [{"GICP_NO_SKIP": "1"}, {"GICP_ACTIVE_LIST": "0"}]:
        _same_bits(ref, env(b.register, **sw), sw)


# ------------------------------------------------------------------------------------------------
# E: robust kernels (the scales and weighted forms are checked by check_stage in test A)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["p31", "p32_tukey"])
def test_robust_loop(name):
    b, _ = _batch(name)
    r = b.register()
    check_loop(b, r, nonconvex=_nonconvex(b), weight=kernel_weights(b, r, ROWS[name][4]))
    if ROWS[name][4][0] == "adaptive":
        p = 0
        extent = float(np.linalg.norm(b.tgts[p].max(0) - b.tgts[p].min(0)))
        _oracle_e2e(b.srcs[p], b.tgts[p], b.params, r.T[p].cpu().numpy(), int(r.n_outer[p]),
                    int(r.converged_at[p]), extent, ROWS[name][4])


# ------------------------------------------------------------------------------------------------
# F: evaluate
# ------------------------------------------------------------------------------------------------
def test_evaluate_matches_the_reduced_form():
    b, Tgs = _batch("p32")
    NQ = _layout(3)[4]
    for T in _transforms(3, Tgs).values():
        red = b.eng.normal_equations(T)
        q = b.eng.evaluate(T)
        assert np.array_equal(q.n_inliers.cpu().numpy(), red[:, NQ + 1].astype(np.int32))
        assert np.array_equal(q.loss.cpu().numpy().view(np.int64), red[:, NQ].view(np.int64))


# ------------------------------------------------------------------------------------------------
# the benchmark's batch and the config-5 pair
# ------------------------------------------------------------------------------------------------
def _device_batch(src, tgt, off, params):
    """A Batch over device tensors that keeps host copies of only the sampled pairs."""
    from generalized_icp_b200.engine import GicpEngine
    b = Batch.__new__(Batch)
    b.dim, b.storage, b.params = 3, "f32", params
    b.eng = GicpEngine(3, "f32")
    b.eng.set_params(**params)
    b.eng.set_target(tgt, off)
    b.eng.set_source(src, off)
    b.off_s = b.off_t = np.asarray(off, np.int64)
    return b


def test_bench_batch_sampled():
    """bench.py's default batch (same generator call and seed, 4096 x 32768, acc_ppt 32): check A on three sampled
    pairs at the three transforms, the whole registration, and those pairs end to end against the float64 oracle."""
    import torch
    from generalized_icp_b200 import synthetic
    cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
    src, tgt, off, T_true = synthetic.patches3d_batch_device(BENCH_PAIRS, n=N_FULL, seed=0, device="cuda", **cfg)
    off = off.cpu().numpy()
    b = _device_batch(src, tgt, off, synthetic.CONFIG4_PARAMS)
    sample = (0, 1777, 4095)
    b.srcs = {p: src[off[p]:off[p + 1]].double().cpu().numpy() for p in sample}
    b.tgts = {p: tgt[off[p]:off[p + 1]].double().cpu().numpy() for p in sample}
    # covariances of the sampled pairs only, at their global rows
    cs, ct = b.eng.covariances(0), b.eng.covariances(1)
    worst = {}
    for tname, T in _transforms(3, T_true.cpu().numpy()).items():
        idx, dist, _ = b.eng.correspond(T, with_W=False)
        red = b.eng.normal_equations(T)
        for p in sample:
            a0, a1 = int(off[p]), int(off[p + 1])
            pi, pdist = idx[a0:a1].cpu().numpy(), dist[a0:a1].cpu().numpy()
            # reference_form indexes the covariances by global row: give it the pair's rows at offset 0
            sub = Batch.__new__(Batch)
            sub.dim, sub.storage, sub.params = 3, "f32", b.params
            sub.srcs, sub.tgts = [b.srcs[p]], [b.tgts[p]]
            sub.off_s = sub.off_t = np.array([0, a1 - a0])
            sub.cs, sub.ct = cs[a0:a1].cpu().numpy(), ct[a0:a1].cpu().numpy()
            NQ = _layout(3)[4]
            mu = red[p, NQ + 2:NQ + 5]
            assert np.array_equal(mu.view(np.int64), _mu(b.tgts[p], 3).view(np.int64))
            want, bound, loss, loss_tol, count = reference_form(sub, 0, T[p], pi, pdist, mu, BENCH_PLAN[0], BENCH_PLAN[3])
            assert int(red[p, NQ + 1]) == count
            assert abs(red[p, NQ] - loss) <= loss_tol
            err = np.abs(red[p, :NQ] - want)
            assert (err <= bound).all(), (tname, p, np.flatnonzero(err > bound))
            worst[tname] = max(worst.get(tname, 0.0), float((err / bound).max()))
    print(f"bench: worst error / bound {worst}")
    r = b.eng.register(history=False)
    torch.cuda.synchronize()
    for p in sample:
        _oracle_e2e(b.srcs[p], b.tgts[p], synthetic.CONFIG4_PARAMS, r.T[p].cpu().numpy(), int(r.n_outer[p]),
                    int(r.converged_at[p]), synthetic.CONFIG4["cube"])


def test_config5_pair_stages():
    """One CONFIG5 pair of 2^24 points per side (acc_ppt 32, 4096 blocks per pair): check A at the identity and the
    generating motion, the reference summed in chunks of 2^20 points."""
    from generalized_icp_b200 import synthetic
    s, t, Tg = synthetic.patches3d_pair(**synthetic.CONFIG5, seed=3)
    assert len(s) == CONFIG5_N
    b = Batch(3, "f32", [s], [t], **synthetic.CONFIG5_PARAMS)
    _host_copies(b)
    worst = {}
    for tname in ("identity", "generating"):
        T = (np.eye(4) if tname == "identity" else Tg)[None]
        _, worst[tname], _, _ = check_stage(b, T, CONFIG5_PLAN[0], CONFIG5_PLAN[3], [0])
    print(f"config5: worst error / bound {worst}")
