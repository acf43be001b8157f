"""Exactness of every correspondence-search path of the registration loop (K3a inside gicpRegister), iteration by
iteration, against exact float64 references.

The stage entry points (gicpKnn, gicpCorrespond) always search from scratch; the loop additionally skips points
whose match cannot have changed (slack bound), seeds tracked lanes with the previous match and compacts the still
active pairs.  These tests pin the loop's matches to an exact 1-NN at every executed iteration (through the
inlier count and the frozen objective the solver minimised), require every diagnostic switch that DESIGN calls an
exact alternative to give bit-identical results, and feed the grid searches adversarial geometry: lattices with
exact ties on cell faces, distances exactly equal to the k-NN radius or the correspondence gate, clouds far from
the origin, size boundaries between kernels and degenerate extents.

Exact 1-NN reference: cKDTree candidates re-ranked by the oracle's float64 key (dx*dx + dy*dy) + dz*dz, then by
index.  Under a general rotation the device's p' = R p + t is computed with FMA contraction and may differ from
numpy's in the last bits, so indices are compared only where the best and second-best keys differ by more than
1e-9 relative plus what a few ulp of |p'| can change (elsewhere the distances must agree to 1e-9 relative plus
that much).  The lattice tests use R = I and dyadic
translations, where every coordinate is exact on both sides and every tie must go to the lower index."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SWITCHES = ("GICP_NO_SKIP", "GICP_TRACK_CELLS", "GICP_SHELL_SEARCH", "GICP_CENTRE_FIRST", "GICP_CORR_SPLIT",
            "GICP_ACTIVE_LIST", "GICP_FUSED_LOOP")
# every alternative DESIGN section 4 calls exact: the loop's results must not change in a single bit
EXACT_ALTERNATIVES = [{"GICP_NO_SKIP": "1"}, {"GICP_TRACK_CELLS": "0"}, {"GICP_TRACK_CELLS": "1"},
                      {"GICP_TRACK_CELLS": "8"}, {"GICP_SHELL_SEARCH": "0"}, {"GICP_CENTRE_FIRST": "0"},
                      {"GICP_CORR_SPLIT": "1"}, {"GICP_CORR_SPLIT": "4"}, {"GICP_ACTIVE_LIST": "0"}]


@pytest.fixture()
def env():
    """env(fn, **switches): run fn with the library's switches set (it re-reads them on every call), then restore
    whatever was set before, also when fn raises."""
    saved = {k: os.environ.get(k) for k in SWITCHES}

    def restore():
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    def run(fn, **kw):
        try:
            for k, v in kw.items():
                os.environ[k] = str(v)
            return fn()
        finally:
            restore()

    yield run
    restore()


# ------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------
def _keys(tgt, q, cand):
    d = tgt[cand] - q[:, None, :]
    k = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
    if tgt.shape[1] == 3:
        k = k + d[..., 2] * d[..., 2]
    return k


def exact_nn(tgt, q):
    """Exact 1-NN of every query under the oracle's rule (float64 key, then lower index).
    Returns (idx (M,), key (M,), key of the runner-up (M,)); idx = -1 and inf keys for an empty target."""
    from scipy.spatial import cKDTree
    from oracle import gicp_oracle as O
    m, n = len(q), len(tgt)
    if n == 0:
        return np.full(m, -1), np.full(m, np.inf), np.full(m, np.inf)
    kk = min(8, n)
    _, cand = cKDTree(tgt).query(q, k=kk, workers=-1)
    cand = cand.reshape(m, kk)
    key = _keys(tgt, q, cand)
    order = np.lexsort((cand, key), axis=-1)
    cand = np.take_along_axis(cand, order, 1)
    key = np.take_along_axis(key, order, 1)
    idx, best = cand[:, 0].copy(), key[:, 0].copy()
    second = key[:, 1].copy() if kk > 1 else np.full(m, np.inf)
    # every candidate the tree returned ties with the best: the lowest index may lie outside them
    full = (kk < n) & (key[:, -1] <= key[:, 0] * (1 + 1e-12))
    if full.any():
        bi, _ = O.knn_bruteforce(tgt, 2, np.inf, queries=q[full])
        idx[full] = bi[:, 0]
        best[full] = _keys(tgt, q[full], bi[:, :1])[:, 0]
        second[full] = _keys(tgt, q[full], bi[:, 1:2])[:, 0]
    return idx, best, second


def _offset(T, dim):
    from oracle import gicp_oracle as O
    if dim == 2:
        return np.array([T[0, 2], T[1, 2], np.arctan2(T[1, 0], T[0, 0])])
    return np.concatenate([T[:3, 3], O.rotvec_from_matrix(T[:3, :3])])


def _bits(x):
    import torch
    return x.contiguous().view(torch.int64 if x.element_size() == 8 else torch.int32)


def _same_bits(a, b, what=""):
    """torch.equal on every output of register(), bit for bit (NaN rows of the history included)."""
    import torch
    for f in ("T", "n_outer", "converged_at", "T_hist", "loss_hist", "inliers"):
        assert torch.equal(_bits(getattr(a, f)), _bits(getattr(b, f))), (what, f)


class Batch:
    """One engine holding a batch of pairs (host copies of what the engine sees, in float64)."""

    def __init__(self, dim, storage, srcs, tgts, **params):
        import torch
        from generalized_icp_b200.engine import GicpEngine
        self.dim, self.storage = dim, storage
        dt = torch.float32 if storage == "f32" else torch.float64
        np_dt = np.float32 if storage == "f32" else np.float64
        self.srcs = [np.asarray(s, dtype=np_dt).reshape(-1, dim).astype(np.float64) for s in srcs]
        self.tgts = [np.asarray(t, dtype=np_dt).reshape(-1, dim).astype(np.float64) for t in tgts]
        self.off_s = np.concatenate([[0], np.cumsum([len(s) for s in self.srcs])]).astype(np.int64)
        self.off_t = np.concatenate([[0], np.cumsum([len(t) for t in self.tgts])]).astype(np.int64)
        self.S = torch.as_tensor(np.concatenate(self.srcs), device="cuda").to(dt)
        self.T = torch.as_tensor(np.concatenate(self.tgts), device="cuda").to(dt)
        self.eng = GicpEngine(dim, storage)
        self.eng.set_params(**params)
        self.params = params
        self.setup()

    def setup(self):
        self.eng.set_target(self.T, self.off_t)
        self.eng.set_source(self.S, self.off_s)

    @property
    def n_pairs(self):
        return len(self.srcs)

    def register(self, T0=None):
        import torch
        r = self.eng.register(T0=T0, history=True)
        torch.cuda.synchronize()
        return r


def check_loop(b, r, T0=None, nonconvex=()):
    """Part 1: every executed iteration k of every pair against the exact 1-NN of the source under T_hist[k]:
    the stage search's indices, the loop's inlier count, and the loop's min_loss as the frozen objective of the exact
    matches at T_hist[k + 1] (at the converged iteration, where T is not updated: the frozen problem's minimum, found
    by the oracle's Newton solver; for the pairs in `nonconvex` the device only has to do at least as well)."""
    from oracle import gicp_oracle as O
    d, d1 = b.dim, b.dim + 1
    d_max = float(b.params.get("max_distance_correspondence", 150.0))
    rel = 2e-5 if b.storage == "f32" else 1e-9
    cs = b.eng.covariances(0).cpu().numpy()
    ct = b.eng.covariances(1).cpu().numpy()
    T_hist = r.T_hist.cpu().numpy()
    loss = r.loss_hist.cpu().numpy()
    inl = r.inliers.cpu().numpy()
    n_out = r.n_outer.cpu().numpy()
    conv = r.converged_at.cpu().numpy()
    if T0 is not None:
        assert np.array_equal(T_hist[:, 0], np.asarray(T0).reshape(-1, d1, d1))
    for k in range(int(n_out.max())):
        Tk_all = np.where(np.isnan(T_hist[:, k]), np.eye(d1), T_hist[:, k])
        idx_dev, dist_dev, _ = b.eng.correspond(Tk_all, with_W=False)
        idx_dev, dist_dev = idx_dev.cpu().numpy(), dist_dev.cpu().numpy()
        for p in range(b.n_pairs):
            if n_out[p] <= k:
                continue
            s, t = b.srcs[p], b.tgts[p]
            Tk = T_hist[p, k]
            pp = s @ Tk[:d, :d].T + Tk[:d, d]
            idx, key, key2 = exact_nn(t, pp)
            dist = np.sqrt(key)
            want = np.where(dist > d_max, -1, idx)
            gi = idx_dev[b.off_s[p]:b.off_s[p + 1]]
            gd = dist_dev[b.off_s[p]:b.off_s[p + 1]]
            # how far the device's p' may lie from numpy's (FMA contraction: a few ulp of |p'|)
            dp = 8 * np.finfo(np.float64).eps * np.abs(pp).max(1)
            band = key2 - key <= 1e-9 * key + 4 * dist * dp          # near-ties at that level: any of them may win
            gate = np.abs(dist - d_max) <= 1e-9 * d_max + dp          # distances at the gate at that level
            ok = ~band & ~gate
            assert np.array_equal(gi[ok], want[ok]), (p, k, np.flatnonzero(gi[ok] != want[ok])[:5])
            both = (gi >= 0) & (want >= 0)
            assert np.all(np.abs(gd[both] - dist[both]) <= 1e-9 * dist[both] + dp[both]), (p, k)
            m = np.where(ok, want, gi)
            g = m >= 0
            assert inl[p, k] == g.sum(), (p, k, inl[p, k], g.sum())
            Rk = Tk[:d, :d]
            q = t[m[g]]
            W = np.linalg.inv(Rk @ cs[b.off_s[p]:b.off_s[p + 1]][g] @ Rk.T + ct[b.off_t[p]:b.off_t[p + 1]][m[g]])
            if conv[p] == k:
                _, want_loss, _, _ = O.inner_newton(_offset(Tk, d), s[g], q, W)
                tol = max(rel, 1e-8)
            else:
                dT = T_hist[p, k + 1] @ np.linalg.inv(Tk)
                res = q - (pp[g] @ dT[:d, :d].T + dT[:d, d])
                want_loss = float(np.einsum("ni,nij,nj->", res, W, res))
                tol = rel
            if b.storage == "f32":
                # fp32 accumulation of the reduced form: its error scales with the loss at the linearisation point
                e = q - pp[g]
                scale = max(abs(want_loss), float(np.einsum("ni,nij,nj->", e, W, e)))
            else:
                scale = abs(want_loss)
            if conv[p] == k and p in nonconvex:
                assert loss[p, k] <= want_loss + tol * scale + 1e-12, (p, k, loss[p, k], want_loss)
            else:
                assert abs(loss[p, k] - want_loss) <= tol * scale + 1e-12, (p, k, loss[p, k], want_loss)
        # the pairs that stopped: nothing written after their last iteration
    for p in range(b.n_pairs):
        assert np.isnan(loss[p, n_out[p]:]).all() and (inl[p, n_out[p]:] == 0).all()


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def _rot_about(c, deg, seed):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    a = np.deg2rad(deg)
    R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = c - R @ c
    return T


def _walls2d(rng, n, box=100.0, n_seg=12):
    """2-D points on random line segments (scan-like structure, well-defined covariances)."""
    a = rng.uniform(0, box, size=(n_seg, 2))
    b = a + rng.normal(size=(n_seg, 2)) * box / 4
    w = rng.integers(0, n_seg, n)
    u = rng.random(n)[:, None]
    return a[w] + u * (b[w] - a[w]) + rng.normal(0, 0.02, size=(n, 2))


def _pair2d(rng, n, deg, shift, uniform=False, box=100.0):
    src = rng.uniform(0, box, size=(n, 2)) if uniform else _walls2d(rng, n, box)
    th = np.deg2rad(deg)
    R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    tgt = (src - box / 2) @ R.T + box / 2 + shift + rng.normal(0, 0.02, size=(n, 2))
    return src, tgt


P3 = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0, max_iterations=40)


def _case(name):
    """The registrations of part 1 (and the switch matrix of part 2): (dim, storage, srcs, tgts, params, T0)."""
    from generalized_icp_b200 import synthetic
    if name == "3d_fused":
        s, t, Tg = synthetic.patches3d_pair(n=1800, n_patches=4, cube=20.0, patch=15.0, seed=3)
        return 3, "f32", [s], [t], P3, (_rot_about(np.full(3, 10.0), 6.0, seed=9) @ Tg)[None]
    if name in ("3d_f32", "3d_f64"):
        storage = name.split("_")[1]
        srcs, tgts, T0s = [], [], []
        for i, deg in enumerate((5.0, 7.5, 10.0)):
            s, t, Tg = synthetic.patches3d_pair(n=20000 + 1111 * i, n_patches=16, cube=40.0, patch=30.0, seed=40 + i)
            srcs.append(s)
            tgts.append(t)
            T0s.append(_rot_about(np.full(3, 20.0), deg, seed=i) @ Tg)
        return 3, storage, srcs, tgts, P3, np.stack(T0s)
    if name == "2d_multi":
        rng = np.random.default_rng(5)
        s, t = _pair2d(rng, 3000, 4.0, (1.0, -0.5))
        return 2, "f64", [s], [t], dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=5.0,
                                        max_iterations=40), None
    raise KeyError(name)


LOOP_CASES = ["3d_f32", "3d_f64", "2d_multi", "3d_fused"]


# ------------------------------------------------------------------------------------------------
# part 1 + 2: the loop's matches, iteration by iteration, and the exact alternatives
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", LOOP_CASES)
def test_loop_matches_are_exact_every_iteration(case, env):
    dim, storage, srcs, tgts, params, T0 = _case(case)
    b = Batch(dim, storage, srcs, tgts, **params)
    r = b.register(T0)
    n_out = r.n_outer.cpu().numpy()
    assert (n_out >= 3).all(), n_out
    check_loop(b, r, T0)
    # the skip (slack bound, compacted work lists) against searching every point in every iteration
    _same_bits(r, env(lambda: b.register(T0), GICP_NO_SKIP=1))


@pytest.mark.parametrize("case", LOOP_CASES)
def test_exact_alternatives_are_bit_identical(case, env):
    dim, storage, srcs, tgts, params, T0 = _case(case)
    b = Batch(dim, storage, srcs, tgts, **params)
    ref = b.register(T0)
    for sw in EXACT_ALTERNATIVES:
        _same_bits(ref, env(lambda: b.register(T0), **sw), sw)


def _big_batch():
    """1152 small 2-D pairs (more than one 1024-pair chunk of the active-list compaction) that stop at very different
    iterations: empty sources and empty targets (stop at iteration 1), unstructured pairs far apart (most run to
    max_iterations), ordinary scan-like pairs."""
    rng = np.random.default_rng(17)
    srcs, tgts = [], []
    for i in range(1152):
        n = int(rng.integers(350, 800))
        if i % 97 == 3:
            s, t = np.zeros((0, 2)), _walls2d(rng, n)
        elif i % 97 == 5:
            s, t = _walls2d(rng, n), np.zeros((0, 2))
        elif i % 7 == 1:
            s, t = _pair2d(rng, n, rng.uniform(-40, 40), rng.uniform(-8, 8, 2), uniform=True)
        else:
            s, t = _pair2d(rng, n, rng.uniform(-4, 4), rng.uniform(-1.5, 1.5, 2))
        srcs.append(s)
        tgts.append(t)
    return srcs, tgts, dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=6.0,
                            max_iterations=15)


def test_big_batch_active_list_and_exact_alternatives(env):
    """Multi-launch loop over 1152 pairs: the active-pair list is on (>= 64 pairs) and its compaction runs two
    1024-pair chunks; 4 points per thread, so GICP_CORR_SPLIT=1 / 4 really change the search's blocks.  Every exact
    alternative is bit-identical.  Every pair against the same pair registered alone: identical iteration counts and
    inlier counts at every iteration, transforms and losses to rounding - not bit for bit, because a cloud's grid
    (hence its sorted point order, hence the order of the fixed-order sums) follows the cell budget, which is sized
    by the largest cloud of the batch."""
    import torch
    srcs, tgts, params = _big_batch()

    def run():
        b = Batch(2, "f64", srcs, tgts, **params)
        ref = b.register()
        n_out = ref.n_outer.cpu().numpy()
        conv = ref.converged_at.cpu().numpy()
        empty = np.array([len(s) == 0 or len(t) == 0 for s, t in zip(srcs, tgts)])
        assert (conv[empty] == 1).all() and (n_out[empty] == 2).all()
        assert (n_out == params["max_iterations"]).sum() >= 3, np.bincount(n_out)
        assert len(np.unique(n_out)) >= 4, np.bincount(n_out)
        for sw in EXACT_ALTERNATIVES:
            _same_bits(ref, env(b.register, GICP_FUSED_LOOP=0, **sw), sw)
        return ref

    ref = env(run, GICP_FUSED_LOOP=0)
    single = Batch(2, "f64", srcs[:1], tgts[:1], **params)
    for i in range(len(srcs)):
        if len(srcs[i]) == 0 or len(tgts[i]) == 0:
            continue                                  # checked above
        single.S = torch.as_tensor(np.asarray(srcs[i], np.float64), device="cuda")
        single.T = torch.as_tensor(np.asarray(tgts[i], np.float64), device="cuda")
        single.off_s = np.array([0, len(srcs[i])], np.int64)
        single.off_t = np.array([0, len(tgts[i])], np.int64)
        r = env(lambda: (single.setup(), single.register())[1], GICP_FUSED_LOOP=0)
        for f in ("n_outer", "converged_at", "inliers"):
            assert torch.equal(getattr(ref, f)[i], getattr(r, f)[0]), (i, f)
        n = int(r.n_outer[0])
        for f in ("T", "T_hist", "loss_hist"):
            a, c = getattr(ref, f)[i], getattr(r, f)[0]
            if f != "T":
                a, c = a[:n], c[:n]
            assert ((a - c).abs() <= 1e-9 * c.abs().clamp(min=1.0)).all(), (i, f)


# ------------------------------------------------------------------------------------------------
# part 3: adversarial geometry
# ------------------------------------------------------------------------------------------------
def _lattice(n=16, spacing=0.5, planar=False, seed=0):
    g = np.arange(n, dtype=np.float64) * spacing
    if planar:
        x, y = np.meshgrid(np.arange(64) * spacing, np.arange(64) * spacing, indexing="ij")
        pts = np.stack([x.ravel(), y.ravel(), np.full(x.size, 3.0)], 1)
    else:
        x, y, z = np.meshgrid(g, g, g, indexing="ij")
        pts = np.stack([x.ravel(), y.ravel(), z.ravel()], 1)
    return pts[np.random.default_rng(seed).permutation(len(pts))]


def _check_knn(b, pts, k, radius, exact_idx=True):
    from oracle import gicp_oracle as O
    idx, dist = b.eng.knn(1)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    want, wd = O.knn_bruteforce(pts, k, radius)
    want = np.where(want == len(pts), -1, want)
    if exact_idx:
        assert np.array_equal(idx, want), np.argwhere(idx != want)[:5]
    m = want >= 0
    assert np.array_equal(idx >= 0, m)
    assert np.all(np.abs(dist[m] - wd[m]) <= 1e-12 * wd[m])
    return want


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("k,radius", [(20, 2.0), (7, 2.0), (24, 2.0), (25, 2.0), (30, 1.0)])
def test_lattice_knn_ties_on_cell_faces(storage, k, radius):
    """16^3 cubic lattice, spacing 0.5, rows permuted (grid path, not the <= 2048-point kernels); the auto cell size
    r/4 puts every point on cell faces.  k = 20 ends inside the 8-way tie of the sqrt(3)/2 shell, k = 7 inside the
    first shell (6 points at 0.5), k = 24/25 straddle the fast path's limit; with r = 1.0 and k = 30 the 6 points at
    exactly 1.0 are excluded (exclusive radius) and the last 3 slots stay empty."""
    pts = _lattice()
    b = Batch(3, storage, [pts], [pts], k=k, max_distance_nearest_neighbors=radius)
    want = _check_knn(b, pts, k, radius)
    if radius == 1.0:
        assert (want >= 0).sum(1).max() == 27           # itself + 6 + 12 + 8 (shells 0.5, 0.71, 0.87); 1.0 is out


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("k", [5, 9])
def test_planar_lattice_knn_and_covariances(storage, k):
    """The lattice in one plane z = 3 (a grid with one z cell): 4-way ties at k = 5 and k = 9; the normal is well
    defined, so the covariances are compared with the oracle's."""
    from oracle import gicp_oracle as O
    pts = _lattice(planar=True)
    b = Batch(3, storage, [pts], [pts], k=k, max_distance_nearest_neighbors=2.0)
    want = _check_knn(b, pts, k, 2.0)
    cov = b.eng.covariances(1).cpu().numpy()
    cw = O.covariances_from_neighbors(pts, np.where(want < 0, len(pts), want))
    assert np.abs(cov - cw).max() < (2e-4 if storage == "f32" else 1e-9)


SHIFTS = [((0.125, 0.0, 0.0), 1), ((0.25, 0.0, 0.0), 2), ((0.25, 0.25, 0.0), 4), ((0.25, 0.25, 0.25), 8)]


@pytest.mark.parametrize("storage", ["f32", "f64"])
@pytest.mark.parametrize("shift,ways", SHIFTS)
def test_lattice_one_nn_ties_and_the_gate(storage, shift, ways, env):
    """Source = the lattice (another row order) under T = translation by a dyadic shift: tie-free, or 2-, 4- and
    8-way ties between target points that all must resolve to the lowest index.  d_max set exactly to the match
    distance keeps every interior point (strict d > d_max gate), one ulp below it drops them.  Checked through the
    stage search, through the loop's first iteration (inlier count), and skip on / off of a whole registration."""
    from oracle import gicp_oracle as O
    tgt = _lattice(seed=0)
    src = _lattice(seed=1)
    T0 = np.eye(4)
    T0[:3, 3] = shift
    moved = src + np.asarray(shift)
    d_nn = float(np.sqrt(np.sum(np.square(shift))))
    for d_max in (d_nn, np.nextafter(d_nn, 0.0), 1.0):
        b = Batch(3, storage, [src], [tgt], k=20, max_distance_nearest_neighbors=2.0, max_distance_correspondence=d_max,
                  max_iterations=1)
        want, wd = O.correspond(moved, tgt, d_max, method="brute")
        idx, dist, _ = b.eng.correspond(T0, with_W=False)
        idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
        assert np.array_equal(idx, want)
        m = want >= 0
        assert np.all(np.abs(dist[m] - wd[m]) <= 1e-12 * wd[m])
        if d_max == d_nn:
            # the points whose neighbours all lie inside the lattice tie `ways` ways and sit exactly at d_max
            interior = np.all((moved > 0.3) & (moved < 7.2), axis=1)
            assert m[interior].all()
            cnt = np.array([(np.abs(np.sqrt(np.sum((tgt - p) ** 2, 1)) - d_nn) == 0).sum() for p in moved[interior][:50]])
            assert (cnt == ways).all()
        elif d_max < d_nn:
            assert m.sum() == 0
        r = b.register(T0[None])
        assert int(r.inliers[0, 0]) == int(m.sum())
    b = Batch(3, storage, [src], [tgt], k=20, max_distance_nearest_neighbors=2.0, max_distance_correspondence=1.0,
              max_iterations=20)
    r = b.register(T0[None])
    _same_bits(r, env(lambda: b.register(T0[None]), GICP_NO_SKIP=1))
    _same_bits(r, env(lambda: b.register(T0[None]), GICP_TRACK_CELLS=0))


@pytest.mark.parametrize("offset", [(1e4, -3e3, 500.0), (1e5, -3e3, 500.0)])
def test_far_from_origin(offset, env):
    """A patch pair translated far from the origin and rounded to fp32 (at 1e5 m the fp32 ulp is ~8 mm and the filter's
    Pf term dominates its margin): k-NN at k = 20, 1-NN at identity and at the generating transform, every iteration
    of the loop, skip on / off, and the end result against the oracle within the north-star tolerance."""
    from generalized_icp_b200 import synthetic
    from oracle import gicp_oracle as O
    s, t, Tg = synthetic.patches3d_pair(n=6000, n_patches=6, cube=30.0, patch=20.0, seed=21)
    off = np.asarray(offset)
    s = (s.astype(np.float64) + off).astype(np.float32).astype(np.float64)
    t = (t.astype(np.float64) + off).astype(np.float32).astype(np.float64)
    Tc = np.eye(4)
    Tc[:3, 3] = off
    Tgen = Tc @ Tg @ np.linalg.inv(Tc)
    params = dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0, max_iterations=40)
    b = Batch(3, "f32", [s], [t], **params)
    _check_knn(b, t, 20, 4.0)
    for T in (np.eye(4), Tgen):
        moved = s @ T[:3, :3].T + T[:3, 3]
        idx, key, key2 = exact_nn(t, moved)
        want = np.where(np.sqrt(key) > 2.0, -1, idx)
        got, dist, _ = b.eng.correspond(T, with_W=False)
        got, dist = got.cpu().numpy(), dist.cpu().numpy()
        ok = (key2 - key > 1e-9 * key) & (np.abs(np.sqrt(key) - 2.0) > 1e-9 * 2.0)
        assert ok.mean() > 0.99
        assert np.array_equal(got[ok], want[ok])
    r = b.register()
    check_loop(b, r)
    _same_bits(r, env(b.register, GICP_NO_SKIP=1))
    ref = O.gicp_oracle(s, t, inner="newton", recompute_src_cov=False, record=False, knn="brute", **params)
    assert int(r.n_outer[0]) == ref["n_outer"]
    Td = r.T[0].cpu().numpy()
    dR = Td[:3, :3].T @ ref["T"][:3, :3]
    assert np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)) <= 1e-5
    assert np.linalg.norm(Td[:3, 3] - ref["T"][:3, 3]) <= 1e-5 * 30.0


@pytest.mark.parametrize("n", [128, 129, 2048, 2049])
def test_size_boundaries(n, env):
    """Clouds on both sides of the kernel boundaries: brute-force k-NN (<= 128 points), general latency kernel
    (<= 2048), grid fast path; fused loop (<= 2048 source points) and multi-launch loop."""
    from generalized_icp_b200 import synthetic
    s, t, Tg = synthetic.patches3d_pair(n=n, n_patches=3, cube=12.0, patch=10.0, seed=n)
    T0 = (_rot_about(np.full(3, 6.0), 4.0, seed=n) @ Tg)[None]
    b = Batch(3, "f32", [s], [t], k=20, max_distance_nearest_neighbors=3.0, max_distance_correspondence=2.0,
              max_iterations=30)
    _check_knn(b, b.tgts[0], 20, 3.0)
    r = b.register(T0)
    check_loop(b, r, T0)
    _same_bits(r, env(lambda: b.register(T0), GICP_NO_SKIP=1))


def test_degenerate_extents(env):
    """A collinear 3-D cloud, a single-point target, a source entirely farther than d_max from its target (all gated
    out: T stays the identity and the loop stops at iteration 1) and d_max larger than the whole cloud (the ball covers
    every cell), as one batch through the multi-launch loop and each pair alone (the fused loop for the pairs of at
    most 2048 points)."""
    rng = np.random.default_rng(31)
    line = np.outer(rng.uniform(0, 50, 3000), [0.6, 0.0, 0.8]) + [1.0, 2.0, 3.0]
    line_t = line + [0.05, -0.02, 0.01]
    blob = rng.normal(size=(1500, 3)) * 3.0
    single = np.array([[0.5, -0.25, 0.125]])
    far = blob + [500.0, 0.0, 0.0]
    srcs = [line, blob, far, blob]
    tgts = [line_t, single, blob, blob + [0.5, 0.3, -0.2]]
    params = dict(k=6, max_distance_nearest_neighbors=2.0, max_distance_correspondence=100.0, max_iterations=25)
    b = Batch(3, "f64", srcs, tgts, **params)
    for p in (0, 3):
        bb = Batch(3, "f64", [srcs[p]], [srcs[p]], k=6, max_distance_nearest_neighbors=2.0)
        _check_knn(bb, srcs[p], 6, 2.0)
    r = b.register()
    # every source point matches the single target point: the frozen objective is not convex in the rotation, and the
    # device's solver may find a lower minimum than the oracle's Newton iteration
    check_loop(b, r, nonconvex={1})
    assert np.array_equal(r.T[2].cpu().numpy(), np.eye(4))
    assert int(r.converged_at[2]) == 1 and (r.inliers[2].cpu().numpy() == 0).all()
    for sw in EXACT_ALTERNATIVES:
        _same_bits(r, env(b.register, **sw), sw)
    for p in range(4):
        one = Batch(3, "f64", [srcs[p]], [tgts[p]], **params)
        ro = one.register()
        check_loop(one, ro, nonconvex={0} if p == 1 else ())
        _same_bits(ro, env(one.register, GICP_NO_SKIP=1))
