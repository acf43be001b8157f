"""Every executed outer iteration's inner solve (K4, csrc/solve.cuh) reaches the minimum of its frozen problem, over
every loop instantiation the library compiles.

check_loop (test_gpu_search_exactness) pins each iteration's matches and asserts that min_loss is the frozen objective
at T_hist[k + 1]: consistency, which a solve that stops early or takes a wrong step still passes.  check_inner_minimum
rebuilds frozen problem k from the exact matches at T_hist[k], the device's own covariances and the kernel's weights,
and asserts at T_hist[k + 1], from per-point float64 residuals:
- the gradient certificate (f64 storage): |J^T w W r| <= 1e-7 of sum_i |J_i^T w_i W_i e_i| at T_hist[k];
- the value: F(T_hist[k + 1]) <= the oracle's Newton minimum + tol * max(that minimum, F(T_hist[k])), tol = 1e-9 for
  f64 and 2e-5 for f32 (check_loop's f32 bound: with f32 storage the solver minimises the f32-accumulated form, so
  only the value bound applies).
Both are inequalities, so a non-convex frozen problem (check_loop's single-point targets) needs no escape here.

ROWS is a table of registrations such that every instantiation of register_loop_kernel (2 dims x 2 storages x plain /
robust / adaptive), accumulate_kernel (dims x storages x plain / robust), scale_select_kernel and solve_kernel runs in
at least one row, and every (dim, storage, covariance_model) appears, models 1 and 2 in both loops.  Small inputs reach
the multi-launch loop with GICP_FUSED_LOOP=0; test_plan_host.py checks that every row's sizes and flags select the
loop named here.  Each row also runs check_loop and is compared end to end with the float64 oracle of its kernel."""
import numpy as np
import pytest

import inner_oracle as IO
from test_gpu_search_exactness import Batch, check_loop, exact_nn, env  # noqa: F401  (env: fixture)

pytestmark = pytest.mark.gpu

# inputs: (generator, dim, source points (an upper bound for the ray-cast scan), parameters)
P_MOVED = dict(k=20, max_distance_nearest_neighbors=4.0, max_distance_correspondence=2.0)
P_SCAN = dict(max_distance_nearest_neighbors=200.0)
P_WALLS = dict(k=6, max_distance_nearest_neighbors=3.0, max_distance_correspondence=5.0, max_iterations=40)
P_BIG = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0, max_iterations=40)
INPUTS = {"moved": (3, 1500, P_MOVED), "scan": (2, 360, P_SCAN), "walls": (2, 3000, P_WALLS),
          "big": (3, 20000, P_BIG)}

# (name, input, storage, loop, kernel, covariance_model); kernel: None, ("fixed", kind, c) or
# ("adaptive", kind, kappa, min_scale).  loop "multi" on a small input sets GICP_FUSED_LOOP=0.
ROWS = [
    ("fused3_f32_plain", "moved", "f32", "fused", None, 0),
    ("fused3_f64_plain", "moved", "f64", "fused", None, 1),
    ("fused3_f32_huber", "moved", "f32", "fused", ("fixed", "huber", 0.2), 2),
    ("fused3_f64_tukey", "moved", "f64", "fused", ("fixed", "tukey", 0.5), 0),
    ("fused3_f32_adaptive", "moved", "f32", "fused", ("adaptive", "cauchy", 0.5, 0.02), 1),
    ("fused3_f64_adaptive", "moved", "f64", "fused", ("adaptive", "tukey", 1.0, 0.02), 2),
    ("fused2_f32_plain", "scan", "f32", "fused", None, 2),
    ("fused2_f64_plain", "scan", "f64", "fused", None, 0),
    ("fused2_f32_huber", "scan", "f32", "fused", ("fixed", "huber", 4.0), 1),
    ("fused2_f64_cauchy", "scan", "f64", "fused", ("fixed", "cauchy", 4.0), 2),
    ("fused2_f32_adaptive", "scan", "f32", "fused", ("adaptive", "huber", 4.5, 1.0), 0),
    ("fused2_f64_adaptive", "scan", "f64", "fused", ("adaptive", "huber", 4.5, 1.0), 1),
    ("multi3_f32_plain", "big", "f32", "multi", None, 0),
    ("multi3_f64_plain", "moved", "f64", "multi", None, 1),
    ("multi3_f32_adaptive", "moved", "f32", "multi", ("adaptive", "huber", 0.5, 0.02), 2),
    ("multi3_f64_adaptive", "big", "f64", "multi", ("adaptive", "tukey", 1.0, 0.02), 0),
    ("multi2_f32_plain", "walls", "f32", "multi", None, 1),
    ("multi2_f64_plain", "scan", "f64", "multi", None, 2),
    ("multi2_f32_adaptive", "scan", "f32", "multi", ("adaptive", "huber", 4.5, 1.0), 0),
    ("multi2_f64_adaptive", "walls", "f64", "multi", ("adaptive", "cauchy", 3.0, 0.05), 2),
]


def _input(name):
    if name == "moved":
        from test_gpu_robust import _moved
        s, t, _ = _moved(n=1500)
    elif name == "scan":
        from test_gpu_robust import _obstacle
        s, t, _ = _obstacle()
    elif name == "walls":
        from test_gpu_search_exactness import _pair2d
        s, t = _pair2d(np.random.default_rng(5), 3000, 4.0, (1.0, -0.5))
    else:
        from generalized_icp_b200 import synthetic
        s, t, _ = synthetic.patches3d_pair(n=20000, n_patches=16, cube=40.0, patch=30.0, seed=40)
    return s, t


def frozen_problems(b, r):
    """For every pair p and executed iteration k: (p, k, p', q, W, distance) of the gated-in exact matches at T_hist[k]
    (check_loop's rule: near-ties and distances at the gate, where either answer is exact, take the device's match),
    with W = inv(R_k C_src R_k^T + C_tgt) from the device's covariances."""
    d = b.dim
    d_max = float(b.params.get("max_distance_correspondence", 150.0))
    cs = b.eng.covariances(0).cpu().numpy()
    ct = b.eng.covariances(1).cpu().numpy()
    T_hist = r.T_hist.cpu().numpy()
    n_out = r.n_outer.cpu().numpy()
    for k in range(int(n_out.max())):
        Tk_all = np.where(np.isnan(T_hist[:, k]), np.eye(d + 1), T_hist[:, k])
        idx_dev, _, _ = b.eng.correspond(Tk_all, with_W=False)
        idx_dev = idx_dev.cpu().numpy()
        for p in range(b.n_pairs):
            if n_out[p] <= k:
                continue
            s, t = b.srcs[p], b.tgts[p]
            Tk = T_hist[p, k]
            pp = s @ Tk[:d, :d].T + Tk[:d, d]
            idx, key, key2 = exact_nn(t, pp)
            dist = np.sqrt(key)
            want = np.where(dist > d_max, -1, idx)
            dp = 8 * np.finfo(np.float64).eps * np.abs(pp).max(1)
            ok = ~(key2 - key <= 1e-9 * key + 4 * dist * dp) & ~(np.abs(dist - d_max) <= 1e-9 * d_max + dp)
            m = np.where(ok, want, idx_dev[b.off_s[p]:b.off_s[p + 1]])
            g = m >= 0
            q = t[m[g]]
            Rk = Tk[:d, :d]
            W = np.linalg.inv(Rk @ cs[b.off_s[p]:b.off_s[p + 1]][g] @ Rk.T + ct[b.off_t[p]:b.off_t[p + 1]][m[g]])
            yield p, k, pp[g], q, W, np.sqrt(np.sum((q - pp[g]) ** 2, axis=1))


def kernel_weights(b, r, weighting):
    """weight(p, k, d): the weights of pair p's gated-in matches at distances d in iteration k - robust_oracle's
    formula at the fixed scale, or at the adaptive scale the library computes at T_hist[k] (gicpRobustScales, bit-exact
    against numpy in test_gpu_robust_adaptive); None without a kernel."""
    import robust_oracle as RO
    if weighting is None:
        return None
    d = b.dim
    T_hist = r.T_hist.cpu().numpy()
    scales = {}

    def weight(p, k, dist):
        if weighting[0] == "fixed":
            return RO.robust_weight(weighting[1], dist, weighting[2])
        if k not in scales:
            scales[k] = b.eng.robust_scales(np.where(np.isnan(T_hist[:, k]), np.eye(d + 1), T_hist[:, k]))
        return RO.robust_weight(weighting[1], dist, scales[k][p])
    return weight


def check_inner_minimum(b, r, weighting):
    """The minimum of every executed, non-converged iteration's frozen problem at T_hist[k + 1] (module docstring).
    weighting: None, ("fixed", kind, c) or ("adaptive", kind, kappa, min_scale).  Returns the worst gradient ratio
    (f64 storage; nan with f32) and the worst value gap F(T_hist[k + 1]) - minimum, relative to the scale."""
    d = b.dim
    f64 = b.storage == "f64"
    tol = 1e-9 if f64 else 2e-5
    T_hist = r.T_hist.cpu().numpy()
    conv = r.converged_at.cpu().numpy()
    weight = kernel_weights(b, r, weighting)
    worst_g, worst_gap, n_checked = 0.0, -np.inf, 0
    for p, k, pp, q, W, dist in frozen_problems(b, r):
        if conv[p] == k:
            continue                                   # T is not updated there; check_loop compares min_loss
        if weight is not None:
            W = weight(p, k, dist)[:, None, None] * W
        dT = T_hist[p, k + 1] @ np.linalg.inv(T_hist[p, k])
        F = IO.objective(pp, q, W, dT)
        F0 = IO.objective(pp, q, W, np.eye(d + 1))
        fmin, _ = IO.newton_minimum(pp, q, W)
        scale = max(fmin, F0)
        gap = (F - fmin) / scale if scale > 0 else 0.0
        assert F <= fmin + tol * scale + 1e-12, (p, k, F, fmin, scale)
        worst_gap = max(worst_gap, gap)
        if f64 and len(q):
            g, _ = IO.gradient_hessian(pp, q, W, dT)
            ratio = np.abs(g).max() / IO.gradient_scale(pp, q, W)
            assert ratio <= 1e-7, (p, k, ratio)
            worst_g = max(worst_g, ratio)
        n_checked += 1
    assert n_checked >= 2, n_checked
    return (worst_g if f64 else float("nan")), worst_gap


def _oracle(s, t, params, kernel, model):
    import adaptive_oracle as AO
    import robust_oracle as RO
    from oracle import gicp_oracle as O
    s, t = np.asarray(s, np.float64), np.asarray(t, np.float64)
    if kernel is None:
        return O.gicp_oracle(s, t, inner="newton", recompute_src_cov=False, record=False, covariance_model=model,
                             **params)
    if kernel[0] == "fixed":
        return RO.gicp_oracle(s, t, robust=kernel[1:], record=False, covariance_model=model, **params)
    return AO.gicp_oracle(s, t, adaptive=kernel[1:], record=False, covariance_model=model, **params)


@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_inner_minimum_every_iteration(row, env):
    import robust_oracle as RO
    name, inp, storage, loop, kernel, model = row
    dim, _, params = INPUTS[inp]
    s, t = _input(inp)
    b = Batch(dim, storage, [s], [t], covariance_model=model, **params)
    if kernel is not None and kernel[0] == "fixed":
        b.eng.set_robust_kernel(kernel[1], kernel[2])
    elif kernel is not None:
        b.eng.set_robust_kernel(kernel[1], adaptive=kernel[2], min_scale=kernel[3])

    def run():
        r = b.register()
        return r, check_inner_minimum(b, r, kernel)
    r, (worst_g, worst_gap) = env(run, GICP_FUSED_LOOP=1 if loop == "fused" else 0)
    n_out, conv = int(r.n_outer[0]), int(r.converged_at[0])
    assert n_out >= 3, n_out
    check_loop(b, r, weight=kernel_weights(b, r, kernel))
    # end to end against the float64 oracle of the same kernel and covariance model (storage-rounded inputs)
    ref = _oracle(b.srcs[0], b.tgts[0], params, kernel, model)
    extent = float(np.linalg.norm(b.tgts[0].max(0) - b.tgts[0].min(0)))
    rot, trans = RO.motion_error(r.T[0].cpu().numpy(), ref["T"])
    print(f"{name}: n_outer {n_out} (oracle {ref['n_outer']}), worst gradient ratio {worst_g:.1e}, worst value gap "
          f"{worst_gap:.1e}, vs oracle {rot:.1e} rad {trans / extent:.1e} extent")
    assert n_out == ref["n_outer"], (n_out, ref["n_outer"])
    assert conv == (-1 if ref["converged_at"] is None else ref["converged_at"]), (conv, ref["converged_at"])
    assert rot <= 1e-5 and trans <= 1e-5 * extent, (rot, trans)
