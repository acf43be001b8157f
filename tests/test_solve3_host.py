"""K4's 3-D inner solver (csrc/solve.cuh inner_solve_warp<3>, the warp-cooperative Levenberg-Marquardt that runs in
every 3-D registration) compiled for the host by tests/host_harness/solve3_host.cu - its 32 lanes as 32 threads - and
checked without a GPU:

- frozen problems whose minimiser is known by construction (q_i = R* p_i + t* exactly, so F >= 0 with F = 0 only at
  (R*, t*)), from 0.1 to 179 degree starts;
- every outer iteration of float64 oracle registrations (plane-to-plane, point-to-point, point-to-plane, Huber and
  Tukey weights), with certificates computed from per-point residuals, not from the reduced form the solver sees:
  a vanishing gradient, a positive semi-definite Hessian and a value no worse than the oracle's Newton minimum;
- degenerate problems (no correspondence, one, two, collinear points, a planar patch), iteration caps, a form rounded
  to float32 as f32 storage accumulates it, and scaled forms.

The stop rules use max(1, |f|) as their floor (solve.cuh), so the solver is deliberately not scale-invariant where
|f| < 1: the scale test stays above that."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import inner_oracle as IO
import quality_oracle as Q
from oracle import gicp_oracle as O

DP = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def solve3(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("solve3_host") / "solve3_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "solve3_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src, "-lpthread"], check=True)
    lib = ctypes.CDLL(out)
    lib.gicp_test_solve3d.argtypes = [DP, ctypes.c_int, DP]

    def run(red, max_it=50):
        red = np.ascontiguousarray(red, dtype=np.float64)
        assert red.shape == (80,)
        o = np.zeros(14)
        assert lib.gicp_test_solve3d(red.ctypes.data_as(DP), max_it, o.ctypes.data_as(DP)) == 0
        return o[:3].copy(), o[3:12].reshape(3, 3).copy(), float(o[13])

    return run


def _rot(axis, deg):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    return O.rot3(np.deg2rad(deg) * axis)


def _spd(rng, n, d=3, cond=30.0):
    """n random SPD matrices with eigenvalues in [1, cond] (scaled like GICP weights: W ~ 1 / (lambda_n + ...))."""
    Qm = np.linalg.qr(rng.normal(size=(n, d, d)))[0]
    ev = np.exp(rng.uniform(0, np.log(cond), size=(n, d))) * 0.05
    return np.einsum("nij,nj,nkj->nik", Qm, ev, Qm)


def _cloud(n=400, seed=0):
    from generalized_icp_b200 import synthetic
    s, _, _ = synthetic.patches3d_pair(n=n, n_patches=5, cube=20.0, patch=12.0, seed=seed)
    return s.astype(np.float64)


def _problem(pp, q, W):
    mu = 0.5 * (q.min(0) + q.max(0))
    return Q.reduced_form(pp, q - pp, W, mu), mu


def _exact(seed, deg, n=400):
    """(pp, q, W, R*, t*, extent) with q = R* p + t* exactly: 3-D patch cloud, random SPD W, rotation by deg about a
    random axis, translation up to the cloud's extent."""
    rng = np.random.default_rng(seed)
    p = _cloud(n, seed)
    ext = float(np.linalg.norm(p.max(0) - p.min(0)))
    R = _rot(rng.normal(size=3), deg)
    t = rng.uniform(-1, 1, 3) * ext / np.sqrt(3)
    return p, p @ R.T + t, _spd(rng, n), R, t, ext


def _check_value(red, dtc, dR, f, what):
    fv = IO.form_value(red, 3, dtc, dR)
    c0 = float(red[72])
    assert abs(fv - f) <= 1e-12 * max(abs(f), c0), (what, f, fv, c0)


# ------------------------------------------------------------------------------------------------
# exact minimiser by construction
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("deg", [0.1, 5.0, 30.0, 60.0, 120.0, 179.0])
@pytest.mark.parametrize("seed", range(6))
def test_exact_minimiser(solve3, seed, deg):
    """Also asserted outright at 120 and 179 degrees, where F is not convex in the rotation: from the identity the
    solver reached (R*, t*) on every seed (rotation error <= 1e-10, |f| <= 1e-15 c0 when this test was written)."""
    p, q, W, R, t, ext = _exact(seed, deg)
    red, mu = _problem(p, q, W)
    c0 = float(red[72])
    dtc, dR, f = solve3(red)
    assert np.isfinite(dtc).all() and np.isfinite(dR).all() and np.isfinite(f)
    T = IO.motion(dtc, dR, mu)
    # the reduced form cancels c0 - 2<G, Z> + <Z, H Z>: an exact minimum comes out as about -1e-15 c0
    assert abs(f) <= 1e-12 * c0, (f, c0)
    assert IO.rotation_error(T[:3, :3], R) <= 1e-9, IO.rotation_error(T[:3, :3], R)
    assert np.abs(T[:3, 3] - t).max() <= 1e-9 * ext, np.abs(T[:3, 3] - t).max()
    _check_value(red, dtc, dR, f, (seed, deg))


# ------------------------------------------------------------------------------------------------
# recorded problems: every outer iteration of float64 oracle registrations
# ------------------------------------------------------------------------------------------------
P3 = dict(k=20, max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0, max_iterations=40)


def _start(seed, deg):
    rng = np.random.default_rng(seed)
    c = np.full(3, 10.0)
    R = _rot(rng.normal(size=3), deg)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = c - R @ c
    return T


def recorded_problems(seed, deg, model, robust):
    """Every outer iteration's frozen problem (p', q, w W) of the float64 oracle loop on a moved-patch pair whose
    source starts deg degrees off: plain or robust (robust_oracle, R_k C_0 R_k^T covariances, Newton inner solve)."""
    import robust_oracle as RO
    from generalized_icp_b200 import synthetic
    s, t, Tg = synthetic.patches3d_pair(n=1500, n_patches=4, cube=20.0, patch=15.0, seed=seed)
    s, t = s.astype(np.float64), t.astype(np.float64)
    T0 = _start(seed + 9, deg) @ Tg
    s0 = s @ T0[:3, :3].T + T0[:3, 3]
    ref = RO.gicp_oracle(s0, t, covariance_model=model, robust=robust, **P3)
    out = []
    for tr in ref["trace"]:
        g = tr["idx"] >= 0
        Tk = tr["T"]
        pp = s0[g] @ Tk[:3, :3].T + Tk[:3, 3]
        out.append((pp, tr["q"][g], tr["w"][g][:, None, None] * tr["W"][g]))
    return out, float(np.linalg.norm(t.max(0) - t.min(0))), 0.5 * (t.min(0) + t.max(0))


def _certify(solve3, pp, q, W, mu, ext, red=None, tol_g=1e-8, what=""):
    """The certificates of one frozen problem at the solver's point; returns (gradient ratio, value gap / c0,
    Hessian condition number)."""
    if red is None:
        red = Q.reduced_form(pp, q - pp, W, mu)
    c0 = float(red[72])
    dtc, dR, f = solve3(red)
    T = IO.motion(dtc, dR, mu)
    _check_value(red, dtc, dR, f, what)
    F = IO.objective(pp, q, W, T)
    g, H = IO.gradient_hessian(pp, q, W, T)
    gs = IO.gradient_scale(pp, q, W)
    ratio = np.abs(g).max() / gs
    assert ratio <= tol_g, (what, ratio)
    ev = np.linalg.eigvalsh(H)
    assert ev[0] >= -1e-9 * ev[-1], (what, ev)
    fmin, Tn = IO.newton_minimum(pp, q, W)
    gap = (F - fmin) / c0
    assert F <= fmin + 1e-9 * c0, (what, F, fmin, c0)
    cond = ev[-1] / ev[0] if ev[0] > 0 else np.inf
    if cond < 1e8:
        assert IO.rotation_error(T[:3, :3], Tn[:3, :3]) <= 1e-7, (what, IO.rotation_error(T[:3, :3], Tn[:3, :3]))
        assert np.abs(T[:3, 3] - Tn[:3, 3]).max() <= 1e-7 * ext, (what, T[:3, 3] - Tn[:3, 3])
    return ratio, gap, cond


RECORDED = [(3, 6.0, 0, None), (40, 5.0, 0, None), (41, 7.5, 1, None), (42, 10.0, 2, None),
            (3, 8.0, 0, ("huber", 0.3)), (40, 6.0, 2, ("tukey", 1.0)), (41, 9.0, 1, ("huber", 0.1))]


@pytest.mark.parametrize("seed,deg,model,robust", RECORDED)
def test_recorded_problems(solve3, seed, deg, model, robust):
    probs, ext, mu = recorded_problems(seed, deg, model, robust)
    assert len(probs) >= 3
    worst = [0.0, -np.inf, 0.0]
    for k, (pp, q, W) in enumerate(probs):
        r, gap, cond = _certify(solve3, pp, q, W, mu, ext, what=(seed, deg, model, robust, k))
        worst = [max(worst[0], r), max(worst[1], gap), max(worst[2], cond)]
    print(f"{len(probs)} iterations: worst gradient ratio {worst[0]:.1e}, value gap / c0 {worst[1]:.1e}, "
          f"Hessian condition {worst[2]:.1e}")


@pytest.mark.parametrize("seed,deg,model,robust", RECORDED)
def test_recorded_problems_converge_like_newton(solve3, seed, deg, model, robust):
    """The Newton term of the rotation block (Cn in inner_solve_warp) makes the iteration converge quadratically:
    every recorded problem is certified after 4 LM iterations (at most 3 were needed when this test was written).
    Gauss-Newton, or a Newton term of the wrong sign, still reaches the minimum within 50 iterations but needs 4-6
    here, so only this cap shows such an error."""
    probs, ext, mu = recorded_problems(seed, deg, model, robust)
    for k, (pp, q, W) in enumerate(probs):
        red = Q.reduced_form(pp, q - pp, W, mu)
        dtc, dR, f = solve3(red, 4)
        g, _ = IO.gradient_hessian(pp, q, W, IO.motion(dtc, dR, mu))
        assert np.abs(g).max() <= 1e-8 * IO.gradient_scale(pp, q, W), (k, np.abs(g).max() / IO.gradient_scale(pp, q, W))


# ------------------------------------------------------------------------------------------------
# degenerate problems
# ------------------------------------------------------------------------------------------------
def test_empty_form(solve3):
    dtc, dR, f = solve3(np.zeros(80))
    assert np.array_equal(dtc, np.zeros(3)) and np.array_equal(dR, np.eye(3)) and f == 0.0


def _degenerate(kind, seed):
    rng = np.random.default_rng(seed)
    R, t = _rot(rng.normal(size=3), 8.0), rng.uniform(-1, 1, 3)
    if kind == "one":
        p, W = rng.uniform(0, 10, (1, 3)), _spd(rng, 1)
    elif kind == "two":
        p, W = rng.uniform(0, 10, (2, 3)), _spd(rng, 2)
    elif kind == "collinear":        # rotation about the line is unconstrained: H is singular
        p = np.outer(rng.uniform(0, 20, 200), [0.6, 0.0, 0.8]) + [1.0, 2.0, 3.0]
        W = np.broadcast_to(np.eye(3), (200, 3, 3)).copy()
    else:                            # planar patch with point-to-point W: in-plane motion weakly constrained
        Fr = np.linalg.qr(rng.normal(size=(3, 3)))[0]
        ab = rng.uniform(-5, 5, (300, 2))
        p = 10.0 + ab[:, :1] * Fr[:, 0] + ab[:, 1:] * Fr[:, 1]
        W = np.broadcast_to(np.eye(3), (300, 3, 3)).copy()
    return p, p @ R.T + t, W


@pytest.mark.parametrize("kind", ["one", "two", "collinear", "planar"])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_degenerate_problems(solve3, kind, seed):
    """Singular H (one, two and collinear correspondences): the damped solve fails and the damping grows.  The true
    minimum is 0 (q = R* p + t* exactly)."""
    p, q, W = _degenerate(kind, seed)
    red, mu = _problem(p, q, W)
    c0 = float(red[72])
    dtc, dR, f = solve3(red)
    assert np.isfinite(dtc).all() and np.isfinite(dR).all() and np.isfinite(f)
    assert -1e-9 * c0 <= f <= c0, (f, c0)
    _check_value(red, dtc, dR, f, kind)
    T = IO.motion(dtc, dR, mu)
    g, H = IO.gradient_hessian(p, q, W, T)
    ev = np.linalg.eigvalsh(H)
    if ev[0] > 1e-9 * ev[-1]:
        assert np.abs(g).max() <= 1e-8 * IO.gradient_scale(p, q, W), (kind, g)


# ------------------------------------------------------------------------------------------------
# iteration caps, float32 rounding, scale
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_it", [1, 3])
def test_iteration_caps(solve3, max_it):
    for seed, deg in ((0, 5.0), (1, 30.0), (2, 60.0)):
        p, q, W, _, _, _ = _exact(seed, deg)
        red, _ = _problem(p, q, W)
        dtc, dR, f = solve3(red, max_it)
        assert f <= float(red[72])
        _check_value(red, dtc, dR, f, (max_it, seed))
    probs, _, mu = recorded_problems(40, 5.0, 0, None)
    for pp, q, W in probs:
        red = Q.reduced_form(pp, q - pp, W, mu)
        prev = float(red[72])
        for it in range(1, max_it + 1):            # no cap gives a worse value than a smaller one
            dtc, dR, f = solve3(red, it)
            assert f <= prev
            prev = f
        _check_value(red, dtc, dR, f, max_it)


def test_float32_rounded_forms(solve3):
    """K3b accumulates the reduced form in float32 with f32 storage: its 72 non-loss entries rounded to float32 perturb
    the problem the way the device sees it.  The output stays finite and no worse than the start."""
    cases = [_problem(*_exact(s, deg)[:3])[0] for s, deg in ((0, 5.0), (1, 30.0), (2, 60.0))]
    probs, _, mu = recorded_problems(42, 10.0, 2, None)
    cases += [Q.reduced_form(pp, q - pp, W, mu) for pp, q, W in probs]
    for red in cases:
        r32 = red.copy()
        r32[:72] = r32[:72].astype(np.float32)
        dtc, dR, f = solve3(r32)
        assert np.isfinite(dtc).all() and np.isfinite(dR).all() and np.isfinite(f)
        assert f <= float(red[72])


@pytest.mark.parametrize("s", [1e-3, 1e6])
def test_scaled_forms(solve3, s):
    """(H, G, c) scaled by s: the same minimiser where |f| >= 1 at both scales (noisy matches keep the minimum large)."""
    rng = np.random.default_rng(5)
    p, q, W, _, _, ext = _exact(3, 20.0)
    q = q + rng.normal(0, 0.5, q.shape)
    W = W * 1e3
    red, _ = _problem(p, q, W)
    dtc, dR, f = solve3(red)
    assert min(abs(f), abs(f) * s) >= 1.0
    rs = red.copy()
    rs[:73] *= s
    dtc_s, dR_s, f_s = solve3(rs)
    assert abs(f_s - s * f) <= 1e-10 * abs(s * f)
    assert np.abs(dR_s - dR).max() <= 1e-10
    assert np.abs(dtc_s - dtc).max() <= 1e-10 * ext
