"""CPU-only checks of the host side: the C ABI library loads and exports every symbol the header
declares, the compat module mirrors the reference's signature, inputs generators are seeded."""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    header = open(os.path.join(ROOT, "include", "gicp_b200.h")).read()
    declared = set(re.findall(r"\b(gicp[A-Z]\w+)\s*\(", header))
    from generalized_icp_b200 import _lib
    assert declared == set(_lib.SYMBOLS)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.gicpVersion() >= 100
    p = _lib.GicpParams()
    assert lib.gicpDefaultParams(ctypes.byref(p)) == 0
    # defaults of gicp.py:78, :5, :11, :24
    assert (p.k, p.max_iterations, p.tolerance) == (6, 100, 1e-6)
    assert (p.max_distance_correspondence, p.max_distance_nearest_neighbors) == (150.0, 50.0)
    assert (p.lambda_tangent, p.lambda_normal) == (100.0, 10.0)


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import gicp as shim
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        shim.gicp(np.zeros((5, 2)), np.ones((5, 2)))
    from generalized_icp_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.gicpCreate(ctypes.byref(h), 0, 2, 1) != 0
    assert b"no CUDA device" in lib.gicpGetLastError()


def test_signature_matches_reference():
    import gicp as shim
    sig = inspect.signature(shim.gicp)
    assert list(sig.parameters) == ["source_points", "target_points", "max_iterations", "tolerance",
                                    "max_distance_correspondence", "max_distance_nearest_neighbors"]
    d = {k: v.default for k, v in sig.parameters.items() if v.default is not inspect._empty}
    assert d == dict(max_iterations=100, tolerance=1e-6, max_distance_correspondence=150,
                     max_distance_nearest_neighbors=50)
    T = np.array([[0.0, -1.0, 2.0], [1.0, 0.0, 3.0], [0, 0, 1.0]])
    cloud = np.array([[1.0, 0.0, 9.0], [0.0, 2.0, 9.0]])          # (N, >=2) accepted, gicp.py:176-177
    assert np.allclose(shim.apply_transformation(cloud, T), [[2.0, 4.0], [0.0, 3.0]])


def test_product_path_does_not_import_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "generalized-icp_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                assert "oracle" not in open(os.path.join(root, f)).read().replace("the oracle", "").replace("CPU oracle", ""), f
    assert "oracle" not in open(os.path.join(ROOT, "gicp.py")).read()


def test_generators_are_seeded(golden):
    import demo_inputs
    from generalized_icp_b200 import synthetic
    g = golden("config1_seed0")
    s, t = demo_inputs.config1_pair(0)
    assert np.array_equal(s, g["src"]) and np.array_equal(t, g["tgt"])
    assert s.shape == (90, 2) and t.shape == (87, 2)
    scans, poses = demo_inputs.lidar_sequence(seed=1, num_rays=90, n_scans=3)
    g2 = golden("config2_rays90_pair0")
    assert np.array_equal(np.asarray(scans[0]), g2["src"]) and np.array_equal(np.asarray(scans[1]), g2["tgt"])
    a, b, T = synthetic.patches3d_pair(n=1000, seed=5)
    a2, b2, T2 = synthetic.patches3d_pair(n=1000, seed=5)
    assert a.dtype == np.float32 and np.array_equal(a, a2) and np.array_equal(b, b2) and np.array_equal(T, T2)


def _reduced_form_numpy(src, q, W, T_lin, mu):
    """The reduced form K3 accumulates (layout: include/gicp_b200.h), evaluated in numpy from the
    reference's own matches q and weights W (rows with W = 0 are gated out)."""
    d = 2
    NP, NS = 3, 3
    pp = src @ T_lin[:d, :d].T + T_lin[:d, d]
    e = q - pp
    pt = np.concatenate([np.ones((len(src), 1)), pp - mu], axis=1)
    red = np.zeros(32)
    ab = 0
    for a in range(NP):
        for b in range(a, NP):
            for cd, (c, dd) in enumerate(((0, 0), (0, 1), (1, 1))):
                red[ab * NS + cd] = np.sum(pt[:, a] * pt[:, b] * W[:, c, dd])
            ab += 1
    We = np.einsum("nij,nj->ni", W, e)
    NH = 18
    for c in range(d):
        for a in range(NP):
            red[NH + c * NP + a] = np.sum(We[:, c] * pt[:, a])
    red[NH + d * NP] = np.sum(e * We)
    red[NH + d * NP + 1] = np.count_nonzero(np.abs(W).sum((1, 2)))
    red[NH + d * NP + 2:NH + d * NP + 4] = mu
    return red


@pytest.mark.parametrize("name", ["config1_seed0", "config1_seed3", "config2_rays90_pair0", "config2_rays360_pair2"])
def test_reduced_form_reproduces_loss_and_grad_loss(name, golden):
    """gicp.py:52-76: the value AND the gradient (tx, ty, theta) of the frozen inner objective follow from the
    32-double reduced form; checked here against what the reference's own loss / grad_loss returned at x0 and
    xopt of every outer iteration (the same helpers are applied to the GPU's reduced form in test_gpu_parity)."""
    from generalized_icp_b200.engine import reduced_form_grad2d, reduced_form_loss
    g = golden(name)
    mu = 0.5 * (g["tgt"].min(0) + g["tgt"].max(0))
    for k in range(len(g["it_fopt"])):
        T = g["all_T"][k]
        red = _reduced_form_numpy(g["src"], g["it_q"][k], g["it_W"][k], T, mu)
        for xk, lk, gk in (("it_x0", "it_loss_at_x0", "it_grad_at_x0"), ("it_xopt", "it_loss_at_xopt", "it_grad_at_xopt")):
            x = g[xk][k]
            Te = np.eye(3)
            Te[:2, :2] = [[np.cos(x[2]), -np.sin(x[2])], [np.sin(x[2]), np.cos(x[2])]]
            Te[:2, 2] = x[:2]
            want = float(g[lk][k])
            assert abs(reduced_form_loss(red, 2, T, Te) - want) <= 1e-9 * max(1.0, abs(want))
            gw = g[gk][k]
            gg = reduced_form_grad2d(red, T, x)
            assert np.abs(gg - gw).max() <= 1e-8 * max(1.0, np.abs(gw).max()), (k, xk, gg, gw)


@pytest.fixture(scope="module")
def solve_host(tmp_path_factory):
    """tests/host_harness/*.cu: the 2-D inner solver and the damped linear solve of csrc/solve.cuh, the covariance
    tail of csrc/knn_cov.cuh and the fp32 search bounds of csrc/objective.cuh (__host__ __device__ functions) compiled
    for the host with nvcc - product source, run here as the thing under test."""
    import ctypes
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    tmp = tmp_path_factory.mktemp("host_harness")
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness")
    libs = []
    for name in ("solve_host", "cov_host", "bounds_host"):
        out = str(tmp / (name + ".so"))
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                        "-shared", "-o", out, os.path.join(here, name + ".cu")], check=True)
        libs.append(ctypes.CDLL(out))
    lib, cov, bounds = libs
    dp = ctypes.POINTER(ctypes.c_double)
    ip = ctypes.POINTER(ctypes.c_int)
    lib.gicp_test_solve2d.argtypes = [dp, ctypes.c_int, dp]
    lib.gicp_test_spd_solve6.argtypes = [dp, dp]
    cov.gicp_test_regularised_cov.argtypes = [ctypes.c_int, dp, ctypes.c_double, ctypes.c_double, dp]
    lib.regularised_cov = cov.gicp_test_regularised_cov
    bounds.gicp_test_filter.argtypes = [ctypes.c_longlong, dp, dp, dp, ctypes.c_int, ip]
    bounds.gicp_test_filter.restype = ctypes.c_longlong
    bounds.gicp_test_slack.argtypes = [ctypes.c_longlong, dp, dp, dp, ctypes.c_int, dp, dp]
    bounds.gicp_test_slack.restype = ctypes.c_longlong
    lib.bounds = bounds
    return lib


@pytest.mark.parametrize("name", ["config1_seed0", "config1_seed3", "config2_rays90_pair0", "config2_rays360_pair2"])
def test_inner_solver_minimises_the_references_inner_problems(name, golden, solve_host):
    """K4's 2-D solver (csrc/solve.cuh inner_solve_2d, compiled for the host) on the reference's own inner problems
    (gicp.py:148-152: matches and weights of every outer iteration of a recorded run): the point it returns is a
    stationary point of the frozen objective (grad_loss of gicp.py:60-76 vanishes there), its value is the reduced
    form's value at that point, and it is at least as good as what the reference's fmin_cg reached."""
    import ctypes
    from generalized_icp_b200.engine import reduced_form_grad2d, reduced_form_loss
    g = golden(name)
    mu = 0.5 * (g["tgt"].min(0) + g["tgt"].max(0))
    dp = ctypes.POINTER(ctypes.c_double)
    n_it = len(g["it_fopt"])
    for k in sorted(set(range(min(n_it, 8))) | {n_it - 1}):     # the first outer iterations and the last one
        T = g["all_T"][k]
        red = np.ascontiguousarray(_reduced_form_numpy(g["src"], g["it_q"][k], g["it_W"][k], T, mu))
        out = np.zeros(8)
        assert solve_host.gicp_test_solve2d(red.ctypes.data_as(dp), 50, out.ctypes.data_as(dp)) == 0
        dtc, dth, fmin, dR = out[:2], out[2], out[3], out[4:].reshape(2, 2)
        assert np.allclose(dR, [[np.cos(dth), -np.sin(dth)], [np.sin(dth), np.cos(dth)]], atol=1e-15)
        # un-centre and compose exactly as solve_pair does: dt = dt_c - (dR - I) mu,  T_new = [dR R | dR t + dt]
        dt = dtc - (dR - np.eye(2)) @ mu
        Tn = np.eye(3)
        Tn[:2, :2] = dR @ T[:2, :2]
        Tn[:2, 2] = dR @ T[:2, 2] + dt
        x_new = np.array([Tn[0, 2], Tn[1, 2], np.arctan2(Tn[1, 0], Tn[0, 0])])
        f_at = reduced_form_loss(red, 2, T, Tn)
        assert abs(f_at - fmin) <= 1e-9 * max(1.0, abs(fmin))
        grad = reduced_form_grad2d(red, T, x_new)
        scale = max(1.0, np.abs(reduced_form_grad2d(red, T, g["it_x0"][k])).max())
        assert np.abs(grad).max() <= 1e-8 * scale, (k, grad, scale)
        assert fmin <= float(g["it_loss_at_xopt"][k]) + 1e-9 * max(1.0, abs(fmin)), (k, fmin, g["it_loss_at_xopt"][k])


def test_damped_solve_host(solve_host):
    """spd_solve<6> (LDL^T, csrc/solve.cuh) against numpy on random SPD systems; an indefinite matrix is reported."""
    import ctypes
    dp = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(7)
    for _ in range(50):
        B = rng.normal(size=(6, 6))
        A = np.ascontiguousarray(B @ B.T + 1e-3 * np.eye(6))
        b = rng.normal(size=6)
        x = b.copy()
        assert solve_host.gicp_test_spd_solve6(A.ctypes.data_as(dp), x.ctypes.data_as(dp)) == 0
        want = np.linalg.solve(A, b)
        assert np.abs(x - want).max() <= 1e-9 * max(1.0, np.abs(want).max())
    A = np.ascontiguousarray(np.diag([1.0, 2.0, -1.0, 1.0, 1.0, 1.0]))
    x = np.ones(6)
    assert solve_host.gicp_test_spd_solve6(A.ctypes.data_as(dp), x.ctypes.data_as(dp)) == 1


def test_covariance_tail_host(solve_host):
    """K2's covariance tail (closed-form symmetric eigen-solve + regularisation, csrc/knn_cov.cuh regularised_cov,
    compiled for the host) against numpy's eigh on the formula of gicp.py:11-16 / the oracle's
    covariances_from_neighbors: generic, nearly planar, nearly collinear and badly scaled scatter matrices; non-finite
    input gives the identity (gicp.py:31-32)."""
    _check_covariance_tail(solve_host, 100.0, 10.0)


# (lambda_tangent, lambda_normal) away from the defaults: the regularisation of fast_gicp / small_gicp, equal lambdas
# (C = lam I exactly), an inverted pair and a ratio of 1e-7
@pytest.mark.parametrize("lam_t,lam_n", [(1.0, 1e-3), (1.0, 1.0), (10.0, 100.0), (1e4, 1e-3)])
def test_covariance_tail_host_lambdas(solve_host, lam_t, lam_n):
    """The same checks with other regularisations."""
    _check_covariance_tail(solve_host, lam_t, lam_n)


def _check_covariance_tail(solve_host, lam_t, lam_n):
    import ctypes
    dp = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(11)

    def want(S, dim):
        evals, evecs = np.linalg.eigh(S)
        if dim == 2:
            v = evecs[:, 1]
            return lam_n * np.eye(2) + (lam_t - lam_n) * np.outer(v, v)
        n = evecs[:, 0]
        return lam_t * np.eye(3) - (lam_t - lam_n) * np.outer(n, n)

    def got(S, dim):
        S6 = np.zeros(6)
        if dim == 2:
            S6[0], S6[1], S6[3] = S[0, 0], S[0, 1], S[1, 1]
        else:
            S6[:] = [S[0, 0], S[0, 1], S[0, 2], S[1, 1], S[1, 2], S[2, 2]]
        C = np.zeros(6)
        solve_host.regularised_cov(dim, S6.ctypes.data_as(dp), lam_t, lam_n, C.ctypes.data_as(dp))
        if dim == 2:
            return np.array([[C[0], C[1]], [C[1], C[2]]])
        return np.array([[C[0], C[1], C[2]], [C[1], C[3], C[4]], [C[2], C[4], C[5]]])

    for dim in (2, 3):
        for case in range(200):
            Q, _ = np.linalg.qr(rng.normal(size=(dim, dim)))
            ev = np.sort(rng.uniform(0.1, 1.0, dim))
            if case % 4 == 1:
                ev[0] = ev[-1] * 1e-6            # nearly planar (3-D) / nearly collinear (2-D)
            if case % 4 == 2 and dim == 3:
                ev[1] = ev[0] * (1 + 1e-3)       # two close small eigenvalues, one dominant direction
                ev[0] *= 1e-2
                ev[1] *= 1e-2
            scale = 10.0 ** rng.integers(-6, 7) if case % 4 == 3 else 1.0
            S = (Q * ev) @ Q.T * scale
            S = 0.5 * (S + S.T)
            gap = (ev[-1] - ev[-2]) if dim == 2 else (ev[1] - ev[0])
            tol = 1e-9 * abs(lam_t - lam_n) / max(gap / ev[-1], 1e-12) * 10
            C = got(S, dim)
            assert np.abs(C - want(S, dim)).max() <= max(tol, 1e-9), (dim, case, ev)
            if lam_t == lam_n:
                assert np.array_equal(C, lam_t * np.eye(dim))
        bad = np.full((dim, dim), np.nan)
        assert np.array_equal(got(bad, dim), np.eye(dim))


def _queries(rng, n):
    """Transformed source points p' (fp64) with |p'| spread log-uniformly over 1 .. 1e5 m (one axis dominant or all
    comparable); half of them are fp32 values (an fp64 query rounded to fp32)."""
    u = rng.normal(size=(n, 3)) * 10.0 ** rng.uniform(-3, 0, size=(n, 3))
    p = u / np.abs(u).max(1, keepdims=True) * 10.0 ** rng.uniform(0, 5, size=(n, 1))
    f = rng.random(n) < 0.5
    p[f] = p[f].astype(np.float32)
    return p


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _key(c, p):
    d = c - p
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def test_search_filter_threshold_is_sound(solve_host):
    """K3a's fp32 candidate filter (csrc/objective.cuh filter_c1 / filter_thr_of, compiled for the host): a target
    point whose exact squared distance - the fp64 key or the __float128 value - is <= the best distance so far always
    passes, for 1.2e6 cases: fp32 targets, |p'| from 1 to 1e5 m (where the filter's Pf term dominates), distances from
    1e-6 m to d_max, best distance equal to the candidate's own key or one ulp below it, and the device's approximate
    rsqrtf modelled by +-2 ulp around the exact reciprocal square root."""
    import ctypes
    dp = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(2024)
    n = 1_200_000
    p = _queries(rng, n)
    d_max = 10.0 ** rng.uniform(0, np.log10(150.0), n)
    d = 10.0 ** rng.uniform(-6, 0, n) * d_max
    c = (p + d[:, None] * _unit(rng, n)).astype(np.float32).astype(np.float64)
    # a third: the worst alignment the bound covers.  p' sits just past the midpoint between two fp32 values on
    # every axis (fp32(p') is half an ulp away), the candidate is m whole ulps beyond the other neighbour, so its fp32
    # distance exceeds the exact one by the full 2 sqrt(3) u P d
    w = np.arange(n) % 3 == 0
    x = p[w].astype(np.float32)
    ulp = np.nextafter(np.abs(x), np.float32(np.inf)) - np.abs(x)
    sgn = np.where(x < 0, -1.0, 1.0)
    p[w] = x + sgn * ulp * (0.5 + 1e-3)                # rounds to the neighbour one ulp out
    m = np.minimum(10.0 ** rng.uniform(0, 6, w.sum()), 0.5 * d_max[w] / ulp.max(1))
    m = np.maximum(np.floor(m), 0.0)[:, None]
    c[w] = (x - sgn * ulp * m).astype(np.float32)
    bd = _key(c, p)
    below = rng.random(n) < 0.3
    bd[below] = np.nextafter(bd[below], 0.0)          # must pass only if the exact value is still <= bd
    p, c, bd = (np.ascontiguousarray(a) for a in (p, c, bd))
    out = np.zeros(n, dtype=np.int32)
    bad = solve_host.bounds.gicp_test_filter(n, p.ctypes.data_as(dp), c.ctypes.data_as(dp), bd.ctypes.data_as(dp), 2,
                                             out.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    assert bad == 0, (p[out == 1][:5], c[out == 1][:5], bd[out == 1][:5])


@pytest.mark.parametrize("f32", [1, 0])
def test_search_slack_is_sound(f32, solve_host):
    """The slack K3a stores for a tracked match (csrc/objective.cuh match_slack: how far the point may move before
    its match could change, which lets the next iterations skip its search) never exceeds half the exact gap between
    the nearest and the runner-up target point (__float128 distances), for 6e5 near-ties per storage type: runner-up
    1 + 1e-7 ... 1 + 1e-3 times as far as the nearest, |p'| from 1 to 1e5 m, distances from 1e-6 m to d_max.  Also
    checks that the bound is not vacuous: well separated pairs get a positive slack."""
    import ctypes
    dp = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(7 + f32)
    n = 600_000
    p = _queries(rng, n)
    d_max = 10.0 ** rng.uniform(0, np.log10(150.0), n)
    d = 10.0 ** rng.uniform(-6, 0, n) * d_max
    gap = 10.0 ** rng.uniform(-7, -3, n)
    a = p + d[:, None] * _unit(rng, n)
    b = p + (d * (1.0 + gap))[:, None] * _unit(rng, n)
    if f32:
        a, b = a.astype(np.float32).astype(np.float64), b.astype(np.float32).astype(np.float64)
    swap = rng.random(n) < 0.5
    a[swap], b[swap] = b[swap].copy(), a[swap].copy()
    p, a, b = (np.ascontiguousarray(x) for x in (p, a, b))
    sl, hg = np.zeros(n), np.zeros(n)
    bad = solve_host.bounds.gicp_test_slack(n, p.ctypes.data_as(dp), a.ctypes.data_as(dp), b.ctypes.data_as(dp), f32,
                                            sl.ctypes.data_as(dp), hg.ctypes.data_as(dp))
    worst = np.argmax(sl - hg)
    assert bad == 0, (p[worst], a[worst], b[worst], sl[worst], hg[worst])
    # not vacuous: where the gap is wide compared with the fp32 resolution at |p'|, the slack is a fair share of it
    wide = hg > 1e-4 * (np.abs(p).max(1) + d)
    assert wide.sum() > 1000 and (sl[wide] > 0.2 * hg[wide]).mean() > 0.9
