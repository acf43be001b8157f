"""CPU checks of the robust kernels (include/gicp_b200.h): the device weight helper compiled for the host against the
float64 formulas of tests/robust_oracle.py, bit for bit, and properties of the robust oracle loop itself."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import robust_oracle as RO
from oracle import gicp_oracle as O

KINDS = ["huber", "cauchy", "tukey"]


@pytest.fixture(scope="module")
def weight_fn(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("robust_host") / "robust_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "robust_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    lib = C.CDLL(out)
    dp = C.POINTER(C.c_double)
    lib.gicp_test_robust_weight.argtypes = [C.c_longlong, C.c_int, dp, dp, dp]

    def w(kind, d, c):
        d, c = np.broadcast_arrays(np.asarray(d, np.float64), np.asarray(c, np.float64))
        d, c = np.ascontiguousarray(d), np.ascontiguousarray(c)
        out = np.empty_like(d)
        lib.gicp_test_robust_weight(d.size, RO.KINDS[kind], d.ctypes.data_as(dp), c.ctypes.data_as(dp),
                                    out.ctypes.data_as(dp))
        return out
    return w


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64))


@pytest.mark.parametrize("kind", [None] + KINDS)
def test_weight_at_zero_and_at_the_scale(weight_fn, kind):
    c = np.array([1e-6, 0.3, 1.0, 2.0, 150.0, 1e6])
    d = np.concatenate([np.zeros_like(c), c, np.nextafter(c, 0), np.nextafter(c, np.inf)])
    cc = np.tile(c, 4)
    got, ref = weight_fn(kind, d, cc), RO.robust_weight(kind, d, cc)
    assert _same_bits(got, ref), (kind, got, ref)
    assert np.all(got[:len(c)] == 1.0)                       # d = 0
    if kind == "huber":
        assert np.all(got[len(c):3 * len(c)] == 1.0)         # d <= c
        assert np.all(got[3 * len(c):] < 1.0)
    if kind == "tukey":
        assert np.all(got[len(c):2 * len(c)] == 0.0)         # u = 1 exactly: weight 0
        assert np.all(got[3 * len(c):] == 0.0)


@pytest.mark.parametrize("kind", ["huber", "cauchy"])
def test_weight_is_exactly_one_at_a_huge_scale(weight_fn, kind):
    d = np.concatenate([[0.0, 5e-324, 1e-300], np.logspace(-12, 150, 400)])
    for c in (1e300, np.finfo(np.float64).max):
        got = weight_fn(kind, d, c)
        assert np.all(got == 1.0), (kind, c, got[got != 1.0][:5])
        assert _same_bits(got, RO.robust_weight(kind, d, c))


@pytest.mark.parametrize("kind", [None] + KINDS)
def test_weight_random_matches_numpy_bit_for_bit(weight_fn, kind):
    rng = np.random.default_rng(11)
    d = 10.0 ** rng.uniform(-6, 6, size=200_000)
    c = 10.0 ** rng.uniform(-6, 6, size=200_000)
    # also near u = 1, where Tukey switches to 0 and Huber to c / d
    d[:20_000] = c[:20_000] * (1.0 + rng.normal(0, 1e-12, size=20_000))
    got, ref = weight_fn(kind, d, c), RO.robust_weight(kind, d, c)
    bad = ~((got == ref) | (np.isnan(got) & np.isnan(ref)))
    assert not bad.any(), (kind, d[bad][:3], c[bad][:3], got[bad][:3], ref[bad][:3])
    assert np.all((got >= 0) & (got <= 1))


def _config1():
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import demo_inputs
    src, tgt = demo_inputs.config1_pair(0)
    return np.asarray(src, np.float64), np.asarray(tgt, np.float64)


def test_oracle_none_and_huge_huber_equal_the_plain_loop():
    src, tgt = _config1()
    plain = O.gicp_oracle(src, tgt, inner="newton", recompute_src_cov=False)
    none = RO.gicp_oracle(src, tgt)
    huge = RO.gicp_oracle(src, tgt, robust=("huber", 1e300))
    for r in (none, huge):
        assert r["n_outer"] == plain["n_outer"] and r["converged_at"] == plain["converged_at"]
        assert _same_bits(r["T"], plain["T"])
        assert _same_bits([t["min_loss"] for t in r["trace"]], [t["min_loss"] for t in plain["trace"]])
        assert all(_same_bits(a, b) for a, b in zip(r["all_T"], plain["all_T"]))


@pytest.mark.parametrize("kind,c", [("huber", 4.0), ("cauchy", 4.0), ("tukey", 12.0)])
def test_oracle_converged_transform_is_an_irls_fixed_point(kind, c):
    """At the converged transform T*, the weights recomputed there give an inner problem whose minimiser is T* again
    (the loop runs until the weighted loss stops changing at 1e-12)."""
    src, tgt = _config1()
    r = RO.gicp_oracle(src, tgt, robust=(kind, c), tolerance=1e-12, max_iterations=300)
    assert r["converged_at"] is not None
    x_star = r["trace"][-1]["offset"]
    T_star = O.offset_to_matrix(x_star, 2)
    moved = O.apply_transformation(src, T_star)
    idx, dist = O.correspond(moved, tgt, 150)
    W = O.weights(T_star[:2, :2] @ r["src_cov0"] @ T_star[:2, :2].T, r["tgt_cov"], idx)
    w = np.where(idx >= 0, RO.robust_weight(kind, dist, c), 1.0)
    x, _, _, _ = O.inner_newton(x_star, src, O.corresponding_points(tgt, idx), w[:, None, None] * W)
    assert np.abs(x - x_star).max() < 1e-9, np.abs(x - x_star).max()


def test_oracle_tukey_with_every_distance_beyond_the_scale_stops_at_identity():
    src, tgt = _config1()
    r = RO.gicp_oracle(src, tgt, robust=("tukey", 1e-9))
    idx, w = r["trace"][0]["idx"], r["trace"][0]["w"]
    assert (idx >= 0).sum() > 10 and np.all(w[idx >= 0] == 0.0)   # gated-in points that weigh nothing
    assert r["n_outer"] == 2 and r["converged_at"] == 1
    assert np.array_equal(r["T"], np.eye(3))
    assert [t["min_loss"] for t in r["trace"]] == [0.0, 0.0]
