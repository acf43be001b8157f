"""CPU checks of the adaptive robust scale (include/gicp_b200.h, gicpSetRobustKernelAdaptive): the device scale helper
compiled for the host against tests/adaptive_oracle.py, bit for bit, and properties of the adaptive oracle loop."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import adaptive_oracle as AO
import robust_oracle as RO
from oracle import gicp_oracle as O

DRIVE = dict(max_distance_nearest_neighbors=200.0, tolerance=1.0)
# median translation error (px) over the 11 pairs of lidar_sequence(seed=0, num_rays=90, n_scans=12), as the oracle
# gives it; adaptive Huber at kappa 4.5 is the setting that beats plain GICP there
PLAIN_MEDIAN_PX = 2.71


@pytest.fixture(scope="module")
def scale_fn(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("adaptive_host") / "adaptive_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "adaptive_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    lib = C.CDLL(out)
    dp = C.POINTER(C.c_double)
    lib.gicp_test_adaptive_scale.argtypes = [C.c_longlong, dp, dp, dp, dp]

    def f(kappa, m, min_scale):
        kappa, m, min_scale = (np.ascontiguousarray(x, dtype=np.float64)
                               for x in np.broadcast_arrays(kappa, m, min_scale))
        out = np.empty_like(m)
        lib.gicp_test_adaptive_scale(m.size, kappa.ctypes.data_as(dp), m.ctypes.data_as(dp),
                                     min_scale.ctypes.data_as(dp), out.ctypes.data_as(dp))
        return out
    return f


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64))


def test_scale_random_matches_numpy_bit_for_bit(scale_fn):
    rng = np.random.default_rng(5)
    n = 200_000
    kappa = 10.0 ** rng.uniform(-3, 3, size=n)
    m = 10.0 ** rng.uniform(-6, 6, size=n)
    min_scale = 10.0 ** rng.uniform(-6, 6, size=n)
    m[:1000] = 0.0                                          # no gated-in correspondence
    kappa[1000:2000] = 1e300                               # kappa * m overflows to inf
    got, ref = scale_fn(kappa, m, min_scale), AO.adaptive_scale(kappa, m, min_scale)
    assert _same_bits(got, ref)
    assert np.all(got[:1000] == min_scale[:1000])
    assert np.all(got >= min_scale)


def test_scale_ties_take_min_scale(scale_fn):
    """kappa * m == min_scale exactly (dyadic values): the result is min_scale, and one ulp either side of it picks
    the larger."""
    kappa = np.array([0.5, 2.0, 4.0, 0.25, 3.0])
    m = np.array([3.0, 0.75, 0.125, 8.0, 1.0])
    tie = kappa * m
    assert _same_bits(scale_fn(kappa, m, tie), tie)
    assert _same_bits(scale_fn(kappa, m, tie), AO.adaptive_scale(kappa, m, tie))
    below, above = np.nextafter(tie, 0), np.nextafter(tie, np.inf)
    assert _same_bits(scale_fn(kappa, m, below), tie)
    assert _same_bits(scale_fn(kappa, m, above), above)


def test_lower_median_rank():
    assert AO.lower_median([]) == 0.0
    assert AO.lower_median([5.0]) == 5.0
    assert AO.lower_median([4.0, 1.0]) == 1.0                  # rank floor((2-1)/2) = 0
    assert AO.lower_median([3.0, 1.0, 2.0]) == 2.0
    assert AO.lower_median([2.0, 2.0, 1.0, 2.0]) == 2.0        # ties count
    d = np.random.default_rng(0).uniform(0, 10, size=1001)
    assert AO.lower_median(d) == np.sort(d)[500]


def _config1():
    import demo_inputs
    src, tgt = demo_inputs.config1_pair(0)
    return np.asarray(src, np.float64), np.asarray(tgt, np.float64)


def _same_loop(a, b):
    assert a["n_outer"] == b["n_outer"] and a["converged_at"] == b["converged_at"]
    assert _same_bits(a["T"], b["T"])
    assert _same_bits([t["min_loss"] for t in a["trace"]], [t["min_loss"] for t in b["trace"]])
    assert all(_same_bits(x, y) for x, y in zip(a["all_T"], b["all_T"]))


@pytest.mark.parametrize("kind", ["huber", "cauchy", "tukey"])
def test_oracle_min_scale_dominant_is_the_fixed_loop(kind):
    src, tgt = _config1()
    c = {"huber": 4.0, "cauchy": 4.0, "tukey": 12.0}[kind]
    ad = AO.gicp_oracle(src, tgt, adaptive=(kind, 1e-300, c))
    assert all(t["c"] == c for t in ad["trace"])
    _same_loop(ad, RO.gicp_oracle(src, tgt, robust=(kind, c)))


@pytest.mark.parametrize("kind", ["huber", "cauchy"])
def test_oracle_huge_kappa_is_the_plain_loop(kind):
    src, tgt = _config1()
    ad = AO.gicp_oracle(src, tgt, adaptive=(kind, 1e300, 1.0))
    assert all(t["c"] > 1e200 for t in ad["trace"])             # m > 0 in every iteration
    _same_loop(ad, O.gicp_oracle(src, tgt, inner="newton", recompute_src_cov=False))


@pytest.mark.parametrize("kind,kappa", [("huber", 3.0), ("cauchy", 4.5), ("tukey", 4.5)])
def test_oracle_converged_transform_is_an_irls_fixed_point(kind, kappa):
    """At the converged T*, the median scale and the weights recomputed there give an inner problem whose minimiser is
    T* again."""
    src, tgt = _config1()
    r = AO.gicp_oracle(src, tgt, adaptive=(kind, kappa, 0.5), tolerance=1e-12, max_iterations=300)
    assert r["converged_at"] is not None
    x_star = r["trace"][-1]["offset"]
    T_star = O.offset_to_matrix(x_star, 2)
    idx, dist = O.correspond(O.apply_transformation(src, T_star), tgt, 150)
    c = AO.scale_at(kappa, 0.5, idx, dist)
    W = O.weights(T_star[:2, :2] @ r["src_cov0"] @ T_star[:2, :2].T, r["tgt_cov"], idx)
    w = np.where(idx >= 0, RO.robust_weight(kind, dist, c), 1.0)
    x, _, _, _ = O.inner_newton(x_star, src, O.corresponding_points(tgt, idx), w[:, None, None] * W)
    assert np.abs(x - x_star).max() < 1e-9, np.abs(x - x_star).max()


def test_oracle_drive_table():
    """The drive of the adaptive scale's motivation: adaptive Huber (kappa 4.5) beats plain GICP in median translation
    error on the 90-ray lidar sequence, and every adaptive kind beats its fixed-scale counterpart."""
    pairs = AO.drive_pairs(seed=0, num_rays=90, n_scans=12)

    def errors(run):
        return np.array([RO.motion_error(run(s, t)["T"], Tg) for s, t, Tg in pairs])
    plain = errors(lambda s, t: RO.gicp_oracle(s, t, record=False, **DRIVE))
    assert abs(np.median(plain[:, 1]) - PLAIN_MEDIAN_PX) < 0.01
    huber = errors(lambda s, t: AO.gicp_oracle(s, t, adaptive=("huber", 4.5, 1.0), record=False, **DRIVE))
    assert np.median(huber[:, 1]) < np.median(plain[:, 1])
    for kind, c in (("cauchy", 4.0), ("tukey", 12.0)):
        fixed = errors(lambda s, t: RO.gicp_oracle(s, t, robust=(kind, c), record=False, **DRIVE))
        ad = errors(lambda s, t: AO.gicp_oracle(s, t, adaptive=(kind, 4.5, 1.0), record=False, **DRIVE))
        assert np.median(ad[:, 1]) < np.median(fixed[:, 1]), kind
