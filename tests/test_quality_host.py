"""CPU checks of gicpEvaluate's map (include/gicp_b200.h): quality_from_reduced (csrc/quality.cuh) compiled for the
host, applied to reduced forms numpy builds from random correspondences, against the direct float64 sums
sum J^T W J and sum J^T W e of tests/quality_oracle.py."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import quality_oracle as QO


@pytest.fixture(scope="module")
def qmap(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("quality_host") / "quality_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "quality_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    lib = C.CDLL(out)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    lib.gicp_test_quality.argtypes = [C.c_int, C.c_longlong, dp, dp, ip, dp, dp, dp]

    def f(dim, red, sum_d2, n_src):
        red = np.ascontiguousarray(red, np.float64)
        sum_d2 = np.ascontiguousarray(sum_d2, np.float64)
        n_src = np.ascontiguousarray(n_src, np.int32)
        n, k = len(red), QO.npar(dim)
        q, H, b = np.empty((n, 4)), np.empty((n, k, k)), np.empty((n, k))
        lib.gicp_test_quality(dim, n, red.ctypes.data_as(dp), sum_d2.ctypes.data_as(dp), n_src.ctypes.data_as(ip),
                              q.ctypes.data_as(dp), H.ctypes.data_as(dp), b.ctypes.data_as(dp))
        return q, H, b
    return f


def _random_pair(rng, dim, n, centre, spread):
    """n correspondences around `centre`: p', e, SPD w W and distances, and the target-box centre mu nearby."""
    pp = centre + rng.uniform(-spread, spread, size=(n, dim))
    e = rng.normal(0, 0.05 * spread, size=(n, dim))
    A = rng.normal(size=(n, dim, dim))
    W = np.einsum("nij,nkj->nik", A, A) + 0.1 * np.eye(dim)
    w = rng.uniform(0, 1, size=n)
    w[: n // 10] = 0.0                                     # Tukey weights of 0 still count
    mu = centre + rng.uniform(-0.5 * spread, 0.5 * spread, size=dim)
    return pp, e, w[:, None, None] * W, np.linalg.norm(e, axis=1), mu


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("far", [0.0, 1e2, 1e4, 1e5])
def test_map_equals_the_direct_sums(qmap, dim, far):
    rng = np.random.default_rng(int(far) + dim)
    reds, d2s, nsrc, refs = [], [], [], []
    for p in range(12):
        n = int(rng.integers(1, 3000))
        centre = far * rng.normal(size=dim) / np.sqrt(dim)
        pp, e, W, dist, mu = _random_pair(rng, dim, n, centre, float(rng.uniform(0.5, 50.0)))
        reds.append(QO.reduced_form(pp, e, W, mu))
        d2s.append(np.sum(dist * dist))
        nsrc.append(n + int(rng.integers(0, 500)))
        refs.append(QO.quality(pp, e, W, dist, nsrc[-1], dim))
    q, H, b = qmap(dim, np.array(reds), np.array(d2s), np.array(nsrc))
    for p, (qr, Hr, br) in enumerate(refs):
        assert q[p, 0] == qr[0] and q[p, 1] == qr[1], (p, q[p], qr)
        assert abs(q[p, 2] - qr[2]) <= 1e-15 * qr[2]
        assert q[p, 3] == reds[p][72 if dim == 3 else 24]           # the loss slot, as it is
        assert QO.block_rel_err(H[p], Hr, dim) < 1e-12, (p, QO.block_rel_err(H[p], Hr, dim))
        assert QO.block_rel_err(b[p], br, dim) < 1e-12, (p, QO.block_rel_err(b[p], br, dim))
        assert np.array_equal(H[p], H[p].T)


@pytest.mark.parametrize("dim", [2, 3])
def test_empty_rows_give_zeros(qmap, dim):
    nred = 80 if dim == 3 else 32
    red = np.zeros((3, nred))
    red[:, nred - 8:] = np.nan            # loss, mu of an empty target box and the padding: never read with n = 0
    red[:, (72 if dim == 3 else 24) + 1] = 0.0
    q, H, b = qmap(dim, red, np.array([0.0, 0.0, 0.0]), np.array([0, 50, 1]))
    assert not np.any(q) and not np.any(H) and not np.any(b)
    assert not np.isnan(q).any()


def test_fitness_of_an_empty_source_and_rmse_are_open3d_s():
    q, _, _ = QO.quality(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 3, 3)), np.zeros(0), 0, 3)
    assert np.array_equal(q, np.zeros(4))
    pp = np.array([[1.0, 2.0, 3.0], [0.0, 1.0, 0.0]])
    e = np.array([[0.3, 0.0, 0.4], [0.0, 0.0, 1.0]])
    q, H, b = QO.quality(pp, e, np.tile(np.eye(3), (2, 1, 1)), np.linalg.norm(e, axis=1), 4, 3)
    assert q[0] == 2 and q[1] == 0.5 and abs(q[2] - np.sqrt((0.25 + 1.0) / 2)) < 1e-15 and abs(q[3] - 1.25) < 1e-15
    assert np.allclose(H, QO.open3d_information(pp), rtol=0, atol=1e-12)   # point-to-point, W = I
