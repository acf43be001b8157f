"""CPU-only checks of voxel distributions' host-compilable parts (tests/host_harness/voxel_cov_host.cu): the per-voxel
finish of gicpSetVoxelized (csrc/voxel.cuh vox_cov_finish, fed the moments the device accumulates) against numpy on
adversarial voxels, and the voxelized set-up plan (csrc/plan.h plan_setup_voxelized)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ZERO, IDENTITY, KNN, VOXEL = 0, 1, 2, 3          # CovSource
NONE = 3                                         # KnnPath::None
SOURCE, TARGET = 0, 1


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("voxel_cov_host") / "voxel_cov_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_harness", "voxel_cov_host.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-Xcompiler", "-fPIC",
                    "-shared", "-o", out, src], check=True)
    L = C.CDLL(out)
    dp = C.POINTER(C.c_double)
    from generalized_icp_b200._lib import GicpParams
    L.gicp_test_voxel_cov.argtypes = [C.c_int, dp, C.c_int, C.c_double, C.c_double, dp]
    L.gicp_test_plan_voxelized.argtypes = [C.POINTER(GicpParams), C.POINTER(C.c_int64), C.c_int, C.c_int, C.c_int, dp,
                                           dp, C.POINTER(C.c_longlong)]
    return L


def _device_cov(lib, X, lam_t, lam_n):
    X = np.ascontiguousarray(X, dtype=np.float64)
    dim = X.shape[1]
    out = np.zeros(6)
    dp = C.POINTER(C.c_double)
    lib.gicp_test_voxel_cov(dim, X.ctypes.data_as(dp), len(X), lam_t, lam_n, out.ctypes.data_as(dp))
    M = np.zeros((dim, dim))
    k = 0
    for i in range(dim):
        for j in range(i, dim):
            M[i, j] = M[j, i] = out[k]
            k += 1
    return M


def _numpy_cov(X, lam_t, lam_n):
    """Reference: np.cov (ddof = 1) + eigh, and the eigen-gap of the end the formula uses (relative to the largest)."""
    dim = X.shape[1]
    if len(X) < 2:
        return np.eye(dim), np.inf
    S = np.cov(X.T, ddof=1)
    if not np.isfinite(S).all():
        return np.eye(dim), np.inf
    w, V = np.linalg.eigh(S)
    top = max(w[-1], 1e-300)
    if dim == 2:
        v = V[:, 1]
        return lam_n * np.eye(2) + (lam_t - lam_n) * np.outer(v, v), (w[1] - w[0]) / top
    n = V[:, 0]
    return lam_t * np.eye(3) - (lam_t - lam_n) * np.outer(n, n), (w[1] - w[0]) / top


def _voxels(dim, rng):
    """(name, points) voxels: general, far from the origin, repeated points, -0.0, rank-deficient, f32-rounded."""
    out = []
    for _ in range(40):
        Q, _ = np.linalg.qr(rng.normal(size=(dim, dim)))
        scale = np.exp(rng.uniform(-3, 0, size=dim))
        X = rng.normal(size=(int(rng.integers(2, 120)), dim)) * scale @ Q.T * 0.2
        out.append(("general", X))
        out.append(("far", X + 1e4 * np.sign(rng.normal(size=dim))))
        out.append(("f32", (X + 37.0).astype(np.float32).astype(np.float64)))
    X = rng.normal(size=(6, dim)) * 0.1
    out.append(("repeated", np.repeat(X, 5, axis=0)))
    out.append(("all_equal", np.repeat(X[:1], 9, axis=0)))
    out.append(("negzero", np.where(rng.random((8, dim)) < 0.5, -0.0, rng.normal(size=(8, dim)) * 0.1)))
    out.append(("single", X[:1]))
    t = rng.uniform(0, 1, size=(10, 1))
    out.append(("collinear", t * rng.normal(size=dim) + 1e4))
    if dim == 3:
        uv = rng.uniform(0, 1, size=(12, 2))
        out.append(("coplanar", np.c_[uv, np.zeros(12)] @ np.linalg.qr(rng.normal(size=(3, 3)))[0].T - 1e4))
    return out


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("lam_t,lam_n", [(100.0, 10.0), (1.0, 1e-3)])
def test_voxel_cov_finish_host(lib, dim, lam_t, lam_n):
    rng = np.random.default_rng(17 + dim)
    lam = max(lam_t, lam_n)
    for name, X in _voxels(dim, rng):
        got = _device_cov(lib, X, lam_t, lam_n)
        want, gap = _numpy_cov(X, lam_t, lam_n)
        assert np.array_equal(got, got.T)
        if len(X) == 1 or np.ptp(X, axis=0).max() == 0:
            # one point, or every point equal: identity (one point) or a zero scatter, which regularised_cov maps to
            # some unit normal; either way a finite regularised form
            if len(X) == 1:
                assert np.array_equal(got, np.eye(dim)), name
            assert np.isfinite(got).all(), name
            continue
        w = np.linalg.eigvalsh(got)
        assert np.allclose(np.sort(w), np.sort([lam_n] + [lam_t] * (dim - 1)) if dim == 3 else
                           np.sort([lam_n, lam_t]), rtol=1e-9, atol=1e-9 * lam), (name, w)
        if gap < 1e-6:
            # rank-deficient at the end the formula uses: the eigenvector is not unique; the regularised form must
            # still hold every direction of the points' span at lam_t (3-D) / the line at lam_t (2-D)
            D = X - X.mean(axis=0)
            _, s, Vt = np.linalg.svd(D, full_matrices=False)
            for v in Vt[s > 1e-9 * s[0]]:
                assert np.allclose(got @ v, lam_t * v, atol=1e-6 * lam), (name, got @ v, v)
            continue
        tol = max(1e-9 * lam * 10 / gap, 1e-9 * lam)
        if name == "far":
            tol *= 1e3          # numpy's np.cov centres by the mean; the device by the first point: both are exact
        assert np.abs(got - want).max() <= tol, (name, np.abs(got - want).max(), tol, gap)


def test_voxel_cov_nonfinite_scatter_is_identity(lib):
    X = np.array([[1e300, 0.0, 0.0], [-1e300, 0.0, 0.0], [0.0, 1.0, 0.0]])
    assert np.array_equal(_device_cov(lib, X, 100.0, 10.0), np.eye(3))


def _plan(lib, which, model, off, f32=True, **prm):
    from generalized_icp_b200._lib import GicpParams
    p = GicpParams(k=6, max_iterations=100, tolerance=1e-6, max_distance_correspondence=150.0,
                   max_distance_nearest_neighbors=50.0, lambda_tangent=100.0, lambda_normal=10.0,
                   inner_max_iterations=50, covariance_model=model)
    for k, v in prm.items():
        setattr(p, k, v)
    off = np.ascontiguousarray(off, dtype=np.int64)
    out = (C.c_longlong * 8)()
    cell, raw_cell = C.c_double(), C.c_double()
    lib.gicp_test_plan_voxelized(C.byref(p), off.ctypes.data_as(C.POINTER(C.c_int64)), len(off) - 1, which, int(f32),
                                 C.byref(cell), C.byref(raw_cell), out)
    return dict(zip(("error", "cov", "knn", "knn_whole", "shared", "same_sizing", "raw_cov", "raw_shared"), out)), \
        cell.value, raw_cell.value


# (which, covariance_model) -> covariance source: models 1 and 2 still force C = I / C = 0
WANT_COV = {(SOURCE, 0): VOXEL, (TARGET, 0): VOXEL, (SOURCE, 1): ZERO, (TARGET, 1): IDENTITY, (SOURCE, 2): ZERO,
            (TARGET, 2): VOXEL}


@pytest.mark.parametrize("which", [SOURCE, TARGET])
@pytest.mark.parametrize("model", [0, 1, 2])
@pytest.mark.parametrize("cells", [dict(), dict(max_distance_nearest_neighbors=5.0, max_distance_correspondence=3.0),
                                   dict(max_distance_nearest_neighbors=50.0, max_distance_correspondence=5.0),
                                   dict(knn_cell=0.3, nn_cell=2.0)])
@pytest.mark.parametrize("off", [[0, 500], [0, 40000, 80000], list(range(0, 3000 * 65, 3000))])
def test_plan_voxelized(lib, which, model, cells, off):
    """The voxel covariance source, one grid (the cell a raw side of the same points searches, sized as the raw plan
    sizes it) and no K2 path."""
    got, cell, raw_cell = _plan(lib, which, model, off, **cells)
    assert got["error"] == 0
    assert got["cov"] == WANT_COV[(which, model)]
    assert got["raw_cov"] == (KNN if WANT_COV[(which, model)] == VOXEL else WANT_COV[(which, model)])
    assert got["knn"] == NONE and got["knn_whole"] == NONE
    assert got["shared"] == 1 and got["same_sizing"] == 1
    assert cell == raw_cell
