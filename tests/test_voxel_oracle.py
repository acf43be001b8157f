"""The voxel-grid oracle (tests/voxel_oracle.py) against a plain dict-based restatement of the
contract in include/gicp_b200.h, and the Python signatures the feature adds.  CPU only."""
import inspect
import math

import numpy as np
import pytest

import voxel_oracle as VO


def _plain(points, offsets, leaf, min_points=1):
    """Row by row: a dict from voxel tuple to the list of its rows, in insertion (= lowest row) order."""
    d = len(points[0]) if len(points) else 3
    out, counts, out_off = [], [], [0]
    voxel_of = [-1] * len(points)
    for c in range(len(offsets) - 1):
        vox = {}
        for r in range(offsets[c], offsets[c + 1]):
            p = [float(x) for x in points[r]]
            if not all(math.isfinite(x) for x in p):
                continue
            vox.setdefault(tuple(math.floor(x / leaf) for x in p), []).append(r)
        for rows in vox.values():
            if len(rows) < min_points:
                continue
            s = [float(points[rows[0]][a]) for a in range(d)]
            for r in rows[1:]:
                s = [s[a] + float(points[r][a]) for a in range(d)]
            for r in rows:
                voxel_of[r] = len(out) - out_off[-1]
            out.append([x / len(rows) for x in s])
            counts.append(len(rows))
        out_off.append(len(out))
    return np.array(out, dtype=np.float64).reshape(-1, d), np.array(out_off), np.array(voxel_of), np.array(counts)


def _check(points, offsets, leaf, min_points=1):
    got = VO.voxel_downsample(points, offsets, leaf, min_points)
    ref = _plain(points, offsets, leaf, min_points)
    assert np.array_equal(got[1], ref[1])
    assert np.array_equal(got[2], ref[2])
    assert np.array_equal(got[3], ref[3])
    assert got[0].shape == ref[0].shape
    # same summation order (sequential from the first point): identical bits, signed zeros included
    assert np.array_equal(got[0].view(np.int64), ref[0].view(np.int64))
    return got


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("leaf", [0.5, 1.0, 2.0, 0.1])
@pytest.mark.parametrize("min_points", [1, 2, 3])
def test_oracle_matches_plain_restatement(dim, leaf, min_points):
    rng = np.random.default_rng(dim * 100 + min_points)
    faces = rng.integers(-6, 7, size=(60, dim)) * 0.5                  # points exactly on voxel faces
    uni = rng.uniform(-3, 3, size=(80, dim))
    bad = rng.uniform(-3, 3, size=(6, dim))
    bad[0, 0], bad[1, -1], bad[2, 0], bad[3] = np.nan, np.inf, -np.inf, np.nan
    pts = np.concatenate([faces, uni, bad, np.full((3, dim), -0.0)])
    pts = pts[rng.permutation(len(pts))]
    # multi-cloud offsets with an empty cloud in the middle and one at the end
    off = [0, 40, 40, 100, len(pts), len(pts)]
    _check(pts, off, leaf, min_points)


def test_negative_coordinates_use_floor():
    pts = np.array([[-0.5, 0.0, 0.0], [-1e-300, 0.0, 0.0], [0.0, 0.0, 0.0], [-1.0, 0.0, 0.0]])
    out, off, vox, cnt = _check(pts, [0, 4], 1.0)
    assert list(vox) == [0, 0, 1, 0] and list(cnt) == [3, 1]


def test_signed_zero_and_identity():
    pts = np.array([[-0.0, -0.0], [1e-9, -2e-9], [0.25, 0.75]])
    out, off, vox, cnt = _check(pts, [0, 3], 1e-9)
    assert np.array_equal(out.view(np.int64), pts.view(np.int64))


def test_non_finite_and_empty_clouds():
    pts = np.array([[np.nan, 0.0, 0.0], [np.inf, 1.0, 1.0], [1.0, 2.0, 3.0]])
    out, off, vox, cnt = _check(pts, [0, 2, 2, 3], 1.0)
    assert list(off) == [0, 0, 0, 1] and list(vox) == [-1, -1, 0]
    out, off, vox, cnt = _check(np.zeros((0, 3)), [0, 0], 1.0)
    assert out.shape == (0, 3) and list(off) == [0, 0]


def test_limits_raise():
    ok = np.array([[0.0, 0.0, 0.0], [(2 ** 21 - 1) + 0.5, 0.0, 0.0]])
    _check(ok, [0, 2], 1.0)
    with pytest.raises(ValueError, match="axis 0"):
        VO.voxel_downsample(np.array([[0.0, 0.0, 0.0], [2.0 ** 21, 0.0, 0.0]]), [0, 2], 1.0)
    with pytest.raises(ValueError, match="axis 1"):
        VO.voxel_downsample(np.array([[0.0, 0.0], [0.0, 2.0 ** 31]]), [0, 2], 1.0)
    _check(np.array([[0.0, 0.0], [0.0, 2.0 ** 31 - 1]]), [0, 2], 1.0)
    with pytest.raises(ValueError, match="int64"):
        VO.voxel_downsample(np.array([[1e300, 0.0, 0.0]]), [0, 1], 1e-10)


def test_signatures():
    from generalized_icp_b200 import compat
    sig = inspect.signature(compat.gicp)
    assert [(p.name, p.default) for p in sig.parameters.values()] == [
        ("source_points", inspect.Parameter.empty), ("target_points", inspect.Parameter.empty),
        ("max_iterations", 100), ("tolerance", 1e-6), ("max_distance_correspondence", 150),
        ("max_distance_nearest_neighbors", 50)]
    assert inspect.signature(compat.gicp_extended).parameters["voxel_size"].default is None
    vs = inspect.signature(compat.voxel_downsample).parameters
    assert list(vs)[:2] == ["cloud", "voxel_size"] and vs["min_points"].default == 1
