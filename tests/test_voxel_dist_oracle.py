"""The voxel-distribution oracle (tests/voxel_dist_oracle.py) against a plain per-voxel restatement: np.cov of each
voxel's finite points and np.linalg.eigh, the formula of gicp.py:11-16 / SURVEY 8c.  CPU only."""
import numpy as np
import pytest

import voxel_dist_oracle as VD


def _plain(points, offsets, leaf, min_points, lam_t, lam_n):
    d = points.shape[1]
    means, covs = [], []
    for c in range(len(offsets) - 1):
        vox = {}
        for r in range(offsets[c], offsets[c + 1]):
            p = points[r]
            if not np.isfinite(p).all():
                continue
            vox.setdefault(tuple(np.floor(p / leaf)), []).append(r)
        for rows in vox.values():                     # insertion order = each voxel's lowest row
            if len(rows) < min_points:
                continue
            X = points[rows]
            means.append(X.mean(axis=0))
            S = np.cov(X.T, ddof=1) if len(rows) > 1 else None
            if S is None or not np.isfinite(S).all():
                covs.append(np.eye(d))
                continue
            _, V = np.linalg.eigh(S)
            if d == 2:
                v = V[:, 1]
                covs.append(lam_n * np.eye(2) + (lam_t - lam_n) * np.outer(v, v))
            else:
                n = V[:, 0]
                covs.append(lam_t * np.eye(3) - (lam_t - lam_n) * np.outer(n, n))
    return np.asarray(means).reshape(-1, d), np.asarray(covs).reshape(-1, d, d)


def _cloud(dim, seed):
    """Voxels of 1, 2, collinear, coplanar and general points, at negative and positive coordinates, a non-finite row."""
    rng = np.random.default_rng(seed)
    parts = [rng.uniform(-3.0, 3.0, size=(400, dim))]                       # general, 1- and 2-point voxels
    base = np.full(dim, -5.25)
    t = rng.uniform(0.05, 0.95, size=(7, 1))
    parts.append(base + t * np.r_[1.0, 0.5, 0.25][:dim] * 0.9)             # collinear in one voxel
    if dim == 3:
        uv = rng.uniform(0.05, 0.95, size=(9, 2))
        parts.append(np.c_[uv, np.full(9, 0.5)] + np.array([7.0, -8.0, 2.0]))   # coplanar, axis-aligned normal
    P = np.concatenate(parts)
    P[5] = np.nan
    P[17, 0] = np.inf
    return P


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("min_points", [1, 3])
def test_oracle_matches_plain_restatement(dim, min_points):
    lam_t, lam_n = 100.0, 10.0
    P = _cloud(dim, 3 + dim)
    off = np.array([0, 250, 250, len(P)])                                  # a middle cloud that is empty
    means, out_off, covs, counts = VD.voxel_distributions(P, off, 1.0, min_points, lam_t, lam_n)
    assert out_off[1] == out_off[2]
    pm, pc = [], []
    for c in range(3):
        m, cv = _plain(P[off[c]:off[c + 1]], [0, off[c + 1] - off[c]], 1.0, min_points, lam_t, lam_n)
        assert len(m) == out_off[c + 1] - out_off[c]
        pm.append(m)
        pc.append(cv)
    pm, pc = np.concatenate(pm), np.concatenate(pc)
    assert np.allclose(means, pm, rtol=0, atol=1e-12)
    assert (counts >= min_points).all()
    lone = counts == 1
    assert np.array_equal(covs[lone], np.broadcast_to(np.eye(dim), (int(lone.sum()), dim, dim)))
    # the eigenvector is unique where the voxel's scatter has distinct eigenvalues at the end the formula uses
    assert len(covs) == len(pc)
    for i in range(len(covs)):
        if counts[i] < 2:
            continue
        err = np.abs(covs[i] - pc[i]).max()
        if err > 1e-9:
            # a degenerate scatter (2 points or collinear in 3-D): any unit normal of the line is valid; check that
            # covs[i] is such a regularised form: eigenvalues (lam_n, lam_t, lam_t) with the tangent block on the line
            w = np.linalg.eigvalsh(covs[i])
            assert dim == 3 and np.allclose(w, [lam_n, lam_t, lam_t]), (i, err, w)
    assert not np.isnan(covs).any()


def test_oracle_min_points_drops_and_empty():
    P = np.zeros((0, 3))
    means, out_off, covs, counts = VD.voxel_distributions(P, [0, 0], 0.5)
    assert means.shape == (0, 3) and covs.shape == (0, 3, 3) and list(out_off) == [0, 0]
    Q = np.array([[0.1, 0.1, 0.1], [0.2, 0.2, 0.3], [5.0, 5.0, 5.0]])
    means, out_off, covs, counts = VD.voxel_distributions(Q, [0, 3], 1.0, min_points=2)
    assert list(out_off) == [0, 1] and list(counts) == [2]
    # two points: the scatter has rank 1; the 3-D normal is any unit vector orthogonal to their difference
    dvec = (Q[1] - Q[0]) / np.linalg.norm(Q[1] - Q[0])
    assert np.allclose(covs[0] @ dvec, 100.0 * dvec)
