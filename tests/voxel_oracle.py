"""float64 restatement of the voxel-grid filter (gicpVoxelDownsample, include/gicp_b200.h) that the GPU tests
compare the device against.  Test infrastructure only: nothing in the package imports it."""
import numpy as np


def voxel_downsample(points, offsets, leaf, min_points=1):
    """float64 restatement of the engine's voxel-grid filter.  For each cloud: voxel = floor(p / leaf) per axis
    (float64 division), non-finite rows dropped, voxels with < min_points points dropped, output point = centroid
    (float64 sum from the voxel's first point, divided by the count), output order = each voxel's lowest row.
    A cloud whose voxel indices leave int64, or span 2^21 voxels or more along an axis in 3-D (2^31 in 2-D), raises
    ValueError.  Returns (out (M, d) f64, out_offsets (P+1,) i64, voxel_of (N,) i64 cloud-local or -1, counts (M,))."""
    P = np.asarray(points)
    off = np.asarray(offsets, dtype=np.int64)
    n, d = P.shape
    bits = 21 if d == 3 else 31
    outs, cnts, out_off = [], [], [0]
    voxel_of = np.full(n, -1, dtype=np.int64)
    for c in range(len(off) - 1):
        Q = P[off[c]:off[c + 1]].astype(np.float64)
        rows = np.nonzero(np.isfinite(Q).all(axis=1))[0]
        if len(rows) == 0:
            out_off.append(out_off[-1])
            continue
        with np.errstate(over="ignore"):                        # an overflow to inf is rejected below
            V = np.floor(Q[rows] / leaf)
        lo, hi = V.min(axis=0), V.max(axis=0)
        for a in range(d):
            if not (-2.0 ** 63 <= lo[a] and hi[a] < 2.0 ** 63):
                raise ValueError(f"cloud {c}, axis {a}: voxel index outside int64; use a larger voxel_size")
            if int(hi[a]) - int(lo[a]) >= 1 << bits:
                raise ValueError(f"cloud {c}, axis {a}: more than 2^{bits} voxels; use a larger voxel_size")
        rel = V.astype(np.int64) - lo.astype(np.int64)
        key = np.zeros(len(rows), dtype=np.int64)
        for a in range(d):
            key = (key << bits) | rel[:, a]
        _, first, inv, count = np.unique(key, return_index=True, return_inverse=True, return_counts=True)
        X = Q[rows][np.argsort(inv, kind="stable")]              # each voxel's points, in ascending row order
        starts = np.concatenate([[0], np.cumsum(count)[:-1]])
        # sequential sums from each voxel's first point (numpy's own reductions sum pairwise): step k adds the k-th
        # point of every voxel that has one, the voxels taken in descending count so that they are a prefix
        desc = np.argsort(-count, kind="stable")
        sums = X[starts[desc]].copy()
        c_desc = count[desc]
        for k in range(1, int(c_desc[0])):
            m = int(np.searchsorted(-c_desc, -k, side="left"))    # voxels with count > k
            sums[:m] += X[starts[desc[:m]] + k]
        cent = np.empty_like(sums)
        cent[desc] = sums / c_desc[:, None]
        kept = np.nonzero(count >= min_points)[0]
        kept = kept[np.argsort(first[kept], kind="stable")]      # output order: lowest row of each voxel
        local = np.full(len(count), -1, dtype=np.int64)
        local[kept] = np.arange(len(kept))
        voxel_of[off[c] + rows] = local[inv]
        outs.append(cent[kept])
        cnts.append(count[kept])
        out_off.append(out_off[-1] + len(kept))
    out = np.concatenate(outs) if outs else np.zeros((0, d))
    counts = np.concatenate(cnts) if cnts else np.zeros(0, dtype=np.int64)
    return out, np.asarray(out_off, dtype=np.int64), voxel_of, counts
