"""Float64 restatement of gicpEvaluate (include/gicp_b200.h): the quality row, H and b of one pair from its
correspondences, and the reduced form (gicpNormalEquations' row) the device maps them from.  Shared by
tests/test_quality_host.py and tests/test_gpu_quality.py.

Conventions: p' = R p + t, e = q - p', left perturbation T(xi) = Exp(xi) T with the rotation first,
J = [J_rot | I], J_rot = -[p']x in 3-D and (-p'_y, p'_x)^T in 2-D; H = sum J^T w W J, b = sum J^T w W e."""
import numpy as np


def npar(dim):
    return 6 if dim == 3 else 3


def skew(x):
    return np.array([[0.0, -x[2], x[1]], [x[2], 0.0, -x[0]], [-x[1], x[0], 0.0]])


def jacobians(pp):
    """(n, d, npar): d(T(xi) p_i) / d xi at xi = 0, evaluated at p'_i."""
    pp = np.asarray(pp, np.float64)
    n, d = pp.shape
    J = np.zeros((n, d, npar(d)))
    if d == 3:
        J[:, 0, 1], J[:, 0, 2] = pp[:, 2], -pp[:, 1]          # -[p']x
        J[:, 1, 0], J[:, 1, 2] = -pp[:, 2], pp[:, 0]
        J[:, 2, 0], J[:, 2, 1] = pp[:, 1], -pp[:, 0]
        J[:, :, 3:] = np.eye(3)
    else:
        J[:, 0, 0], J[:, 1, 0] = -pp[:, 1], pp[:, 0]
        J[:, :, 1:] = np.eye(2)
    return J


def hessian_gradient(pp, e, W):
    """H = sum J^T W J, b = sum J^T W e over the rows given (W already carries the robust weight)."""
    J = jacobians(pp)
    WJ = np.einsum("nkl,nlj->nkj", W, J)
    H = np.einsum("nki,nkj->ij", J, WJ)
    b = np.einsum("nki,nk->i", J, np.einsum("nkl,nl->nk", W, e))
    return H, b


def gradient_magnitude(pp, e, W):
    """sum_i |J_i^T W_i e_i| elementwise: the scale of b's rounding error.  b itself goes to 0 where the registration
    converged, so its error is judged against the size of the terms it sums."""
    J = jacobians(pp)
    return np.abs(np.einsum("nki,nk->ni", J, np.einsum("nkl,nl->nk", W, e))).sum(axis=0)


def quality(pp, e, W, dist, n_src, d):
    """(quality row [n, fitness, rmse, loss], H, b) of one pair from its gated-in rows: p', e, w W, distance."""
    pp, e, W, dist = (np.asarray(x, np.float64) for x in (pp, e, W, dist))
    n = len(dist)
    if n == 0:
        return np.zeros(4), np.zeros((npar(d), npar(d))), np.zeros(npar(d))
    H, b = hessian_gradient(pp, e, W)
    loss = float(np.einsum("nk,nkl,nl->", e, W, e))
    return np.array([n, n / n_src if n_src else 0.0, np.sqrt(np.sum(dist * dist) / n), loss]), H, b


def open3d_information(points):
    """Open3D's get_information_matrix_from_point_clouds: sum G_r^T G_r over three rows per point (3-D, rotation
    first), evaluated here at the given points."""
    GTG = np.zeros((6, 6))
    for t in np.asarray(points, np.float64):
        for G in ([0.0, t[2], -t[1], 1.0, 0.0, 0.0], [-t[2], 0.0, t[0], 0.0, 1.0, 0.0],
                  [t[1], -t[0], 0.0, 0.0, 0.0, 1.0]):
            G = np.asarray(G)
            GTG += np.outer(G, G)
    return GTG


def reduced_form(pp, e, W, mu):
    """gicpNormalEquations' row (layout in include/gicp_b200.h) of the gated-in rows p', e, w W, centred on mu."""
    pp, e, W, mu = (np.asarray(x, np.float64) for x in (pp, e, W, mu))
    d = len(mu)
    NP, NS = d + 1, d * (d + 1) // 2
    ab = [(a, b) for a in range(NP) for b in range(a, NP)]
    cd = [(c, k) for c in range(d) for k in range(c, d)]
    NH = len(ab) * NS
    red = np.zeros(80 if d == 3 else 32)
    pt = np.concatenate([np.ones((len(pp), 1)), pp - mu], axis=1)
    for i, (a, b) in enumerate(ab):
        for j, (c, k) in enumerate(cd):
            red[i * NS + j] = np.sum(pt[:, a] * pt[:, b] * W[:, c, k])
    v = np.einsum("nkl,nl->nk", W, e)
    for c in range(d):
        for a in range(NP):
            red[NH + c * NP + a] = np.sum(v[:, c] * pt[:, a])
    red[NH + d * NP] = float(np.einsum("nk,nk->", e, v))
    red[NH + d * NP + 1] = len(pp)
    red[NH + d * NP + 2:NH + d * NP + 2 + d] = mu
    return red


def blocks(M, dim):
    """The (rotation-rotation, rotation-translation, translation-translation) blocks of an (npar, npar) matrix, or the
    (rotation, translation) parts of an (npar,) vector."""
    r = 3 if dim == 3 else 1
    M = np.asarray(M)
    if M.ndim == 1:
        return M[:r], M[r:]
    return M[:r, :r], M[:r, r:], M[r:, r:]


def block_rel_err(got, ref, dim, scale=None):
    """max over the blocks of |got - ref| / |ref| (Frobenius; an all-zero reference block compares absolutely), or
    / |scale| per block when a scale of the same shape is given."""
    out = 0.0
    for g, f, s in zip(blocks(got, dim), blocks(ref, dim), blocks(ref if scale is None else scale, dim)):
        nf = np.linalg.norm(s)
        out = max(out, np.linalg.norm(g - f) / (nf if nf > 0 else 1.0))
    return out
