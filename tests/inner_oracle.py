"""Float64 checks of K4's inner solve (csrc/solve.cuh) that do not depend on the solver: the reduced form's value at a
returned point, and the gradient and Hessian of the frozen objective from per-point residuals.  Shared by
tests/test_solve3_host.py, tests/test_host.py and tests/test_gpu_inner_minimum.py.

A frozen problem is (p', q, W): linearised points p'_i = T_k p_i, matches q_i and weights W_i (the robust weight already
folded in).  The objective of a motion (dR, dt) applied on the left is  F = sum r_i^T W_i r_i,  r_i = q_i - dR p'_i - dt.
The certificates use the chart  x -> exp([w]x) x + tau  around the returned point (rotation first, as
quality_oracle.jacobians); at a stationary point the Hessian's inertia does not depend on the chart."""
import numpy as np

import quality_oracle as Q
from oracle import gicp_oracle as O


def dense_H(red, d):
    """The dense (D * NP)^2 form Hd[c * NP + a][e * NP + b] = H(a, b, c, e) of the packed reduced Hessian (solve.cuh
    dense_H_entry)."""
    NP, NS = d + 1, d * (d + 1) // 2

    def sym(n, a, b):
        a, b = min(a, b), max(a, b)
        return a * n - a * (a - 1) // 2 + (b - a)

    DN = d * NP
    Hd = np.empty((DN, DN))
    for row in range(DN):
        for col in range(DN):
            c, a, e, b = row // NP, row % NP, col // NP, col % NP
            Hd[row, col] = red[sym(NP, a, b) * NS + sym(d, c, e)]
    return Hd


def split(red, d):
    """(Hd, G, c0, mu) of a packed reduced form."""
    NP = d + 1
    NH = (NP * (NP + 1) // 2) * (d * (d + 1) // 2)
    NQ = NH + d * NP
    return dense_H(red, d), np.asarray(red[NH:NQ]), float(red[NQ]), np.asarray(red[NQ + 2:NQ + 2 + d])


def form_value(red, d, dtc, dR):
    """f(Z) = c - 2 <G, Z> + <Z, H Z>,  Z = [dt_c | dR - I]: the value the solver reports for its returned point."""
    Hd, G, c0, _ = split(red, d)
    Z = np.concatenate([np.asarray(dtc)[:, None], np.asarray(dR) - np.eye(d)], axis=1).ravel()
    return c0 - 2.0 * float(G @ Z) + float(Z @ Hd @ Z)


def motion(dtc, dR, mu):
    """The left motion [dR | dt] the solver's centred (dt_c, dR) stands for: dt = dt_c - (dR - I) mu (solve_pair)."""
    d = len(mu)
    T = np.eye(d + 1)
    T[:d, :d] = dR
    T[:d, d] = np.asarray(dtc) - (np.asarray(dR) - np.eye(d)) @ np.asarray(mu)
    return T


def objective(pp, q, W, T):
    """F at the motion T, from per-point residuals."""
    d = pp.shape[1]
    r = q - (pp @ T[:d, :d].T + T[:d, d])
    return float(np.einsum("ni,nij,nj->", r, W, r))


def _gens(d):
    if d == 2:
        return [np.array([[0.0, -1.0], [1.0, 0.0]])]
    return [Q.skew(e) for e in np.eye(3)]


def gradient_hessian(pp, q, W, T):
    """(J^T W r summed, the Hessian of F) at the motion T, in the chart x -> exp([w]x) x + tau (rotation first).
    grad F = -2 sum J_i^T W_i r_i, so the first value is -grad F / 2."""
    d = pp.shape[1]
    x = pp @ T[:d, :d].T + T[:d, d]
    r = q - x
    J = Q.jacobians(x)
    Wr = np.einsum("nij,nj->ni", W, r)
    g = np.einsum("nki,nk->i", J, Wr)
    H = 2.0 * np.einsum("nki,nkl,nlj->ij", J, W, J)
    E = _gens(d)
    nr = len(E)
    for k in range(nr):
        for l in range(nr):
            S = 0.5 * (E[k] @ E[l] + E[l] @ E[k])     # d2 exp([w]x) x / dw_k dw_l at w = 0
            H[k, l] -= 2.0 * float(np.einsum("ni,ni->", Wr, x @ S.T))
    return g, H


def gradient_scale(pp, q, W):
    """max over the parameters of sum_i |J_i^T W_i e_i| at the linearisation point: what the gradient is judged
    against (it goes to 0 at a minimum, so a relative error has no other natural scale)."""
    return float(Q.gradient_magnitude(pp, q - pp, W).max())


def newton_minimum(pp, q, W):
    """The oracle's minimum of the frozen problem (inner_newton from the linearisation point): (f, motion T)."""
    d = pp.shape[1]
    x, f, _, _ = O.inner_newton(np.zeros(3 if d == 2 else 6), pp, q, W)
    return f, O.offset_to_matrix(x, d)


def rotation_error(Ra, Rb):
    """|Ra^T Rb - I| (Frobenius): resolves errors near zero, unlike the arccos of the trace."""
    return float(np.linalg.norm(Ra.T @ Rb - np.eye(len(Ra))))
