// K4: per-pair tail of one outer iteration.  Replaces fmin_cg (gicp.py:152) and the
// convergence / bookkeeping block gicp.py:153-167.
//   1. sums the blocks' partial reductions of K3 in a fixed order (deterministic),
//   2. minimises the frozen inner objective  f(Z) = c - 2<G,Z> + <Z, H Z>,  Z = [dt | dR - I],
//      over (dt, dR in SO(D)) by Levenberg-Marquardt on the (D + D(D-1)/2)-parameter normal
//      equations  2 J^T H J  (3x3 in 2-D, 6x6 in 3-D), to convergence - the well-defined target
//      of the reference's "minimise loss with W fixed",
//   3. applies the stop rule |last - min_loss| < tolerance BEFORE updating T (gicp.py:160-167),
//      records the history and updates the pair's transform.
#pragma once
#include "common.cuh"

namespace gicp {

// entry e of the dense form Hd[c * NP + a][d * NP + b] = H(a, b, c, d) of the packed reduced Hessian Hq [NAB][NS]
// (K3b's layout): the solver applies H 5-8 times per LM iteration, as dense matrix-vector products
template <int D> __host__ __device__ __forceinline__ double dense_H_entry(const double* Hq, int e) {
    using DD = Dim<D>;
    constexpr int DN = D * DD::NP;
    const int row = e / DN, col = e % DN;
    const int c_ = row / DD::NP, a = row % DD::NP, d = col / DD::NP, b = col % DD::NP;
    return Hq[symidx(DD::NP, a, b) * DD::NS + symidx(D, c_, d)];
}

// shared-memory scratch of one warp's solve
template <int D> struct SolveScratch {
    static constexpr int NP = D + 1, DN = D * NP, NPAR = Dim<D>::NPAR;
    double Hd[DN * DN];
    double Z[DN], Zn[DN], Gam[DN];
    double dZ[NPAR][DN], HdZ[NPAR][DN];
    double A[NPAR][NPAR], g[NPAR];
    double dR[D][D], dt[D];
    double f, lam, dtheta;
    int go;
};

// Solves A x = b for a symmetric positive definite A through A = L D L^T (in place: unit lower L below the diagonal, D
// on it); returns false when A is not positive definite (same pivots as a Cholesky factorisation).  No square roots and
// one reciprocal per pivot: in float64 a division or a square root is a ~20-instruction dependent chain, and the damped
// solve sits on the critical path of every LM iteration of a small registration (one lane, everybody else waits).
template <int N> __host__ __device__ inline bool spd_solve(double A[N][N], double b[N]) {
    double inv[N];
    for (int j = 0; j < N; ++j) {
        double d = A[j][j];
        for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k] * A[k][k];
        if (!(d > 0.0) || !isfinite(d)) return false;
        A[j][j] = d;
        inv[j] = 1.0 / d;
        for (int i = j + 1; i < N; ++i) {
            double s = A[i][j];
            for (int k = 0; k < j; ++k) s -= A[i][k] * A[j][k] * A[k][k];
            A[i][j] = s * inv[j];
        }
    }
    for (int i = 0; i < N; ++i) {          // L y = b
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= A[i][k] * b[k];
        b[i] = s;
    }
    for (int i = 0; i < N; ++i) b[i] *= inv[i];   // D z = y
    for (int i = N - 1; i >= 0; --i) {     // L^T x = z
        double s = b[i];
        for (int k = i + 1; k < N; ++k) s -= A[k][i] * b[k];
        b[i] = s;
    }
    return true;
}

__host__ __device__ inline void rodrigues(const double w[3], double R[3][3]) {
    const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    double A, B;  // R = I + A K + B K^2
    if (th2 < 1e-16) { A = 1.0 - th2 / 6.0; B = 0.5 - th2 / 24.0; }
    else { const double th = sqrt(th2); A = sin(th) / th; B = (1.0 - cos(th)) / th2; }
    const double K[3][3] = {{0, -w[2], w[1]}, {w[2], 0, -w[0]}, {-w[1], w[0], 0}};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double k2 = 0.0;
            for (int k = 0; k < 3; ++k) k2 += K[i][k] * K[k][j];
            R[i][j] = (i == j ? 1.0 : 0.0) + A * K[i][j] + B * k2;
        }
}

// dR for the candidate step; dim 2 keeps the accumulated angle so dR is always an exact rot(dtheta)
template <int D>
__host__ __device__ inline void compose_rotation(const double* step_rot, const double dR[D][D], double dtheta,
                                                 double dRn[D][D], double* dtheta_n) {
    if constexpr (D == 2) {
        const double th = dtheta + step_rot[0];
        double s, c;
        sincos(th, &s, &c);
        dRn[0][0] = c; dRn[0][1] = -s; dRn[1][0] = s; dRn[1][1] = c;
        *dtheta_n = th;
    } else {
        double E[3][3];
        rodrigues(step_rot, E);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) dRn[i][j] = E[i][0] * dR[0][j] + E[i][1] * dR[1][j] + E[i][2] * dR[2][j];
        *dtheta_n = 0.0;
    }
}

// (spd_solve, dense_H_entry, inner_solve_2d and inner_solve_warp are __host__ __device__: tests/test_host.py and
// tests/test_solve3_host.py compile them for the host and check the minimiser without a GPU.)
// 2-D, ONE LANE: Levenberg-Marquardt on the reduced form  f(Z) = c - 2<G,Z> + <Z, H Z>,  Z = [dt | dR - I]  (the same
// iteration as the warp-cooperative 3-D version below: same damping, acceptance and stop rules), evaluated on the
// projection of the form onto the four numbers Z depends on.  With dR = rot(th):
//     Z = [[tx, p, -q], [ty, q, p]],  u = (tx, ty, p, q) = (tx, ty, cos th - 1, sin th),  Z_flat = B u,
// so f = c - 2 (B^T G).u + u^T (B^T H B) u with a constant 6x4 matrix B of 0 / +-1 entries.  M = B^T H B (10 distinct
// numbers) and B^T G are formed once; an LM iteration then costs ~150 register-resident flops.  (The first version
// applied the packed 6x6 form five times per LM iteration with its index arithmetic: ~3 k instructions of one lane,
// 2/3 of the time of a small registration - every other warp of the fused loop waits for this lane.  The
// warp-cooperative formulation was measured slower than one lane in 2-D: its hand-overs cost more than 3 parameters
// can save.)
__host__ __device__ inline void inner_solve_2d(const double* Hq, const double* G, double c0, int max_it, double dR[2][2],
                                      double dt[2], double* dtheta, double* fmin) {
    auto Hd = [&](int e, int f) { return dense_H_entry<2>(Hq, e * 6 + f); };
    const double M00 = Hd(0, 0), M01 = Hd(0, 3), M02 = Hd(0, 1) + Hd(0, 5), M03 = Hd(0, 4) - Hd(0, 2);
    const double M11 = Hd(3, 3), M12 = Hd(3, 1) + Hd(3, 5), M13 = Hd(3, 4) - Hd(3, 2);
    const double M22 = Hd(1, 1) + 2.0 * Hd(1, 5) + Hd(5, 5);
    const double M23 = (Hd(1, 4) - Hd(1, 2)) + (Hd(5, 4) - Hd(5, 2));
    const double M33 = Hd(4, 4) - 2.0 * Hd(4, 2) + Hd(2, 2);
    const double b0 = G[0], b1 = G[3], b2 = G[1] + G[5], b3 = G[4] - G[2];
    double tx = 0.0, ty = 0.0, th = 0.0, cs = 1.0, sn = 0.0;   // dR = rot(th) = [[cs, -sn], [sn, cs]]
    double f = c0;
    double lam = 1e-9;
    for (int it = 0; it < max_it; ++it) {
        // gradient wrt u: r = 2 (M u - b);  tangents: d/dtx = e0, d/dty = e1, d/dth = (0, 0, -sin th, cos th)
        const double p = cs - 1.0, q = sn;
        const double r0 = 2.0 * (M00 * tx + M01 * ty + M02 * p + M03 * q - b0);
        const double r1 = 2.0 * (M01 * tx + M11 * ty + M12 * p + M13 * q - b1);
        const double r2 = 2.0 * (M02 * tx + M12 * ty + M22 * p + M23 * q - b2);
        const double r3 = 2.0 * (M03 * tx + M13 * ty + M23 * p + M33 * q - b3);
        const double w2 = -sn, w3 = cs;
        const double g[3] = {r0, r1, r2 * w2 + r3 * w3};
        double A[3][3];
        A[0][0] = 2.0 * M00;
        A[1][0] = A[0][1] = 2.0 * M01;
        A[1][1] = 2.0 * M11;
        A[2][0] = A[0][2] = 2.0 * (M02 * w2 + M03 * w3);
        A[2][1] = A[1][2] = 2.0 * (M12 * w2 + M13 * w3);
        const double a22_gn = 2.0 * (w2 * (M22 * w2 + M23 * w3) + w3 * (M23 * w2 + M33 * w3));
        // u is linear in (tx, ty), so the only second-order term the Gauss-Newton matrix misses is r . d2u/dth2 =
        // -(r2 cos th + r3 sin th) in the (th, th) entry.  With it the iteration is Newton's (quadratic instead of
        // linear convergence to the same minimiser: 3-4 instead of 5-9 iterations); it is dropped for an iteration
        // whose matrix it makes indefinite.
        const double a22_newton = a22_gn - (r2 * cs + r3 * sn);
        bool newton = a22_newton > 0.0;
        const double gmax = fmax(fabs(g[0]), fmax(fabs(g[1]), fabs(g[2])));
        if (!(gmax > 1e-11 * fmax(1.0, fabs(f)))) break;
        bool accepted = false;
        double stepmax = 0.0;
        for (int tries = 0; tries < 40; ++tries) {
            double L[3][3], step[3];
            A[2][2] = newton ? a22_newton : a22_gn;
            for (int x = 0; x < 3; ++x) {
                for (int y = 0; y < 3; ++y) L[x][y] = A[x][y];
                L[x][x] += lam * A[x][x];
                step[x] = -g[x];
            }
            if (!spd_solve<3>(L, step)) {
                if (newton) { newton = false; continue; }
                lam = fmax(lam * 10.0, 1e-6);
                continue;
            }
            const double thn = th + step[2];
            double sn_n, cs_n;
            sincos(thn, &sn_n, &cs_n);
            const double txn = tx + step[0], tyn = ty + step[1], pn = cs_n - 1.0, qn = sn_n;
            const double m0 = M00 * txn + M01 * tyn + M02 * pn + M03 * qn;
            const double m1 = M01 * txn + M11 * tyn + M12 * pn + M13 * qn;
            const double m2 = M02 * txn + M12 * tyn + M22 * pn + M23 * qn;
            const double m3 = M03 * txn + M13 * tyn + M23 * pn + M33 * qn;
            const double lin = b0 * txn + b1 * tyn + b2 * pn + b3 * qn;
            const double quad = txn * m0 + tyn * m1 + pn * m2 + qn * m3;
            const double fn = c0 - 2.0 * lin + quad;
            const double pred = -(g[0] * step[0] + g[1] * step[1] + g[2] * step[2]);
            if (fn <= f || pred <= 1e-11 * fabs(f)) {
                tx = txn; ty = tyn; th = thn; cs = cs_n; sn = sn_n;
                f = fn;
                lam = fmax(lam * 0.1, 1e-12);
                accepted = true;
                stepmax = fmax(fabs(step[0]), fmax(fabs(step[1]), fabs(step[2])));
                break;
            }
            lam = fmax(lam * 10.0, 1e-9);
        }
        if (!accepted || stepmax < 1e-14) break;
    }
    dt[0] = tx; dt[1] = ty;
    dR[0][0] = cs; dR[0][1] = -sn; dR[1][0] = sn; dR[1][1] = cs;
    *dtheta = th;
    *fmin = f;
}

// Host builds of inner_solve_warp (tests/host_harness/solve3_host.cu) run its 32 lanes as 32 threads; the harness
// defines this hook as a barrier over them.  The library never calls the solver on the host.
extern void (*g_host_warp_sync)();

// the warp's barrier between the solver's phases: __syncwarp() on the device, the harness's barrier on the host
__host__ __device__ __forceinline__ void solve_warp_sync() {
#ifdef __CUDA_ARCH__
    __syncwarp();
#else
    g_host_warp_sync();
#endif
}

// Minimise the reduced form  f(Z) = c - 2<G,Z> + <Z, H Z>,  Z = [dt | dR - I]  (flat index c * NP + a), over
// (dt, dR in SO(D)) by Levenberg-Marquardt.  WARP-COOPERATIVE: all 32 lanes of one warp call this with the same
// arguments; the matrix-vector products, tangents and normal equations are spread over the lanes (one row or one
// entry per lane, every sum in a fixed order), lane 0 runs the damped solve and the acceptance test.  A one-lane
// version of the same algorithm executed ~17 k instructions per LM iteration in 3-D (it was the slowest kernel of a
// small registration: 37 us per launch); this one executes ~1.3 k.  Results in sc.dR, sc.dt, sc.dtheta, sc.f.
template <int D>
__host__ __device__ void inner_solve_warp(SolveScratch<D>& sc, const double* G, double c0, int max_it, int lane) {
    using SS = SolveScratch<D>;
    constexpr int NP = SS::NP, DN = SS::DN, NPAR = SS::NPAR;
    if (lane == 0) {
        for (int i = 0; i < D; ++i) {
            sc.dt[i] = 0.0;
            for (int j = 0; j < D; ++j) sc.dR[i][j] = (i == j) ? 1.0 : 0.0;
        }
        sc.dtheta = 0.0;
        sc.f = c0;
        sc.lam = 1e-9;
    }
    if (lane < DN) sc.Z[lane] = 0.0;
    solve_warp_sync();
    for (int it = 0; it < max_it; ++it) {
        // gradient wrt Z: Gam = 2 (H Z - G)
        if (lane < DN) {
            const double* row = sc.Hd + lane * DN;
            double s = 0.0;
            for (int e = 0; e < DN; ++e) s += row[e] * sc.Z[e];
            sc.Gam[lane] = 2.0 * (s - G[lane]);
        }
        // tangent directions dZ_x: translations, then rotations [0 | E_k dR]
        for (int q = lane; q < NPAR * DN; q += 32) {
            const int x = q / DN, e = q % DN, c_ = e / NP, a = e % NP;
            double v = 0.0;
            if (x < D) {
                v = (c_ == x && a == 0) ? 1.0 : 0.0;
            } else if (a > 0) {
                if constexpr (D == 2) {
                    // E = [[0,-1],[1,0]]
                    v = (c_ == 0) ? -sc.dR[1][a - 1] : sc.dR[0][a - 1];
                } else {
                    const int k = x - 3, k1 = (k + 1) % 3, k2 = (k + 2) % 3;  // (E_k M)[k1] = -M[k2], (E_k M)[k2] = M[k1]
                    if (c_ == k1) v = -sc.dR[k2][a - 1];
                    else if (c_ == k2) v = sc.dR[k1][a - 1];
                }
            }
            sc.dZ[x][e] = v;
        }
        solve_warp_sync();
        for (int q = lane; q < NPAR * DN; q += 32) {
            const int x = q / DN, r = q % DN;
            const double* row = sc.Hd + r * DN;
            double s = 0.0;
            for (int e = 0; e < DN; ++e) s += row[e] * sc.dZ[x][e];
            sc.HdZ[x][r] = s;
        }
        solve_warp_sync();
        if (lane < NPAR) {
            double s = 0.0;
            for (int e = 0; e < DN; ++e) s += sc.Gam[e] * sc.dZ[lane][e];
            sc.g[lane] = s;
        }
        for (int q = lane; q < NPAR * NPAR; q += 32) {
            const int x = q / NPAR, y = q % NPAR;
            if (y <= x) {
                double s = 0.0;
                for (int e = 0; e < DN; ++e) s += sc.dZ[x][e] * sc.HdZ[y][e];
                sc.A[x][y] = sc.A[y][x] = 2.0 * s;
            }
        }
        solve_warp_sync();
        if (lane == 0) {
            double f = sc.f, lam = sc.lam;
            double gmax = 0.0;
            for (int x = 0; x < NPAR; ++x) gmax = fmax(gmax, fabs(sc.g[x]));
            bool go = gmax > 1e-11 * fmax(1.0, fabs(f));
            if (go) {
                // Second-order term the Gauss-Newton matrix 2 J^T H J misses: Z is linear in dt, and for the left
                // perturbation dR <- exp([eta]x) dR,  d2 dR / d eta_k d eta_l = (E_k E_l + E_l E_k) dR / 2  with
                // E_k E_l = e_l e_k^T - delta_kl I, so  Gam . d2Z = (P_kl + P_lk) / 2 - delta_kl tr P,  P = dR Gam_R^T
                // (Gam_R: the rotation columns of the gradient wrt Z).  With it the iteration is Newton's (quadratic
                // instead of linear convergence to the same minimiser); it is dropped for an iteration whose matrix it
                // makes indefinite.
                double Cn[3][3] = {};
                bool newton = false;
                if constexpr (D == 3) {
                    double P[3][3], trP = 0.0;
                    for (int k = 0; k < 3; ++k)
                        for (int l = 0; l < 3; ++l) {
                            double v = 0.0;
                            for (int j = 0; j < 3; ++j) v += sc.dR[k][j] * sc.Gam[l * NP + 1 + j];
                            P[k][l] = v;
                        }
                    trP = P[0][0] + P[1][1] + P[2][2];
                    for (int k = 0; k < 3; ++k)
                        for (int l = 0; l < 3; ++l) Cn[k][l] = 0.5 * (P[k][l] + P[l][k]) - (k == l ? trP : 0.0);
                    newton = true;
                }
                bool accepted = false;
                double stepmax = 0.0;
                for (int tries = 0; tries < 40; ++tries) {
                    double L[NPAR][NPAR], step[NPAR];
                    for (int x = 0; x < NPAR; ++x) {
                        for (int y = 0; y < NPAR; ++y) {
                            L[x][y] = sc.A[x][y];
                            if (newton && x >= D && y >= D) L[x][y] += Cn[x - D][y - D];
                        }
                        L[x][x] += lam * sc.A[x][x];
                        step[x] = -sc.g[x];
                    }
                    if (!spd_solve<NPAR>(L, step)) {
                        if (newton) { newton = false; continue; }
                        lam = fmax(lam * 10.0, 1e-6);
                        continue;
                    }
                    double dRn[D][D], dtn[D], thn;
                    compose_rotation<D>(step + D, sc.dR, sc.dtheta, dRn, &thn);
                    for (int c_ = 0; c_ < D; ++c_) {
                        dtn[c_] = sc.dt[c_] + step[c_];
                        sc.Zn[c_ * NP] = dtn[c_];
                        for (int j = 0; j < D; ++j) sc.Zn[c_ * NP + 1 + j] = dRn[c_][j] - (c_ == j ? 1.0 : 0.0);
                    }
                    // f(Zn) = c - 2 <G, Zn> + <Zn, H Zn>
                    double lin = 0.0, quad = 0.0;
                    for (int r = 0; r < DN; ++r) {
                        const double* row = sc.Hd + r * DN;
                        double hz = 0.0;
                        for (int e = 0; e < DN; ++e) hz += row[e] * sc.Zn[e];
                        lin += G[r] * sc.Zn[r];
                        quad += sc.Zn[r] * hz;
                    }
                    const double fn = c0 - 2.0 * lin + quad;
                    double pred = 0.0;
                    for (int x = 0; x < NPAR; ++x) pred -= sc.g[x] * step[x];
                    if (fn <= f || pred <= 1e-11 * fabs(f)) {
                        for (int c_ = 0; c_ < D; ++c_) {
                            sc.dt[c_] = dtn[c_];
                            for (int j = 0; j < D; ++j) sc.dR[c_][j] = dRn[c_][j];
                        }
                        for (int e = 0; e < DN; ++e) sc.Z[e] = sc.Zn[e];
                        sc.dtheta = thn;
                        f = fn;
                        lam = fmax(lam * 0.1, 1e-12);
                        accepted = true;
                        for (int x = 0; x < NPAR; ++x) stepmax = fmax(stepmax, fabs(step[x]));
                        break;
                    }
                    lam = fmax(lam * 10.0, 1e-9);
                }
                if (!accepted || stepmax < 1e-14) go = false;
            }
            sc.f = f;
            sc.lam = lam;
            sc.go = go ? 1 : 0;
        }
        solve_warp_sync();
        if (!sc.go) break;
    }
}

struct SolveArgs {
    const double* partial;  // [n_pairs][blocks_per_pair][NRED]
    int blocks_per_pair;
    int n_pairs;
    double* sum_out;        // if set: write the summed rows [n_pairs][NRED] (+mu) and return
    PairState* state;
    int max_iterations;
    int inner_max_iterations;
    double tolerance;
    double* d_T;            // [n_pairs][(D+1)^2]
    int* d_n_outer;
    int* d_converged;
    double* d_loss_hist;    // optional [n_pairs][max_iterations]
    double* d_T_hist;       // optional [n_pairs][max_iterations+1][(D+1)^2]
    int* d_inliers;         // optional [n_pairs][max_iterations]
    int* n_active;
    const int* active_list;   // optional (see ObjArgs): warp w of the grid handles pair active_list[w]
    const int* n_list;
};

template <int D> __device__ inline void write_T(double* out, const PairState& st) {
    for (int i = 0; i < D; ++i) {
        for (int j = 0; j < D; ++j) out[i * (D + 1) + j] = st.R[i * 3 + j];
        out[i * (D + 1) + D] = st.t[i];
    }
    for (int j = 0; j < D; ++j) out[D * (D + 1) + j] = 0.0;
    out[D * (D + 1) + D] = 1.0;
}

constexpr int SOLVE_WARPS = 4;
constexpr int PRESUM_SPAN = 64;   // block partials folded into one row by presum_kernel

// Large pairs have thousands of block partials per pair and K4 sums them with one warp: fold PRESUM_SPAN consecutive
// rows into one first (fixed order: bitwise reproducible).  grid (ceil(blocks_per_pair / PRESUM_SPAN), n_pairs), NRED threads.
template <int D>
__global__ void presum_kernel(const double* __restrict__ partial, int blocks_per_pair, double* __restrict__ out,
                              int out_per_pair, const PairState* __restrict__ state) {
    constexpr int NRED = Dim<D>::NRED;
    const int pair = blockIdx.y;
    if (state[pair].status != PAIR_ACTIVE) return;
    const int b0 = blockIdx.x * PRESUM_SPAN, b1 = min(b0 + PRESUM_SPAN, blocks_per_pair);
    const double* p = partial + ((size_t)pair * blocks_per_pair + b0) * NRED + threadIdx.x;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;   // four chains, combined in a fixed order
    int b = b0;
    for (; b + 4 <= b1; b += 4) {
        s0 += p[0]; s1 += p[NRED]; s2 += p[2 * NRED]; s3 += p[3 * NRED];
        p += 4 * NRED;
    }
    for (; b < b1; ++b) { s0 += p[0]; p += NRED; }
    out[((size_t)pair * out_per_pair + blockIdx.x) * NRED + threadIdx.x] = (s0 + s1) + (s2 + s3);
}

// Tail of one outer iteration of one pair, run by ONE WARP (all 32 lanes call it): `sums` is the pair's summed reduced
// form ([NRED] doubles, shared memory), `sc` the warp's scratch, `st` the pair's state (read by the caller).
// The updated state goes to `stp` (a.state + pair; the fused loop keeps the state in shared memory).
template <int D>
__device__ void solve_pair(const SolveArgs& a, const int pair, PairState st, const double* sums, SolveScratch<D>& sc,
                           PairState* stp) {
    using DD = Dim<D>;
    constexpr int NQ = DD::NQ, DN2 = SolveScratch<D>::DN * SolveScratch<D>::DN;
    const int lane = threadIdx.x & 31;
    double dR[D][D], dtc[D], dtheta, fmin;
    if constexpr (D == 2) {
        if (lane != 0) return;
        inner_solve_2d(sums, sums + DD::NH, sums[NQ], a.inner_max_iterations, dR, dtc, &dtheta, &fmin);
    } else {
        for (int e = lane; e < DN2; e += 32) sc.Hd[e] = dense_H_entry<D>(sums, e);
        __syncwarp();
        inner_solve_warp<D>(sc, sums + DD::NH, sums[NQ], a.inner_max_iterations, lane);
        if (lane != 0) return;
        for (int i = 0; i < D; ++i) {
            dtc[i] = sc.dt[i];
            for (int j = 0; j < D; ++j) dR[i][j] = sc.dR[i][j];
        }
        dtheta = sc.dtheta;
        fmin = sc.f;
    }
    const int inliers = (int)(sums[NQ + 1] + 0.5);

    const int it = st.iter;
    const double delta = fabs(st.last_loss - fmin);  // gicp.py:155
    if (a.d_loss_hist) a.d_loss_hist[(size_t)pair * a.max_iterations + it] = fmin;
    if (a.d_inliers) a.d_inliers[(size_t)pair * a.max_iterations + it] = inliers;
    a.d_n_outer[pair] = it + 1;
    if (delta < a.tolerance) {  // gicp.py:160-162: stop WITHOUT applying this iteration's offset
        st.status = PAIR_CONVERGED;
        st.converged_at = it;
    } else {
        st.last_loss = fmin;
        // un-centre:  r = q - dR p' - dt,  dt = dt_c - (dR - I) mu
        double dt[D];
        for (int i = 0; i < D; ++i) {
            double s = dtc[i];
            for (int j = 0; j < D; ++j) s -= (dR[i][j] - (i == j ? 1.0 : 0.0)) * st.mu[j];
            dt[i] = s;
        }
        // T_{k+1} = [dR R_k | dR t_k + dt]
        double Rn[D][D], tn[D];
        for (int i = 0; i < D; ++i) {
            double s = dt[i];
            for (int j = 0; j < D; ++j) s += dR[i][j] * st.t[j];
            tn[i] = s;
        }
        if constexpr (D == 2) {
            st.theta += dtheta;  // the reference rebuilds T from (tx, ty, theta), gicp.py:166
            double s, c;
            sincos(st.theta, &s, &c);
            Rn[0][0] = c; Rn[0][1] = -s; Rn[1][0] = s; Rn[1][1] = c;
        } else {
            for (int i = 0; i < D; ++i)
                for (int j = 0; j < D; ++j) {
                    double s = 0.0;
                    for (int k = 0; k < D; ++k) s += dR[i][k] * st.R[k * 3 + j];
                    Rn[i][j] = s;
                }
        }
        for (int i = 0; i < 9; ++i) st.Rp[i] = st.R[i];
        for (int i = 0; i < 3; ++i) st.tp[i] = st.t[i];
        for (int i = 0; i < D; ++i) {
            for (int j = 0; j < D; ++j) st.R[i * 3 + j] = Rn[i][j];
            st.t[i] = tn[i];
        }
        st.iter = it + 1;
        if (a.d_T_hist) write_T<D>(a.d_T_hist + ((size_t)pair * (a.max_iterations + 1) + it + 1) * (D + 1) * (D + 1), st);
        if (st.iter >= a.max_iterations) st.status = PAIR_MAXITER;
    }
    write_T<D>(a.d_T + (size_t)pair * (D + 1) * (D + 1), st);
    a.d_converged[pair] = st.converged_at;
    *stp = st;
    if (st.status != PAIR_ACTIVE && a.n_active) atomicSub(a.n_active, 1);
}

template <int D>
__global__ void __launch_bounds__(SOLVE_WARPS * 32) solve_kernel(const SolveArgs a) {
    using DD = Dim<D>;
    constexpr int NRED = DD::NRED, NQ = DD::NQ;
    __shared__ double s_red[SOLVE_WARPS][NRED];
    __shared__ SolveScratch<D> s_sc[SOLVE_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int pair = blockIdx.x * SOLVE_WARPS + warp;
    if (a.active_list) {
        if (pair >= *a.n_list) return;
        pair = a.active_list[pair];
    }
    if (pair >= a.n_pairs) return;
    PairState st = a.state[pair];
    if (!a.sum_out && st.status != PAIR_ACTIVE) return;
    for (int j = lane; j < NRED; j += 32) {
        double s = 0.0;
        const double* p = a.partial + (size_t)pair * a.blocks_per_pair * NRED + j;
        for (int b = 0; b < a.blocks_per_pair; ++b) s += p[(size_t)b * NRED];
        s_red[warp][j] = s;
    }
    __syncwarp();
    if (a.sum_out) {
        for (int j = lane; j < NRED; j += 32) {
            double v = s_red[warp][j];
            if (j >= NQ + 2 && j < NQ + 2 + D) v = st.mu[j - NQ - 2];
            a.sum_out[(size_t)pair * NRED + j] = v;
        }
        return;
    }
    solve_pair<D>(a, pair, st, s_red[warp], s_sc[warp], a.state + pair);
}

// One block: the pairs that are still iterating, in ascending order -> list[0 .. *n_list)
constexpr int COMPACT_THREADS = 1024;
__global__ void __launch_bounds__(COMPACT_THREADS) compact_active_kernel(const PairState* __restrict__ state, int n_pairs,
                                                                         int* __restrict__ list, int* __restrict__ n_list) {
    __shared__ int s_warp[COMPACT_THREADS / 32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int p0 = 0; p0 < n_pairs; p0 += COMPACT_THREADS) {
        const int p = p0 + threadIdx.x;
        const bool act = p < n_pairs && state[p].status == PAIR_ACTIVE;
        const unsigned bal = __ballot_sync(0xffffffffu, act);
        if (lane == 0) s_warp[w] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int i = 0; i < COMPACT_THREADS / 32; ++i) {
            const int c = s_warp[i];
            if (i < w) before += c;
            total += c;
        }
        if (act) list[s_base + before + __popc(bal & ((1u << lane) - 1u))] = p;
        __syncthreads();
        if (threadIdx.x == 0) s_base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_list = s_base;
}

// initialise the state of one pair (gicp.py:107-110): T = T0 or identity, last_loss = inf
template <int D>
__device__ inline void init_pair_state(PairState* stp, const double* T0, const double* tgt_bbox, int pair, double* d_T,
                                       double* d_T_hist, int max_iterations, int* d_n_outer, int* d_converged) {
    PairState st;
    for (int i = 0; i < 9; ++i) st.R[i] = (i % 4 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 3; ++i) { st.t[i] = 0.0; st.mu[i] = 0.5 * (tgt_bbox[pair * 6 + i] + tgt_bbox[pair * 6 + 3 + i]); }
    st.theta = 0.0;
    if (T0) {
        const double* T = T0 + (size_t)pair * (D + 1) * (D + 1);
        for (int i = 0; i < D; ++i) {
            for (int j = 0; j < D; ++j) st.R[i * 3 + j] = T[i * (D + 1) + j];
            st.t[i] = T[i * (D + 1) + D];
        }
        if (D == 2) st.theta = atan2(st.R[3], st.R[0]);
    }
    for (int i = 0; i < 9; ++i) st.Rp[i] = st.R[i];
    for (int i = 0; i < 3; ++i) st.tp[i] = st.t[i];
    st.last_loss = INFINITY;
    st.iter = 0;
    st.status = PAIR_ACTIVE;
    st.converged_at = -1;
    st.pad = 0;
    *stp = st;
    if (d_T) write_T<D>(d_T + (size_t)pair * (D + 1) * (D + 1), st);
    if (d_T_hist) write_T<D>(d_T_hist + (size_t)pair * (max_iterations + 1) * (D + 1) * (D + 1), st);
    if (d_n_outer) d_n_outer[pair] = 0;
    if (d_converged) d_converged[pair] = -1;
}

template <int D>
__global__ void init_state_kernel(PairState* state, const double* T0, const double* tgt_bbox, int n_pairs,
                                  double* d_T, double* d_T_hist, int max_iterations, int* d_n_outer,
                                  int* d_converged, int* n_active) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair == 0 && n_active) *n_active = n_pairs;   // pairs still iterating (K4 counts it down, the host polls it)
    if (pair >= n_pairs) return;
    init_pair_state<D>(state + pair, T0, tgt_bbox, pair, d_T, d_T_hist, max_iterations, d_n_outer, d_converged);
}

}  // namespace gicp
