// Registration quality at given transforms (gicpEvaluate; semantics in include/gicp_b200.h).  The correspondences and
// the reduced form come from the stage path's own kernels (correspond_kernel, accumulate_kernel, solve_kernel's
// sum_out fold); this file adds the one per-pair kernel that turns them into the quality row, H and b.
#pragma once
#include "common.cuh"

namespace gicp {

constexpr int GICP_NQ = 4;   // GICP_NQUALITY: n, fitness, inlier RMSE, loss

// Coefficient of p'_a in row k of the Jacobian column of rotation parameter i: J_rot(i)_k = sum_a g * p'_a.  3-D: the
// derivative of (w x p')_k by w_i, Levi-Civita eps(k, i, a).  2-D: the one rotation is about the (absent) z axis,
// d(R(theta) p')/dtheta = (-p'_y, p'_x) = eps(k, z, a).
template <int D> __host__ __device__ __forceinline__ double rot_gen(int i, int k, int a) {
    const int j = D == 3 ? i : 2;
    return 0.5 * (double)((k - j) * (j - a) * (a - k));
}

// The map from one pair's folded reduced form (gicpNormalEquations' row: sums over p~ = (1, d), d = p' - mu, and mu)
// to the quality row, H (NPAR x NPAR, rotation first) and b (NPAR).  H = sum J^T W J and b = sum J^T W e with
// J = [J_rot | I] are exact linear functions of the sums once the centring is undone:
//   sum p'_a W = mu_a sum W + sum d_a W,   sum p'_a p'_b W = mu_a mu_b sum W + mu_a sum d_b W + mu_b sum d_a W + sum d_a d_b W,
//   sum p'_a v = mu_a sum v + sum d_a v.
// Host-callable: tests/host_harness/quality_host.cu checks it against numpy without a GPU.  With n = 0 every output is
// 0 and mu (from an empty target's bounding box, possibly not finite) is not read.
template <int D>
__host__ __device__ inline void quality_from_reduced(const double* red, double sum_d2, int n_src, double* q, double* H,
                                                     double* b) {
    using DD = Dim<D>;
    constexpr int NP = DD::NP, NS = DD::NS, NH = DD::NH, NQ = DD::NQ, NPAR = DD::NPAR, NR = NPAR - D;
    const double n = red[NQ + 1];
    if (!(n > 0.0)) {
        for (int i = 0; i < GICP_NQ; ++i) q[i] = 0.0;
        for (int i = 0; i < NPAR * NPAR; ++i) H[i] = 0.0;
        for (int i = 0; i < NPAR; ++i) b[i] = 0.0;
        return;
    }
    q[0] = n;
    q[1] = n_src > 0 ? n / (double)n_src : 0.0;
    q[2] = sqrt(sum_d2 / n);
    q[3] = red[NQ];
    const double* mu = red + NQ + 2;
    // S(a, b, k, l) = sum p~_a p~_b W_kl, V(k, a) = sum v_k p~_a (p~_0 = 1)
    auto S = [&](int a, int bb, int k, int l) { return red[symidx(NP, a, bb) * NS + symidx(D, k, l)]; };
    auto V = [&](int k, int a) { return red[NH + k * NP + a]; };
    auto A = [&](int a, int k, int l) { return mu[a] * S(0, 0, k, l) + S(0, a + 1, k, l); };   // sum p'_a W_kl
    auto B = [&](int a, int bb, int k, int l) {                                                 // sum p'_a p'_b W_kl
        return mu[a] * mu[bb] * S(0, 0, k, l) + mu[a] * S(0, bb + 1, k, l) + mu[bb] * S(0, a + 1, k, l) +
               S(a + 1, bb + 1, k, l);
    };
#pragma unroll
    for (int i = 0; i < NR; ++i) {
#pragma unroll
        for (int j = i; j < NR; ++j) {   // rotation x rotation: sum J_rot(i)^T W J_rot(j)
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k)
#pragma unroll
                for (int a = 0; a < D; ++a) {
                    const double gi = rot_gen<D>(i, k, a);
                    if (gi == 0.0) continue;
#pragma unroll
                    for (int l = 0; l < D; ++l)
#pragma unroll
                        for (int c = 0; c < D; ++c) {
                            const double gj = rot_gen<D>(j, l, c);
                            if (gj != 0.0) s += gi * gj * B(a, c, k, l);
                        }
                }
            H[i * NPAR + j] = H[j * NPAR + i] = s;
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {    // rotation x translation: sum J_rot(i)^T W e_j
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k)
#pragma unroll
                for (int a = 0; a < D; ++a) {
                    const double gi = rot_gen<D>(i, k, a);
                    if (gi != 0.0) s += gi * A(a, k, j);
                }
            H[i * NPAR + NR + j] = H[(NR + j) * NPAR + i] = s;
        }
        double s = 0.0;                  // sum J_rot(i)^T v
#pragma unroll
        for (int k = 0; k < D; ++k)
#pragma unroll
            for (int a = 0; a < D; ++a) {
                const double gi = rot_gen<D>(i, k, a);
                if (gi != 0.0) s += gi * (mu[a] * V(k, 0) + V(k, a + 1));
            }
        b[i] = s;
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
#pragma unroll
        for (int l = 0; l < D; ++l) H[(NR + k) * NPAR + NR + l] = S(0, 0, k, l);
        b[NR + k] = V(k, 0);
    }
}

constexpr int QUALITY_THREADS = 256;

// One block per pair: sum d_i^2 over the pair's gated-in rows (idx >= 0) of the correspondence pass, in a fixed order
// (per-thread strided sums, warp shuffles, the warps in order: bitwise reproducible), then quality_from_reduced on the
// pair's folded row `red`.  idx / dist are in input order; the pair's rows are [pt_begin, pt_end) of its source meta.
// Any of quality / H / b may be null.
template <int D>
__global__ void __launch_bounds__(QUALITY_THREADS) quality_kernel(const double* __restrict__ red,
                                                                  const CloudMeta* __restrict__ src_meta,
                                                                  const int* __restrict__ idx,
                                                                  const double* __restrict__ dist,
                                                                  double* __restrict__ quality, double* __restrict__ H,
                                                                  double* __restrict__ b) {
    constexpr int NRED = Dim<D>::NRED, NPAR = Dim<D>::NPAR;
    const int pair = blockIdx.x;
    const CloudMeta ms = src_meta[pair];
    double s = 0.0;
    for (int i = ms.pt_begin + (int)threadIdx.x; i < ms.pt_end; i += QUALITY_THREADS)
        if (idx[i] >= 0) s += dist[i] * dist[i];
    __shared__ double s_part[QUALITY_THREADS / 32];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x != 0) return;
    double sum_d2 = 0.0;
#pragma unroll
    for (int w = 0; w < QUALITY_THREADS / 32; ++w) sum_d2 += s_part[w];
    double q[GICP_NQ], h[NPAR * NPAR], g[NPAR];
    quality_from_reduced<D>(red + (size_t)pair * NRED, sum_d2, ms.pt_end - ms.pt_begin, q, h, g);
    if (quality)
        for (int i = 0; i < GICP_NQ; ++i) quality[(size_t)pair * GICP_NQ + i] = q[i];
    if (H)
        for (int i = 0; i < NPAR * NPAR; ++i) H[(size_t)pair * NPAR * NPAR + i] = h[i];
    if (b)
        for (int i = 0; i < NPAR; ++i) b[(size_t)pair * NPAR + i] = g[i];
}

}  // namespace gicp
