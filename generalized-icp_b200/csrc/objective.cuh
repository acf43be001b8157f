// K3: the fused per-iteration pass.  Replaces, per outer iteration of the reference loop,
//   apply_transformation (gicp.py:119), the per-point 1-NN query + d_max gate (gicp.py:129-138),
//   W_i = inv(C_src,k[i] + C_tgt[j]) (gicp.py:143-145; C_src,k = R_k C_src,0 R_k^T, which equals the
//   reference's recomputation on the transformed cloud, gicp.py:120) and every loss / grad_loss
//   evaluation of the inner minimisation (gicp.py:52-76): with W and the matches frozen, the
//   residual  r_i = e_i - Z p~_i  (e_i = q_i - p'_i, p~_i = (1, p'_i - mu), Z = [dt | dR - I])  is
//   linear in Z, so one streaming pass that reduces  sum p~p~^T (x) W,  sum (W e) p~^T  and
//   sum e^T W e  gives the inner objective exactly; K4 then minimises it without touching the
//   points again.
//
// One thread per source point; a warp owns 32 consecutive points of the source's Morton order (a
// compact blob), stages the target cells around the blob's image with TMA bulk copies
// (stream.cuh) and every lane scans the staged candidates (broadcast LDS.128).
// Exactness: an fp32 distance with a proven error margin filters candidates, the ranked
// key is the float64 squared distance of the oracle, ties go to the lower target index.
// Per-point algebra runs in fp64; products are accumulated per thread in the storage precision,
// reduced with warp shuffles, then across warps and blocks in fp64 in a fixed order (bitwise
// reproducible, no float atomics).
#pragma once
#include "../../include/gicp_b200.h"
#include "common.cuh"
#include "stream.cuh"

namespace gicp {

constexpr int OBJ_THREADS = 128;
constexpr int OBJ_STAGE_BYTES = 2048;  // per warp (small: occupancy matters more than window size here)
constexpr int OBJ_GROUP_REACH = 4;
constexpr int OBJ_MAX_PPT = 16;   // search blocks and the fused loop; the accumulation alone runs up to twice that

template <typename Real> struct ObjArgs {
    const CloudMeta* src_meta;
    const PRec<Real>* src_spts;
    const Real* src_cov;
    const CloudMeta* tgt_meta;
    const int* tgt_cell_start;
    const int* tgt_lut;
    const PRec<Real>* tgt_spts;   // records carry the cloud-local input index in .idx (tie-break key)
    const Real* tgt_cov;
    const int* tgt_inv_perm;      // input row (global) -> sorted position
    int* match;                   // [n_src_total], source nn order: matched target position or -1.  Written by
                                  // correspond_kernel, read by accumulate_kernel; with use_prev the previous
                                  // iteration's match bounds the next search
    int use_prev;
    float* slack;                 // [n_src_total]: how far a point may still move before its match can change
    const PairState* state;
    const double* T_override;  // optional [n_pairs][(D+1)^2], device
    double* partial;           // [n_pairs][blocks_per_pair][NRED]
    int blocks_per_pair;
    int ppt;
    double d_max;
    int* out_idx;
    double* out_dist;
    double* out_W;
    int slice_begin, slice_end;
    int ignore_status;
    int track_max_cells;      // per-lane walk only when the ball spans at most this many cells
    int centre_first;
    int shell_search;         // untracked lanes search per-lane shells before the cooperative phase
    // optional compacted list of the pairs that are still iterating (compact_active_kernel): blockIdx.y is then a
    // slot of that list, and slots beyond *n_list return at once - in the convergence tail of a large batch a launch
    // otherwise starts (and immediately retires) tens of thousands of blocks of finished pairs
    const int* active_list;
    const int* n_list;
    // robust kernel (gicpSetRobustKernel): read only by the Robust instantiations of accumulate_block
    int robust_kind;
    double robust_scale;
    // adaptive scale (gicpSetRobustKernelAdaptive, scale.cuh): c_p = adaptive_scale(scale_kappa, median, scale_min).
    // pair_scale: the scale of every pair at this iteration, written by the select of the multi-launch loop and read by
    // the Robust accumulation instead of robust_scale when set
    const double* pair_scale;
    double scale_kappa, scale_min;
};

// dynamic shared memory of the search blocks: one mbarrier per warp (128 B), the warps' TMA stages, the work list of
// ppt * OBJ_THREADS indices.  The fused loop with an adaptive scale appends the select's keys behind it.
__host__ __device__ inline size_t obj_smem(int ppt) {
    return 128 + (size_t)(OBJ_THREADS / 32) * OBJ_STAGE_BYTES + (size_t)OBJ_THREADS * ppt * sizeof(int);
}

// ---- the two fp32 bounds of the exact search (host-callable: tests/host_harness/bounds_host.cu checks them) ----
// Filter: for a candidate c, a query p' (fp64) and its fp32 rounding f, d2_32 = |c - f|^2 in fp32 satisfies
// |d2_32 - d2| <= 2 sqrt(3) d u P + 6 u d2  (u = 2^-24, P >= max|f_i|).  c1 is the coefficient of d in that bound.
__host__ __device__ __forceinline__ float filter_c1(float Pf) { return 5e-7f * Pf * 1.0001f; }
// Threshold on d2_32 that every candidate with exact d2 <= bd passes: b = bd rounded up to fp32, rs ~ 1/sqrt(max(b,
// 1e-30)).  The device passes rsqrtf (2 ulp of error, covered by the 1.0001 in c1).
__host__ __device__ __forceinline__ float filter_thr_of(float b, float rs, float c1) {
    const float sq = fmaxf(b, 1e-30f) * rs;           // sqrt(max(b, 1e-30)) >= sqrt(b): never under the bound
    return fmaf(b, 1.000002f, c1 * sq) + 1e-30f;
}
// Slack of a tracked, matched point: how far it may move before its match can change.  d1 = its match distance
// rounded up, m2 = second smallest fp32 squared distance seen (INFINITY: none), rad32 = lower bound of the distance
// to every target point outside the examined cell box.  Never more than half the gap to the true runner-up.
__host__ __device__ __forceinline__ float match_slack(float d1, float m2, float rad32, float c1, float Pf) {
    // runner-up: at least lb2 away (fp32 error bound of the filter), or outside the examined ball
    const float lb2 = m2 * 0.999999f - c1 * sqrtf(m2);
    const float d2e = fminf(sqrtf(fmaxf(lb2, 0.f)) * 0.999999f, rad32);
    float sl = fmaxf(0.f, 0.5f * (d2e - d1) * 0.99999f - 1e-6f * (Pf + d1));
    if (!(m2 < INFINITY)) sl = fmaxf(0.f, 0.5f * (fminf(rad32, 1e30f) - d1) * 0.99999f - 1e-6f * (Pf + d1));
    return sl;
}

// ---- robust kernel weight (IRLS; semantics in include/gicp_b200.h), host-callable: tests/host_harness/robust_host.cu
// checks it bit for bit against the float64 formulas of the oracle.  Every product and sum is rounded on its own (no
// FMA contraction), so the device, the host and numpy agree, and a huge scale gives w == 1.0 exactly for Huber and
// Cauchy (u * u underflows to 0). ----
__host__ __device__ __forceinline__ double robust_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double robust_weight(int kind, double d, double c) {
    const double u = d / c;
    if (kind == GICP_ROBUST_HUBER) return d <= c ? 1.0 : c / d;
    if (kind == GICP_ROBUST_CAUCHY) return 1.0 / (1.0 + robust_mul(u, u));
    if (kind == GICP_ROBUST_TUKEY) {
        const double a = 1.0 - robust_mul(u, u);
        return u < 1.0 ? robust_mul(a, a) : 0.0;
    }
    return 1.0;
}

// ---- adaptive scale (semantics in include/gicp_b200.h): c = max(min_scale, kappa * m), kappa * m rounded once, and
// min_scale when the two are equal.  m = 0 (no gated-in correspondence) gives min_scale.  Host-callable:
// tests/host_harness/adaptive_host.cu checks it bit for bit against numpy. ----
__host__ __device__ __forceinline__ double adaptive_scale(double kappa, double m, double min_scale) {
    const double c = robust_mul(kappa, m);
    return c > min_scale ? c : min_scale;
}

// p' = R p + t (gicp.py:119).  K3b and the scale select (scale.cuh) both form it here, so the distance the select
// orders is bit for bit the one K3b gates on and weights with (the device contracts these products into FMAs).
template <int D, typename Real>
__device__ __forceinline__ void transform_point(const double (&R)[D][D], const double (&t)[D], const PRec<Real>& p,
                                                double (&pp)[3]) {
    const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double v = R[i][0] * px + R[i][1] * py + t[i];
        if constexpr (D == 3) v += R[i][2] * pz;
        pp[i] = v;
    }
}

template <typename Real>
__device__ __forceinline__ int obj_pair_of_block(const ObjArgs<Real>& a) {
    if (!a.active_list) return (int)blockIdx.y;
    return ((int)blockIdx.y < *a.n_list) ? a.active_list[blockIdx.y] : -1;
}

// One block of the search: points [bx * ppt * OBJ_THREADS, ...) of pair `pair`.  `ws` is the warp's TMA stage
// (buffer, mbarrier, phase); it is carried by the caller so that the fused registration loop (register_loop_kernel)
// can call this once per outer iteration on one initialised mbarrier.
// `stp`: the pair's state (a.state + pair; the fused loop keeps it in shared memory instead).
template <int D, typename Real>
__device__ __forceinline__ void correspond_block(const ObjArgs<Real>& a, const int pair, const int bx,
                                                 WarpStage<Real>& ws, unsigned char* smem_raw, const PairState* stp) {
    const PairState st = *stp;
    if (!a.ignore_status && st.status != PAIR_ACTIVE) return;

    double R[D][D], t[D];
    if (a.T_override) {
        const double* T = a.T_override + (size_t)pair * (D + 1) * (D + 1);
#pragma unroll
        for (int i = 0; i < D; ++i) {
#pragma unroll
            for (int j = 0; j < D; ++j) R[i][j] = T[i * (D + 1) + j];
            t[i] = T[i * (D + 1) + D];
        }
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) {
#pragma unroll
            for (int j = 0; j < D; ++j) R[i][j] = st.R[i * 3 + j];
            t[i] = st.t[i];
        }
    }
    const CloudMeta ms = a.src_meta[pair];
    const CloudMeta mt = a.tgt_meta[pair];
    int begin = ms.pt_begin, end = ms.pt_end;
    if (a.slice_begin >= 0) { begin = max(begin, a.slice_begin); end = min(end, a.slice_end); }
    const double d2cap = a.d_max * a.d_max * (1.0 + 1e-9);
    const float pad = cell_box_pad(mt);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- pass 1 (tracking iterations): decide for every point of the block whether its match can have
    //      changed at all, and compact the ones that need a search into a dense work list, so that the
    //      search below runs with full warps instead of a few busy lanes per warp.
    //      Exact skip: at its last search the point's nearest neighbour was d1 away and every other
    //      target point at least d2 away.  While it has moved less than (d2 - d1) / 2 in total since
    //      then, the same target point is still strictly the nearest. ----
    int* s_list = reinterpret_cast<int*>(smem_raw + 128 + (OBJ_THREADS / 32) * OBJ_STAGE_BYTES);   // [OBJ_THREADS * ppt]
    __shared__ int s_count;
    const int blk_begin = begin + bx * a.ppt * OBJ_THREADS;
    const int blk_end = min(end, blk_begin + a.ppt * OBJ_THREADS);
    const bool compact = a.use_prev && a.slack != nullptr;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    if (compact) {
        for (int sbase = blk_begin + warp * 32; sbase < blk_end; sbase += OBJ_THREADS) {
            const int s = sbase + lane;
            bool need_search = false;
            if (s < blk_end) {
                need_search = true;
                const int pm = a.match[s];
                float sl = a.slack[s];
                if (pm >= 0 && sl > 0.f) {
                    const PRec<Real> p = a.src_spts[s];
                    const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
                    double mv2 = 0.0;
#pragma unroll
                    for (int i = 0; i < D; ++i) {
                        double vn = R[i][0] * px + R[i][1] * py + t[i];
                        double vo = st.Rp[i * 3 + 0] * px + st.Rp[i * 3 + 1] * py + st.tp[i];
                        if constexpr (D == 3) { vn += R[i][2] * pz; vo += st.Rp[i * 3 + 2] * pz; }
                        mv2 += (vn - vo) * (vn - vo);
                    }
                    sl -= __double2float_ru(sqrt(mv2) * (1.0 + 1e-6)) + 1e-30f;
                    a.slack[s] = fmaxf(sl, 0.f);
                    need_search = !(sl > 0.f);
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, need_search);
            int wpos = 0;
            if (lane == 0 && bal) wpos = atomicAdd(&s_count, __popc(bal));
            wpos = __shfl_sync(0xffffffffu, wpos, 0);
            if (need_search) s_list[wpos + __popc(bal & ((1u << lane) - 1u))] = s;
        }
        __syncthreads();
    }
    const int n_work = compact ? s_count : max(blk_end - blk_begin, 0);

    for (int w0 = warp * 32; w0 < n_work; w0 += OBJ_THREADS) {   // warp-uniform
        const bool valid = w0 + lane < n_work;
        const int wi = valid ? w0 + lane : n_work - 1;
        const int s = compact ? s_list[wi] : blk_begin + wi;
        constexpr bool skip = false;
        const PRec<Real> p = a.src_spts[s];
        double pp[3] = {0.0, 0.0, 0.0};  // p' = R p + t (gicp.py:119)
        {
            const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
#pragma unroll
            for (int i = 0; i < D; ++i) {
                double v = R[i][0] * px + R[i][1] * py + t[i];
                if constexpr (D == 3) v += R[i][2] * pz;
                pp[i] = v;
            }
        }
        // ---- 1-NN in the target grid, bounded by d_max (exactly equivalent to the unbounded
        //      query + gate of gicp.py:132-138, SURVEY appendix A rule 6).  The match of the previous
        //      outer iteration gives an upper bound on the new nearest distance, so only the cells
        //      that intersect the ball of that radius around p' are searched (still exact). ----
        double bestd = d2cap;
        int bestidx = -1;      // cloud-local input index of the best target point so far (-1: none)
        int prevpos = -1;      // sorted position of the previous iteration's match when it seeds the search
        int previdx = -1;
        if (a.use_prev) {
            const int pm = a.match[s];
            if (pm >= 0) {
                const PRec<Real> qo = a.tgt_spts[pm];
                const double e2 = exact_d2((double)qo.x - pp[0], (double)qo.y - pp[1], (double)qo.z - pp[2]);
                if (e2 <= d2cap) { bestd = e2; bestidx = (int)qo.idx; prevpos = pm; previdx = bestidx; }
            }
        }
        const float fx = (float)pp[0], fy = (float)pp[1], fz = (float)pp[2];
        const float Pf = fmaxf(fabsf(fx), fmaxf(fabsf(fy), fabsf(fz))) * 1.0000002f;
        const float c1 = filter_c1(Pf);
        auto filter_thr = [&](double bd) {
            const float b = __double2float_ru(bd);
            // sqrt(b) through the reciprocal-square-root unit (2 instructions instead of the IEEE sequence; it is
            // re-evaluated on every improvement of the best distance)
            return filter_thr_of(b, rsqrtf(fmaxf(b, 1e-30f)), c1);
        };
        float thr32 = filter_thr(bestd);
        float m1 = INFINITY, m2 = INFINITY;   // two smallest fp32 squared distances seen (slack of the next iterations)
        auto test = [&](const PRec<Real>& c) {
            bool pass = true;
            double e2 = 0.0;
            if (sizeof(Real) == 4) {
                const float dx = (float)c.x - fx, dy = (float)c.y - fy, dz = (float)c.z - fz;
                const float d32 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
                m2 = fminf(m2, fmaxf(m1, d32));
                m1 = fminf(m1, d32);
                pass = d32 <= thr32;
            } else {
                e2 = exact_d2((double)c.x - pp[0], (double)c.y - pp[1], (double)c.z - pp[2]);
                const float d32 = __double2float_rd(e2);
                m2 = fminf(m2, fmaxf(m1, d32));
                m1 = fminf(m1, d32);
            }
            if (pass) {
                if (sizeof(Real) == 4) e2 = exact_d2((double)c.x - pp[0], (double)c.y - pp[1], (double)c.z - pp[2]);
                const int cidx = (int)c.idx;
                // exact ties (same float64 distance) go to the lower input index, like the oracle
                if (e2 < bestd || (e2 == bestd && bestidx >= 0 && cidx < bestidx)) {
                    bestd = e2; bestidx = cidx;
                    thr32 = filter_thr(bestd);
                }
            }
        };
        // the points of one cell, the next record already in flight while the current one is tested
        auto run_cell = [&](int j0, int j1) {
            if (j0 >= j1) return;
            PRec<Real> c = a.tgt_spts[j0];
            for (int j = j0 + 1; j < j1; ++j) {
                const PRec<Real> nx = a.tgt_spts[j];
                test(c);
                c = nx;
            }
            test(c);
        };
        const double rad = sqrt(bestd) * (1.0 + 1e-9) + 1e-300;
        int mylo[3], myhi[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            mylo[i] = (i < D) ? cell_coord(pp[i] - rad, mt.origin[i], mt.inv_h) : 0;
            myhi[i] = (i < D) ? cell_coord(pp[i] + rad, mt.origin[i], mt.inv_h) : 0;
        }
        // a lane walks its own cells only when they are few; wide balls (no previous match, or a
        // match that moved far) are searched by the whole warp through the TMA stage
        const int x0 = max(mylo[0], 0), x1 = min(myhi[0], mt.dims[0] - 1);
        const int y0 = max(mylo[1], 0), y1 = min(myhi[1], mt.dims[1] - 1);
        const int z0 = max(mylo[2], 0), z1 = min(myhi[2], mt.dims[2] - 1);
        const int ncell = max(x1 - x0 + 1, 0) * max(y1 - y0 + 1, 0) * max(z1 - z0 + 1, 0);
        const bool tracked = !skip && bestidx >= 0 && ncell <= a.track_max_cells;
        // a tracked lane examines every point of the cell box [mylo, myhi]; everything outside that box is
        // at least `rad32` away (distance from p' to the nearest box face that has cells behind it)
        float rad32 = INFINITY;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            if (mylo[i] > 0) rad32 = fminf(rad32, __double2float_rd(pp[i] - (mt.origin[i] + mylo[i] * mt.h)));
            if (myhi[i] < mt.dims[i] - 1)
                rad32 = fminf(rad32, __double2float_rd(mt.origin[i] + (myhi[i] + 1) * mt.h - pp[i]));
        }
        rad32 = fmaxf(rad32 * 0.999999f - pad, 0.f);
        if (tracked) {
            // ---- phase A: per-lane walk over the (few) cells that intersect the ball ----
            const int* L = a.tgt_lut + mt.lut_base;
            for (int z = z0; z <= z1; ++z) {
                const int lz = __ldg(L + 2 * GICP_LUT_N + z);
                for (int y = y0; y <= y1; ++y) {
                    const int lyz = lz | __ldg(L + GICP_LUT_N + y);
                    for (int x = x0; x <= x1; ++x) {
                        const int* cs = a.tgt_cell_start + mt.cell_base + (lyz | __ldg(L + x));
                        const int j0 = __ldg(cs), j1 = __ldg(cs + 1);
                        run_cell(j0, j1);
                    }
                }
            }
        }
        // ---- phase A': lanes without a usable previous match (first iteration, gated-out points) search
        //      shell by shell around their own cell; every hit shrinks the ball, cells beyond it are
        //      skipped, and the search stops as soon as the searched box covers the best distance ----
        bool shell_done = tracked || skip;
        if (a.shell_search && !shell_done) {
            const int scx = cell_coord(pp[0], mt.origin[0], mt.inv_h);
            const int scy = cell_coord(pp[1], mt.origin[1], mt.inv_h);
            const int scz = (D == 3) ? cell_coord(pp[2], mt.origin[2], mt.inv_h) : 0;
            const int* L = a.tgt_lut + mt.lut_base;
            auto shell_cell = [&](int x, int y, int z) {
                if (x < 0 || y < 0 || z < 0 || x >= mt.dims[0] || y >= mt.dims[1] || z >= mt.dims[2]) return;
                if (cell_box_dist2(mt, pad, fx, fy, fz, x, y, z, x, y, z) > thr32) return;
                const int* cs = a.tgt_cell_start + mt.cell_base +
                                (__ldg(L + x) | __ldg(L + GICP_LUT_N + y) | __ldg(L + 2 * GICP_LUT_N + z));
                const int j0 = __ldg(cs), j1 = __ldg(cs + 1);
                run_cell(j0, j1);
            };
            constexpr int ZR = (D == 3) ? 1 : 0;
            const int sc[3] = {scx, scy, scz};
            for (int rho = 0; rho <= 2; ++rho) {
                for (int dz = -rho * ZR; dz <= rho * ZR; ++dz)
                    for (int dy = -rho; dy <= rho; ++dy) {
                        const bool outer = abs(dz) == rho || abs(dy) == rho;
                        if (outer) {
                            for (int dx = -rho; dx <= rho; ++dx) shell_cell(scx + dx, scy + dy, scz + dz);
                        } else {
                            shell_cell(scx - rho, scy + dy, scz + dz);
                            shell_cell(scx + rho, scy + dy, scz + dz);
                        }
                    }
                // distance from p' to the nearest face of the searched box that has cells behind it
                double cover = INFINITY;
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    if (sc[i] - rho > 0) cover = fmin(cover, pp[i] - (mt.origin[i] + (sc[i] - rho) * mt.h));
                    if (sc[i] + rho < mt.dims[i] - 1) cover = fmin(cover, mt.origin[i] + (sc[i] + rho + 1) * mt.h - pp[i]);
                }
                cover *= (1.0 - 1e-9);
                if ((bestidx >= 0 && bestd <= cover * cover) || cover >= a.d_max) { shell_done = true; break; }
            }
        }
        // ---- phase B: warp-cooperative search through the TMA stage (what the shells could not settle).
        //      First the cells the group's points fall into (a near match shrinks every lane's ball at
        //      once), then the rest of the union box, staging only the blocks that still reach into some
        //      lane's ball ----
        unsigned pending = __ballot_sync(0xffffffffu, !shell_done);
        if (pending) {
            const int cx = cell_coord(pp[0], mt.origin[0], mt.inv_h);
            const int cy = cell_coord(pp[1], mt.origin[1], mt.inv_h);
            const int cz = (D == 3) ? cell_coord(pp[2], mt.origin[2], mt.inv_h) : 0;
            const int mycell[3] = {cx, cy, cz};
            const int none[3] = {0, 0, 0};
            while (pending) {
                const unsigned grp = next_group(pending, cx, cy, cz, OBJ_GROUP_REACH);
                pending &= ~grp;
                const bool mine = (grp >> lane) & 1u;
                auto window = [&](const PRec<Real>* w, int n) {
                    for (int j = 0; j < n; ++j) {
                        const PRec<Real> c = w[j];
                        if (mine) test(c);
                    }
                };
                auto need = [&](int bx0, int by0, int bz0, int bx1, int by1, int bz1) {
                    // only blocks that reach into some lane's current best-distance ball are staged
                    return mine && cell_box_dist2(mt, pad, fx, fy, fz, bx0, by0, bz0, bx1, by1, bz1) <= thr32;
                };
                int clo[3], chi[3], lo[3], hi[3];
                group_union(grp, lane, mycell, mycell, mt, clo, chi);
                bool has_c = false;
                if (a.centre_first) {
                    stream_cells<Real>(mt, a.tgt_cell_start, a.tgt_lut, a.tgt_spts, clo, chi, none, none, false, ws,
                                       lane, window, need);
                    has_c = !(chi[0] < clo[0] || chi[1] < clo[1] || chi[2] < clo[2]);
                }
                group_union(grp, lane, mylo, myhi, mt, lo, hi);
                stream_cells<Real>(mt, a.tgt_cell_start, a.tgt_lut, a.tgt_spts, lo, hi, clo, chi, has_c, ws, lane,
                                   window, need);
            }
        }
        if (!valid || skip) continue;
        const double dist = (bestidx >= 0) ? sqrt(bestd) : INFINITY;
        const bool matched = (bestidx >= 0) && !(dist > a.d_max);  // gicp.py:136 rejects d > d_max
        // the match is kept as the target's sorted position (what K3b gathers by): one look-up when it changed
        int bestpos = -1;
        if (matched) bestpos = (bestidx == previdx) ? prevpos : a.tgt_inv_perm[mt.pt_begin + bestidx];
        a.match[s] = bestpos;
        if (a.slack) {
            float sl = 0.f;
            if (tracked && matched) sl = match_slack(__double2float_ru(dist), m2, rad32, c1, Pf);
            a.slack[s] = sl;
        }
        if (a.out_idx || a.out_dist) {
            const size_t out_row = (size_t)ms.pt_begin + (size_t)p.idx;
            if (a.out_idx) a.out_idx[out_row] = matched ? bestidx : -1;
            if (a.out_dist) a.out_dist[out_row] = dist;
        }
    }
}

// the warp's TMA stage inside the block's dynamic shared memory (obj_smem() bytes); lane 0 initialises the mbarrier
template <typename Real>
__device__ __forceinline__ WarpStage<Real> obj_warp_stage(unsigned char* smem_raw) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpStage<Real> ws;
    ws.buf = reinterpret_cast<PRec<Real>*>(smem_raw + 128 + warp * OBJ_STAGE_BYTES);
    ws.bar = reinterpret_cast<uint64_t*>(smem_raw) + warp;
    ws.phase = 0;
    ws.cap = OBJ_STAGE_BYTES / (int)sizeof(PRec<Real>);
    if (lane == 0) { mbar_init(ws.bar, 1); mbar_fence_init(); }
    __syncwarp();
    return ws;
}

// Occupancy decides this kernel (divergent dependent loads): 3-D fp32 is compiled for 10 blocks per SM = 48 registers
// (measured per 512 pairs: natural 64 registers 14.73 ms, 48 registers 13.83 ms, 40 registers 14.26 ms; 128
// registers 21.6 ms).  The other instantiations keep 8 blocks per SM (64 registers, what the compiler chose unprompted).
template <int D, typename Real>
__global__ void __launch_bounds__(OBJ_THREADS, (D == 3 && sizeof(Real) == 4) ? 10 : 8) correspond_kernel(const ObjArgs<Real> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int pair = obj_pair_of_block(a);
    if (pair < 0) return;
    WarpStage<Real> ws = obj_warp_stage<Real>(smem_raw);
    correspond_block<D, Real>(a, pair, blockIdx.x, ws, smem_raw, a.state + pair);
}

// One block of the accumulation: points [bx * ppt * OBJ_THREADS, ...) of pair `pair` -> out[NRED]
// (a.partial[pair][bx]; the fused loop passes its shared-memory sum and state instead).
// Robust: every gated-in correspondence is weighted by robust_weight(kind, d, c) - W, v = W e and e^T W e are scaled by
// w before they enter the accumulators, so the reduced form is that of sum w_i r_i^T W_i r_i.  A compile-time switch:
// the Robust = false instantiations are the unweighted kernels, instruction for instruction.  `c` is the pair's scale
// (the fixed robust_scale, or this iteration's adaptive one); Robust = false ignores it.
template <int D, typename Real, bool Robust = false>
__device__ __forceinline__ void accumulate_block(const ObjArgs<Real>& a, const int pair, const int bx,
                                                 const PairState* stp, double* out, const double c = 0.0) {
    using DD = Dim<D>;
    using AccT = Real;
    constexpr int NP = DD::NP, NS = DD::NS, NH = DD::NH, NQ = DD::NQ, NRED = DD::NRED;
    const PairState st = *stp;
    if (!a.ignore_status && st.status != PAIR_ACTIVE) return;

    double R[D][D], t[D];
    if (a.T_override) {
        const double* T = a.T_override + (size_t)pair * (D + 1) * (D + 1);
#pragma unroll
        for (int i = 0; i < D; ++i) {
#pragma unroll
            for (int j = 0; j < D; ++j) R[i][j] = T[i * (D + 1) + j];
            t[i] = T[i * (D + 1) + D];
        }
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) {
#pragma unroll
            for (int j = 0; j < D; ++j) R[i][j] = st.R[i * 3 + j];
            t[i] = st.t[i];
        }
    }
    const CloudMeta ms = a.src_meta[pair];
    const CloudMeta mt = a.tgt_meta[pair];
    int begin = ms.pt_begin, end = ms.pt_end;
    if (a.slice_begin >= 0) { begin = max(begin, a.slice_begin); end = min(end, a.slice_end); }

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (begin >= end) {
        // empty source cloud (or empty shard slice): nothing to gather - the pipeline below would read the record
        // before `begin`.  The pair's partial rows are zero.
        if (threadIdx.x < NRED) out[threadIdx.x] = 0.0;
        return;
    }
    AccT acc[NQ];
#pragma unroll
    for (int i = 0; i < NQ; ++i) acc[i] = AccT(0);
    double loss_acc = 0.0;
    int cnt = 0;

    // software pipeline over the thread's points: while point `it` is being processed, the gather of
    // point it+1 (target record + covariance, addressed by its match) and the match index of point it+2
    // are already in flight - the kernel is bound by dependent-load latency otherwise
    const int s_first = begin + bx * a.ppt * OBJ_THREADS + threadIdx.x;
    auto load_match = [&](int it) {
        const int s = s_first + it * OBJ_THREADS;
        return (it < a.ppt && s < end) ? a.match[s] : -1;
    };
    struct Gathered { PRec<Real> q; Real ct[NS]; PRec<Real> p; Real cs[NS]; };
    auto gather = [&](int m, int it) {
        Gathered g;
        {   // the source side of the same point: streamed, but just as far away as the gathered target
            const int s = min(s_first + it * OBJ_THREADS, end - 1);
            g.p = a.src_spts[s];
            const Real* cs = a.src_cov + (size_t)s * NS;
            if constexpr (sizeof(Real) == 4 && NS == 6) {
                // 24-byte records, 8-byte aligned: three 64-bit loads instead of six 32-bit ones
                const float2* c2 = reinterpret_cast<const float2*>(cs);
                const float2 u0 = __ldg(c2), u1 = __ldg(c2 + 1), u2 = __ldg(c2 + 2);
                g.cs[0] = u0.x; g.cs[1] = u0.y; g.cs[2] = u1.x; g.cs[3] = u1.y; g.cs[4] = u2.x; g.cs[5] = u2.y;
            } else {
#pragma unroll
                for (int i = 0; i < NS; ++i) g.cs[i] = cs[i];
            }
        }
        if (m >= 0) {
            g.q = a.tgt_spts[m];
            const Real* ct = a.tgt_cov + (size_t)m * NS;
            if constexpr (sizeof(Real) == 4 && NS == 6) {
                const float2* t2 = reinterpret_cast<const float2*>(ct);
                const float2 u0 = __ldg(t2), u1 = __ldg(t2 + 1), u2 = __ldg(t2 + 2);
                g.ct[0] = u0.x; g.ct[1] = u0.y; g.ct[2] = u1.x; g.ct[3] = u1.y; g.ct[4] = u2.x; g.ct[5] = u2.y;
            } else {
#pragma unroll
                for (int i = 0; i < NS; ++i) g.ct[i] = ct[i];
            }
        } else {
            g.q.x = g.q.y = g.q.z = Real(0); g.q.idx = 0;
#pragma unroll
            for (int i = 0; i < NS; ++i) g.ct[i] = Real(0);
        }
        return g;
    };
    int m_cur = load_match(0);
    Gathered g_cur = gather(m_cur, 0);
    int m_next = load_match(1);
    for (int it = 0; it < a.ppt; ++it) {
        const int s = s_first + it * OBJ_THREADS;
        if (s >= end) break;
        const int bestpos = m_cur;
        const Gathered g = g_cur;
        g_cur = gather(m_next, it + 1);   // in flight during this iteration's arithmetic
        m_cur = m_next;
        m_next = load_match(it + 2);
        const size_t out_row = (size_t)ms.pt_begin + (size_t)g.p.idx;
        if (bestpos < 0) {
            if (a.out_W) {
                for (int i = 0; i < D * D; ++i) a.out_W[out_row * D * D + i] = 0.0;
            }
            continue;
        }
        double pp[3] = {0.0, 0.0, 0.0};  // p' = R p + t (gicp.py:119)
        transform_point<D, Real>(R, t, g.p, pp);
        // ---- W = inv(C_tgt[j] + R C_src[i] R^T), e = q - p' ----
        const PRec<Real> q = g.q;
        double w_rob = 1.0;   // robust kernel weight at the current distance (Robust only)
        {   // gicp.py:136: the gate applies to the CURRENT distance (a kept match may have drifted out)
            const double d2 = exact_d2((double)q.x - pp[0], (double)q.y - pp[1], (double)q.z - pp[2]);
            if (sqrt(d2) > a.d_max) {
                if (a.out_W) {
                    for (int i = 0; i < D * D; ++i) a.out_W[out_row * D * D + i] = 0.0;
                }
                continue;
            }
            if constexpr (Robust) w_rob = robust_weight(a.robust_kind, sqrt(d2), c);
        }
        double Cs[NS], M[NS], W[NS], e[D], v[D];
        {
#pragma unroll
            for (int i = 0; i < NS; ++i) Cs[i] = (double)g.cs[i];
#pragma unroll
            for (int i = 0; i < NS; ++i) M[i] = (double)g.ct[i];
        }
        if constexpr (D == 3) {
            const double C[3][3] = {{Cs[0], Cs[1], Cs[2]}, {Cs[1], Cs[3], Cs[4]}, {Cs[2], Cs[4], Cs[5]}};
            double A[3][3];
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) A[i][j] = R[i][0] * C[0][j] + R[i][1] * C[1][j] + R[i][2] * C[2][j];
            int k = 0;
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = i; j < 3; ++j) M[k++] += A[i][0] * R[j][0] + A[i][1] * R[j][1] + A[i][2] * R[j][2];
            sym_inv3(M, W);
            e[0] = (double)q.x - pp[0]; e[1] = (double)q.y - pp[1]; e[2] = (double)q.z - pp[2];
            v[0] = W[0] * e[0] + W[1] * e[1] + W[2] * e[2];
            v[1] = W[1] * e[0] + W[3] * e[1] + W[4] * e[2];
            v[2] = W[2] * e[0] + W[4] * e[1] + W[5] * e[2];
        } else {
            const double C[2][2] = {{Cs[0], Cs[1]}, {Cs[1], Cs[2]}};
            double A[2][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) A[i][j] = R[i][0] * C[0][j] + R[i][1] * C[1][j];
            M[0] += A[0][0] * R[0][0] + A[0][1] * R[0][1];
            M[1] += A[0][0] * R[1][0] + A[0][1] * R[1][1];
            M[2] += A[1][0] * R[1][0] + A[1][1] * R[1][1];
            sym_inv2(M, W);
            e[0] = (double)q.x - pp[0]; e[1] = (double)q.y - pp[1];
            v[0] = W[0] * e[0] + W[1] * e[1];
            v[1] = W[1] * e[0] + W[2] * e[1];
        }
        double li = 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i) li += e[i] * v[i];
        if constexpr (Robust) {   // w W replaces W: the gated-in count below still counts this point
            li *= w_rob;
#pragma unroll
            for (int i = 0; i < NS; ++i) W[i] *= w_rob;
#pragma unroll
            for (int i = 0; i < D; ++i) v[i] *= w_rob;
        }
        loss_acc += li;
        ++cnt;
        if (a.out_W) {
            double* o = a.out_W + out_row * D * D;
#pragma unroll
            for (int i = 0; i < D; ++i)
#pragma unroll
                for (int j = 0; j < D; ++j) o[i * D + j] = W[symidx(D, i, j)];
        }
        // ---- accumulate the reduced form ----
        AccT pt[NP], Wa[NS], va[D];
        pt[0] = AccT(1);
#pragma unroll
        for (int i = 0; i < D; ++i) { pt[1 + i] = (AccT)(pp[i] - st.mu[i]); va[i] = (AccT)v[i]; }
#pragma unroll
        for (int i = 0; i < NS; ++i) Wa[i] = (AccT)W[i];
        {
            int ab = 0;
#pragma unroll
            for (int i = 0; i < NP; ++i)
#pragma unroll
                for (int j = i; j < NP; ++j) {
                    const AccT sij = pt[i] * pt[j];
#pragma unroll
                    for (int cd = 0; cd < NS; ++cd) acc[ab * NS + cd] += sij * Wa[cd];
                    ++ab;
                }
#pragma unroll
            for (int c = 0; c < D; ++c)
#pragma unroll
                for (int i = 0; i < NP; ++i) acc[NH + c * NP + i] += va[c] * pt[i];
        }
    }

    // ---- block reduction: warp shuffles, then the warps' sums in fixed order in fp64 ----
    __shared__ double s_red[OBJ_THREADS / 32][NQ + 2];
#pragma unroll
    for (int i = 0; i < NQ; ++i) {
        const AccT r = warp_sum(acc[i]);
        if (lane == 0) s_red[warp][i] = (double)r;
    }
    {
        const double l = warp_sum(loss_acc);
        const int c = warp_sum(cnt);
        if (lane == 0) { s_red[warp][NQ] = l; s_red[warp][NQ + 1] = (double)c; }
    }
    __syncthreads();
    if (threadIdx.x < NRED) {
        double r = 0.0;
        if (threadIdx.x < NQ + 2) {
#pragma unroll
            for (int w = 0; w < OBJ_THREADS / 32; ++w) r += s_red[w][threadIdx.x];
        }
        out[threadIdx.x] = r;
    }
}

// f32 storage: 128 registers, 4 blocks per SM.  f64 storage carries 72 fp64 accumulators per thread: 2 blocks per SM
// and 255 registers instead of ~1.2 KB of spills per thread under the 128-register cap
template <int D, typename Real, bool Robust = false>
__global__ void __launch_bounds__(OBJ_THREADS, (sizeof(Real) == 8 && D == 3) ? 2 : 4) accumulate_kernel(const ObjArgs<Real> a) {
    const int pair = obj_pair_of_block(a);
    if (pair < 0) return;
    double c = 0.0;
    if constexpr (Robust) c = a.pair_scale ? a.pair_scale[pair] : a.robust_scale;
    accumulate_block<D, Real, Robust>(a, pair, blockIdx.x, a.state + pair,
                              a.partial + ((size_t)pair * a.blocks_per_pair + blockIdx.x) * Dim<D>::NRED, c);
}

}  // namespace gicp
