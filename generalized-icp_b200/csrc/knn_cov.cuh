// K2: fixed-radius k-NN over the uniform grid + plane-to-plane regularised covariance.
// Replaces compute_covariance_matrix / compute_covariance_matrix_single_point
// (reference gicp.py:19-35, 5-17): tree.query(k, distance_upper_bound) per point,
// np.cov, np.linalg.eig, R diag(100,10) R^T.
//
// Work decomposition: one warp = 32 consecutive points of the Morton-sorted order (a compact
// blob of a few cells).  The warp stages the cell blocks around its queries with TMA bulk copies
// (stream.cuh) and every lane scans the staged candidates (broadcast LDS.128).
//
// Fast path (knn_hist_kernel): three sweeps, no long selection network.
//   1. ring by ring (ring 0 = the queries' own cells) every lane histograms the fp32 distance of
//      each candidate into 64 distance bins (lane-private column in shared memory); after a ring
//      the bin holding the k-th candidate bounds the lane's k-th neighbour distance, and the
//      search stops once the searched box covers that bound for every lane;
//   2. the box is streamed once more and each lane keeps the candidates under its bound (k plus
//      the few that share the last bin) in a lane-private list;
//   3. everything below the bin of the k-th candidate is in the set; the entries of that bin are marked and
//      then ranked among themselves by counting, all lanes side by side.  The ranked key is the float64
//      squared distance (dx*dx + dy*dy) + dz*dz of the oracle, ties to the lower point index: fp32 keys
//      decide every comparison that falls outside their rounding band, exact keys the rest.  The moments of
//      the selected neighbours are accumulated in a loop of their own (next gather in flight).
// General path (knn_general_kernel): exact sorted top-k in registers fed through a per-lane queue;
// used when k is too large for the fast path's list and for the warps whose list overflowed.
#pragma once
#include "common.cuh"
#include "stream.cuh"

namespace gicp {

constexpr int KNN_WARPS = 4;
constexpr int KNN_THREADS = KNN_WARPS * 32;
constexpr int KNN_STAGE_BYTES = 8192;   // per warp
constexpr int KNN_QUEUE = 24;           // general path: parked survivors per lane
constexpr int KNN_WARP_SMEM = KNN_STAGE_BYTES + KNN_QUEUE * 32 * 12;
constexpr int KNN_GROUP_REACH = 4;
constexpr int KNN_BINS = 64;            // fast path: distance bins per lane (uint8 counters)
constexpr int KNN_LIST_BYTES = 8192;    // fast path: lane-private candidate list, per warp
// fast cooperative path: 1 KB stage + 8 KB list per warp = 37 KB per block -> 6 blocks (24 warps) per SM at the
// kernel's 80 registers; measured 24.8 ms (1 KB) / 26.7 (2 KB, 5 blocks) / 25.9 (512 B) per 2 x 256 clouds
constexpr int KNN_HSTAGE_BYTES = 1024;
constexpr int KNN_HIST_WARP_SMEM = KNN_HSTAGE_BYTES + KNN_LIST_BYTES;   // histogram aliases the list

template <typename Real> struct KnnArgs {
    const CloudMeta* meta;
    const int* cell_start;
    const int* lut;
    const PRec<Real>* spts;
    const Real* raw;     // caller's (n_total, D) array: neighbour coordinates for the covariance
    Real* cov_sorted;    // [n_total][NS], cell-sorted order
    int* knn_idx;        // optional [n_total][k], input order, cloud-local, -1 missing
    double* knn_dist;    // optional [n_total][k]
    int k;
    double radius;
    double lam_t, lam_n;
    int slice_begin, slice_end;  // sorted-position slice handled by this rank (<0: whole clouds)
    int* overflow_count;         // fast path -> general path hand-over
    int2* overflow_list;         // (cloud, chunk base)
    int overflow_cap;
};

// fast path list capacity per lane: 32 (float keys) / 21 (double keys)
template <typename Real> __host__ __device__ constexpr int knn_list_cap() { return KNN_LIST_BYTES / (32 * ((int)sizeof(Real) + 4)); }

__device__ __forceinline__ bool key_less(double d, int i, double dd, int ii) {
    return d < dd || (d == dd && i < ii);
}

// gicp.py:11-16 / SURVEY 8c: regularised covariance from the neighbourhood's scatter matrix
// S (00 01 02 11 12 22, already divided by cnt-1).  C: D(D+1)/2 entries.
template <int D>
__host__ __device__ __forceinline__ void regularised_cov(const double S[6], bool ident, double lam_t, double lam_n, double* C) {
    bool finite = true;
#pragma unroll
    for (int i = 0; i < 6; ++i) finite = finite && isfinite(S[i]);
    if (!finite) ident = true;  // gicp.py:31-32
    if (!ident) {
        if constexpr (D == 2) {
            // eigenvector of the largest eigenvalue (gicp.py:14-16): C = lam_n I + (lam_t-lam_n) v v^T
            const double phi = 0.5 * atan2(2.0 * S[1], S[0] - S[3]);
            double sn, cs;
            sincos(phi, &sn, &cs);
            const double dl = lam_t - lam_n;
            C[0] = lam_n + dl * cs * cs;
            C[1] = dl * cs * sn;
            C[2] = lam_n + dl * sn * sn;
        } else {
            // normal = eigenvector of the smallest eigenvalue: C = lam_t I - (lam_t-lam_n) n n^T
            double n[3];
            smallest_eigvec3(S[0], S[1], S[2], S[3], S[4], S[5], n);
            const double dl = lam_t - lam_n;
            C[0] = lam_t - dl * n[0] * n[0];
            C[1] = -dl * n[0] * n[1];
            C[2] = -dl * n[0] * n[2];
            C[3] = lam_t - dl * n[1] * n[1];
            C[4] = -dl * n[1] * n[2];
            C[5] = lam_t - dl * n[2] * n[2];
        }
    } else {
        if constexpr (D == 2) { C[0] = 1.0; C[1] = 0.0; C[2] = 1.0; }
        else { C[0] = 1.0; C[1] = 0.0; C[2] = 0.0; C[3] = 1.0; C[4] = 0.0; C[5] = 1.0; }
    }
}

// moments about the query point (count, sum of offsets, sum of outer products) -> sample covariance
// (ddof = 1) -> regularised covariance of sorted position s
template <int D, typename Real>
__device__ __forceinline__ void knn_finish_cov(const KnnArgs<Real>& a, int s, int n_valid, const double mean[3],
                                               double S[6]) {
    constexpr int NS = Dim<D>::NS;
    double C[NS];
    const bool ident = n_valid <= 1;     // gicp.py:27,33-34
    if (!ident) {
        const double inv = 1.0 / n_valid;
        const double m0 = mean[0] * inv, m1 = mean[1] * inv, m2 = mean[2] * inv;
        const double f = 1.0 / (n_valid - 1);   // ddof = 1 (np.cov default, gicp.py:12)
        S[0] = (S[0] - n_valid * m0 * m0) * f; S[1] = (S[1] - n_valid * m0 * m1) * f;
        S[2] = (S[2] - n_valid * m0 * m2) * f; S[3] = (S[3] - n_valid * m1 * m1) * f;
        S[4] = (S[4] - n_valid * m1 * m2) * f; S[5] = (S[5] - n_valid * m2 * m2) * f;
    }
    regularised_cov<D>(S, ident, a.lam_t, a.lam_n, C);
    Real* out = a.cov_sorted + (size_t)s * NS;
#pragma unroll
    for (int i = 0; i < NS; ++i) out[i] = (Real)C[i];
}

// sweep 3 of the fast paths: rank a lane's candidate list by counting, accumulate the moments of the
// winners (rank < k, inside the radius), write the optional index/distance outputs and the
// regularised covariance of sorted position s.
template <int D, typename Real>
__device__ __forceinline__ void knn_rank_and_finish(const KnnArgs<Real>& a, const CloudMeta& m, int s, int my_idx,
                                                    Real mx, Real my, Real mz, const Real* lk, const int* li,
                                                    int lane, int mcount, float edge_lo) {
    using KeyT = Real;
    // ---- sweep 3: rank the list by counting; winners (rank < k) go to their sorted slot ----
    const size_t cloud_row0 = (size_t)m.pt_begin;
    auto exact_key = [&](int idx) {
        const Real* q = a.raw + (cloud_row0 + idx) * D;
        const double dz = (D == 3) ? (double)q[D - 1] - (double)mz : 0.0;
        return exact_d2((double)q[0] - (double)mx, (double)q[1] - (double)my, dz);
    };
    int n_valid = 0;            // neighbours that pass the exact radius test
    double mean[3] = {0.0, 0.0, 0.0};
    double S[6] = {0, 0, 0, 0, 0, 0};
    int* out_idx = a.knn_idx ? a.knn_idx + (cloud_row0 + my_idx) * (size_t)a.k : nullptr;
    double* out_d = a.knn_dist ? a.knn_dist + (cloud_row0 + my_idx) * (size_t)a.k : nullptr;
    // Only the SET of the k nearest matters for the covariance.  Every candidate below the k-th
    // histogram bin is in it for sure (fewer than k candidates lie below that bin); only the candidates
    // of the k-th bin compete for the remaining k - n_sure places and need ranking.  The 4e-6 margin
    // keeps "sure" exact under fp32 rounding: an excluded candidate is farther than some candidate of
    // the k-th bin, hence farther than every sure one.  With index output the whole list is ranked.
    const bool need_order = a.knn_idx != nullptr;
    float sure_thr = need_order ? -1.0f : ((sizeof(Real) == 4) ? edge_lo * (1.0f - 4e-6f) : edge_lo);
    int n_sure = 0;
    for (int j = 0; j < mcount; ++j) n_sure += ((float)lk[j * 32 + lane] < sure_thr) ? 1 : 0;
    if (n_sure >= a.k) sure_thr = -1.0f;   // only possible if an 8-bit histogram counter wrapped: rank everything
    // pass A: the sure entries are selected as they come; the entries that need ranking are only marked.
    // (Ranking them inside this loop would run every lane's counting loop on its own - the marked
    // positions differ from lane to lane - at a few active lanes per instruction.)
    unsigned amb = 0, sel = 0;
    for (int i = 0; i < mcount; ++i) {
        if ((float)lk[i * 32 + lane] < sure_thr) sel |= 1u << i;
        else amb |= 1u << i;
    }
    // pass B: every lane ranks its next marked entry by counting, all lanes side by side.  Only the marked
    // entries are compared: every sure entry is closer than every marked one by more than the rounding of
    // the fp32 keys, except within 5e-7 of the threshold itself, where both are below the k-th bin and the
    // rank (at most n_sure + marked-below-the-bin - 1 <= k - 2) selects the entry either way.
    const unsigned marked = amb;
    if (n_sure >= a.k) n_sure = 0;
    while (amb) {
        const int i = __ffs(amb) - 1;
        amb &= amb - 1;
        const KeyT ki = lk[i * 32 + lane];
        const int ii = li[i * 32 + lane];
        int r = n_sure;
        if (sizeof(Real) == 4) {
            const float lo_k = (float)ki * 0.999999f, hi_k = (float)ki * 1.000001f;
            int below = 0, upto = 0;
            for (unsigned mm = marked; mm; mm &= mm - 1) {
                const float kj = (float)lk[(__ffs(mm) - 1) * 32 + lane];
                below += (kj < lo_k) ? 1 : 0;
                upto += (kj <= hi_k) ? 1 : 0;
            }
            r += below;
            if (upto - below > 1) {   // another candidate inside the fp32 rounding band: exact keys decide
                const double ei = exact_key(ii);
                for (unsigned mm = marked; mm; mm &= mm - 1) {
                    const int j = __ffs(mm) - 1;
                    const float kj = (float)lk[j * 32 + lane];
                    if (j != i && kj >= lo_k && kj <= hi_k) {
                        const int ij = li[j * 32 + lane];
                        r += key_less(exact_key(ij), ij, ei, ii) ? 1 : 0;
                    }
                }
            }
        } else {
            for (unsigned mm = marked; mm; mm &= mm - 1) {
                const int j = __ffs(mm) - 1;
                r += key_less((double)lk[j * 32 + lane], li[j * 32 + lane], (double)ki, ii) ? 1 : 0;
            }
        }
        if (r < a.k) {
            sel |= 1u << i;
            if (out_idx) {   // index output: every entry comes through here (sure_thr = -1)
                const double dist = sqrt(exact_key(ii));
                const bool ok = dist < a.radius;
                out_idx[r] = ok ? ii : -1;
                if (out_d) out_d[r] = ok ? dist : INFINITY;
            }
        }
    }
    // pass C: moments of the selected entries, in list order; the coordinates of the next one are
    // fetched (a random 12-byte gather) while the current one is accumulated
    {
        auto fetch = [&](unsigned mask, Real& x, Real& y, Real& z) {
            const Real* q = a.raw + (cloud_row0 + li[(__ffs(mask) - 1) * 32 + lane]) * D;
            x = q[0]; y = q[1]; z = (D == 3) ? q[D - 1] : Real(0);
        };
        Real nx = 0, ny = 0, nz = 0;
        if (sel) fetch(sel, nx, ny, nz);
        while (sel) {
            const Real qx = nx, qy = ny, qz = nz;
            sel &= sel - 1;
            if (sel) fetch(sel, nx, ny, nz);
            const double d0 = (double)qx - (double)mx, d1 = (double)qy - (double)my;
            const double d2 = (D == 3) ? (double)qz - (double)mz : 0.0;
            const double dist = sqrt(exact_d2(d0, d1, d2));
            if (dist < a.radius) {         // exclusive bound, gicp.py:24
                ++n_valid;
                // moments about the query point keep the scatter matrix accurate
                mean[0] += d0; mean[1] += d1; mean[2] += d2;
                S[0] += d0 * d0; S[1] += d0 * d1; S[2] += d0 * d2;
                S[3] += d1 * d1; S[4] += d1 * d2; S[5] += d2 * d2;
            }
        }
    }
    if (out_idx) {
        for (int o = min(mcount, a.k); o < a.k; ++o) {
            out_idx[o] = -1;
            if (out_d) out_d[o] = INFINITY;
        }
    }
    knn_finish_cov<D, Real>(a, s, n_valid, mean, S);
}

// ================================================================================================
// fast path
// ================================================================================================
template <int D, typename Real>
__global__ void __launch_bounds__(KNN_THREADS) knn_hist_kernel(const KnnArgs<Real> a) {
    using KeyT = Real;  // list key: the fp32 filter distance (float storage) / the exact key (double storage)
    constexpr int CAP = knn_list_cap<Real>();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char* wbase = smem_raw + 128 + warp * KNN_HIST_WARP_SMEM;
    WarpStage<Real> ws;
    ws.buf = reinterpret_cast<PRec<Real>*>(wbase);
    ws.bar = bars + warp;
    ws.phase = 0;
    ws.cap = KNN_HSTAGE_BYTES / (int)sizeof(PRec<Real>);
    unsigned char* hist = wbase + KNN_HSTAGE_BYTES;                                 // [KNN_BINS][32] uint8, sweep 1
    KeyT* lk = reinterpret_cast<KeyT*>(wbase + KNN_HSTAGE_BYTES);                   // [CAP][32], sweeps 2-3 (aliases hist)
    int* li = reinterpret_cast<int*>(wbase + KNN_HSTAGE_BYTES + CAP * 32 * sizeof(KeyT));  // [CAP][32]

    const int cloud = blockIdx.y;
    const CloudMeta m = a.meta[cloud];
    int begin = m.pt_begin, end = m.pt_end;
    if (a.slice_begin >= 0) { begin = max(begin, a.slice_begin); end = min(end, a.slice_end); }
    const int base = begin + (blockIdx.x * KNN_WARPS + warp) * 32;
    if (base >= end) return;
    if (lane == 0) { mbar_init(ws.bar, 1); mbar_fence_init(); }
    __syncwarp();

    const bool valid = base + lane < end;
    const PRec<Real> me = a.spts[valid ? base + lane : end - 1];
    const int my_idx = (int)me.idx;
    const Real mx = me.x, my = me.y, mz = me.z;
    const int cx = min(max(cell_coord((double)mx, m.origin[0], m.inv_h), 0), m.dims[0] - 1);
    const int cy = min(max(cell_coord((double)my, m.origin[1], m.inv_h), 0), m.dims[1] - 1);
    const int cz = (D == 3) ? min(max(cell_coord((double)mz, m.origin[2], m.inv_h), 0), m.dims[2] - 1) : 0;

    const double r2cap = a.radius * a.radius * (1.0 + 1e-12);
    const float r2cap32 = __double2float_ru(r2cap * (1.0 + 1e-6));
    // logarithmic distance bins straight from the float bit pattern: 8 bins per octave of d^2 (3
    // mantissa bits), the last bin holds the radius; everything closer than radius/16 shares bin 0
    const int ubase = (int)(__float_as_uint(r2cap32) >> 20) - (KNN_BINS - 1);
    const float pad = cell_box_pad(m);
    const int rho_max = max(1, (int)ceil(a.radius / (m.h * (1.0 - 1e-9))));
    float bound32 = r2cap32;   // squared-distance bound under which at least k candidates lie
    float edge_lo = 0.0f;      // lower edge of the histogram bin that holds the k-th candidate
    bool overflow = false;
    const size_t sorted_pos = (size_t)(base + lane);

    // fp32 distance of a candidate (float storage), or the float image of the exact one (double storage)
    auto dist32 = [&](const PRec<Real>& c) {
        if (sizeof(Real) == 4) {
            const float dx = (float)c.x - (float)mx, dy = (float)c.y - (float)my, dz = (float)c.z - (float)mz;
            return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        } else {
            return (float)exact_d2((double)c.x - (double)mx, (double)c.y - (double)my, (double)c.z - (double)mz);
        }
    };

    unsigned pending = 0xffffffffu;
    while (pending) {
        const unsigned grp = next_group(pending, cx, cy, cz, KNN_GROUP_REACH);
        pending &= ~grp;
        const bool mine = (grp >> lane) & 1u;
        // the histogram shares its memory with the list of the previous group: start clean
#pragma unroll
        for (int b = 0; b < KNN_BINS; ++b) hist[b * 32 + lane] = 0;
        __syncwarp();
        const int mycell[3] = {cx, cy, cz};
        int qlo[3], qhi[3];
        group_union(grp, lane, mycell, mycell, m, qlo, qhi);
        int plo[3] = {0, 0, 0}, phi[3] = {-1, -1, -1};
        int lo[3] = {0, 0, 0}, hi[3] = {-1, -1, -1};
        // ---- sweep 1: histogram the distances ring by ring.  After every ring the histogram bounds
        //      the lane's k-th distance; blocks beyond every lane's bound are not staged ----
        float prov32 = r2cap32;
        float lim = mine ? r2cap32 : -1.0f;   // candidates beyond the lane's provisional bound are not binned
        int seen = 0;
        for (int rho = 0; rho <= rho_max; ++rho) {
#pragma unroll
            for (int c = 0; c < 3; ++c) { lo[c] = max(qlo[c] - rho, 0); hi[c] = min(qhi[c] + rho, m.dims[c] - 1); }
            stream_cells<Real>(m, a.cell_start, a.lut, a.spts, lo, hi, plo, phi, rho > 0, ws, lane,
                               [&](const PRec<Real>* w, int n) {
                // `lim` is -1 for lanes outside the group, so one compare gates both conditions; the bin index only
                // needs clamping from below (d2 <= r2cap32 bounds it from above)
                int j = 0;
                for (; j + 4 <= n; j += 4) {     // 4 candidates in flight: the histogram update is a dependent chain
                    const PRec<Real> c0 = w[j], c1 = w[j + 1], c2 = w[j + 2], c3 = w[j + 3];
                    const float e0 = dist32(c0), e1 = dist32(c1), e2 = dist32(c2), e3 = dist32(c3);
                    const int g0 = max((int)(__float_as_uint(e0) >> 20) - ubase, 0);
                    const int g1 = max((int)(__float_as_uint(e1) >> 20) - ubase, 0);
                    const int g2 = max((int)(__float_as_uint(e2) >> 20) - ubase, 0);
                    const int g3 = max((int)(__float_as_uint(e3) >> 20) - ubase, 0);
                    if (e0 <= lim) { hist[g0 * 32 + lane] += 1; ++seen; }
                    if (e1 <= lim) { hist[g1 * 32 + lane] += 1; ++seen; }
                    if (e2 <= lim) { hist[g2 * 32 + lane] += 1; ++seen; }
                    if (e3 <= lim) { hist[g3 * 32 + lane] += 1; ++seen; }
                }
                for (; j < n; ++j) {
                    const float e0 = dist32(w[j]);
                    const int g0 = max((int)(__float_as_uint(e0) >> 20) - ubase, 0);
                    if (e0 <= lim) { hist[g0 * 32 + lane] += 1; ++seen; }
                }
            }, [&](int x0, int y0, int z0, int x1, int y1, int z1) {
                return mine && cell_box_dist2(m, pad, (float)mx, (float)my, (float)mz, x0, y0, z0, x1, y1, z1) <= prov32;
            });
#pragma unroll
            for (int c = 0; c < 3; ++c) { plo[c] = lo[c]; phi[c] = hi[c]; }
            // bin that holds the k-th candidate -> bound on the k-th neighbour distance.  (A counter
            // that wrapped at 256 only makes the bound larger, never wrong.)
            int kb = KNN_BINS - 1;
            bool have = false;
            if (seen >= a.k) {
                int cum = 0;
                for (int b = 0; b < KNN_BINS; ++b) {
                    cum += hist[b * 32 + lane];
                    if (cum >= a.k) { kb = b; break; }
                }
                have = kb < KNN_BINS - 1;
            }
            // every candidate of bins <= kb has d2 < edge2 (exact: bin edges are float bit patterns)
            const float edge2 = have ? __uint_as_float((unsigned)(ubase + kb + 1) << 20) : r2cap32;
            prov32 = fminf(prov32, edge2);
            if (mine) lim = prov32;
            if (rho == 0) continue;
            const double cover = rho * m.h * (1.0 - 1e-9);
            const bool mine_done = !mine || (have && (double)prov32 <= cover * cover);
            if (__all_sync(0xffffffffu, mine_done) || cover >= a.radius) {
                if (mine) {
                    bound32 = prov32;
                    edge_lo = (have && kb > 0) ? __uint_as_float((unsigned)(ubase + kb) << 20) : 0.0f;
                }
                break;
            }
        }
        __syncwarp();
        // ---- sweep 2: keep the candidates under the bound ----
        const int none[3] = {0, 0, 0};
        int cnt_l = 0;
        // The list takes every candidate up to the bound widened by the rounding of the fp32 keys: a candidate
        // that is left out is then farther - in exact arithmetic - than the k candidates known to lie under the bound.
        const float list32 = bound32 * 1.000002f;
        const float lim2 = mine ? list32 : -1.0f;
        stream_cells<Real>(m, a.cell_start, a.lut, a.spts, lo, hi, none, none, false, ws, lane,
                           [&](const PRec<Real>* w, int n) {
            auto key_of = [&](const PRec<Real>& c) -> KeyT {
                if (sizeof(Real) == 4) return (KeyT)dist32(c);
                return (KeyT)exact_d2((double)c.x - (double)mx, (double)c.y - (double)my, (double)c.z - (double)mz);
            };
            auto keep = [&](KeyT key, const PRec<Real>& c) {
                if ((float)key <= lim2) {
                    if (cnt_l < CAP) { lk[cnt_l * 32 + lane] = key; li[cnt_l * 32 + lane] = (int)c.idx; }
                    ++cnt_l;
                }
            };
            int j = 0;
            for (; j + 4 <= n; j += 4) {     // 4 candidates in flight (shared-memory load latency)
                const PRec<Real> c0 = w[j], c1 = w[j + 1], c2 = w[j + 2], c3 = w[j + 3];
                const KeyT k0 = key_of(c0), k1 = key_of(c1), k2 = key_of(c2), k3 = key_of(c3);
                keep(k0, c0); keep(k1, c1); keep(k2, c2); keep(k3, c3);
            }
            for (; j < n; ++j) {
                const PRec<Real> c = w[j];
                keep(key_of(c), c);
            }
        }, [&](int x0, int y0, int z0, int x1, int y1, int z1) {
            // only blocks that reach into some lane's ball are staged
            return mine && cell_box_dist2(m, pad, (float)mx, (float)my, (float)mz, x0, y0, z0, x1, y1, z1) <= list32;
        });
        // ---- sweep 3 for this group's lanes (the list memory is recycled by the next group) ----
        const bool ovf = mine && cnt_l > CAP;
        overflow = overflow || ovf;
        if (mine && valid && !ovf)
            knn_rank_and_finish<D, Real>(a, m, (int)sorted_pos, my_idx, mx, my, mz, lk, li, lane, min(cnt_l, CAP), edge_lo);
        __syncwarp();
    }
    // hand the whole warp to the general path if any lane's list overflowed (it recomputes all 32 lanes)
    if (__any_sync(0xffffffffu, overflow)) {
        if (lane == 0) {
            const int slot = atomicAdd(a.overflow_count, 1);
            if (slot < a.overflow_cap) a.overflow_list[slot] = make_int2(cloud, base);
        }
    }
}

// Sorted top-k (slots [KCAP-k, KCAP) live, INT_MAX = empty) -> radius test, optional index / distance outputs,
// sample covariance about the mean (ddof = 1) and its regularised form, written for sorted position s_pos.
template <int D, typename Real, int KCAP>
__device__ __forceinline__ void topk_finish(const KnnArgs<Real>& a, const CloudMeta& m, int s_pos, int my_idx,
                                            double (&ad)[KCAP], int (&ai)[KCAP]) {
    // ---- covariance of the surviving neighbours (gicp.py:25-34, 5-17) ----
    const size_t cloud_row0 = (size_t)m.pt_begin;
    int cnt = 0;
    double mean[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int s = 0; s < KCAP; ++s) {
        const bool ok = (s >= KCAP - a.k) && ai[s] != INT_MAX && sqrt(ad[s]) < a.radius;
        if (!ok && s >= KCAP - a.k) ai[s] = INT_MAX;
        if (ok) {
            ++cnt;
            const Real* q = a.raw + (cloud_row0 + ai[s]) * D;
#pragma unroll
            for (int c = 0; c < D; ++c) mean[c] += (double)q[c];
        }
    }
    if (a.knn_idx) {
        int o = 0;
        int* out = a.knn_idx + (cloud_row0 + my_idx) * (size_t)a.k;
        double* outd = a.knn_dist ? a.knn_dist + (cloud_row0 + my_idx) * (size_t)a.k : nullptr;
#pragma unroll
        for (int s = 0; s < KCAP; ++s) {
            if (s >= KCAP - a.k && ai[s] != INT_MAX) {
                out[o] = ai[s];
                if (outd) outd[o] = sqrt(ad[s]);
                ++o;
            }
        }
        for (; o < a.k; ++o) {
            out[o] = -1;
            if (outd) outd[o] = INFINITY;
        }
    }
    constexpr int NS = Dim<D>::NS;
    double C[NS];
    bool ident = cnt <= 1;
    if (!ident) {
        const double inv = 1.0 / cnt;
#pragma unroll
        for (int c = 0; c < D; ++c) mean[c] *= inv;
        double S[6] = {0, 0, 0, 0, 0, 0};  // 00 01 02 11 12 22
#pragma unroll
        for (int s = 0; s < KCAP; ++s) {
            if (s >= KCAP - a.k && ai[s] != INT_MAX) {
                const Real* q = a.raw + (cloud_row0 + ai[s]) * D;
                const double d0 = (double)q[0] - mean[0], d1 = (double)q[1] - mean[1];
                const double d2 = (D == 3) ? (double)q[D - 1] - mean[2] : 0.0;
                S[0] += d0 * d0; S[1] += d0 * d1; S[2] += d0 * d2;
                S[3] += d1 * d1; S[4] += d1 * d2; S[5] += d2 * d2;
            }
        }
        const double f = 1.0 / (cnt - 1);  // ddof = 1 (np.cov default, gicp.py:12)
#pragma unroll
        for (int i = 0; i < 6; ++i) S[i] *= f;
        bool finite = true;
#pragma unroll
        for (int i = 0; i < 6; ++i) finite = finite && isfinite(S[i]);
        if (!finite) {
            ident = true;  // gicp.py:31-32
        } else if constexpr (D == 2) {
            // eigenvector of the largest eigenvalue (gicp.py:14-16): C = lam_n I + (lam_t-lam_n) v v^T
            const double phi = 0.5 * atan2(2.0 * S[1], S[0] - S[3]);
            double sn, cs;
            sincos(phi, &sn, &cs);
            const double dl = a.lam_t - a.lam_n;
            C[0] = a.lam_n + dl * cs * cs;
            C[1] = dl * cs * sn;
            C[2] = a.lam_n + dl * sn * sn;
        } else {
            // normal = eigenvector of the smallest eigenvalue: C = lam_t I - (lam_t-lam_n) n n^T
            double n[3];
            smallest_eigvec3(S[0], S[1], S[2], S[3], S[4], S[5], n);
            const double dl = a.lam_t - a.lam_n;
            C[0] = a.lam_t - dl * n[0] * n[0];
            C[1] = -dl * n[0] * n[1];
            C[2] = -dl * n[0] * n[2];
            C[3] = a.lam_t - dl * n[1] * n[1];
            C[4] = -dl * n[1] * n[2];
            C[5] = a.lam_t - dl * n[2] * n[2];
        }
    }
    if (ident) {
        if constexpr (D == 2) { C[0] = 1.0; C[1] = 0.0; C[2] = 1.0; }
        else { C[0] = 1.0; C[1] = 0.0; C[2] = 0.0; C[3] = 1.0; C[4] = 0.0; C[5] = 1.0; }
    }
    Real* out = a.cov_sorted + (size_t)s_pos * NS;
#pragma unroll
    for (int i = 0; i < NS; ++i) out[i] = (Real)C[i];
}

// ================================================================================================
// general path
// ================================================================================================
template <int D, typename Real, int KCAP>
__device__ __forceinline__ void knn_general_chunk(const KnnArgs<Real>& a, int cloud, int base, int end,
                                                  unsigned char* wbase, WarpStage<Real>& ws, int lane) {
    double* qd = reinterpret_cast<double*>(wbase + KNN_STAGE_BYTES);                 // [KNN_QUEUE][32]
    int* qi = reinterpret_cast<int*>(wbase + KNN_STAGE_BYTES + KNN_QUEUE * 32 * 8);  // [KNN_QUEUE][32]
    const CloudMeta m = a.meta[cloud];

    const bool valid = base + lane < end;
    const PRec<Real> me = a.spts[valid ? base + lane : end - 1];
    const int my_idx = (int)me.idx;
    const int cx = min(max(cell_coord((double)me.x, m.origin[0], m.inv_h), 0), m.dims[0] - 1);
    const int cy = min(max(cell_coord((double)me.y, m.origin[1], m.inv_h), 0), m.dims[1] - 1);
    const int cz = (D == 3) ? min(max(cell_coord((double)me.z, m.origin[2], m.inv_h), 0), m.dims[2] - 1) : 0;

    // sorted top-k: slots [KCAP-k, KCAP) are live, the ones before hold -1 sentinels
    double ad[KCAP];
    int ai[KCAP];
    const double r2cap = a.radius * a.radius * (1.0 + 1e-12);
#pragma unroll
    for (int s = 0; s < KCAP; ++s) {
        const bool live = s >= KCAP - a.k;
        ad[s] = live ? r2cap : -1.0;
        ai[s] = live ? INT_MAX : -1;
    }
    float thr32 = __double2float_ru(r2cap * (1.0 + 1e-6));
    const Real mx = me.x, my = me.y, mz = me.z;
    int qn = 0;

    auto drain = [&]() {
        const int nmax = warp_max(qn);
        for (int i = 0; i < nmax; ++i) {
            if (i < qn) {
                const double e2 = qd[i * 32 + lane];
                const int ci = qi[i * 32 + lane];
                bool lt_s = key_less(e2, ci, ad[KCAP - 1], ai[KCAP - 1]);
                if (lt_s) {
#pragma unroll
                    for (int s = KCAP - 1; s > 0; --s) {
                        const bool lt_prev = key_less(e2, ci, ad[s - 1], ai[s - 1]);
                        if (lt_prev) { ad[s] = ad[s - 1]; ai[s] = ai[s - 1]; }
                        else if (lt_s) { ad[s] = e2; ai[s] = ci; }
                        lt_s = lt_prev;
                    }
                    if (lt_s) { ad[0] = e2; ai[0] = ci; }
                }
            }
        }
        qn = 0;
        thr32 = __double2float_ru(ad[KCAP - 1] * (1.0 + 1e-6));
    };

    const int rho_max = max(1, (int)ceil(a.radius / (m.h * (1.0 - 1e-9))));
    unsigned pending = 0xffffffffu;
    while (pending) {
        const unsigned grp = next_group(pending, cx, cy, cz, KNN_GROUP_REACH);
        pending &= ~grp;
        const bool mine = (grp >> lane) & 1u;
        const int mycell[3] = {cx, cy, cz};
        int qlo[3], qhi[3];
        group_union(grp, lane, mycell, mycell, m, qlo, qhi);
        int plo[3] = {0, 0, 0}, phi[3] = {-1, -1, -1};
        for (int rho = 0; rho <= rho_max; ++rho) {
            int lo[3], hi[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) { lo[c] = max(qlo[c] - rho, 0); hi[c] = min(qhi[c] + rho, m.dims[c] - 1); }
            stream_cells<Real>(m, a.cell_start, a.lut, a.spts, lo, hi, plo, phi, rho > 0, ws, lane,
                               [&](const PRec<Real>* w, int n) {
                for (int j = 0; j < n; ++j) {
                    const PRec<Real> c = w[j];
                    bool pass = mine;
                    if (sizeof(Real) == 4) {
                        const float dx = (float)c.x - (float)mx, dy = (float)c.y - (float)my, dz = (float)c.z - (float)mz;
                        pass = pass && (fmaf(dz, dz, fmaf(dy, dy, dx * dx)) <= thr32);
                    }
                    if (pass) {
                        const double e2 = exact_d2((double)c.x - (double)mx, (double)c.y - (double)my,
                                                   (double)c.z - (double)mz);
                        const int ci = (int)c.idx;
                        if (key_less(e2, ci, ad[KCAP - 1], ai[KCAP - 1])) {
                            qd[qn * 32 + lane] = e2;
                            qi[qn * 32 + lane] = ci;
                            ++qn;
                        }
                    }
                    if (__any_sync(0xffffffffu, qn == KNN_QUEUE)) drain();
                }
            });
            drain();
#pragma unroll
            for (int c = 0; c < 3; ++c) { plo[c] = lo[c]; phi[c] = hi[c]; }
            if (rho == 0) continue;
            // done when the searched box covers every lane's k-th distance, or the radius
            const double cover = rho * m.h * (1.0 - 1e-9);
            const bool mine_done = !mine || ((ai[KCAP - 1] != INT_MAX) && (ad[KCAP - 1] <= cover * cover));
            if (__all_sync(0xffffffffu, mine_done) || cover >= a.radius) break;
        }
    }

    if (!valid) return;
    topk_finish<D, Real, KCAP>(a, m, base + lane, my_idx, ad, ai);
}

// from_list = 0: grid (blocks, n_clouds), one warp per 32 sorted points.
// from_list = 1: grid-stride over the fast path's overflow list.
template <int D, typename Real, int KCAP>
__global__ void __launch_bounds__(KNN_THREADS) knn_general_kernel(const KnnArgs<Real> a, int from_list) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char* wbase = smem_raw + 128 + warp * KNN_WARP_SMEM;
    // one mbarrier per warp for the whole kernel: the phase carries over from chunk to chunk
    WarpStage<Real> ws;
    ws.buf = reinterpret_cast<PRec<Real>*>(wbase);
    ws.bar = bars + warp;
    ws.phase = 0;
    ws.cap = KNN_STAGE_BYTES / (int)sizeof(PRec<Real>);
    if (lane == 0) { mbar_init(ws.bar, 1); mbar_fence_init(); }
    __syncwarp();
    if (!from_list) {
        const CloudMeta m = a.meta[blockIdx.y];
        int begin = m.pt_begin, end = m.pt_end;
        if (a.slice_begin >= 0) { begin = max(begin, a.slice_begin); end = min(end, a.slice_end); }
        const int base = begin + (blockIdx.x * KNN_WARPS + warp) * 32;
        if (base >= end) return;
        knn_general_chunk<D, Real, KCAP>(a, blockIdx.y, base, end, wbase, ws, lane);
    } else {
        const int n = min(*a.overflow_count, a.overflow_cap);
        for (int e = blockIdx.x * KNN_WARPS + warp; e < n; e += gridDim.x * KNN_WARPS) {
            const int2 it = a.overflow_list[e];
            const CloudMeta m = a.meta[it.x];
            int end = m.pt_end;
            if (a.slice_begin >= 0) end = min(end, a.slice_end);
            knn_general_chunk<D, Real, KCAP>(a, it.x, it.y, end, wbase, ws, lane);
            __syncwarp();
        }
    }
}

// ================================================================================================
// brute force for small clouds (latency path): one thread per query, every point of the cloud streamed
// from shared memory (a broadcast read), exact float64 keys, sorted top-k in registers.  Measured per cloud
// (grid build + k-NN, stream synchronised): 48-point scans 77 -> 60 us, 192-360-point scans 95 -> 102 us - n serial
// fp64 candidate tests per thread overtake the grid walk's ~20 TMA round trips at ~150 points, hence the cap.
// grid (n_clouds), KNN_BRUTE_THREADS threads; dynamic shared memory n_max * sizeof(PRec<Real>).
// ================================================================================================
constexpr int KNN_BRUTE_MAX = 128;
constexpr int KNN_BRUTE_THREADS = 128;

template <int D, typename Real, int KCAP>
__global__ void __launch_bounds__(KNN_BRUTE_THREADS) knn_brute_kernel(const KnnArgs<Real> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PRec<Real>* pts = reinterpret_cast<PRec<Real>*>(smem_raw);
    const CloudMeta m = a.meta[blockIdx.x];
    const int n = m.pt_end - m.pt_begin;
    for (int i = threadIdx.x; i < n; i += KNN_BRUTE_THREADS) pts[i] = a.spts[m.pt_begin + i];
    __syncthreads();
    const double r2cap = a.radius * a.radius * (1.0 + 1e-12);
    for (int q = threadIdx.x; q < n; q += KNN_BRUTE_THREADS) {
        const PRec<Real> me = pts[q];
        double ad[KCAP];
        int ai[KCAP];
#pragma unroll
        for (int s = 0; s < KCAP; ++s) {
            const bool live = s >= KCAP - a.k;
            ad[s] = live ? r2cap : -1.0;
            ai[s] = live ? INT_MAX : -1;
        }
        for (int j = 0; j < n; ++j) {
            const PRec<Real> c = pts[j];
            const double e2 = exact_d2((double)c.x - (double)me.x, (double)c.y - (double)me.y, (double)c.z - (double)me.z);
            const int ci = (int)c.idx;
            bool lt_s = key_less(e2, ci, ad[KCAP - 1], ai[KCAP - 1]);
            if (lt_s) {
#pragma unroll
                for (int s = KCAP - 1; s > 0; --s) {
                    const bool lt_prev = key_less(e2, ci, ad[s - 1], ai[s - 1]);
                    if (lt_prev) { ad[s] = ad[s - 1]; ai[s] = ai[s - 1]; }
                    else if (lt_s) { ad[s] = e2; ai[s] = ci; }
                    lt_s = lt_prev;
                }
                if (lt_s) { ad[0] = e2; ai[0] = ci; }
            }
        }
        topk_finish<D, Real, KCAP>(a, m, m.pt_begin + q, (int)me.idx, ad, ai);
    }
}

}  // namespace gicp
