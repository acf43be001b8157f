// K0: voxel-grid downsampling of a batch (gicpVoxelDownsample).  Semantics (include/gicp_b200.h):
//   voxel of a point = floor((double)p_a / L) per axis, lattice anchored at the origin; rows with a non-finite
//   coordinate are dropped; a voxel with >= min_points points becomes its fp64 centroid; a cloud's output rows
//   are ordered by each voxel's lowest input row.
// Pipeline: per-cloud voxel bounds -> 64-bit key per row (cloud | cloud-relative voxel coordinates) -> stable sort
// of (key, row) -> run heads / tails in sorted order -> keep flag at each kept voxel's head row (input order) ->
// exclusive scan = output row -> fixed-order fp64 centroid per run.
// gicpSetVoxelized runs the same pipeline with Stats = true: the centroid pass also accumulates each voxel's second
// moments and writes its regularised covariance (vox_cov_finish).
#pragma once
#include "common.cuh"
#include "knn_cov.cuh"

namespace gicp {

constexpr int VOX_THREADS = 256;
constexpr int VOX_ITEMS = 16;        // points per thread of the bounds pass
constexpr int VOX_SEQ_MAX = 32;      // runs up to this long are summed by one thread, longer ones by a block
constexpr unsigned long long VOX_SENTINEL = ~0ull;   // key of a non-finite row: sorts after every voxel

template <int D, typename Real>
__device__ __forceinline__ bool vox_load(const Real* __restrict__ pts, long long g, double v[D]) {
    bool fin = true;
#pragma unroll
    for (int c = 0; c < D; ++c) {
        v[c] = (double)pts[(size_t)g * D + c];
        fin = fin && isfinite(v[c]);
    }
    return fin;
}

// grid (chunks, n_clouds): min / max of each coordinate over the chunk's FINITE rows -> part[cloud][chunk][6]
template <int D, typename Real>
__global__ void __launch_bounds__(VOX_THREADS) voxel_bounds_partial_kernel(const Real* __restrict__ pts,
                                                                           const int* __restrict__ offsets,
                                                                           double* __restrict__ part, int chunks) {
    const int cloud = blockIdx.y;
    const int b = offsets[cloud], e = offsets[cloud + 1];
    const int c0 = b + blockIdx.x * (VOX_THREADS * VOX_ITEMS);
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < VOX_ITEMS; ++i) {
        const int g = c0 + i * VOX_THREADS + threadIdx.x;
        if (g >= e) break;
        double v[D];
        if (!vox_load<D, Real>(pts, g, v)) continue;
#pragma unroll
        for (int c = 0; c < D; ++c) { lo[c] = fmin(lo[c], v[c]); hi[c] = fmax(hi[c], v[c]); }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fmin(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmax(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
    }
    __shared__ double s_lo[VOX_THREADS / 32][3], s_hi[VOX_THREADS / 32][3];
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0)
        for (int c = 0; c < 3; ++c) { s_lo[w][c] = lo[c]; s_hi[w][c] = hi[c]; }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int c = threadIdx.x;
        double l = s_lo[0][c], h = s_hi[0][c];
        for (int i = 1; i < VOX_THREADS / 32; ++i) { l = fmin(l, s_lo[i][c]); h = fmax(h, s_hi[i][c]); }
        double* o = part + ((size_t)cloud * chunks + blockIdx.x) * 6;
        o[c] = l;
        o[3 + c] = h;
    }
}

// one warp per cloud: vb[cloud] = (floor(lo / L), floor(hi / L)) per axis.  floor(x / L) is monotone in x (IEEE
// division rounds monotonically), so these are the smallest and largest voxel indices of the cloud's finite rows.
// An empty cloud keeps lo = +inf > hi = -inf.
__global__ void voxel_bounds_kernel(const double* __restrict__ part, int chunks, int n_clouds, double leaf,
                                    double* __restrict__ vb) {
    const int cloud = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (cloud >= n_clouds) return;
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int k = lane; k < chunks; k += 32) {
        const double* p = part + ((size_t)cloud * chunks + k) * 6;
        for (int c = 0; c < 3; ++c) { lo[c] = fmin(lo[c], p[c]); hi[c] = fmax(hi[c], p[3 + c]); }
    }
    for (int c = 0; c < 3; ++c)
        for (int o = 16; o > 0; o >>= 1) {
            lo[c] = fmin(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmax(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
    if (lane == 0)
        for (int c = 0; c < 3; ++c) {
            vb[(size_t)cloud * 6 + c] = (lo[c] <= hi[c]) ? floor(lo[c] / leaf) : INFINITY;
            vb[(size_t)cloud * 6 + 3 + c] = (lo[c] <= hi[c]) ? floor(hi[c] / leaf) : -INFINITY;
        }
}

// grid (ceil(max_n / 256), n_clouds): key and sort value (the row) of every row.  The host has checked that every
// cloud-relative voxel index fits its field: shift[c] places axis c, the cloud index sits at cloud_shift (or is left
// out when cloud_shift < 0: the segmented sort keeps the clouds apart).
struct VoxKeyGeom {
    int shift[3];
    int cloud_shift;
};
template <int D, typename Real>
__global__ void voxel_key_kernel(const Real* __restrict__ pts, const int* __restrict__ offsets,
                                 const double* __restrict__ vb, double leaf, VoxKeyGeom geo,
                                 unsigned long long* __restrict__ keys, int* __restrict__ vals) {
    const int cloud = blockIdx.y;
    const int g = offsets[cloud] + blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= offsets[cloud + 1]) return;
    double v[D];
    unsigned long long k = VOX_SENTINEL;
    if (vox_load<D, Real>(pts, g, v)) {
        k = geo.cloud_shift >= 0 ? (unsigned long long)cloud << geo.cloud_shift : 0ull;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const long long q = (long long)floor(v[c] / leaf) - (long long)vb[(size_t)cloud * 6 + c];
            k |= (unsigned long long)q << geo.shift[c];
        }
    }
    keys[g] = k;
    vals[g] = g;
}

// segmented sort: equal coordinate keys of two clouds can meet at a segment boundary; the first row of every
// non-empty segment starts a run (rid doubles as the head flag array before the scan)
__global__ void voxel_segment_heads_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ offsets,
                                           int n_clouds, int* __restrict__ head) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_clouds) return;
    const int b = offsets[c];
    if (b < offsets[c + 1] && keys[b] != VOX_SENTINEL) head[b] = 1;
}

// head[i] = 1 where sorted position i starts a voxel (a finite row whose key differs from its predecessor's); the
// array has n + 1 entries, the last stays 0
__global__ void voxel_head_kernel(const unsigned long long* __restrict__ keys, int n, int* __restrict__ head) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    int f = 0;
    if (i < n) {
        const unsigned long long k = keys[i];
        f = k != VOX_SENTINEL && (i == 0 || keys[i - 1] != k);
    }
    head[i] = f;
}

// after the exclusive scan of the head flags (rid[i] = voxels starting before position i, rid[n] = voxel count):
// run_begin / run_end of every voxel in sorted order
__global__ void voxel_runs_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ rid, int n,
                                  int* __restrict__ run_begin, int* __restrict__ run_end) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || keys[i] == VOX_SENTINEL) return;
    const bool head = rid[i + 1] != rid[i];
    const int run = head ? rid[i] : rid[i] - 1;
    if (head) run_begin[run] = i;
    const bool tail = i + 1 == n || keys[i + 1] == VOX_SENTINEL || rid[i + 2] != rid[i + 1];
    if (tail) run_end[run] = i + 1;
}

// keep[row] = 1 at the lowest input row of every voxel with >= min_points points (keep is zeroed before)
__global__ void voxel_keep_kernel(const int* __restrict__ rid, int n, const int* __restrict__ run_begin,
                                  const int* __restrict__ run_end, const int* __restrict__ rows, int min_points,
                                  int* __restrict__ keep) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rid[n]) return;
    const int b = run_begin[r];
    if (run_end[r] - b >= min_points) keep[rows[b]] = 1;
}

// out_off[c] = output rows before cloud c (orow is the exclusive scan of keep, orow[n] the total)
__global__ void voxel_out_offsets_kernel(const int* __restrict__ orow, const int* __restrict__ offsets, int n_clouds,
                                         int* __restrict__ out_off) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= n_clouds) out_off[c] = orow[offsets[c]];
}

// cloud of output row o: the last c with out_off[c] <= o (empty clouds share their offset with the next one)
__device__ __forceinline__ int vox_cloud_of(const int* __restrict__ out_off, int n_clouds, int o) {
    int lo = 0, hi = n_clouds;   // out_off[lo] <= o < out_off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (out_off[mid] <= o) lo = mid; else hi = mid;
    }
    return lo;
}

struct VoxOutArgs {
    const int* rid;         // rid[n] = number of voxels
    int n;
    const int* run_begin;
    const int* run_end;
    const int* rows;        // sorted rows (ascending within a voxel: the sorts are stable)
    const int* orow;        // output row of a kept voxel, at its lowest row
    const int* out_off;     // (n_clouds + 1) output offsets
    int n_clouds;
    int min_points;
    int* voxel_of;          // optional (n) cloud-local output row, -1 prefilled
    int* counts;            // optional (M) points per output row
    int* big_list;          // voxels longer than VOX_SEQ_MAX, for voxel_centroid_block_kernel
    int* big_count;
};

template <int D, typename Real>
__device__ __forceinline__ void vox_write(const VoxOutArgs& a, Real* __restrict__ out, int o, const double s[D],
                                          int count) {
#pragma unroll
    for (int c = 0; c < D; ++c) out[(size_t)o * D + c] = (Real)(s[c] / (double)count);
    if (a.counts) a.counts[o] = count;
}

// where the Stats kernels write the covariance of output row o (cov + o * NS) and its regularisation
template <typename Real>
struct VoxCovArgs {
    Real* cov;
    double lam_t, lam_n;
};

// The covariance of one voxel from its moments about its first point p0: n points, sd = sum (p - p0), sq = sum
// (p - p0)(p - p0)^T (packed upper triangle, Dim<D>::NS entries).  The sample covariance (ddof = 1) about the mean
// is (sq - n m m^T) / (n - 1) with m = sd / n - the formula of knn_finish_cov, whose moments are about the query
// point - then regularised_cov; a voxel of one point, or a non-finite scatter, gets the identity (gicp.py:27, 31-34).
// The shift by p0 bounds the cancellation by the voxel's extent instead of its distance from the origin.
template <int D>
__host__ __device__ inline void vox_cov_finish(int n, const double sd[D], const double sq[Dim<D>::NS], double lam_t,
                                               double lam_n, double C[Dim<D>::NS]) {
    double S[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // regularised_cov's layout: 00 01 02 11 12 22 (2-D: 00 01 11)
    const bool ident = n <= 1;
    if (!ident) {
        const double inv = 1.0 / n;
        const double f = 1.0 / (n - 1);   // ddof = 1 (np.cov default, gicp.py:12)
        double m[D];
#pragma unroll
        for (int c = 0; c < D; ++c) m[c] = sd[c] * inv;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j) S[symidx(3, i, j)] = (sq[symidx(D, i, j)] - n * m[i] * m[j]) * f;
    }
    regularised_cov<D>(S, ident, lam_t, lam_n, C);
}

template <int D, typename Real>
__device__ __forceinline__ void vox_write_cov(const VoxCovArgs<Real>& cv, int o, int count, const double sd[D],
                                              const double sq[Dim<D>::NS]) {
    constexpr int NS = Dim<D>::NS;
    double C[NS];
    vox_cov_finish<D>(count, sd, sq, cv.lam_t, cv.lam_n, C);
#pragma unroll
    for (int i = 0; i < NS; ++i) cv.cov[(size_t)o * NS + i] = (Real)C[i];
}

// one thread per voxel: the centroid of a voxel of <= VOX_SEQ_MAX points, summed in fp64 in ascending row order
// starting from the first point (a -0.0 coordinate survives); longer voxels go to the block kernel.  With Stats the
// same pass accumulates the moments about the first point and writes the voxel's covariance.
template <int D, typename Real, bool Stats>
__global__ void voxel_centroid_kernel(VoxOutArgs a, const Real* __restrict__ pts, Real* __restrict__ out,
                                      VoxCovArgs<Real> cv) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.rid[a.n]) return;
    const int b = a.run_begin[r], e = a.run_end[r];
    const int count = e - b;
    if (count < a.min_points) return;
    if (count > VOX_SEQ_MAX) {
        a.big_list[atomicAdd(a.big_count, 1)] = r;
        return;
    }
    const int head = a.rows[b];
    const int o = a.orow[head];
    const int local = a.voxel_of ? o - a.out_off[vox_cloud_of(a.out_off, a.n_clouds, o)] : 0;
    constexpr int NS = Dim<D>::NS;
    double s[D], p0[D], sd[D], sq[NS];
    vox_load<D, Real>(pts, head, s);
    if constexpr (Stats) {
#pragma unroll
        for (int c = 0; c < D; ++c) { p0[c] = s[c]; sd[c] = 0.0; }
#pragma unroll
        for (int i = 0; i < NS; ++i) sq[i] = 0.0;
    }
    if (a.voxel_of) a.voxel_of[head] = local;
#pragma unroll 4
    for (int j = b + 1; j < e; ++j) {
        const int row = a.rows[j];
        double v[D];
        vox_load<D, Real>(pts, row, v);
#pragma unroll
        for (int c = 0; c < D; ++c) s[c] += v[c];
        if constexpr (Stats) {
            double d[D];
#pragma unroll
            for (int c = 0; c < D; ++c) { d[c] = v[c] - p0[c]; sd[c] += d[c]; }
#pragma unroll
            for (int i = 0, k = 0; i < D; ++i)
#pragma unroll
                for (int jj = i; jj < D; ++jj, ++k) sq[k] += d[i] * d[jj];
        }
        if (a.voxel_of) a.voxel_of[row] = local;
    }
    vox_write<D, Real>(a, out, o, s, count);
    if constexpr (Stats) vox_write_cov<D, Real>(cv, o, count, sd, sq);
}

// one block per long voxel (persistent over the list): thread t sums points t, t + 256, ... in row order, then a
// fixed shared-memory tree.  The order depends only on the voxel's own points, so a batch and its clouds one at a
// time give identical bits.  -0.0 is the identity of IEEE addition (-0.0 + x == x for every x, +0.0 included).
// With Stats every thread also sums its points' moments about the voxel's first point, and the tree reduces them too:
// rows [0, D) of sm hold the sums, [D, 2D) the offsets from p0, [2D, 2D + NS) their outer products.
template <int D, typename Real, bool Stats>
__global__ void __launch_bounds__(VOX_THREADS) voxel_centroid_block_kernel(VoxOutArgs a, const Real* __restrict__ pts,
                                                                           Real* __restrict__ out, VoxCovArgs<Real> cv) {
    constexpr int NS = Dim<D>::NS;
    constexpr int NM = Stats ? 2 * D + NS : D;
    __shared__ double sm[NM][VOX_THREADS];
    const int n_big = *a.big_count;
    for (int k = blockIdx.x; k < n_big; k += gridDim.x) {
        const int r = a.big_list[k];
        const int b = a.run_begin[r], e = a.run_end[r];
        const int o = a.orow[a.rows[b]];
        const int local = a.voxel_of ? o - a.out_off[vox_cloud_of(a.out_off, a.n_clouds, o)] : 0;
        double s[D], p0[D], sd[D], sq[NS];
#pragma unroll
        for (int c = 0; c < D; ++c) s[c] = -0.0;
        if constexpr (Stats) {
            vox_load<D, Real>(pts, a.rows[b], p0);
#pragma unroll
            for (int c = 0; c < D; ++c) sd[c] = 0.0;
#pragma unroll
            for (int i = 0; i < NS; ++i) sq[i] = 0.0;
        }
#pragma unroll 4
        for (int j = b + threadIdx.x; j < e; j += VOX_THREADS) {
            const int row = a.rows[j];
            double v[D];
            vox_load<D, Real>(pts, row, v);
#pragma unroll
            for (int c = 0; c < D; ++c) s[c] += v[c];
            if constexpr (Stats) {
                double d[D];
#pragma unroll
                for (int c = 0; c < D; ++c) { d[c] = v[c] - p0[c]; sd[c] += d[c]; }
#pragma unroll
                for (int i = 0, k = 0; i < D; ++i)
#pragma unroll
                    for (int jj = i; jj < D; ++jj, ++k) sq[k] += d[i] * d[jj];
            }
            if (a.voxel_of) a.voxel_of[row] = local;
        }
#pragma unroll
        for (int c = 0; c < D; ++c) sm[c][threadIdx.x] = s[c];
        if constexpr (Stats) {
#pragma unroll
            for (int c = 0; c < D; ++c) sm[D + c][threadIdx.x] = sd[c];
#pragma unroll
            for (int i = 0; i < NS; ++i) sm[2 * D + i][threadIdx.x] = sq[i];
        }
        __syncthreads();
        for (int w = VOX_THREADS / 2; w > 0; w >>= 1) {
            if (threadIdx.x < w)
#pragma unroll
                for (int c = 0; c < NM; ++c) sm[c][threadIdx.x] += sm[c][threadIdx.x + w];
            __syncthreads();
        }
        if (threadIdx.x == 0) {
#pragma unroll
            for (int c = 0; c < D; ++c) s[c] = sm[c][0];
            vox_write<D, Real>(a, out, o, s, e - b);
            if constexpr (Stats) {
#pragma unroll
                for (int c = 0; c < D; ++c) sd[c] = sm[D + c][0];
#pragma unroll
                for (int i = 0; i < NS; ++i) sq[i] = sm[2 * D + i][0];
                vox_write_cov<D, Real>(cv, o, e - b, sd, sq);
            }
        }
        __syncthreads();
    }
}

}  // namespace gicp
