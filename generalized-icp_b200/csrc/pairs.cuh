// gicpSetPairList: the sources of a pair list gathered into pair order.
//
// The loop's per-point state (match, slack), the select's keys, the output rows and gicpEvaluate's correspondences are
// all indexed by src_meta[pair].pt_begin + i, so two pairs that share a source cannot share its rows.  Instead of a
// second base threaded through every kernel, every pair's source is copied once, in its grid order and with its
// cloud-local .idx, to rows [offsets[p], offsets[p+1]) of a pair-ordered array, and every pair gets metadata of its own.
// The existing kernels then run over the pair list exactly as over a one-to-one batch, unchanged.
#pragma once
#include "common.cuh"

namespace gicp {

constexpr int PAIR_GATHER_THREADS = 256;
constexpr int PAIR_GATHER_ROWS = 1024;   // source rows per block

template <typename Real> struct PairGatherArgs {
    const int* list;               // [n_pairs][3]: source cloud, target cloud, first row of the pair
    const CloudMeta* set_meta;     // the source set's search-grid metadata (CloudSet::nng)
    const PRec<Real>* set_spts;    // ... its records in that grid's order
    const Real* set_cov;           // ... its covariances in the same order; nullptr: the pairs' sources get C = 0
    const CloudMeta* tgt_set_meta;
    const double* tgt_set_bbox;    // [n_tgt][6]: min xyz, max xyz of the k-NN grid (the centring point's source)
    CloudMeta* src_meta;           // [n_pairs] outputs
    CloudMeta* tgt_meta;
    double* tgt_bbox;
    PRec<Real>* spts;
    Real* cov;
};

// bytes [0, n) from s to d by the block, in the widest word that both addresses and the length allow
template <typename W> __device__ __forceinline__ void block_copy(const char* __restrict__ s, char* __restrict__ d, size_t n) {
    const W* sw = reinterpret_cast<const W*>(s);
    W* dw = reinterpret_cast<W*>(d);
    for (size_t i = threadIdx.x; i < n / sizeof(W); i += PAIR_GATHER_THREADS) dw[i] = __ldg(sw + i);
}
__device__ __forceinline__ void block_copy_any(const char* s, char* d, size_t n) {
    const size_t a = (size_t)s | (size_t)d | n;
    if (a % 16 == 0) block_copy<uint4>(s, d, n);
    else if (a % 8 == 0) block_copy<uint2>(s, d, n);
    else block_copy<unsigned>(s, d, n);
}
__device__ __forceinline__ void block_zero_any(char* d, size_t n) {
    if (((size_t)d | n) % 16 == 0) {
        for (size_t i = threadIdx.x; i < n / 16; i += PAIR_GATHER_THREADS) reinterpret_cast<uint4*>(d)[i] = make_uint4(0, 0, 0, 0);
    } else {
        for (size_t i = threadIdx.x; i < n / 4; i += PAIR_GATHER_THREADS) reinterpret_cast<unsigned*>(d)[i] = 0u;
    }
}

// grid (blocks over the largest source, n_pairs): block x of pair p copies rows [x * PAIR_GATHER_ROWS, ...) of the
// pair's source; block 0 also writes the pair's metadata: the source's with its rows rebased (the kernels read only
// pt_begin / pt_end of it), the target cloud's unchanged (it addresses the target set's shared grid arrays, which the
// search reads in place) and the target cloud's box.
template <int D, typename Real>
__global__ void __launch_bounds__(PAIR_GATHER_THREADS) pair_gather_kernel(PairGatherArgs<Real> a) {
    constexpr int NS = Dim<D>::NS;
    const int p = blockIdx.y;
    const int s = a.list[3 * p], t = a.list[3 * p + 1], first = a.list[3 * p + 2];
    const CloudMeta ms = a.set_meta[s];
    const int n = ms.pt_end - ms.pt_begin;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        CloudMeta m = ms;
        m.pt_begin = first;
        m.pt_end = first + n;
        a.src_meta[p] = m;
        a.tgt_meta[p] = a.tgt_set_meta[t];
    }
    if (blockIdx.x == 0 && threadIdx.x < 6) a.tgt_bbox[p * 6 + threadIdx.x] = a.tgt_set_bbox[t * 6 + threadIdx.x];
    const int r0 = blockIdx.x * PAIR_GATHER_ROWS;
    const int rows = min(n - r0, PAIR_GATHER_ROWS);
    if (rows <= 0) return;
    block_copy<uint4>(reinterpret_cast<const char*>(a.set_spts + ms.pt_begin + r0),
                      reinterpret_cast<char*>(a.spts + first + r0), (size_t)rows * sizeof(PRec<Real>));
    char* dc = reinterpret_cast<char*>(a.cov + (size_t)(first + r0) * NS);
    const size_t cov_bytes = (size_t)rows * NS * sizeof(Real);
    if (a.set_cov) block_copy_any(reinterpret_cast<const char*>(a.set_cov + (size_t)(ms.pt_begin + r0) * NS), dc, cov_bytes);
    else block_zero_any(dc, cov_bytes);
}

}  // namespace gicp
