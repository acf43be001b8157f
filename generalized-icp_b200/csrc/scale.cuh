// K3s: the adaptive robust scale (gicpSetRobustKernelAdaptive).  Between the search (K3a) and the accumulation (K3b)
// of every outer iteration, pair p's scale becomes c_p = max(min_scale, kappa * m_p), m_p the lower median (rank
// floor((n-1)/2), ascending) of the float64 distances d_i of its n gated-in correspondences.
//
// The order statistic is an exact radix select.  A non-negative double orders like its bit pattern read as uint64, so
// the key of a point is the bits of its d_i (NO_KEY when it has no gated-in match), and the median's key is found one
// 8-bit digit at a time, from the top: a histogram of the digit over the keys that share the digits found so far, and
// the bin that holds the wanted rank.  As soon as that bin holds a single key, one sweep finds it.  Integer counts only:
// the result is exact and the same on every run.
//   - fused loop: block_pair_scale, the whole select inside the pair's block, keys in shared memory;
//   - multi-launch loop / stage entry points: scale_select_kernel, one launch per digit over the active pairs, keys in a
//     per-point scratch written by the first launch (later launches read only the keys, never the targets), block
//     histograms summed per pair in global memory, and the last block of a pair to finish picks the bin.
#pragma once
#include "objective.cuh"

namespace gicp {

constexpr unsigned long long NO_KEY = ~0ull;   // above every finite distance's bits
constexpr int SEL_BINS = 256;
constexpr int SEL_PASSES = 8;                   // 8-bit digits of a 64-bit key

// per pair, between the launches of the multi-launch select
struct SelState {
    unsigned long long prefix;   // the digits of the median's key found so far (lower bits 0)
    unsigned k;                  // rank of the median among the keys that share them
    int shift;                   // the lowest bit found so far
    int phase;                   // SEL_RUNNING, SEL_UNIQUE (one key shares the prefix: the next launch finds it), SEL_DONE
};
enum { SEL_RUNNING = 0, SEL_UNIQUE = 1, SEL_DONE = 2 };

struct ScaleArgs {
    unsigned long long* keys;   // [n_src_total] (source nn order)
    unsigned* hist;             // [n_pairs][SEL_BINS], zero between uses
    unsigned* arrived;          // [n_pairs] blocks of the current launch that are done, zero between uses
    SelState* sel;              // [n_pairs]
    double* scale;              // [n_pairs] the result (ObjArgs::pair_scale)
};

template <int D, typename Real>
__device__ __forceinline__ void pair_transform(const ObjArgs<Real>& a, const int pair, const PairState& st, double (&R)[D][D],
                                               double (&t)[D]) {
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
}

// the key of source point s (its match from K3a, the distance and the gate exactly as accumulate_block forms them)
template <int D, typename Real>
__device__ __forceinline__ unsigned long long scale_key(const ObjArgs<Real>& a, const double (&R)[D][D],
                                                        const double (&t)[D], const int s) {
    const int m = a.match[s];
    if (m < 0) return NO_KEY;
    const PRec<Real> q = a.tgt_spts[m];
    double pp[3] = {0.0, 0.0, 0.0};
    transform_point<D, Real>(R, t, a.src_spts[s], pp);
    const double d = sqrt(exact_d2((double)q.x - pp[0], (double)q.y - pp[1], (double)q.z - pp[2]));
    return d > a.d_max ? NO_KEY : (unsigned long long)__double_as_longlong(d);
}

// does `key` share the digits above bit `shift` with `prefix` (shift 64: every key does)
__device__ __forceinline__ bool sel_match(unsigned long long key, unsigned long long prefix, int shift) {
    return key != NO_KEY && (shift >= 64 || (key >> shift) == (prefix >> shift));
}

// warp 0, all lanes: the bin of `hist` that holds rank k (0 <= k < total): its index, the count of the bins below it and
// its own count.  `total` (every lane) is the sum of all bins.
__device__ __forceinline__ void sel_pick_bin(const unsigned* hist, const unsigned k, int& bin, unsigned& below,
                                             unsigned& in_bin) {
    const int lane = threadIdx.x & 31;
    unsigned c[SEL_BINS / 32], sum = 0;
#pragma unroll
    for (int j = 0; j < SEL_BINS / 32; ++j) { c[j] = hist[lane * (SEL_BINS / 32) + j]; sum += c[j]; }
    unsigned inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    const unsigned exc = inc - sum;
    const bool mine = exc <= k && k < inc;
    const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
    int b = 0;
    unsigned acc = exc, cnt = 0;
    if (mine) {
        bool found = false;
#pragma unroll
        for (int j = 0; j < SEL_BINS / 32; ++j) {
            if (!found && k < acc + c[j]) { b = j; cnt = c[j]; found = true; }
            if (!found) acc += c[j];
        }
    }
    bin = __shfl_sync(0xffffffffu, lane * (SEL_BINS / 32) + b, src);
    below = __shfl_sync(0xffffffffu, acc, src);
    in_bin = __shfl_sync(0xffffffffu, cnt, src);
}

__device__ __forceinline__ unsigned warp_total(unsigned v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- fused loop: the scale of pair `pair` at its current state, computed by the whole block.  `keys`: at least as
// many slots as the pair has source points (shared memory).  Every thread returns the same c. ----
template <int D, typename Real>
__device__ __forceinline__ double block_pair_scale(const ObjArgs<Real>& a, const int pair, const PairState* stp,
                                                   unsigned long long* keys) {
    __shared__ unsigned s_hist[SEL_BINS];
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned s_k;
    __shared__ int s_shift, s_phase;
    double R[D][D], t[D];
    pair_transform<D, Real>(a, pair, *stp, R, t);
    const CloudMeta ms = a.src_meta[pair];
    const int n_pts = ms.pt_end - ms.pt_begin;
    for (int i = threadIdx.x; i < n_pts; i += OBJ_THREADS) keys[i] = scale_key<D, Real>(a, R, t, ms.pt_begin + i);
    if (threadIdx.x == 0) { s_prefix = 0; s_shift = 64; s_phase = SEL_RUNNING; }
    for (int pass = 0; pass < SEL_PASSES; ++pass) {
        for (int b = threadIdx.x; b < SEL_BINS; b += OBJ_THREADS) s_hist[b] = 0;
        __syncthreads();                                       // keys, cleared bins and the last pick are visible
        const unsigned long long prefix = s_prefix;
        const int above = s_shift, shift = above - 8;
        for (int i = threadIdx.x; i < n_pts; i += OBJ_THREADS) {
            const unsigned long long key = keys[i];
            if (sel_match(key, prefix, above)) atomicAdd(&s_hist[(key >> shift) & (SEL_BINS - 1)], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            unsigned k = s_k;
            bool empty = false;
            if (pass == 0) {
                unsigned n = 0;
                for (int b = threadIdx.x; b < SEL_BINS; b += 32) n += s_hist[b];
                n = warp_total(n);
                k = n ? (n - 1) / 2 : 0;
                empty = n == 0;
                if (empty && threadIdx.x == 0) s_phase = SEL_DONE;   // no gated-in match: m = 0, c = min_scale
            }
            if (!empty) {
                int bin;
                unsigned below, in_bin;
                sel_pick_bin(s_hist, k, bin, below, in_bin);
                if (threadIdx.x == 0) {
                    s_prefix = prefix | ((unsigned long long)bin << shift);
                    s_k = k - below;
                    s_shift = shift;
                    s_phase = shift == 0 ? SEL_DONE : in_bin == 1 ? SEL_UNIQUE : SEL_RUNNING;
                }
            }
        }
        __syncthreads();
        if (s_phase != SEL_RUNNING) break;
    }
    if (s_phase == SEL_UNIQUE) {                               // the one key that shares the prefix is the median
        const unsigned long long prefix = s_prefix;
        const int shift = s_shift;
        __syncthreads();
        for (int i = threadIdx.x; i < n_pts; i += OBJ_THREADS)
            if (sel_match(keys[i], prefix, shift)) s_prefix = keys[i];
        __syncthreads();
    }
    const double m = s_shift == 64 ? 0.0 : __longlong_as_double((long long)s_prefix);
    return adaptive_scale(a.scale_kappa, m, a.scale_min);
}

// The same as a call: the 2-D fused loop calls it, so that the loop keeps its registers (inlined, ptxas caps the 2-D
// f32 loop at 128 registers and spills; the 3-D loops spill less with the select inlined).
template <int D, typename Real>
__device__ __noinline__ double block_pair_scale_call(const ObjArgs<Real>& a, const int pair, const PairState* stp,
                                                     unsigned long long* keys) {
    return block_pair_scale<D, Real>(a, pair, stp, keys);
}

// ---- multi-launch loop: digit `pass` of every pair's select.  Grid (blocks_per_pair, pairs or active-list slots), the
// blocks of the accumulation (a.ppt points per thread).  Launched SEL_PASSES times per iteration; the launches after a
// pair's median is known return at once. ----
template <int D, typename Real>
__global__ void __launch_bounds__(OBJ_THREADS) scale_select_kernel(const ObjArgs<Real> a, const ScaleArgs sc,
                                                                   const int pass) {
    __shared__ unsigned s_hist[SEL_BINS];
    __shared__ bool s_last;
    const int pair = obj_pair_of_block(a);
    if (pair < 0) return;
    const PairState st = a.state[pair];
    if (!a.ignore_status && st.status != PAIR_ACTIVE) return;
    SelState ss;
    if (pass == 0) {
        ss.prefix = 0; ss.k = 0; ss.shift = 64; ss.phase = SEL_RUNNING;
    } else {
        ss = sc.sel[pair];
        if (ss.phase == SEL_DONE) return;
    }
    const CloudMeta ms = a.src_meta[pair];
    const int begin = ms.pt_begin + blockIdx.x * a.ppt * OBJ_THREADS;
    const int end = min(ms.pt_end, begin + a.ppt * OBJ_THREADS);
    if (ss.phase == SEL_UNIQUE) {
        for (int s = begin + threadIdx.x; s < end; s += OBJ_THREADS) {
            const unsigned long long key = sc.keys[s];
            if (sel_match(key, ss.prefix, ss.shift)) {   // exactly one point of the pair
                sc.scale[pair] = adaptive_scale(a.scale_kappa, __longlong_as_double((long long)key), a.scale_min);
                sc.sel[pair].phase = SEL_DONE;
            }
        }
        return;
    }
    const int shift = ss.shift - 8;
    for (int b = threadIdx.x; b < SEL_BINS; b += OBJ_THREADS) s_hist[b] = 0;
    __syncthreads();
    if (pass == 0) {
        double R[D][D], t[D];
        pair_transform<D, Real>(a, pair, st, R, t);
        for (int s = begin + threadIdx.x; s < end; s += OBJ_THREADS) {
            const unsigned long long key = scale_key<D, Real>(a, R, t, s);
            sc.keys[s] = key;
            if (key != NO_KEY) atomicAdd(&s_hist[key >> shift], 1u);
        }
    } else {
        for (int s = begin + threadIdx.x; s < end; s += OBJ_THREADS) {
            const unsigned long long key = sc.keys[s];
            if (sel_match(key, ss.prefix, ss.shift)) atomicAdd(&s_hist[(key >> shift) & (SEL_BINS - 1)], 1u);
        }
    }
    __syncthreads();
    unsigned* gh = sc.hist + (size_t)pair * SEL_BINS;
    for (int b = threadIdx.x; b < SEL_BINS; b += OBJ_THREADS)
        if (s_hist[b]) atomicAdd(gh + b, s_hist[b]);
    __threadfence();                                          // this block's counts before its arrival
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(sc.arrived + pair, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    // the last block of the pair: every other block's counts are in gh
    __threadfence();
    for (int b = threadIdx.x; b < SEL_BINS; b += OBJ_THREADS) s_hist[b] = __ldcg(gh + b);
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned k = ss.k;
        bool empty = false;
        if (pass == 0) {
            unsigned n = 0;
            for (int b = threadIdx.x; b < SEL_BINS; b += 32) n += s_hist[b];
            n = warp_total(n);
            k = n ? (n - 1) / 2 : 0;
            empty = n == 0;
        }
        if (empty) {
            if (threadIdx.x == 0) {                          // no gated-in match: c = min_scale
                sc.scale[pair] = adaptive_scale(a.scale_kappa, 0.0, a.scale_min);
                ss.phase = SEL_DONE;
                sc.sel[pair] = ss;
            }
        } else {
            int bin;
            unsigned below, in_bin;
            sel_pick_bin(s_hist, k, bin, below, in_bin);
            if (threadIdx.x == 0) {
                ss.prefix |= (unsigned long long)bin << shift;
                ss.k = k - below;
                ss.shift = shift;
                ss.phase = shift == 0 ? SEL_DONE : in_bin == 1 ? SEL_UNIQUE : SEL_RUNNING;
                if (shift == 0)
                    sc.scale[pair] = adaptive_scale(a.scale_kappa, __longlong_as_double((long long)ss.prefix), a.scale_min);
                sc.sel[pair] = ss;
            }
        }
    }
    for (int b = threadIdx.x; b < SEL_BINS; b += OBJ_THREADS) gh[b] = 0;   // ready for the next launch
    if (threadIdx.x == 0) sc.arrived[pair] = 0;
}

}  // namespace gicp
