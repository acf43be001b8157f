// Fused registration loop for small pairs (the reference's own workloads: visualization.py's ~90-point pair,
// robot-visualization.py's 90-360-beam scans): the whole outer loop of gicp() (gicp.py:116-167) in ONE launch.
// One block per pair runs  K3a search -> K3b accumulation -> K4 solve  until the pair's stop rule fires; the
// stages are the very block functions of the multi-launch path (objective.cuh, solve.cuh), separated by
// __syncthreads() instead of kernel boundaries, so there is no launch, no poll and no host round trip inside a
// registration.  Requires every source cloud to fit one block (<= OBJ_THREADS * OBJ_MAX_PPT points).
#pragma once
#include "objective.cuh"
#include "scale.cuh"
#include "solve.cuh"

namespace gicp {

// `init_bbox` != nullptr: the kernel also initialises its pair (identity start, what init_state_kernel and the two
// memsets of the match / slack arrays do on the multi-launch path) - a small registration is then ONE launch.
// Robust: the accumulation weights every correspondence by its robust kernel weight (accumulate_block).  Adaptive
// (with Robust): the block first selects the pair's scale of the iteration (block_pair_scale, scale.cuh).
// Adaptive is a template argument of its own, so that the fixed-scale loop keeps its registers.
template <int D, typename Real, bool Robust = false, bool Adaptive = false>
__global__ void __launch_bounds__(OBJ_THREADS) register_loop_kernel(const ObjArgs<Real> oa, const SolveArgs sa,
                                                                    const double* init_bbox) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int NRED = Dim<D>::NRED;
    // the pair's state and the reduced form live in shared memory for the whole loop: on the multi-launch path they
    // travel through global memory between the stages, which costs a block that owns the pair four dependent L2 round
    // trips per outer iteration
    __shared__ double s_sum[NRED];
    __shared__ SolveScratch<D> s_sc;
    __shared__ PairState s_state;
    const int pair = blockIdx.x;
    WarpStage<Real> ws = obj_warp_stage<Real>(smem_raw);   // one mbarrier per warp for the whole loop
    if (init_bbox) {
        if (threadIdx.x == 0)
            init_pair_state<D>(&s_state, nullptr, init_bbox, pair, sa.d_T, sa.d_T_hist, sa.max_iterations, sa.d_n_outer,
                               sa.d_converged);
        const CloudMeta ms = oa.src_meta[pair];
        for (int s = ms.pt_begin + (int)threadIdx.x; s < ms.pt_end; s += OBJ_THREADS) {
            oa.match[s] = -1;
            if (oa.slack) oa.slack[s] = 0.f;
        }
    } else if (threadIdx.x == 0) {
        s_state = sa.state[pair];                          // initialised by init_state_kernel (start transform given)
    }
    __syncthreads();
    for (int it = 0; it < sa.max_iterations; ++it) {
        correspond_block<D, Real>(oa, pair, 0, ws, smem_raw, &s_state);
        __syncthreads();                                   // this block's matches are visible to the block
        double c = 0.0;                                    // the robust scale of this iteration
        if constexpr (Adaptive) {
            // the keys live behind the search's shared memory (obj_smem(ppt) + 8 B per point)
            unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw + obj_smem(oa.ppt));
            if constexpr (D == 2) c = block_pair_scale_call<D, Real>(oa, pair, &s_state, keys);
            else c = block_pair_scale<D, Real>(oa, pair, &s_state, keys);
        } else if constexpr (Robust) {
            c = oa.robust_scale;
        }
        accumulate_block<D, Real, Robust>(oa, pair, 0, &s_state, s_sum, c);
        __syncthreads();
        if (threadIdx.x < 32) solve_pair<D>(sa, pair, s_state, s_sum, s_sc, &s_state);   // warp 0, all lanes
        __syncthreads();                                   // the new state is visible to the block
        if (s_state.status != PAIR_ACTIVE) break;
    }
    if (threadIdx.x == 0) sa.state[pair] = s_state;        // what later calls on the handle read
}

}  // namespace gicp
