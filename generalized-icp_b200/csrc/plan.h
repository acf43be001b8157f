// Host-side plans: which kernels a set-up, a registration and a stage call run, and how their work is split.  Every
// path decision of the library is taken here, once per call, from the parameters, the input shape and the
// environment switches; gicp_b200.cu only sizes buffers and launches what a plan says.  No kernels: the .cuh
// headers are included for their constants.  tests/host_harness/plan_host.cu compiles this header for the host.
#pragma once

#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <vector>

#include "../../include/gicp_b200.h"
#include "grid.cuh"
#include "knn_cov.cuh"
#include "objective.cuh"
#include "solve.cuh"

namespace gicp {

// Environment switches.  Each one is either the reference a test compares the default path against, or the way a
// test reaches a path at sizes it can afford.  The defaults are the library's behaviour.
struct Switches {
    bool no_skip = false;            // GICP_NO_SKIP=1: K3a searches every point in every iteration (no slack skip)
    int track_max_cells = 1 << 30;   // GICP_TRACK_CELLS=n: a tracked K3a lane walks at most n cells on its own
    int shell_search = 1;            // GICP_SHELL_SEARCH=0: untracked K3a lanes go straight to the cooperative search
    int centre_first = 1;            // GICP_CENTRE_FIRST=0: the cooperative search does not stream the centre cells first
    int corr_split = 2;              // GICP_CORR_SPLIT=n: K3a blocks per K3b block (before the rounding of plan_loop)
    bool active_list = true;         // GICP_ACTIVE_LIST=0: every pair's blocks are launched in every iteration
    bool fused_loop = true;          // GICP_FUSED_LOOP=0: small pairs take the multi-launch loop
    bool small_grid = true;          // GICP_SMALL_GRID=0: small clouds take the multi-kernel grid build and grid k-NN
    bool knn_brute = true;           // GICP_KNN_BRUTE=0: clouds of <= KNN_BRUTE_MAX points take the grid k-NN
    int64_t pair_overlap_max = 1LL << 20;   // GICP_PAIR_OVERLAP_MAX=n: gicpSetPair overlaps sides of <= n points
};

// The library's only environment reads.  Called at the top of every entry point that launches, so that a switch
// changed between two calls takes effect at the next one; gicpSetPair gives both sides one snapshot.
inline Switches read_switches() {
    Switches s;
    if (const char* v = getenv("GICP_NO_SKIP")) s.no_skip = atoi(v) != 0;
    if (const char* v = getenv("GICP_TRACK_CELLS")) s.track_max_cells = atoi(v);
    if (const char* v = getenv("GICP_SHELL_SEARCH")) s.shell_search = atoi(v);
    if (const char* v = getenv("GICP_CENTRE_FIRST")) s.centre_first = atoi(v);
    if (const char* v = getenv("GICP_CORR_SPLIT")) s.corr_split = atoi(v);
    if (const char* v = getenv("GICP_ACTIVE_LIST")) s.active_list = atoi(v) != 0;
    if (const char* v = getenv("GICP_FUSED_LOOP")) s.fused_loop = atoi(v) != 0;
    if (const char* v = getenv("GICP_SMALL_GRID")) s.small_grid = atoi(v) != 0;
    if (const char* v = getenv("GICP_KNN_BRUTE")) s.knn_brute = atoi(v) != 0;
    if (const char* v = getenv("GICP_PAIR_OVERLAP_MAX")) s.pair_overlap_max = atoll(v);
    return s;
}

// The communicator of a sharded handle (gicpCommInit); `on` = false without one.
struct Ranks {
    bool on = false;
    int n = 1, rank = 0;
};

// nullptr when `off` describes n_clouds clouds the library takes (and then *max_n is the largest), else why not
inline const char* check_offsets(const int64_t* off, int n_clouds, int* max_n) {
    if (n_clouds <= 0 || n_clouds > 65535) return "n_clouds must be in [1, 65535]";
    if (off[0] != 0) return "offsets[0] must be 0";
    *max_n = 0;
    for (int i = 1; i <= n_clouds; ++i) {
        if (off[i] < off[i - 1]) return "offsets must be non-decreasing";
        if (off[i] >= (1LL << 31) - 1024) return "more than 2^31 points in one batch";
        *max_n = std::max<int>(*max_n, (int)(off[i] - off[i - 1]));
    }
    return nullptr;
}

// C = 0, C = I, estimated by K2, or the covariance of the voxel's own points (gicpSetVoxelized, voxel.cuh)
enum class CovSource { Zero, Identity, Knn, Voxel };
// knn_brute_kernel (one block per cloud, one launch); knn_general_kernel alone (one launch); knn_hist_kernel with
// the overflow hand-over to knn_general_kernel (two launches); None: a voxelized side, which has no k-NN lists
enum class KnnPath { Brute, General, HistGeneral, None };

struct SetupPlan {
    const char* error = nullptr;   // why the clouds cannot be set up; nothing below is valid then
    int n_clouds = 0, max_n = 0;
    int64_t n_total = 0;
    double knn_cell = 0, nn_cell = 0;   // cell edges of the k-NN grid and of the correspondence-search grid
    bool shared = true;                 // the k-NN grid also serves the search: one grid, no covariance re-ordering
    long long budget = 0;               // cells per cloud of either grid
    bool single_block = false;          // small_grid_kernel builds a grid in one launch, else the multi-kernel build
    int inline_n = -1;   // >= 0: one cloud of that many points, passed to small_grid_kernel; the offsets are never uploaded
    CovSource cov = CovSource::Knn;
    KnnPath knn = KnnPath::General;        // K2 of the set-up (the rank's slice when sharded)
    KnnPath knn_whole = KnnPath::General;  // K2 of gicpKnn, which always covers the whole cloud set
    int kc = 6;                            // top-k capacity of knn_brute_kernel / knn_general_kernel
    bool sharded = false;   // every rank estimates one equal slice of the covariances, then they are all-gathered
    int slice_begin = -1, slice_end = -1;   // that slice (sharding.equal_slice), -1 when not sharded
    int64_t slice_len = 0;                  // the length of every rank's slice, the last one padded
};

// The one choice of the k-NN kernel.  Latency mode (a few small clouds) runs one launch and no overflow hand-over.
inline KnnPath pick_knn(const SetupPlan& p, const Switches& sw, int k, bool f32, bool sliced) {
    const bool latency = p.max_n <= SMALL_GRID_MAX && p.n_total <= 65536 && sw.small_grid;
    if (latency && p.max_n <= KNN_BRUTE_MAX && !sliced && sw.knn_brute) return KnnPath::Brute;
    const int cap = f32 ? knn_list_cap<float>() : knn_list_cap<double>();
    return (k + 8 <= cap && !latency) ? KnnPath::HistGeneral : KnnPath::General;
}

inline SetupPlan plan_setup(const gicpParams& prm, const Switches& sw, const int64_t* off, int n_clouds, int which,
                            bool f32, const Ranks& ranks) {
    SetupPlan p;
    if ((p.error = check_offsets(off, n_clouds, &p.max_n))) return p;
    p.n_clouds = n_clouds;
    p.n_total = off[n_clouds];

    // cell edges; never smaller than (search radius)/8 so that a lane's ball spans <= 17 cells per axis.  The k-NN
    // default is the measured optimum of the cooperative fast path on the bench workload (r = 5 m -> 1.25 m cells).
    const double r = prm.max_distance_nearest_neighbors, d_max = prm.max_distance_correspondence;
    p.knn_cell = prm.knn_cell > 0 ? std::max(prm.knn_cell, r / 8.0) : 0.25 * r;
    p.nn_cell = prm.nn_cell > 0 ? std::max(prm.nn_cell, d_max / 8.0) : 0.5 * d_max;
    // one grid for both stages when the k-NN cell suits the correspondence search: not larger than twice the search's
    // own choice (d_max / 2) and not smaller than d_max / 8 (a lane's ball then spans <= 17 cells per axis).  Measured
    // on the bench workload (k-NN cell 1.25 m, search cell 1.0 m): K3a 14.97 vs 15.16 ms per 512 pairs - no loss.
    p.shared = p.knn_cell <= 2.0 * p.nn_cell && p.knn_cell >= d_max / 8.0;

    long long budget = prm.max_cells_per_cloud;
    if (budget <= 0) {
        budget = 4096;   // Morton padding can cost up to 8x the occupied box
        while (budget < 8LL * p.max_n) budget <<= 1;
        // Large batches: the tables (memset + scan + 4 B per cell) of all clouds together stay within 2^30 cells -
        // a cloud's table shrinks towards one cell per point instead of eight, and grid_meta_kernel enlarges the cell
        // edge by the few per cent that save the Morton bits.  Tables of 2^15-2^17 instead of 2^18 cells per bench
        // cloud were measured slower (the larger cells cost K2 more than K1 gains), hence the 2^30 limit.
        while (budget * n_clouds > (1LL << 30) && budget > 4096 && budget / 2 >= p.max_n) budget >>= 1;
    }
    if (budget * n_clouds > (1LL << 30)) {
        budget = (1LL << 30) / n_clouds;
        if (budget < 64) {
            p.error = "too many clouds for the cell table";
            return p;
        }
    }
    p.budget = budget;

    // small clouds (the reference's own workloads): the whole build of a cloud in one block, one launch.  One small
    // cloud takes its point count as a kernel argument, so the offsets upload and its copy-engine hop disappear.
    p.single_block = p.max_n <= SMALL_GRID_MAX && budget <= (1LL << 20) && p.n_total > 0 && sw.small_grid;
    p.inline_n = (n_clouds == 1 && p.single_block) ? (int)p.n_total : -1;

    // covariance model (ICP family): GICP estimates both sides; point-to-point uses C_src = 0, C_tgt = I;
    // point-to-plane uses C_src = 0 and the estimated target covariances
    const int model = prm.covariance_model;
    if (model == GICP_POINT_TO_POINT) p.cov = which == GICP_TARGET ? CovSource::Identity : CovSource::Zero;
    else if (model == GICP_POINT_TO_PLANE && which == GICP_SOURCE) p.cov = CovSource::Zero;
    else p.cov = CovSource::Knn;

    // sharded: every rank computes an equal slice (k-NN grid order) of BOTH clouds and the slices are all-gathered -
    // the correspondence stage walks the clouds in a different (1-NN grid) order, so every rank needs every covariance
    p.sharded = ranks.on && n_clouds == 1;
    if (p.sharded) {
        p.slice_len = (p.n_total + ranks.n - 1) / ranks.n;   // ncclAllGather needs equal-sized slices
        p.slice_begin = (int)std::min<int64_t>(p.n_total, p.slice_len * ranks.rank);
        p.slice_end = (int)std::min<int64_t>(p.n_total, p.slice_len * (ranks.rank + 1));
    }
    p.knn = pick_knn(p, sw, prm.k, f32, p.sharded);
    p.knn_whole = pick_knn(p, sw, prm.k, f32, false);
    p.kc = prm.k <= 6 ? 6 : prm.k <= 20 ? 20 : 32;
    return p;
}

// gicpSetVoxelized: a side of voxel means (`off` are the output offsets of the voxel pass) whose covariances come from
// each voxel's own points.  It needs one grid only, the one a raw side of the same points would search
// (CloudSet::nng()): the k-NN-cell grid under a shared plan, else the nn_cell grid, so K3a keeps its cell choice and a
// voxelized source keeps the grid order, and with it the accumulation order, of a raw set-up of the same array.  That
// grid sits in the k-NN grid's slot (shared = true), where gicpCovariances, gicpSourceCovariancesAt and the loop's
// centring read a side.  No K2 runs: covariance_model 1 and 2 still force C = I / C = 0 as they do for a raw side.
inline SetupPlan plan_setup_voxelized(const gicpParams& prm, const Switches& sw, const int64_t* off, int n_clouds,
                                      int which, bool f32) {
    SetupPlan p = plan_setup(prm, sw, off, n_clouds, which, f32, Ranks{});
    if (p.error) return p;
    if (!p.shared) p.knn_cell = p.nn_cell;
    p.shared = true;
    if (p.cov == CovSource::Knn) p.cov = CovSource::Voxel;
    p.knn = p.knn_whole = KnnPath::None;
    return p;
}

struct LoopPlan {
    int slice_begin = -1, slice_end = -1;   // the rank's source slice when sharded (sharding.source_slice), else -1
    int acc_ppt = 1;       // K3b points per thread
    int bpp = 1;           // K3b blocks per pair (and of the stage entry points' K3a)
    int search_ppt = 1;    // K3a points per thread in the multi-launch loop
    int search_bpp = 1;    // K3a blocks per pair in the multi-launch loop
    bool fused = false;    // register_loop_kernel runs the whole loop of every pair in one launch
    bool self_init = false;   // ... and initialises its pair itself (no start transform)
    int fused_ppt = 1;        // its points per thread
    bool presum = false;      // fold the block partials PRESUM_SPAN to 1 before K4
    int bpp2 = 1;             // rows per pair after the fold
    bool active_list = false;   // compact the still-active pairs after every iteration
    bool sharded = false;       // all-reduce between K3b and K4; blocking polls every poll_every-th iteration
    int poll_every = 1;
    bool robust = false;        // the accumulation weights the correspondences: the Robust instantiations of K3b / the fused loop
    bool adaptive = false;      // ... at a scale selected every iteration: the select (scale.cuh) runs before K3b
};

// `sliced`: the registration loop of a sharded handle covers the rank's slice; the stage entry points always cover the
// whole source, so that their outputs are complete.
inline LoopPlan plan_loop(const Switches& sw, const SetupPlan& src, bool sliced, const Ranks& ranks, bool prof_on,
                          bool has_T0, bool robust = false, bool adaptive = false) {
    LoopPlan p;
    // a robust kernel other than GICP_ROBUST_NONE: every launch of the accumulation takes its Robust instantiation (the
    // unweighted kernels are left exactly as they are); nothing else of the loop changes
    p.robust = robust;
    // an adaptive scale: the fused loop selects it inside its Robust instantiation, the multi-launch loop and the stage
    // entry points launch scale_select_kernel between K3a and K3b
    p.adaptive = robust && adaptive;
    const int np = src.n_clouds;
    p.sharded = ranks.on && np == 1;
    int span = src.max_n;
    if (sliced && p.sharded) {
        p.slice_begin = (int)(src.n_total * ranks.rank / ranks.n);
        p.slice_end = (int)(src.n_total * (ranks.rank + 1) / ranks.n);
        span = p.slice_end - p.slice_begin;
    }
    // enough blocks to fill the machine, as many points per thread as that allows.  The accumulation's software
    // pipeline has a fill bubble per thread (match index -> gathered record): longer per-thread runs amortise it when
    // the batch is large enough.  Measured per 1024 pairs of the bench workload: 16 / 32 / 64 points per thread ->
    // 9.66 / 9.16 / 9.31 ms.
    const long long total_pts = (long long)std::max(span, 1) * np;
    p.acc_ppt = std::max(1, std::min(2 * OBJ_MAX_PPT, (int)(total_pts / (148LL * 8 * OBJ_THREADS))));
    p.bpp = std::max(1, (span + OBJ_THREADS * p.acc_ppt - 1) / (OBJ_THREADS * p.acc_ppt));

    // Small pairs (every source cloud fits one block): the whole outer loop in one launch (fused.cuh).  Not with a
    // communicator (the all-reduce sits between the stages) and not while per-stage timing is on.
    p.fused = !p.sharded && !prof_on && src.max_n <= OBJ_THREADS * OBJ_MAX_PPT && sw.fused_loop;
    p.self_init = p.fused && !has_T0;
    p.fused_ppt = std::max(1, (src.max_n + OBJ_THREADS - 1) / OBJ_THREADS);

    // thousands of block partials per pair (one large pair): fold them 64 to 1 before the one-warp sum of K4
    p.presum = p.bpp > 2 * PRESUM_SPAN;
    p.bpp2 = (p.bpp + PRESUM_SPAN - 1) / PRESUM_SPAN;

    // the search runs on smaller blocks than the accumulation (its work per point is uneven: better balance and a
    // shorter tail), the accumulation keeps the longer per-thread pipeline.  The split must divide acc_ppt, so an
    // acc_ppt without a small divisor (17, 19, 23, ...) leaves the search unsplit at more than OBJ_MAX_PPT / 2 points
    // per thread.  Kept as measured: changing it changes the search's blocks.
    int split = sw.corr_split;
    while (p.acc_ppt / split > OBJ_MAX_PPT / 2) split *= 2;
    while (split > 1 && p.acc_ppt % split) --split;
    p.search_ppt = p.acc_ppt / std::max(split, 1);
    p.search_bpp = p.bpp * (p.acc_ppt / p.search_ppt);

    // Large batches: after every iteration the still-active pairs are compacted into a list (one small block), and
    // the next launches cover only as many slots of it as the latest poll counted.  Without it every launch of the
    // convergence tail starts tens of thousands of blocks that return at once (4096 pairs: 131 k blocks per search).
    p.active_list = !p.sharded && np >= 64 && sw.active_list;
    // with a communicator every rank must issue the same all-reduces: a blocking poll on a fixed schedule
    p.poll_every = p.sharded ? 2 : 1;
    return p;
}

// A set-up side as gicpSetPairList sees it: its host offsets (n_clouds + 1), or off = nullptr when it is not set up
struct SetSizes {
    const int64_t* off = nullptr;
    int n_clouds = 0;
};

struct PairPlan {
    const char* error = nullptr;   // why the list is refused; nothing below is valid then
    std::vector<int64_t> offsets;  // n_pairs + 1: pair p's rows of the pair-ordered sources and per-point outputs
    SetupPlan view;                // what plan_loop takes: n_clouds = n_pairs, max_n and n_total over the pairs' sources
};

// gicpSetPairList: pair p registers cloud src_cloud[p] of the set `source_set` names (the source set, or the target
// set itself) onto cloud tgt_cloud[p] of the target set.  The view is the source plan of the one-to-one batch whose
// p-th source is that cloud: plan_loop then makes every choice of the loop (ppt, blocks per pair, fused, active list,
// presum) exactly as for that batch.
inline PairPlan plan_pairs(int n_pairs, const int32_t* src_cloud, const int32_t* tgt_cloud, int source_set,
                           const SetSizes& source, const SetSizes& target, bool comm) {
    PairPlan p;
    if (comm) {
        p.error = "a handle with a communicator (gicpCommInit) registers one-to-one only";
        return p;
    }
    if (n_pairs < 1 || n_pairs > 65535) {
        p.error = "n_pairs must be in [1, 65535]";
        return p;
    }
    if (source_set != GICP_SOURCE && source_set != GICP_TARGET) {
        p.error = "source_set must be GICP_SOURCE 0 or GICP_TARGET 1";
        return p;
    }
    const SetSizes& from = source_set == GICP_TARGET ? target : source;
    if (!target.off || !from.off) {
        p.error = source_set == GICP_TARGET ? "set the target first" : "set source and target first";
        return p;
    }
    if (!src_cloud || !tgt_cloud) {
        p.error = "null cloud index array";
        return p;
    }
    p.offsets.assign(n_pairs + 1, 0);
    int max_n = 0;
    for (int i = 0; i < n_pairs; ++i) {
        const int s = src_cloud[i], t = tgt_cloud[i];
        if (s < 0 || s >= from.n_clouds || t < 0 || t >= target.n_clouds) {
            p.error = "a cloud index is out of range";
            return p;
        }
        const int64_t n = from.off[s + 1] - from.off[s];
        p.offsets[i + 1] = p.offsets[i] + n;
        if (p.offsets[i + 1] >= (1LL << 31) - 1024) {
            p.error = "more than 2^31 points over the pairs' sources";
            return p;
        }
        max_n = std::max<int>(max_n, (int)n);
    }
    p.view.n_clouds = n_pairs;
    p.view.max_n = max_n;
    p.view.n_total = p.offsets[n_pairs];
    return p;
}

// gicpSetPair sets the two sides up side by side while one side alone cannot fill the GPU: the single-block set-ups
// of small clouds, and up to ~1 M points per side (a 100k cloud's k-NN is one partial wave of blocks whose duration is
// its slowest chunk).  Larger sides saturate the device on their own: one after the other.
inline bool pair_overlap(const Switches& sw, const Ranks& ranks, bool prof_on, int64_t n_target, int64_t n_source) {
    return !ranks.on && !prof_on && n_target <= sw.pair_overlap_max && n_source <= sw.pair_overlap_max;
}

}  // namespace gicp
