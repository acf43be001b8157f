// libgicp_b200.so - host side of the C ABI declared in include/gicp_b200.h.
// Orchestrates the kernels K1 (grid.cuh), K2 (knn_cov.cuh), K3 (objective.cuh), K4 (solve.cuh).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>   // header-only NVTX: ranges per stage for nsys / ncu timelines

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/gicp_b200.h"
#include "grid.cuh"
#include "knn_cov.cuh"
#include "objective.cuh"
#include "raycast.cuh"
#include "solve.cuh"
#include "fused.cuh"
#include "scale.cuh"
#include "voxel.cuh"
#include "quality.cuh"
#include "pairs.cuh"
#include "plan.h"

using namespace gicp;

namespace {

thread_local std::string g_last_error;

int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return 1;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Grid {
    DevBuf meta, cell_start, spts, inv_perm, bbox, lut;
    bool built = false;
    void release() { meta.release(); cell_start.release(); spts.release(); inv_perm.release(); bbox.release(); lut.release(); }
};

struct CloudSet {
    const void* raw = nullptr;
    SetupPlan plan;           // sizes, grids and kernels of this cloud set, fixed by its set-up
    std::vector<int> off32;   // staging copy of the offsets for the asynchronous upload (must outlive the call)
    std::vector<int64_t> h_off;   // the set-up's offsets on the host (n_clouds + 1): the sizes gicpSetPairList reads
    DevBuf d_offsets;   // int32 [n_clouds+1]; not uploaded when plan.inline_n >= 0
    Grid knn;           // grid of the covariance neighbourhoods (cell ~ knn radius / 4)
    Grid nn;            // grid of the correspondence search (cell ~ d_max / 2): the target is searched in it,
                        // the source is only ORDERED by it (compact warps in K3).  Built only when the k-NN
                        // grid's cells do not suit the search (plan.shared = false)
    DevBuf cov_knn;     // covariances in knn-grid order (written by K2)
    DevBuf cov_nn;      // the same covariances in nn-grid order (read by K3); unused when shared
    bool ready = false;
    Grid& nng() { return plan.shared ? knn : nn; }
    DevBuf& covnn() { return plan.shared ? cov_knn : cov_nn; }
    void release() { d_offsets.release(); knn.release(); nn.release(); cov_knn.release(); cov_nn.release(); }
};

// gicpSetPairList: the listed pairs' sources gathered into pair order with per-pair metadata (pairs.cuh).  While `on`,
// the loop and the stage entry points run over the pairs (loop_view) instead of source cloud i against target cloud i.
struct PairList {
    bool on = false;
    SetupPlan view;            // plan_pairs: n_clouds = n_pairs, max_n and n_total over the pairs' sources
    std::vector<int> h_list;   // staging of the upload: [n_pairs][3] source cloud, target cloud, first row
    DevBuf list, src_meta, tgt_meta, tgt_bbox, spts, cov;
    void release() {
        for (DevBuf* b : {&list, &src_meta, &tgt_meta, &tgt_bbox, &spts, &cov}) b->release();
        on = false;
    }
};

// NCCL through dlopen: the engine must load without NCCL when no communicator is requested.
struct Id128 { char b[128]; };  // ncclUniqueId is 128 opaque bytes, passed by value
typedef int (*nccl_init_fn)(void**, int, Id128, int);
struct Nccl {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    nccl_init_fn CommInitRank = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
Nccl g_nccl;

int load_nccl() {
    if (g_nccl.lib) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) return fail("cannot dlopen libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(void*))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (nccl_init_fn)dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.AllGather || !g_nccl.CommDestroy)
        return fail("libnccl is missing a required symbol");
    return 0;
}
constexpr int NCCL_FLOAT64 = 8, NCCL_SUM = 0, NCCL_INT8 = 0;

}  // namespace

// scratch of one set-up (grid build + k-NN) in flight: sort keys / values, CUB storage, bounding-box partials, the
// k-NN overflow hand-over list
struct SetupScratch {
    DevBuf keys, keys_alt, vals, vals_alt, cub_tmp, bbox_part, ovf_count, ovf_list;
    void release() {
        for (DevBuf* b : {&keys, &keys_alt, &vals, &vals_alt, &cub_tmp, &bbox_part, &ovf_count, &ovf_list}) b->release();
    }
};

// scratch of gicpVoxelDownsample: its own, so a downsample between gicpSetPair and gicpRegister leaves both sides alone
struct VoxelScratch {
    DevBuf offsets, part, vb, keys, keys_alt, vals, vals_alt, rid, orow, out_off, big, cub_tmp;
    DevBuf cov;                 // gicpSetVoxelized: each output row's covariance, in output-row order
    double* h_vb = nullptr;     // pinned: per-cloud voxel bounds
    int* h_out_off = nullptr;   // pinned: output offsets
    int h_cap = 0;              // clouds the pinned buffers hold
    std::vector<int> off32;
    void release() {
        for (DevBuf* b : {&offsets, &part, &vb, &keys, &keys_alt, &vals, &vals_alt, &rid, &orow, &out_off, &big, &cub_tmp, &cov})
            b->release();
        if (h_vb) cudaFreeHost(h_vb);
        if (h_out_off) cudaFreeHost(h_out_off);
        h_vb = nullptr;
        h_out_off = nullptr;
        h_cap = 0;
    }
};

struct gicpContext {
    int device = 0, dim = 2, storage = GICP_STORAGE_F64;
    gicpParams prm;
    int robust_kind = GICP_ROBUST_NONE;   // gicpSetRobustKernel
    double robust_scale = 0.0;
    bool robust_adaptive = false;         // gicpSetRobustKernelAdaptive: c = max(robust_min_scale, robust_kappa * median)
    double robust_kappa = 0.0, robust_min_scale = 0.0;
    CloudSet src, tgt;
    PairList pairs;   // gicpSetPairList; discarded whenever a side or the parameters change
    // [0]: every call on the caller's stream; [1]: the source side of gicpSetPair while it runs on the internal stream
    SetupScratch scr[2];
    VoxelScratch vox;
    DevBuf state, partial, partial2, red, T_dev, n_active, prev_match, slack, active_list;
    DevBuf sel_keys, sel_hist, sel_arrived, sel_state, pair_scale;   // the adaptive scale's select (scale.cuh)
    DevBuf eval_idx, eval_dist;   // gicpEvaluate: the correspondences at the evaluated transforms (input order)
    static constexpr int NPOLL = 8;
    int* h_poll = nullptr;  // pinned [NPOLL]: progress polls in flight
    cudaEvent_t poll_ev[NPOLL] = {};
    cudaStream_t last_stream = nullptr;   // stream of the last gicpSet*/gicpRegister call (gicpPromoteTargetToSource has none)
    int64_t launches = 0;
    // per-stage CUDA-event timing (off by default): stage ids in include/gicp_b200.h
    bool prof_on = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct ProfRec { int stage; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_recs;
    cudaEvent_t prof_event() {
        if (ev_used == ev_pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev_pool.push_back(e);
        }
        return ev_pool[ev_used++];
    }
    // sharded-source mode
    void* comm = nullptr;
    int n_ranks = 1, rank = 0;
    // gicpSetPair: the source side of a small pair is set up on this stream while the target side runs on the caller's
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

namespace {

int ns_of(int dim) { return dim * (dim + 1) / 2; }

const char* const kStageNames[GICP_N_STAGES_ALL] = {"gicp:grid_build", "gicp:knn_cov", "gicp:correspond",
                                                     "gicp:accumulate", "gicp:solve", "gicp:scale_select"};

struct ProfScope {
    gicpContext* h;
    cudaStream_t st;
    cudaEvent_t b = nullptr;
    ProfScope(gicpContext* h_, int stage, cudaStream_t st_) : h(h_), st(st_) {
        nvtxRangePushA(kStageNames[stage]);   // a no-op unless a profiler is attached
        if (!h->prof_on) return;
        cudaEvent_t a = h->prof_event();
        b = h->prof_event();
        cudaEventRecord(a, st);
        h->prof_recs.push_back({stage, a, b});
    }
    ~ProfScope() {
        if (b) cudaEventRecord(b, st);
        nvtxRangePop();
    }
};

template <int D, typename Real>
int build_grid(gicpContext* h, CloudSet& cs, Grid& g, double h_target, cudaStream_t st, SetupScratch& sc) {
    const SetupPlan& p = cs.plan;
    const int nc = p.n_clouds;
    const int64_t n = p.n_total;
    const long long budget = p.budget;
    const long long total_cells = budget * nc;
    const int chunks = std::max(1, (p.max_n + BBOX_THREADS * BBOX_ITEMS - 1) / (BBOX_THREADS * BBOX_ITEMS));
    CU(sc.bbox_part.ensure((size_t)nc * chunks * 6 * sizeof(double)));
    CU(g.meta.ensure((size_t)nc * sizeof(CloudMeta)));
    CU(g.bbox.ensure((size_t)nc * 6 * sizeof(double)));
    CU(g.cell_start.ensure((size_t)(total_cells + 1) * sizeof(int)));
    CU(g.spts.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(PRec<Real>)));
    CU(g.inv_perm.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(int)));
    CU(sc.keys.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.keys_alt.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.vals.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.vals_alt.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    const Real* pts = static_cast<const Real*>(cs.raw);
    const int* offs = cs.d_offsets.as<int>();
    ProfScope prof(h, GICP_STAGE_GRID, st);

    if (p.single_block) {   // the whole build of a cloud in one block, one launch
        CU(g.lut.ensure((size_t)nc * 3 * GICP_LUT_N * sizeof(int)));
        small_grid_kernel<D, Real><<<nc, SMALL_GRID_THREADS, 0, st>>>(pts, offs, h_target, budget, g.meta.as<CloudMeta>(),
                                                                      g.bbox.as<double>(), g.lut.as<int>(),
                                                                      g.cell_start.as<int>(), g.spts.as<PRec<Real>>(),
                                                                      g.inv_perm.as<int>(), 1, p.inline_n);
        h->launches += 1;
        CU(cudaGetLastError());
        g.built = true;
        return 0;
    }

    bbox_partial_kernel<D, Real><<<dim3(chunks, nc), BBOX_THREADS, 0, st>>>(pts, offs, sc.bbox_part.as<double>(), chunks);
    grid_meta_kernel<D><<<(nc + 3) / 4, 128, 0, st>>>(sc.bbox_part.as<double>(), chunks, offs, nc, h_target, budget,
                                                          g.meta.as<CloudMeta>(), g.bbox.as<double>());
    CU(g.lut.ensure((size_t)nc * 3 * GICP_LUT_N * sizeof(int)));
    morton_lut_kernel<<<dim3(3 * GICP_LUT_N / 256, nc), 256, 0, st>>>(g.meta.as<CloudMeta>(), g.lut.as<int>());
    // the cell histogram is built in the table itself and scanned in place (no second 4-byte-per-cell buffer)
    CU(cudaMemsetAsync(g.cell_start.p, 0, (size_t)(total_cells + 1) * sizeof(int), st));
    h->launches += 3;
    if (n > 0) {
        const int bx = (p.max_n + 255) / 256;
        cell_key_kernel<D, Real><<<dim3(bx, nc), 256, 0, st>>>(pts, g.meta.as<CloudMeta>(), sc.keys.as<unsigned>(),
                                                               sc.vals.as<int>(), g.cell_start.as<int>());
        h->launches += 1;
    }
    {   // cell_start = exclusive scan of the histogram
        size_t tmp = 0;
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, g.cell_start.as<int>(), g.cell_start.as<int>(),
                                         (int)(total_cells + 1), st));
        CU(sc.cub_tmp.ensure(tmp));
        CU(cub::DeviceScan::ExclusiveSum(sc.cub_tmp.p, tmp, g.cell_start.as<int>(), g.cell_start.as<int>(),
                                         (int)(total_cells + 1), st));
        h->launches += 2;
    }
    if (n > 0) {
        int bits = 1;
        while ((1LL << bits) < total_cells) ++bits;
        cub::DoubleBuffer<unsigned> dk(sc.keys.as<unsigned>(), sc.keys_alt.as<unsigned>());
        cub::DoubleBuffer<int> dv(sc.vals.as<int>(), sc.vals_alt.as<int>());
        size_t tmp = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (int)n, 0, bits, st));
        CU(sc.cub_tmp.ensure(tmp));
        CU(cub::DeviceRadixSort::SortPairs(sc.cub_tmp.p, tmp, dk, dv, (int)n, 0, bits, st));
        h->launches += (bits + 7) / 8 + 2;
        const int bx = (p.max_n + 255) / 256;
        gather_sorted_kernel<D, Real><<<dim3(bx, nc), 256, 0, st>>>(pts, g.meta.as<CloudMeta>(), dv.Current(),
                                                                    g.spts.as<PRec<Real>>(), g.inv_perm.as<int>());
        h->launches += 1;
    }
    CU(cudaGetLastError());
    g.built = true;
    return 0;
}

template <int D, typename Real>
__global__ void regather_cov_kernel(const CloudMeta* __restrict__ meta, const PRec<Real>* __restrict__ spts_dst,
                                    const int* __restrict__ inv_perm_src, const Real* __restrict__ cov_src,
                                    Real* __restrict__ cov_dst) {
    constexpr int NS = Dim<D>::NS;
    const CloudMeta m = meta[blockIdx.y];
    const int s = m.pt_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m.pt_end) return;
    const int g = m.pt_begin + (int)spts_dst[s].idx;
    const int ss = inv_perm_src[g];
#pragma unroll
    for (int i = 0; i < NS; ++i) cov_dst[(size_t)s * NS + i] = cov_src[(size_t)ss * NS + i];
}

// ICP variants: a side whose covariance is a constant multiple of the identity (0 or 1) skips K2
template <int D, typename Real>
__global__ void fill_cov_kernel(Real* __restrict__ cov, size_t n, Real diag) {
    constexpr int NS = Dim<D>::NS;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int a = 0, k = 0; a < D; ++a)
        for (int b = a; b < D; ++b, ++k) cov[i * NS + k] = (a == b) ? diag : Real(0);
}

template <int D, typename Real>
__global__ void export_cov_kernel(const CloudMeta* __restrict__ meta, const PRec<Real>* __restrict__ spts,
                                  const Real* __restrict__ cov_sorted, double* __restrict__ out) {
    constexpr int NS = Dim<D>::NS;
    const CloudMeta m = meta[blockIdx.y];
    const int s = m.pt_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m.pt_end) return;
    const size_t g = (size_t)m.pt_begin + (size_t)spts[s].idx;
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) out[g * D * D + i * D + j] = (double)cov_sorted[(size_t)s * NS + symidx(D, i, j)];
}

// out[t][g] = R_t C[g] R_t^T in input order (gicp.py:120-121)
template <int D, typename Real>
__global__ void rotated_cov_kernel(const CloudMeta* __restrict__ meta, const PRec<Real>* __restrict__ spts,
                                   const Real* __restrict__ cov_sorted, const double* __restrict__ T, int n_clouds,
                                   size_t n_total, double* __restrict__ out) {
    constexpr int NS = Dim<D>::NS;
    const CloudMeta m = meta[blockIdx.y];
    const int s = m.pt_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m.pt_end) return;
    const int t = blockIdx.z;
    const double* Tm = T + ((size_t)t * n_clouds + blockIdx.y) * (D + 1) * (D + 1);
    double C[D][D], A[D][D];
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) C[i][j] = (double)cov_sorted[(size_t)s * NS + symidx(D, i, j)];
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            double v = 0.0;
            for (int k = 0; k < D; ++k) v += Tm[i * (D + 1) + k] * C[k][j];
            A[i][j] = v;
        }
    const size_t g = (size_t)m.pt_begin + (size_t)spts[s].idx;
    double* o = out + ((size_t)t * n_total + g) * D * D;
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            double v = 0.0;
            for (int k = 0; k < D; ++k) v += A[i][k] * Tm[j * (D + 1) + k];
            o[i * D + j] = v;
        }
}

// K2 along `path` (pick_knn), over the slice [slice_b, slice_e) of a single cloud or, with slice_b < 0, every cloud
template <int D, typename Real>
int launch_knn(gicpContext* h, CloudSet& cs, KnnPath path, int* d_idx, double* d_dist, cudaStream_t st, int slice_b,
               int slice_e, SetupScratch& sc) {
    const SetupPlan& p = cs.plan;
    KnnArgs<Real> a;
    a.meta = cs.knn.meta.as<CloudMeta>();
    a.cell_start = cs.knn.cell_start.as<int>();
    a.lut = cs.knn.lut.as<int>();
    a.spts = cs.knn.spts.as<PRec<Real>>();
    a.raw = static_cast<const Real*>(cs.raw);
    a.cov_sorted = cs.cov_knn.as<Real>();
    a.knn_idx = d_idx;
    a.knn_dist = d_dist;
    a.k = h->prm.k;
    a.radius = h->prm.max_distance_nearest_neighbors;
    a.lam_t = h->prm.lambda_tangent;
    a.lam_n = h->prm.lambda_normal;
    a.slice_begin = slice_b;
    a.slice_end = slice_e;
    if (p.n_total == 0) return 0;
    const int span = (slice_b >= 0) ? (slice_e - slice_b) : p.max_n;
    if (span <= 0) return 0;
    const int bx = (span + KNN_THREADS - 1) / KNN_THREADS;
    dim3 grid(bx, p.n_clouds);
    // fast path's overflow hand-over: worst case every warp
    const long long n_chunks = (long long)bx * KNN_WARPS * p.n_clouds;
    CU(sc.ovf_count.ensure(sizeof(int)));
    CU(sc.ovf_list.ensure((size_t)n_chunks * sizeof(int2)));
    a.overflow_count = sc.ovf_count.as<int>();
    a.overflow_list = sc.ovf_list.as<int2>();
    a.overflow_cap = (int)std::min<long long>(n_chunks, INT_MAX);
    const size_t smem_g = 128 + (size_t)KNN_WARPS * KNN_WARP_SMEM;
    const size_t smem_h = 128 + (size_t)KNN_WARPS * KNN_HIST_WARP_SMEM;
    ProfScope prof(h, GICP_STAGE_KNN_COV, st);
#define KNN_LAUNCH(KC, GRID, FROM_LIST)                                                                      \
    do {                                                                                                     \
        CU(cudaFuncSetAttribute(knn_general_kernel<D, Real, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                (int)smem_g));                                                               \
        knn_general_kernel<D, Real, KC><<<GRID, KNN_THREADS, smem_g, st>>>(a, FROM_LIST);                    \
    } while (0)
    if (path == KnnPath::Brute) {
        // tiny clouds: brute force from shared memory, one block per cloud, one launch
        const size_t smem_b = (size_t)p.max_n * sizeof(PRec<Real>);
        if (p.kc == 6) knn_brute_kernel<D, Real, 6><<<p.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        else if (p.kc == 20) knn_brute_kernel<D, Real, 20><<<p.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        else knn_brute_kernel<D, Real, 32><<<p.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        h->launches += 1;
    } else if (path == KnnPath::HistGeneral) {
        CU(cudaMemsetAsync(sc.ovf_count.p, 0, sizeof(int), st));
        CU(cudaFuncSetAttribute(knn_hist_kernel<D, Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
        CU(cudaFuncSetAttribute(knn_hist_kernel<D, Real>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        knn_hist_kernel<D, Real><<<grid, KNN_THREADS, smem_h, st>>>(a);
        const dim3 lgrid(296, 1);
        if (p.kc == 6) KNN_LAUNCH(6, lgrid, 1);
        else if (p.kc == 20) KNN_LAUNCH(20, lgrid, 1);
        else KNN_LAUNCH(32, lgrid, 1);
        h->launches += 2;
    } else {
        if (p.kc == 6) KNN_LAUNCH(6, grid, 0);
        else if (p.kc == 20) KNN_LAUNCH(20, grid, 0);
        else KNN_LAUNCH(32, grid, 0);
        h->launches += 1;
    }
#undef KNN_LAUNCH
    CU(cudaGetLastError());
    return 0;
}

// the side's offsets to the device, unless its plan passes a single cloud's size as a kernel argument
int upload_offsets(CloudSet& cs, const int64_t* h_offsets, cudaStream_t st) {
    const int n_clouds = cs.plan.n_clouds;
    CU(cs.d_offsets.ensure((size_t)(n_clouds + 1) * sizeof(int)));
    cs.h_off.assign(h_offsets, h_offsets + n_clouds + 1);
    // no stream synchronisation here: a copy from pageable memory is staged by the driver before the call returns,
    // and the staging vector lives in the handle
    if (cs.plan.inline_n < 0) {
        cs.off32.assign(h_offsets, h_offsets + n_clouds + 1);
        CU(cudaMemcpyAsync(cs.d_offsets.p, cs.off32.data(), cs.off32.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    }
    return 0;
}

template <int D, typename Real>
int set_cloud(gicpContext* h, const Switches& sw, int which, const void* d_points, const int64_t* h_offsets,
              int n_clouds, cudaStream_t st, int scratch_slot) {
    SetupScratch& sc = h->scr[scratch_slot];
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    cs.ready = false;
    h->pairs.on = false;
    h->last_stream = st;
    cs.plan = plan_setup(h->prm, sw, h_offsets, n_clouds, which, std::is_same<Real, float>::value,
                         Ranks{h->comm != nullptr, h->n_ranks, h->rank});
    const SetupPlan& p = cs.plan;
    if (p.error) return fail("%s (%d clouds)", p.error, n_clouds);
    if (p.n_total > 0 && !d_points) return fail("null point array");
    cs.raw = d_points;
    if (upload_offsets(cs, h_offsets, st)) return 1;

    if (build_grid<D, Real>(h, cs, cs.knn, p.knn_cell, st, sc)) return 1;
    const size_t n_cov = (size_t)std::max<int64_t>(p.sharded ? p.slice_len * h->n_ranks : p.n_total, 1);
    CU(cs.cov_knn.ensure(n_cov * ns_of(D) * sizeof(Real)));
    if (p.cov != CovSource::Knn) {
        const size_t n = (size_t)std::max<int64_t>(p.n_total, 1);
        const Real diag = p.cov == CovSource::Identity ? Real(1) : Real(0);
        fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_knn.as<Real>(), n, diag);
        h->launches += 1;
    } else {
        if (launch_knn<D, Real>(h, cs, p.knn, nullptr, nullptr, st, p.slice_begin, p.slice_end, sc)) return 1;
        if (p.sharded) {
            const size_t bytes = (size_t)p.slice_len * ns_of(D) * sizeof(Real);
            char* basep = cs.cov_knn.as<char>();
            int rc = g_nccl.AllGather(basep + bytes * h->rank, basep, bytes, NCCL_INT8, h->comm, st);
            if (rc) return fail("ncclAllGather failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
        }
    }
    if (!p.shared) {   // second ordering for the correspondence stage + the covariances carried over to it
        if (build_grid<D, Real>(h, cs, cs.nn, p.nn_cell, st, sc)) return 1;
        CU(cs.cov_nn.ensure((size_t)std::max<int64_t>(p.n_total, 1) * ns_of(D) * sizeof(Real)));
        if (p.n_total > 0) {
            const int bx = (p.max_n + 255) / 256;
            regather_cov_kernel<D, Real><<<dim3(bx, n_clouds), 256, 0, st>>>(
                cs.nn.meta.as<CloudMeta>(), cs.nn.spts.as<PRec<Real>>(), cs.knn.inv_perm.as<int>(), cs.cov_knn.as<Real>(),
                cs.cov_nn.as<Real>());
            h->launches += 1;
        }
    }
    CU(cudaGetLastError());
    cs.ready = true;
    return 0;
}

// gicpPromoteTargetToSource with an ICP-family model: the promoted side keeps its grids, but its covariances
// were the TARGET's (I for point-to-point, the estimated ones for point-to-plane); a source has C = 0 in both.
template <int D, typename Real>
int zero_source_cov(gicpContext* h, cudaStream_t st) {
    CloudSet& cs = h->src;
    const size_t n = (size_t)std::max<int64_t>(cs.plan.n_total, 1);
    fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_knn.as<Real>(), n, Real(0));
    if (!cs.plan.shared) fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_nn.as<Real>(), n, Real(0));
    h->launches += cs.plan.shared ? 1 : 2;
    CU(cudaGetLastError());
    return 0;
}

// What the loop and the pair-indexed entry points run over: source cloud i against target cloud i, or the pair list.
// `plan` sizes the loop (n_clouds = pairs, max_n and n_total of the sources), `tgt_bbox` holds every pair's target box
// (the centring point and the fused loop's self-initialisation).
struct LoopView {
    const SetupPlan& plan;
    const double* tgt_bbox;
    bool ready;   // something to register: both sides set up, or a pair list (which needs no source set)
};
LoopView loop_view(gicpContext* h) {
    if (h->pairs.on) return LoopView{h->pairs.view, h->pairs.tgt_bbox.as<double>(), true};
    return LoopView{h->src.plan, h->tgt.knn.bbox.as<double>(), h->src.ready && h->tgt.ready};
}

template <int D, typename Real>
int objective_args(gicpContext* h, const Switches& sw, bool sliced, bool has_T0, ObjArgs<Real>& a, LoopPlan& lp) {
    CloudSet &S = h->src, &T = h->tgt;
    const PairList& pl = h->pairs;
    const LoopView lv = loop_view(h);
    if (!lv.ready) return fail("set source and target first");
    const int np = lv.plan.n_clouds;
    if (!pl.on && np != T.plan.n_clouds) return fail("source has %d clouds, target %d", np, T.plan.n_clouds);
    lp = plan_loop(sw, lv.plan, sliced, Ranks{h->comm != nullptr, h->n_ranks, h->rank}, h->prof_on, has_T0,
                   h->robust_kind != GICP_ROBUST_NONE, h->robust_adaptive);
    a.src_meta = pl.on ? pl.src_meta.as<CloudMeta>() : S.nng().meta.as<CloudMeta>();
    a.src_spts = pl.on ? pl.spts.as<PRec<Real>>() : S.nng().spts.as<PRec<Real>>();
    a.src_cov = pl.on ? pl.cov.as<Real>() : S.covnn().as<Real>();
    a.tgt_meta = pl.on ? pl.tgt_meta.as<CloudMeta>() : T.nng().meta.as<CloudMeta>();
    a.tgt_cell_start = T.nng().cell_start.as<int>();
    a.tgt_lut = T.nng().lut.as<int>();
    a.tgt_spts = T.nng().spts.as<PRec<Real>>();
    a.tgt_cov = T.covnn().as<Real>();
    a.tgt_inv_perm = T.nng().inv_perm.as<int>();
    a.match = nullptr;
    a.use_prev = 0;
    CU(h->state.ensure((size_t)np * sizeof(PairState)));
    a.state = h->state.as<PairState>();
    a.T_override = nullptr;
    a.d_max = h->prm.max_distance_correspondence;
    a.out_idx = nullptr;
    a.out_dist = nullptr;
    a.out_W = nullptr;
    a.slice_begin = lp.slice_begin;
    a.slice_end = lp.slice_end;
    a.ignore_status = 0;
    a.track_max_cells = sw.track_max_cells;
    a.centre_first = sw.centre_first;
    a.shell_search = sw.shell_search;
    a.active_list = nullptr;
    a.n_list = nullptr;
    a.robust_kind = h->robust_kind;
    a.robust_scale = h->robust_scale;
    a.pair_scale = nullptr;
    a.scale_kappa = h->robust_kappa;
    a.scale_min = h->robust_min_scale;
    a.ppt = lp.acc_ppt;
    a.blocks_per_pair = lp.bpp;
    CU(h->partial.ensure((size_t)np * lp.bpp * Dim<D>::NRED * sizeof(double)));
    CU(h->red.ensure((size_t)np * Dim<D>::NRED * sizeof(double)));
    a.partial = h->partial.as<double>();
    CU(h->prev_match.ensure((size_t)std::max<int64_t>(lv.plan.n_total, 1) * sizeof(int)));
    a.match = h->prev_match.as<int>();
    CU(h->slack.ensure((size_t)std::max<int64_t>(lv.plan.n_total, 1) * sizeof(float)));
    a.slack = nullptr;
    return 0;
}

// the host transforms to T_dev, complete before the call returns (the caller's buffer may go away)
int upload_T(gicpContext* h, const double* h_T, size_t bytes, cudaStream_t st) {
    CU(h->T_dev.ensure(bytes));
    CU(cudaMemcpyAsync(h->T_dev.p, h_T, bytes, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

template <int D, typename Real>
int ensure_state(gicpContext* h, const double* h_T0, double* d_T, double* d_T_hist, int* d_n_outer,
                 int* d_converged, cudaStream_t st) {
    const LoopView lv = loop_view(h);
    const int np = lv.plan.n_clouds;
    CU(h->state.ensure((size_t)np * sizeof(PairState)));
    CU(h->n_active.ensure(sizeof(int)));
    const double* d_T0 = nullptr;
    if (h_T0) {
        if (upload_T(h, h_T0, (size_t)np * (D + 1) * (D + 1) * sizeof(double), st)) return 1;
        d_T0 = h->T_dev.as<double>();
    }
    init_state_kernel<D><<<(np + 127) / 128, 128, 0, st>>>(h->state.as<PairState>(), d_T0, lv.tgt_bbox, np,
                                                           d_T, d_T_hist, h->prm.max_iterations, d_n_outer, d_converged,
                                                           h->n_active.as<int>());
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

// the multi-launch select's scratch: the histograms and arrival counters start at zero (the last block of every pair
// leaves them so); a.pair_scale is where the accumulation reads the scale
template <int D, typename Real>
int prepare_select(gicpContext* h, ObjArgs<Real>& a, ScaleArgs& sc, cudaStream_t st) {
    const SetupPlan& sp = loop_view(h).plan;
    const int np = sp.n_clouds;
    CU(h->sel_keys.ensure((size_t)std::max<int64_t>(sp.n_total, 1) * sizeof(unsigned long long)));
    CU(h->sel_hist.ensure((size_t)np * SEL_BINS * sizeof(unsigned)));
    CU(h->sel_arrived.ensure((size_t)np * sizeof(unsigned)));
    CU(h->sel_state.ensure((size_t)np * sizeof(SelState)));
    CU(h->pair_scale.ensure((size_t)np * sizeof(double)));
    CU(cudaMemsetAsync(h->sel_hist.p, 0, (size_t)np * SEL_BINS * sizeof(unsigned), st));
    CU(cudaMemsetAsync(h->sel_arrived.p, 0, (size_t)np * sizeof(unsigned), st));
    sc.keys = h->sel_keys.as<unsigned long long>();
    sc.hist = h->sel_hist.as<unsigned>();
    sc.arrived = h->sel_arrived.as<unsigned>();
    sc.sel = h->sel_state.as<SelState>();
    sc.scale = h->pair_scale.as<double>();
    a.pair_scale = sc.scale;
    return 0;
}

// every pair's scale at its current matches: SEL_PASSES launches over the accumulation's blocks (a.ppt, bpp x gy)
template <int D, typename Real>
int launch_select(gicpContext* h, const ObjArgs<Real>& a, const ScaleArgs& sc, int bpp, int gy, cudaStream_t st) {
    for (int pass = 0; pass < SEL_PASSES; ++pass)
        scale_select_kernel<D, Real><<<dim3(bpp, gy), OBJ_THREADS, 0, st>>>(a, sc, pass);
    h->launches += SEL_PASSES;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_register(gicpContext* h, const Switches& sw, const double* h_T0, double* d_T, int* d_n_outer, int* d_converged,
                double* d_loss_hist, double* d_T_hist, int* d_inliers, cudaStream_t st) {
    ObjArgs<Real> oa;
    LoopPlan lp;
    if (objective_args<D, Real>(h, sw, true, h_T0 != nullptr, oa, lp)) return 1;
    if (lp.adaptive && lp.sharded)
        return fail("an adaptive robust scale needs every source point on one rank: sharded-source registration "
                    "(gicpCommInit) takes a fixed scale (gicpSetRobustKernel) or none");
    const LoopView lv = loop_view(h);
    const int np = lv.plan.n_clouds;
    const int bpp = lp.bpp;
    h->last_stream = st;
    if (lp.self_init) {
        CU(h->state.ensure((size_t)np * sizeof(PairState)));
    } else {
        if (ensure_state<D, Real>(h, h_T0, d_T, d_T_hist, d_n_outer, d_converged, st)) return 1;
        // last iteration's match per source point (bounds the next search); -1 = none yet
        CU(cudaMemsetAsync(h->prev_match.p, 0xFF, (size_t)std::max<int64_t>(lv.plan.n_total, 1) * sizeof(int), st));
        CU(cudaMemsetAsync(h->slack.p, 0, (size_t)std::max<int64_t>(lv.plan.n_total, 1) * sizeof(float), st));
    }
    oa.use_prev = 1;
    oa.slack = sw.no_skip ? nullptr : h->slack.as<float>();
    SolveArgs sa;
    sa.partial = h->partial.as<double>();
    sa.blocks_per_pair = bpp;
    sa.n_pairs = np;
    sa.sum_out = nullptr;
    sa.state = h->state.as<PairState>();
    sa.max_iterations = h->prm.max_iterations;
    sa.inner_max_iterations = h->prm.inner_max_iterations;
    sa.tolerance = h->prm.tolerance;
    sa.d_T = d_T;
    sa.d_n_outer = d_n_outer;
    sa.d_converged = d_converged;
    sa.d_loss_hist = d_loss_hist;
    sa.d_T_hist = d_T_hist;
    sa.d_inliers = d_inliers;
    sa.n_active = h->n_active.as<int>();
    sa.active_list = nullptr;
    sa.n_list = nullptr;
    if (lp.fused) {
        oa.ppt = lp.fused_ppt;
        oa.blocks_per_pair = 1;
        sa.blocks_per_pair = 1;
        sa.n_active = nullptr;   // nobody polls
        // with an adaptive scale the select's keys (8 B per source point) follow the search's shared memory
        const size_t smem = obj_smem(oa.ppt) + (lp.adaptive ? (size_t)OBJ_THREADS * oa.ppt * sizeof(unsigned long long) : 0);
        auto loop_kernel = lp.adaptive ? register_loop_kernel<D, Real, true, true>
                           : lp.robust ? register_loop_kernel<D, Real, true> : register_loop_kernel<D, Real, false>;
        CU(cudaFuncSetAttribute(loop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ProfScope prof(h, GICP_STAGE_CORRESPOND, st);
        loop_kernel<<<np, OBJ_THREADS, smem, st>>>(oa, sa, lp.self_init ? lv.tgt_bbox : nullptr);
        h->launches += 1;
        CU(cudaGetLastError());
        return 0;
    }
    const int bpp2 = lp.bpp2;
    if (lp.presum) {
        CU(h->partial2.ensure((size_t)np * bpp2 * Dim<D>::NRED * sizeof(double)));
        sa.partial = h->partial2.as<double>();
        sa.blocks_per_pair = bpp2;
    }
    ScaleArgs sc{};
    if (lp.adaptive && prepare_select<D, Real>(h, oa, sc, st)) return 1;
    ObjArgs<Real> oc = oa;
    oc.ppt = lp.search_ppt;
    auto acc_kernel = lp.robust ? accumulate_kernel<D, Real, true> : accumulate_kernel<D, Real, false>;
    const int sgrid = (np + SOLVE_WARPS - 1) / SOLVE_WARPS;
    const bool sharded = lp.sharded;
    // Progress polls (4 bytes each, the only host<->device traffic inside the loop).  A single-process registration
    // does not wait for them: the count of still-active pairs is copied to pinned memory after every iteration and
    // looked at (cudaEventQuery) before later iterations are launched, so the host runs a few iterations ahead and the
    // GPU never idles on a round trip; an iteration launched after everything converged is a no-op (every block
    // returns on the pair's status).  With a communicator every rank must issue the same all-reduces, so the sharded
    // mode keeps a blocking poll on a fixed schedule (all ranks see the same count: they solve bit-identical forms).
    constexpr int LOOK = 3;
    int issued = 0, checked = 0;
    // with the active-pair list the launches cover `known_active` slots of it: the latest polled count, an upper
    // bound of the list's length since the count only falls
    const bool use_list = lp.active_list;
    int known_active = np;
    if (use_list) {
        CU(h->active_list.ensure((size_t)(np + 1) * sizeof(int)));
        int* lst = h->active_list.as<int>();
        compact_active_kernel<<<1, COMPACT_THREADS, 0, st>>>(h->state.as<PairState>(), np, lst + 1, lst);
        h->launches += 1;
        oa.active_list = oc.active_list = sa.active_list = lst + 1;
        oa.n_list = oc.n_list = sa.n_list = lst;
    }
    for (int it = 0; it < h->prm.max_iterations; ++it) {
        bool done = false;
        while (checked < issued && !done) {
            const int slot = checked % gicpContext::NPOLL;
            cudaError_t q = (sharded || issued - checked > LOOK) ? cudaEventSynchronize(h->poll_ev[slot])
                                                                 : cudaEventQuery(h->poll_ev[slot]);
            if (q == cudaErrorNotReady) { cudaGetLastError(); break; }
            CU(q);
            done = h->h_poll[slot] <= 0;
            known_active = std::min(known_active, std::max(h->h_poll[slot], 1));
            ++checked;
        }
        if (done) break;
        const int gy = use_list ? known_active : np;
        {
            ProfScope prof(h, GICP_STAGE_CORRESPOND, st);
            correspond_kernel<D, Real><<<dim3(lp.search_bpp, gy), OBJ_THREADS, obj_smem(oc.ppt), st>>>(oc);
        }
        if (lp.adaptive) {
            ProfScope prof(h, GICP_STAGE_SCALE_SELECT, st);
            if (launch_select<D, Real>(h, oa, sc, bpp, gy, st)) return 1;
        }
        {
            ProfScope prof(h, GICP_STAGE_ACCUMULATE, st);
            acc_kernel<<<dim3(bpp, gy), OBJ_THREADS, 0, st>>>(oa);
        }
        {
            ProfScope prof(h, GICP_STAGE_SOLVE, st);
            if (lp.presum) {
                presum_kernel<D><<<dim3(bpp2, np), Dim<D>::NRED, 0, st>>>(h->partial.as<double>(), bpp, h->partial2.as<double>(),
                                                                        bpp2, h->state.as<PairState>());
                h->launches += 1;
            }
            if (sharded) {
                SolveArgs s1 = sa;
                s1.sum_out = h->red.as<double>();
                solve_kernel<D><<<sgrid, SOLVE_WARPS * 32, 0, st>>>(s1);
                int rc = g_nccl.AllReduce(h->red.p, h->red.p, (size_t)Dim<D>::NRED, NCCL_FLOAT64, NCCL_SUM, h->comm, st);
                if (rc) return fail("ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
                SolveArgs s2 = sa;
                s2.partial = h->red.as<double>();
                s2.blocks_per_pair = 1;
                solve_kernel<D><<<sgrid, SOLVE_WARPS * 32, 0, st>>>(s2);
                h->launches += 4;
            } else {
                solve_kernel<D><<<use_list ? (gy + SOLVE_WARPS - 1) / SOLVE_WARPS : sgrid, SOLVE_WARPS * 32, 0, st>>>(sa);
                h->launches += 3;
                if (use_list) {
                    int* lst = h->active_list.as<int>();
                    compact_active_kernel<<<1, COMPACT_THREADS, 0, st>>>(h->state.as<PairState>(), np, lst + 1, lst);
                    h->launches += 1;
                }
            }
        }
        if ((it + 1) % lp.poll_every == 0) {
            const int slot = issued % gicpContext::NPOLL;
            CU(cudaMemcpyAsync(h->h_poll + slot, h->n_active.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(h->poll_ev[slot], st));
            ++issued;
        }
    }
    CU(cudaGetLastError());
    return 0;
}

// One stage pass at the DEVICE transforms d_T, enqueued on `st` without a synchronisation: the correspondences
// (d_idx / d_dist in input order), with an adaptive scale every pair's scale (sc.scale), the weight matrices d_W and,
// with `fold`, every pair's reduced form (+mu) in h->red.  `oa` / `lp` come from objective_args.
template <int D, typename Real>
int stage_pass(gicpContext* h, ObjArgs<Real>& oa, const LoopPlan& lp, const double* d_T, int* d_idx, double* d_dist,
               double* d_W, bool fold, ScaleArgs& sc, cudaStream_t st) {
    const int np = loop_view(h).plan.n_clouds;
    const int bpp = lp.bpp;
    if (ensure_state<D, Real>(h, nullptr, nullptr, nullptr, nullptr, nullptr, st)) return 1;
    oa.T_override = d_T;
    oa.out_idx = d_idx;
    oa.out_dist = d_dist;
    oa.out_W = d_W;
    oa.ignore_status = 1;
    if (lp.adaptive && prepare_select<D, Real>(h, oa, sc, st)) return 1;
    correspond_kernel<D, Real><<<dim3(bpp, np), OBJ_THREADS, obj_smem(oa.ppt), st>>>(oa);
    if (lp.adaptive && launch_select<D, Real>(h, oa, sc, bpp, np, st)) return 1;
    auto acc_kernel = lp.robust ? accumulate_kernel<D, Real, true> : accumulate_kernel<D, Real, false>;
    if (d_W || fold) acc_kernel<<<dim3(bpp, np), OBJ_THREADS, 0, st>>>(oa);
    h->launches += 2;
    if (fold) {
        SolveArgs sa;
        memset(&sa, 0, sizeof sa);
        sa.partial = h->partial.as<double>();
        sa.blocks_per_pair = bpp;
        sa.n_pairs = np;
        sa.sum_out = h->red.as<double>();
        sa.state = h->state.as<PairState>();
        solve_kernel<D><<<(np + SOLVE_WARPS - 1) / SOLVE_WARPS, SOLVE_WARPS * 32, 0, st>>>(sa);
        h->launches += 1;
    }
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_stage(gicpContext* h, const Switches& sw, const double* h_T, int* d_idx, double* d_dist, double* d_W,
             double* h_out, double* h_scale, cudaStream_t st) {
    ObjArgs<Real> oa;
    LoopPlan lp;
    // stage entry points always cover the whole source (no slicing), so their outputs are complete
    if (objective_args<D, Real>(h, sw, false, true, oa, lp)) return 1;
    const int np = loop_view(h).plan.n_clouds;
    if (!h_T) return fail("h_T is required");
    if (upload_T(h, h_T, (size_t)np * (D + 1) * (D + 1) * sizeof(double), st)) return 1;
    ScaleArgs sc{};
    if (stage_pass<D, Real>(h, oa, lp, h->T_dev.as<double>(), d_idx, d_dist, d_W, h_out != nullptr, sc, st)) return 1;
    if (h_scale) CU(cudaMemcpyAsync(h_scale, sc.scale, (size_t)np * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (h_out)
        CU(cudaMemcpyAsync(h_out, h->red.p, (size_t)np * Dim<D>::NRED * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return 0;
}

// gicpEvaluate: a stage pass at the caller's device transforms into the handle's own correspondence scratch, then one
// quality_kernel block per pair.  Stream-ordered, no synchronisation.
template <int D, typename Real>
int do_evaluate(gicpContext* h, const Switches& sw, const double* d_T, double* d_quality, double* d_H, double* d_b,
                cudaStream_t st) {
    ObjArgs<Real> oa;
    LoopPlan lp;
    if (objective_args<D, Real>(h, sw, false, true, oa, lp)) return 1;
    const SetupPlan& sp = loop_view(h).plan;
    const int np = sp.n_clouds;
    const size_t n_src = (size_t)std::max<int64_t>(sp.n_total, 1);
    CU(h->eval_idx.ensure(n_src * sizeof(int)));
    CU(h->eval_dist.ensure(n_src * sizeof(double)));
    ScaleArgs sc{};
    if (stage_pass<D, Real>(h, oa, lp, d_T, h->eval_idx.as<int>(), h->eval_dist.as<double>(), nullptr, true, sc, st))
        return 1;
    quality_kernel<D><<<np, QUALITY_THREADS, 0, st>>>(h->red.as<double>(), oa.src_meta, h->eval_idx.as<int>(),
                                                      h->eval_dist.as<double>(), d_quality, d_H, d_b);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_knn(gicpContext* h, int which, int* d_idx, double* d_dist, cudaStream_t st) {
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    if (!cs.ready) return fail("cloud not set");
    if (cs.plan.knn_whole == KnnPath::None)
        return fail("the %s was set up by gicpSetVoxelized: a voxelized side has no k-NN lists",
                    which == GICP_TARGET ? "target" : "source");
    // re-runs K2 over the whole cloud set with the index outputs enabled; the covariances are rewritten with the
    // values of that run (the set-up's own values unless the set-up ran a constant model or a sharded slice)
    return launch_knn<D, Real>(h, cs, cs.plan.knn_whole, d_idx, d_dist, st, -1, -1, h->scr[0]);
}

template <int D, typename Real>
int do_cov(gicpContext* h, int which, double* d_cov, cudaStream_t st) {
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    if (!cs.ready) return fail("cloud not set");
    const SetupPlan& p = cs.plan;
    if (p.n_total == 0) return 0;
    const int bx = (p.max_n + 255) / 256;
    export_cov_kernel<D, Real><<<dim3(bx, p.n_clouds), 256, 0, st>>>(cs.knn.meta.as<CloudMeta>(),
                                                                      cs.knn.spts.as<PRec<Real>>(),
                                                                      cs.cov_knn.as<Real>(), d_cov);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_rotcov(gicpContext* h, const double* h_T, int n_T, double* d_out, cudaStream_t st) {
    CloudSet& cs = h->src;
    const PairList& pl = h->pairs;
    if (!pl.on && !cs.ready) return fail("source not set");
    const SetupPlan& p = loop_view(h).plan;
    if (n_T <= 0 || p.n_total == 0) return 0;
    if (n_T > 65535) return fail("n_T too large");
    if (upload_T(h, h_T, (size_t)n_T * p.n_clouds * (D + 1) * (D + 1) * sizeof(double), st)) return 1;
    const int bx = (p.max_n + 255) / 256;
    // a pair list's sources: the gathered copies (search-grid order; the output is in input order either way)
    rotated_cov_kernel<D, Real><<<dim3(bx, p.n_clouds, n_T), 256, 0, st>>>(
        pl.on ? pl.src_meta.as<CloudMeta>() : cs.knn.meta.as<CloudMeta>(),
        pl.on ? pl.spts.as<PRec<Real>>() : cs.knn.spts.as<PRec<Real>>(), pl.on ? pl.cov.as<Real>() : cs.cov_knn.as<Real>(),
        h->T_dev.as<double>(), p.n_clouds, (size_t)p.n_total, d_out);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

int bit_length(unsigned long long v) {
    int b = 0;
    while (b < 64 && (v >> b)) ++b;
    return b;
}

// gicpVoxelDownsample (voxel.cuh).  Two host synchronisations: the per-cloud voxel bounds (they size the key fields and
// are checked against the limits) and the output offsets.
// With `stats` (gicpSetVoxelized) the centroid kernels also write every output row's covariance to h->vox.cov.
template <int D, typename Real>
int do_voxel(gicpContext* h, const void* d_points, const int64_t* h_off, int nc, double leaf, int min_points,
             void* d_out, int64_t* h_out_off, int* d_voxel_of, int* d_counts, cudaStream_t st, bool stats = false) {
    VoxelScratch& v = h->vox;
    int max_n = 0;
    if (const char* e = check_offsets(h_off, nc, &max_n)) return fail("%s (%d clouds)", e, nc);
    const int n = (int)h_off[nc];
    if (n == 0) {
        for (int i = 0; i <= nc; ++i) h_out_off[i] = 0;
        return 0;
    }
    if (!d_points || !d_out) return fail("null point or output array");
    const Real* pts = static_cast<const Real*>(d_points);
    v.off32.assign(h_off, h_off + nc + 1);
    if (nc + 1 > v.h_cap) {
        if (v.h_vb) cudaFreeHost(v.h_vb);
        if (v.h_out_off) cudaFreeHost(v.h_out_off);
        v.h_vb = nullptr;
        v.h_out_off = nullptr;
        v.h_cap = 0;
        CU(cudaMallocHost(&v.h_vb, (size_t)(nc + 1) * 6 * sizeof(double)));
        CU(cudaMallocHost(&v.h_out_off, (size_t)(nc + 1) * sizeof(int)));
        v.h_cap = nc + 1;
    }
    const int chunks = (max_n + VOX_THREADS * VOX_ITEMS - 1) / (VOX_THREADS * VOX_ITEMS);
    CU(v.offsets.ensure((size_t)(nc + 1) * sizeof(int)));
    CU(v.part.ensure((size_t)nc * std::max(chunks, 1) * 6 * sizeof(double)));
    CU(v.vb.ensure((size_t)nc * 6 * sizeof(double)));
    const int* offs = v.offsets.as<int>();
    CU(cudaMemcpyAsync(v.offsets.p, v.off32.data(), (size_t)(nc + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
    // 1. voxel bounds of every cloud's finite rows -> host
    voxel_bounds_partial_kernel<D, Real><<<dim3(chunks, nc), VOX_THREADS, 0, st>>>(pts, offs, v.part.as<double>(), chunks);
    voxel_bounds_kernel<<<(nc + 3) / 4, 128, 0, st>>>(v.part.as<double>(), chunks, nc, leaf, v.vb.as<double>());
    CU(cudaMemcpyAsync(v.h_vb, v.vb.p, (size_t)nc * 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
    h->launches += 2;
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    // every voxel index an int64, every cloud-relative index below the per-axis limit; then the narrowest key fields
    const double two63 = 9223372036854775808.0;
    const int limit_bits = D == 3 ? 21 : 31;
    long long max_ext[3] = {0, 0, 0};
    for (int c = 0; c < nc; ++c) {
        const double* b = v.h_vb + (size_t)c * 6;
        if (!(b[0] <= b[3])) continue;   // no finite row
        for (int a = 0; a < D; ++a) {
            for (double q : {b[a], b[3 + a]})
                if (!(q >= -two63 && q < two63))
                    return fail("voxel_size %g: cloud %d has voxel index %g along axis %c, outside int64; use a larger "
                                "voxel_size", leaf, c, q, "xyz"[a]);
            const __int128 ext = (__int128)(long long)b[3 + a] - (__int128)(long long)b[a];
            if (ext >= ((__int128)1 << limit_bits))
                return fail("voxel_size %g: cloud %d spans %.0f voxels along axis %c, the limit is 2^%d per axis in %d-D; "
                            "use a larger voxel_size", leaf, c, (double)ext + 1.0, "xyz"[a], limit_bits, D);
            max_ext[a] = std::max<long long>(max_ext[a], (long long)ext);
        }
    }
    VoxKeyGeom geo;
    int coord_bits = 0;
    for (int a = 2; a >= 0; --a) {
        geo.shift[a] = coord_bits;
        if (a < D) coord_bits += bit_length((unsigned long long)max_ext[a]);
    }
    // the cloud index above the coordinates, sized so that the all-ones sentinel exceeds every finite row's key; when
    // it does not fit 64 bits the clouds are sorted as segments on the coordinates alone
    const int end_bit = coord_bits + bit_length((unsigned long long)nc);
    const bool segmented = end_bit > 64;
    geo.cloud_shift = segmented ? -1 : coord_bits;

    // 2. keys, stable sort
    CU(v.keys.ensure((size_t)n * 8));
    CU(v.keys_alt.ensure((size_t)n * 8));
    CU(v.vals.ensure((size_t)(n + 1) * 4));
    CU(v.vals_alt.ensure((size_t)(n + 1) * 4));
    CU(v.rid.ensure((size_t)(n + 1) * 4));
    CU(v.orow.ensure((size_t)(n + 1) * 4));
    CU(v.out_off.ensure((size_t)(nc + 1) * 4));
    CU(v.big.ensure((size_t)(n / (VOX_SEQ_MAX + 1) + 2) * 4));
    voxel_key_kernel<D, Real><<<dim3((max_n + 255) / 256, nc), 256, 0, st>>>(pts, offs, v.vb.as<double>(), leaf, geo,
                                                                             v.keys.as<unsigned long long>(), v.vals.as<int>());
    h->launches += 1;
    const unsigned long long* K;
    const int* R;
    int* free_vals;
    unsigned long long* free_keys;
    if (!segmented) {
        cub::DoubleBuffer<unsigned long long> dk(v.keys.as<unsigned long long>(), v.keys_alt.as<unsigned long long>());
        cub::DoubleBuffer<int> dv(v.vals.as<int>(), v.vals_alt.as<int>());
        size_t tmp = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, n, 0, end_bit, st));
        CU(v.cub_tmp.ensure(tmp));
        CU(cub::DeviceRadixSort::SortPairs(v.cub_tmp.p, tmp, dk, dv, n, 0, end_bit, st));
        h->launches += (end_bit + 7) / 8 + 2;
        K = dk.Current();
        R = dv.Current();
        free_keys = dk.Alternate();
        free_vals = dv.Alternate();
    } else {
        size_t tmp = 0;
        CU(cub::DeviceSegmentedSort::StableSortPairs(nullptr, tmp, v.keys.as<unsigned long long>(),
                                                     v.keys_alt.as<unsigned long long>(), v.vals.as<int>(),
                                                     v.vals_alt.as<int>(), n, nc, offs, offs + 1, st));
        CU(v.cub_tmp.ensure(tmp));
        CU(cub::DeviceSegmentedSort::StableSortPairs(v.cub_tmp.p, tmp, v.keys.as<unsigned long long>(),
                                                     v.keys_alt.as<unsigned long long>(), v.vals.as<int>(),
                                                     v.vals_alt.as<int>(), n, nc, offs, offs + 1, st));
        h->launches += 3;
        K = v.keys_alt.as<unsigned long long>();
        R = v.vals_alt.as<int>();
        free_keys = v.keys.as<unsigned long long>();
        free_vals = v.vals.as<int>();
    }
    // 3. voxels as runs of the sorted keys: run id by a scan of the head flags, begin / end per run
    int* rid = v.rid.as<int>();
    int* run_begin = reinterpret_cast<int*>(free_keys);   // the sort's other key buffer holds 2n ints
    int* run_end = run_begin + n;
    voxel_head_kernel<<<(n + 1 + 255) / 256, 256, 0, st>>>(K, n, rid);
    h->launches += 1;
    if (segmented) {
        voxel_segment_heads_kernel<<<(nc + 255) / 256, 256, 0, st>>>(K, offs, nc, rid);
        h->launches += 1;
    }
    auto excl_scan = [&](int* a, int len) -> int {
        size_t tmp = 0;
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, a, a, len, st));
        CU(v.cub_tmp.ensure(tmp));
        CU(cub::DeviceScan::ExclusiveSum(v.cub_tmp.p, tmp, a, a, len, st));
        h->launches += 2;
        return 0;
    };
    if (excl_scan(rid, n + 1)) return 1;
    const int nb = (n + 255) / 256;
    voxel_runs_kernel<<<nb, 256, 0, st>>>(K, rid, n, run_begin, run_end);
    // 4. keep flag at each kept voxel's lowest row; its scan in input order is the output row
    int* orow = v.orow.as<int>();
    CU(cudaMemsetAsync(orow, 0, (size_t)(n + 1) * 4, st));
    voxel_keep_kernel<<<nb, 256, 0, st>>>(rid, n, run_begin, run_end, R, min_points, orow);
    h->launches += 2;
    if (excl_scan(orow, n + 1)) return 1;
    voxel_out_offsets_kernel<<<(nc + 1 + 255) / 256, 256, 0, st>>>(orow, offs, nc, v.out_off.as<int>());
    h->launches += 1;
    // 5. centroids, counts and the row -> output map
    if (d_voxel_of) CU(cudaMemsetAsync(d_voxel_of, 0xFF, (size_t)n * 4, st));
    int* big_count = free_vals + n;    // the sort's other value buffer: n + 1 ints, the list lives in v.big
    CU(cudaMemsetAsync(big_count, 0, sizeof(int), st));
    VoxOutArgs oa{rid, n, run_begin, run_end, R, orow, v.out_off.as<int>(), nc, min_points, d_voxel_of, d_counts,
                  v.big.as<int>(), big_count};
    const int big_blocks = std::max(1, std::min(n / (VOX_SEQ_MAX + 1), 148 * 8));
    if (stats) {
        CU(v.cov.ensure((size_t)n * ns_of(D) * sizeof(Real)));
        const VoxCovArgs<Real> cv{v.cov.as<Real>(), h->prm.lambda_tangent, h->prm.lambda_normal};
        ProfScope prof(h, GICP_STAGE_KNN_COV, st);
        voxel_centroid_kernel<D, Real, true><<<nb, 256, 0, st>>>(oa, pts, static_cast<Real*>(d_out), cv);
        voxel_centroid_block_kernel<D, Real, true><<<big_blocks, VOX_THREADS, 0, st>>>(oa, pts, static_cast<Real*>(d_out), cv);
    } else {
        voxel_centroid_kernel<D, Real, false><<<nb, 256, 0, st>>>(oa, pts, static_cast<Real*>(d_out), VoxCovArgs<Real>{});
        voxel_centroid_block_kernel<D, Real, false><<<big_blocks, VOX_THREADS, 0, st>>>(oa, pts, static_cast<Real*>(d_out),
                                                                                        VoxCovArgs<Real>{});
    }
    h->launches += 2;
    CU(cudaMemcpyAsync(v.h_out_off, v.out_off.p, (size_t)(nc + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    for (int i = 0; i <= nc; ++i) h_out_off[i] = v.h_out_off[i];
    return 0;
}

// a voxelized side's covariances, computed in output-row order, in the order of its grid
template <int D, typename Real>
__global__ void sort_cov_kernel(const CloudMeta* __restrict__ meta, const PRec<Real>* __restrict__ spts,
                                const Real* __restrict__ cov_rows, Real* __restrict__ cov_sorted) {
    constexpr int NS = Dim<D>::NS;
    const CloudMeta m = meta[blockIdx.y];
    const int s = m.pt_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m.pt_end) return;
    const size_t g = (size_t)m.pt_begin + (size_t)spts[s].idx;
#pragma unroll
    for (int i = 0; i < NS; ++i) cov_sorted[(size_t)s * NS + i] = cov_rows[g * NS + i];
}

// gicpSetVoxelized: the voxel pass with moments into the handle's voxel scratch, then - only once it has succeeded and
// the voxel means have a plan - the side: its one grid over d_out and the covariances in that grid's order.  A refused
// call leaves both sides as they were.
template <int D, typename Real>
int set_voxelized(gicpContext* h, const Switches& sw, int which, const void* d_points, const int64_t* h_off, int nc,
                  double leaf, int min_points, void* d_out, int64_t* h_out_off, cudaStream_t st) {
    if (do_voxel<D, Real>(h, d_points, h_off, nc, leaf, min_points, d_out, h_out_off, nullptr, nullptr, st, true)) return 1;
    const SetupPlan plan = plan_setup_voxelized(h->prm, sw, h_out_off, nc, which, std::is_same<Real, float>::value);
    if (plan.error) return fail("%s (%d clouds)", plan.error, nc);
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    cs.ready = false;
    h->pairs.on = false;
    h->last_stream = st;
    cs.plan = plan;
    cs.raw = d_out;
    if (upload_offsets(cs, h_out_off, st)) return 1;
    const SetupPlan& p = cs.plan;
    if (build_grid<D, Real>(h, cs, cs.knn, p.knn_cell, st, h->scr[0])) return 1;
    const size_t n = (size_t)std::max<int64_t>(p.n_total, 1);
    CU(cs.cov_knn.ensure(n * ns_of(D) * sizeof(Real)));
    if (p.cov != CovSource::Voxel) {
        const Real diag = p.cov == CovSource::Identity ? Real(1) : Real(0);
        fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_knn.as<Real>(), n, diag);
        h->launches += 1;
    } else if (p.n_total > 0) {
        sort_cov_kernel<D, Real><<<dim3((p.max_n + 255) / 256, nc), 256, 0, st>>>(
            cs.knn.meta.as<CloudMeta>(), cs.knn.spts.as<PRec<Real>>(), h->vox.cov.as<Real>(), cs.cov_knn.as<Real>());
        h->launches += 1;
    }
    CU(cudaGetLastError());
    cs.ready = true;
    return 0;
}

// gicpSetPairList: validate (plan_pairs), then gather the pairs' sources and metadata on `st`.  A refused list leaves
// the handle as it was.
template <int D, typename Real>
int set_pair_list(gicpContext* h, int n_pairs, const int32_t* src_cloud, const int32_t* tgt_cloud, int source_set,
                  int64_t* h_pair_offsets, cudaStream_t st) {
    auto sizes = [](const CloudSet& cs) { return cs.ready ? SetSizes{cs.h_off.data(), cs.plan.n_clouds} : SetSizes{}; };
    PairPlan pp = plan_pairs(n_pairs, src_cloud, tgt_cloud, source_set, sizes(h->src), sizes(h->tgt), h->comm != nullptr);
    if (pp.error) return fail("gicpSetPairList refused: %s", pp.error);
    PairList& pl = h->pairs;
    pl.on = false;   // until the new list is in place: a CUDA failure below leaves the handle one-to-one
    CloudSet& from = source_set == GICP_TARGET ? h->tgt : h->src;
    const size_t n = (size_t)std::max<int64_t>(pp.view.n_total, 1);
    CU(pl.list.ensure((size_t)n_pairs * 3 * sizeof(int)));
    CU(pl.src_meta.ensure((size_t)n_pairs * sizeof(CloudMeta)));
    CU(pl.tgt_meta.ensure((size_t)n_pairs * sizeof(CloudMeta)));
    CU(pl.tgt_bbox.ensure((size_t)n_pairs * 6 * sizeof(double)));
    CU(pl.spts.ensure(n * sizeof(PRec<Real>)));
    CU(pl.cov.ensure(n * ns_of(D) * sizeof(Real)));
    pl.h_list.resize((size_t)n_pairs * 3);
    for (int p = 0; p < n_pairs; ++p) {
        pl.h_list[3 * p] = src_cloud[p];
        pl.h_list[3 * p + 1] = tgt_cloud[p];
        pl.h_list[3 * p + 2] = (int)pp.offsets[p];
    }
    CU(cudaMemcpyAsync(pl.list.p, pl.h_list.data(), pl.h_list.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    // a target set's covariances are those of a target (I, or the estimated ones under covariance_model 1 / 2); a
    // source set up as such has C = 0 there
    const bool zero_cov = source_set == GICP_TARGET && h->prm.covariance_model != GICP_PLANE_TO_PLANE;
    PairGatherArgs<Real> a{pl.list.as<int>(), from.nng().meta.as<CloudMeta>(), from.nng().spts.as<PRec<Real>>(),
                           zero_cov ? nullptr : from.covnn().as<Real>(), h->tgt.nng().meta.as<CloudMeta>(),
                           h->tgt.knn.bbox.as<double>(), pl.src_meta.as<CloudMeta>(), pl.tgt_meta.as<CloudMeta>(),
                           pl.tgt_bbox.as<double>(), pl.spts.as<PRec<Real>>(), pl.cov.as<Real>()};
    const int bx = std::max(1, (pp.view.max_n + PAIR_GATHER_ROWS - 1) / PAIR_GATHER_ROWS);
    pair_gather_kernel<D, Real><<<dim3(bx, n_pairs), PAIR_GATHER_THREADS, 0, st>>>(a);
    h->launches += 1;
    CU(cudaGetLastError());
    h->last_stream = st;
    pl.view = pp.view;
    pl.on = true;
    if (h_pair_offsets) std::copy(pp.offsets.begin(), pp.offsets.end(), h_pair_offsets);
    return 0;
}

#define DISPATCH(h, FN, ...)                                                               \
    ((h)->dim == 2 ? ((h)->storage == GICP_STORAGE_F32 ? FN<2, float>(__VA_ARGS__) : FN<2, double>(__VA_ARGS__)) \
                   : ((h)->storage == GICP_STORAGE_F32 ? FN<3, float>(__VA_ARGS__) : FN<3, double>(__VA_ARGS__)))

int check(gicpHandle h) {
    if (!h) return fail("null handle");
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return fail("cudaSetDevice(%d): %s", h->device, cudaGetErrorString(e));
    return 0;
}

}  // namespace

extern "C" {

const char* gicpGetLastError(void) { return g_last_error.c_str(); }
int gicpVersion(void) { return 106; }

int gicpDefaultParams(gicpParams* p) {
    if (!p) return fail("null params");
    memset(p, 0, sizeof *p);
    p->k = 6;
    p->max_iterations = 100;
    p->tolerance = 1e-6;
    p->max_distance_correspondence = 150.0;
    p->max_distance_nearest_neighbors = 50.0;
    p->lambda_tangent = 100.0;
    p->lambda_normal = 10.0;
    p->inner_max_iterations = 50;
    return 0;
}

int gicpCreate(gicpHandle* out, int device, int dim, int storage) {
    if (!out) return fail("null out");
    if (dim != 2 && dim != 3) return fail("dim must be 2 or 3 (got %d)", dim);
    if (storage != GICP_STORAGE_F32 && storage != GICP_STORAGE_F64) return fail("bad storage %d", storage);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail("no CUDA device available (%s): this engine has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail("device %d out of range (%d devices)", device, count);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail("device %d is sm_%d%d; this library holds sm_100a code only (B200)", device, prop.major, prop.minor);
    gicpContext* h = new gicpContext();
    h->device = device;
    h->dim = dim;
    h->storage = storage;
    gicpDefaultParams(&h->prm);
    CU(cudaMallocHost(&h->h_poll, gicpContext::NPOLL * sizeof(int)));
    for (int i = 0; i < gicpContext::NPOLL; ++i) CU(cudaEventCreateWithFlags(&h->poll_ev[i], cudaEventDisableTiming));
    *out = h;
    return 0;
}

int gicpDestroy(gicpHandle h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    h->src.release();
    h->tgt.release();
    h->pairs.release();
    for (SetupScratch& sc : h->scr) sc.release();
    h->vox.release();
    DevBuf* bufs[] = {&h->state, &h->partial, &h->partial2, &h->red, &h->T_dev, &h->n_active, &h->prev_match, &h->slack,
                      &h->active_list, &h->sel_keys, &h->sel_hist, &h->sel_arrived, &h->sel_state, &h->pair_scale,
                      &h->eval_idx, &h->eval_dist};
    for (DevBuf* b : bufs) b->release();
    if (h->h_poll) cudaFreeHost(h->h_poll);
    for (cudaEvent_t e : h->poll_ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    delete h;
    return 0;
}

int gicpSetParams(gicpHandle h, const gicpParams* p) {
    if (check(h)) return 1;
    if (!p) return fail("null params");
    if (p->k < 1 || p->k > 32) return fail("k must be in [1, 32] (got %d)", p->k);
    if (p->max_iterations < 1) return fail("max_iterations must be >= 1");
    if (!(p->max_distance_nearest_neighbors > 0)) return fail("max_distance_nearest_neighbors must be > 0");
    if (!(p->max_distance_correspondence > 0)) return fail("max_distance_correspondence must be > 0");
    if (p->covariance_model < 0 || p->covariance_model > 2) return fail("covariance_model must be 0, 1 or 2");
    // a zero lambda_normal makes C_B + R C_A R^T singular wherever two normals align, a negative one makes W indefinite
    if (!(std::isfinite(p->lambda_tangent) && p->lambda_tangent > 0))
        return fail("lambda_tangent must be finite and > 0 (got %g)", p->lambda_tangent);
    if (!(std::isfinite(p->lambda_normal) && p->lambda_normal > 0))
        return fail("lambda_normal must be finite and > 0 (got %g)", p->lambda_normal);
    h->prm = *p;
    if (h->prm.inner_max_iterations <= 0) h->prm.inner_max_iterations = 50;
    h->src.ready = false;
    h->tgt.ready = false;
    h->pairs.on = false;
    return 0;
}

int gicpSetRobustKernel(gicpHandle h, int kind, double scale) {
    if (check(h)) return 1;
    if (kind < GICP_ROBUST_NONE || kind > GICP_ROBUST_TUKEY)
        return fail("unknown robust kernel %d (GICP_ROBUST_NONE 0, HUBER 1, CAUCHY 2, TUKEY 3)", kind);
    if (kind != GICP_ROBUST_NONE && !(std::isfinite(scale) && scale > 0))
        return fail("robust kernel scale must be finite and > 0 (got %g)", scale);
    // the set-up source and target stay valid: the weights enter only the accumulation of later calls
    h->robust_kind = kind;
    h->robust_scale = kind == GICP_ROBUST_NONE ? 0.0 : scale;
    h->robust_adaptive = false;
    return 0;
}

int gicpSetRobustKernelAdaptive(gicpHandle h, int kind, double kappa, double min_scale) {
    if (check(h)) return 1;
    if (kind < GICP_ROBUST_HUBER || kind > GICP_ROBUST_TUKEY)
        return fail("adaptive robust kernel must be GICP_ROBUST_HUBER 1, CAUCHY 2 or TUKEY 3 (got %d; switch the kernel "
                    "off with gicpSetRobustKernel(h, GICP_ROBUST_NONE, 0))", kind);
    if (!(std::isfinite(kappa) && kappa > 0)) return fail("adaptive robust kappa must be finite and > 0 (got %g)", kappa);
    if (!(std::isfinite(min_scale) && min_scale > 0))
        return fail("adaptive robust min_scale must be finite and > 0 (got %g)", min_scale);
    h->robust_kind = kind;
    h->robust_scale = 0.0;
    h->robust_adaptive = true;
    h->robust_kappa = kappa;
    h->robust_min_scale = min_scale;
    return 0;
}

int gicpSetTarget(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_offsets) return fail("null offsets");
    return DISPATCH(h, set_cloud, h, read_switches(), GICP_TARGET, d_points, h_offsets, n_clouds, (cudaStream_t)stream, 0);
}

int gicpSetSource(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_offsets) return fail("null offsets");
    return DISPATCH(h, set_cloud, h, read_switches(), GICP_SOURCE, d_points, h_offsets, n_clouds, (cudaStream_t)stream, 0);
}

int gicpSetPair(gicpHandle h, const void* d_target, const int64_t* h_target_offsets, const void* d_source,
                const int64_t* h_source_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_target_offsets || !h_source_offsets) return fail("null offsets");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_clouds <= 0) return fail("n_clouds must be positive");
    const Switches sw = read_switches();
    // side by side (pair_overlap), each side with its own scratch (scr[0] / scr[1]), or one after the other
    if (!pair_overlap(sw, Ranks{h->comm != nullptr, h->n_ranks, h->rank}, h->prof_on, h_target_offsets[n_clouds],
                      h_source_offsets[n_clouds])) {
        if (DISPATCH(h, set_cloud, h, sw, GICP_TARGET, d_target, h_target_offsets, n_clouds, st, 0)) return 1;
        return DISPATCH(h, set_cloud, h, sw, GICP_SOURCE, d_source, h_source_offsets, n_clouds, st, 0);
    }
    if (!h->side_stream) {
        CU(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    // fork: the side stream sees everything the caller queued on `stream` so far (the upload of the clouds);
    // join: `stream` continues only after the source side is set up
    CU(cudaEventRecord(h->ev_fork, st));
    CU(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    const int rc_t = DISPATCH(h, set_cloud, h, sw, GICP_TARGET, d_target, h_target_offsets, n_clouds, st, 0);
    const int rc_s =
        rc_t ? 1 : DISPATCH(h, set_cloud, h, sw, GICP_SOURCE, d_source, h_source_offsets, n_clouds, h->side_stream, 1);
    CU(cudaEventRecord(h->ev_join, h->side_stream));
    CU(cudaStreamWaitEvent(st, h->ev_join, 0));
    h->last_stream = st;
    return rc_t || rc_s;
}

int gicpPromoteTargetToSource(gicpHandle h) {
    if (check(h)) return 1;
    if (!h->tgt.ready) return fail("no target to promote");
    std::swap(h->src, h->tgt);   // both sides own the same kind of state (two grids + covariances)
    h->tgt.ready = false;
    h->pairs.on = false;
    if (h->prm.covariance_model != GICP_PLANE_TO_PLANE) return DISPATCH(h, zero_source_cov, h, h->last_stream);
    return 0;
}

int gicpSetPairList(gicpHandle h, int32_t n_pairs, const int32_t* h_source_cloud, const int32_t* h_target_cloud,
                    int source_set, int64_t* h_pair_offsets, void* stream) {
    if (check(h)) return 1;
    return DISPATCH(h, set_pair_list, h, n_pairs, h_source_cloud, h_target_cloud, source_set, h_pair_offsets,
                    (cudaStream_t)stream);
}

int gicpRegister(gicpHandle h, const double* h_T0, double* d_T, int32_t* d_n_outer, int32_t* d_converged,
                 double* d_loss_hist, double* d_T_hist, int32_t* d_inliers, void* stream) {
    if (check(h)) return 1;
    if (!d_T || !d_n_outer || !d_converged) return fail("d_T, d_n_outer and d_converged are required");
    return DISPATCH(h, do_register, h, read_switches(), h_T0, d_T, d_n_outer, d_converged, d_loss_hist, d_T_hist, d_inliers,
                    (cudaStream_t)stream);
}

int gicpKnn(gicpHandle h, int which, int32_t* d_idx, double* d_dist, void* stream) {
    if (check(h)) return 1;
    if (!d_idx) return fail("d_idx is required");
    return DISPATCH(h, do_knn, h, which, d_idx, d_dist, (cudaStream_t)stream);
}

int gicpCovariances(gicpHandle h, int which, double* d_cov, void* stream) {
    if (check(h)) return 1;
    if (!d_cov) return fail("d_cov is required");
    return DISPATCH(h, do_cov, h, which, d_cov, (cudaStream_t)stream);
}

int gicpCorrespond(gicpHandle h, const double* h_T, int32_t* d_idx, double* d_dist, double* d_W, void* stream) {
    if (check(h)) return 1;
    return DISPATCH(h, do_stage, h, read_switches(), h_T, d_idx, d_dist, d_W, (double*)nullptr, (double*)nullptr,
                    (cudaStream_t)stream);
}

int gicpNormalEquations(gicpHandle h, const double* h_T, double* h_out, void* stream) {
    if (check(h)) return 1;
    if (!h_out) return fail("h_out is required");
    return DISPATCH(h, do_stage, h, read_switches(), h_T, (int*)nullptr, (double*)nullptr, (double*)nullptr, h_out,
                    (double*)nullptr, (cudaStream_t)stream);
}

int gicpRobustScales(gicpHandle h, const double* h_T, double* h_scale, void* stream) {
    if (check(h)) return 1;
    if (!h_T || !h_scale) return fail("h_T and h_scale are required");
    const LoopView lv = loop_view(h);
    if (!lv.ready) return fail("set source and target first");
    if (!h->robust_adaptive) {   // a fixed scale, or 0 without a kernel: nothing to compute
        for (int p = 0; p < lv.plan.n_clouds; ++p) h_scale[p] = h->robust_scale;
        return 0;
    }
    return DISPATCH(h, do_stage, h, read_switches(), h_T, (int*)nullptr, (double*)nullptr, (double*)nullptr,
                    (double*)nullptr, h_scale, (cudaStream_t)stream);
}

int gicpEvaluate(gicpHandle h, const double* d_T, double* d_quality, double* d_H, double* d_b, void* stream) {
    if (check(h)) return 1;
    if (!d_T) return fail("d_T is required");
    return DISPATCH(h, do_evaluate, h, read_switches(), d_T, d_quality, d_H, d_b, (cudaStream_t)stream);
}

int gicpSourceCovariancesAt(gicpHandle h, const double* h_T, int32_t n_T, double* d_out, void* stream) {
    if (check(h)) return 1;
    if (!h_T || !d_out) return fail("h_T and d_out are required");
    return DISPATCH(h, do_rotcov, h, h_T, n_T, d_out, (cudaStream_t)stream);
}

int gicpVoxelDownsample(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds,
                        double voxel_size, int32_t min_points, void* d_out, int64_t* h_out_offsets,
                        int32_t* d_voxel_of, int32_t* d_counts, void* stream) {
    if (check(h)) return 1;
    if (!h_offsets || !h_out_offsets) return fail("null offsets");
    if (d_points && d_out == d_points) return fail("d_out must not alias d_points");
    if (!(std::isfinite(voxel_size) && voxel_size > 0)) return fail("voxel_size must be finite and > 0 (got %g)", voxel_size);
    if (min_points < 1) return fail("min_points must be >= 1 (got %d)", min_points);
    return DISPATCH(h, do_voxel, h, d_points, h_offsets, n_clouds, voxel_size, min_points, d_out, h_out_offsets,
                    d_voxel_of, d_counts, (cudaStream_t)stream);
}

int gicpSetVoxelized(gicpHandle h, int which, const void* d_points, const int64_t* h_offsets, int32_t n_clouds,
                     double voxel_size, int32_t min_points, void* d_out, int64_t* h_out_offsets, void* stream) {
    if (check(h)) return 1;
    if (which != GICP_SOURCE && which != GICP_TARGET)
        return fail("which must be GICP_SOURCE 0 or GICP_TARGET 1 (got %d)", which);
    if (h->comm) return fail("gicpSetVoxelized: a handle with a communicator (gicpCommInit) takes raw sides only");
    if (!h_offsets || !h_out_offsets) return fail("null offsets");
    if (d_points && d_out == d_points) return fail("d_out must not alias d_points");
    if (!(std::isfinite(voxel_size) && voxel_size > 0)) return fail("voxel_size must be finite and > 0 (got %g)", voxel_size);
    if (min_points < 1) return fail("min_points must be >= 1 (got %d)", min_points);
    return DISPATCH(h, set_voxelized, h, read_switches(), which, d_points, h_offsets, n_clouds, voxel_size, min_points,
                    d_out, h_out_offsets, (cudaStream_t)stream);
}

int gicpCommGetUniqueId(char id[128]) {
    if (load_nccl()) return 1;
    int rc = g_nccl.GetUniqueId(id);
    if (rc) return fail("ncclGetUniqueId failed (%d)", rc);
    return 0;
}

int gicpCommInit(gicpHandle h, int32_t n_ranks, int32_t rank, const char id[128]) {
    if (check(h)) return 1;
    if (load_nccl()) return 1;
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail("bad rank %d / %d", rank, n_ranks);
    Id128 u;
    memcpy(u.b, id, 128);
    void* comm = nullptr;
    int rc = g_nccl.CommInitRank(&comm, n_ranks, u, rank);
    if (rc) return fail("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    h->comm = comm;
    h->n_ranks = n_ranks;
    h->rank = rank;
    h->src.ready = h->tgt.ready = false;
    h->pairs.on = false;
    return 0;
}

int gicpCommDestroy(gicpHandle h) {
    if (check(h)) return 1;
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    h->comm = nullptr;
    h->n_ranks = 1;
    h->rank = 0;
    return 0;
}

int gicpRayCast(int device, const double* d_poses, int32_t n_poses, int32_t num_rays, const double* d_segments,
                int32_t n_seg, const double* d_circles, int32_t n_circ, double max_range, const double* d_noise,
                double* d_rel_xy, int32_t* d_hit, void* stream) {
    if (n_poses <= 0 || num_rays <= 0 || 360 % num_rays != 0) return fail("need n_poses > 0 and num_rays dividing 360");
    if (!d_poses || !d_rel_xy || !d_hit) return fail("null pointer");
    CU(cudaSetDevice(device));
    RayCastArgs a{d_poses, n_poses, num_rays, d_segments, n_seg, d_circles, n_circ, max_range, d_noise, d_rel_xy, d_hit};
    const long long n = (long long)n_poses * num_rays;
    raycast_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
    CU(cudaGetLastError());
    return 0;
}

int64_t gicpLaunchCount(gicpHandle h) { return h ? h->launches : 0; }

int gicpProfile(gicpHandle h, int enable) {
    if (check(h)) return 1;
    h->prof_on = enable != 0;
    h->prof_recs.clear();
    h->ev_used = 0;
    return 0;
}

int gicpProfileReadStages(gicpHandle h, int32_t n_stages, double* ms_out, int64_t* count_out) {
    if (check(h)) return 1;
    if (n_stages < 0 || n_stages > GICP_N_STAGES_ALL) return fail("n_stages must be in [0, %d]", GICP_N_STAGES_ALL);
    if (n_stages && (!ms_out || !count_out)) return fail("ms_out and count_out are required");
    CU(cudaDeviceSynchronize());
    for (int i = 0; i < n_stages; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
    for (auto& r : h->prof_recs) {
        if (r.stage >= n_stages) continue;
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, r.a, r.b));
        ms_out[r.stage] += ms;
        count_out[r.stage] += 1;
    }
    h->prof_recs.clear();
    h->ev_used = 0;
    return 0;
}

int gicpProfileRead(gicpHandle h, double ms_out[GICP_N_STAGES], int64_t count_out[GICP_N_STAGES]) {
    return gicpProfileReadStages(h, GICP_N_STAGES, ms_out, count_out);
}

}  // extern "C"

