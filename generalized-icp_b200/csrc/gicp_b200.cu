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
#include <vector>

#include "../../include/gicp_b200.h"
#include "grid.cuh"
#include "knn_cov.cuh"
#include "objective.cuh"
#include "raycast.cuh"
#include "solve.cuh"
#include "fused.cuh"
#include "voxel.cuh"

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
    long long budget = 0;
    long long total_cells = 0;
    double h_target = 0;
    bool built = false;
    void release() { meta.release(); cell_start.release(); spts.release(); inv_perm.release(); bbox.release(); lut.release(); }
};

struct CloudSet {
    const void* raw = nullptr;
    std::vector<int64_t> offsets;
    std::vector<int> off32;   // staging copy of the offsets for the asynchronous upload (must outlive the call)
    int n_clouds = 0;
    int64_t n_total = 0;
    int max_n = 0;
    DevBuf d_offsets;   // int32 [n_clouds+1]
    int inline_n = -1;  // >= 0: one small cloud of that many points, its offsets travel as a kernel argument (no upload)
    Grid knn;           // grid of the covariance neighbourhoods (cell ~ knn radius / 4)
    Grid nn;            // grid of the correspondence search (cell ~ d_max / 2): the target is searched in it,
                        // the source is only ORDERED by it (compact warps in K3).  Built only when the k-NN
                        // grid's cells do not suit the search (`shared` = false)
    DevBuf cov_knn;     // covariances in knn-grid order (written by K2)
    DevBuf cov_nn;      // the same covariances in nn-grid order (read by K3); unused when shared
    bool shared = true; // one grid serves both stages: half the grid builds, no covariance re-ordering
    bool ready = false;
    Grid& nng() { return shared ? knn : nn; }
    DevBuf& covnn() { return shared ? cov_knn : cov_nn; }
    void release() { d_offsets.release(); knn.release(); nn.release(); cov_knn.release(); cov_nn.release(); }
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
    double* h_vb = nullptr;     // pinned: per-cloud voxel bounds
    int* h_out_off = nullptr;   // pinned: output offsets
    int h_cap = 0;              // clouds the pinned buffers hold
    std::vector<int> off32;
    void release() {
        for (DevBuf* b : {&offsets, &part, &vb, &keys, &keys_alt, &vals, &vals_alt, &rid, &orow, &out_off, &big, &cub_tmp})
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
    CloudSet src, tgt;
    // [0]: every call on the caller's stream; [1]: the source side of gicpSetPair while it runs on the internal stream
    SetupScratch scr[2];
    VoxelScratch vox;
    DevBuf state, partial, partial2, red, T_dev, n_active, prev_match, slack, active_list;
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

const char* const kStageNames[GICP_N_STAGES] = {"gicp:grid_build", "gicp:knn_cov", "gicp:correspond", "gicp:accumulate",
                                                 "gicp:solve"};

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
    const int nc = cs.n_clouds;
    const int64_t n = cs.n_total;
    long long budget = h->prm.max_cells_per_cloud;
    if (budget <= 0) {
        budget = 4096;  // Morton padding can cost up to 8x the occupied box
        while (budget < 8LL * cs.max_n) budget <<= 1;
    }
    // Large batches: the table (memset + scan + 4 B per cell, per cloud set) is sized for one cell per point instead
    // of eight - grid_meta_kernel then enlarges the cell edge by the few per cent that save the Morton bits (a 40 m
    // cloud at 1.25 m cells needs 33-36 cells per axis = 2^18 padded; at 1.3-1.4 m it fits 2^15)
    if (h->prm.max_cells_per_cloud <= 0) {
        long long cap_total = 1LL << 30;   // default: no shrinking (measured: the larger cells cost K2 more than K1 gains)
        if (getenv("GICP_CELL_TABLE_LOG2") && atoi(getenv("GICP_CELL_TABLE_LOG2")) > 0) cap_total = 1LL << atoi(getenv("GICP_CELL_TABLE_LOG2"));
        while (budget * (long long)nc > cap_total && budget > 4096 && budget / 2 >= cs.max_n) budget >>= 1;
    }
    if (budget * (long long)nc > (1LL << 30)) {
        budget = (1LL << 30) / nc;
        if (budget < 64) return fail("too many clouds for the cell table (%d)", nc);
    }
    g.budget = budget;
    g.total_cells = budget * nc;
    g.h_target = h_target;
    const int chunks = std::max(1, (cs.max_n + BBOX_THREADS * BBOX_ITEMS - 1) / (BBOX_THREADS * BBOX_ITEMS));
    CU(sc.bbox_part.ensure((size_t)nc * chunks * 6 * sizeof(double)));
    CU(g.meta.ensure((size_t)nc * sizeof(CloudMeta)));
    CU(g.bbox.ensure((size_t)nc * 6 * sizeof(double)));
    CU(g.cell_start.ensure((size_t)(g.total_cells + 1) * sizeof(int)));
    CU(g.spts.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(PRec<Real>)));
    CU(g.inv_perm.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(int)));
    CU(sc.keys.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.keys_alt.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.vals.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    CU(sc.vals_alt.ensure((size_t)std::max<int64_t>(n, 1) * 4));
    const Real* pts = static_cast<const Real*>(cs.raw);
    const int* offs = cs.d_offsets.as<int>();
    ProfScope prof(h, GICP_STAGE_GRID, st);

    // small clouds (the reference's own workloads): the whole build of a cloud in one block, one launch
    if (cs.max_n <= SMALL_GRID_MAX && budget <= (1LL << 20) && n > 0 &&
        !(getenv("GICP_SMALL_GRID") && atoi(getenv("GICP_SMALL_GRID")) == 0)) {
        CU(g.lut.ensure((size_t)nc * 3 * GICP_LUT_N * sizeof(int)));
        small_grid_kernel<D, Real><<<nc, SMALL_GRID_THREADS, 0, st>>>(pts, offs, h_target, budget, g.meta.as<CloudMeta>(),
                                                                      g.bbox.as<double>(), g.lut.as<int>(),
                                                                      g.cell_start.as<int>(), g.spts.as<PRec<Real>>(),
                                                                      g.inv_perm.as<int>(), 1, cs.inline_n);
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
    CU(cudaMemsetAsync(g.cell_start.p, 0, (size_t)(g.total_cells + 1) * sizeof(int), st));
    h->launches += 3;
    if (n > 0) {
        const int bx = (cs.max_n + 255) / 256;
        cell_key_kernel<D, Real><<<dim3(bx, nc), 256, 0, st>>>(pts, g.meta.as<CloudMeta>(), sc.keys.as<unsigned>(),
                                                               sc.vals.as<int>(), g.cell_start.as<int>());
        h->launches += 1;
    }
    {   // cell_start = exclusive scan of the histogram
        size_t tmp = 0;
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, g.cell_start.as<int>(), g.cell_start.as<int>(),
                                         (int)(g.total_cells + 1), st));
        CU(sc.cub_tmp.ensure(tmp));
        CU(cub::DeviceScan::ExclusiveSum(sc.cub_tmp.p, tmp, g.cell_start.as<int>(), g.cell_start.as<int>(),
                                         (int)(g.total_cells + 1), st));
        h->launches += 2;
    }
    if (n > 0) {
        int bits = 1;
        while ((1LL << bits) < g.total_cells) ++bits;
        cub::DoubleBuffer<unsigned> dk(sc.keys.as<unsigned>(), sc.keys_alt.as<unsigned>());
        cub::DoubleBuffer<int> dv(sc.vals.as<int>(), sc.vals_alt.as<int>());
        size_t tmp = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp, dk, dv, (int)n, 0, bits, st));
        CU(sc.cub_tmp.ensure(tmp));
        CU(cub::DeviceRadixSort::SortPairs(sc.cub_tmp.p, tmp, dk, dv, (int)n, 0, bits, st));
        h->launches += (bits + 7) / 8 + 2;
        const int bx = (cs.max_n + 255) / 256;
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

template <int D, typename Real>
int launch_knn(gicpContext* h, CloudSet& cs, int* d_idx, double* d_dist, cudaStream_t st, int slice_b, int slice_e,
               SetupScratch& sc) {
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
    if (cs.n_total == 0) return 0;
    const int span = (slice_b >= 0) ? (slice_e - slice_b) : cs.max_n;
    if (span <= 0) return 0;
    const int bx = (span + KNN_THREADS - 1) / KNN_THREADS;
    dim3 grid(bx, cs.n_clouds);
    // fast path's overflow hand-over: worst case every warp
    const long long n_chunks = (long long)bx * KNN_WARPS * cs.n_clouds;
    CU(sc.ovf_count.ensure(sizeof(int)));
    CU(sc.ovf_list.ensure((size_t)n_chunks * sizeof(int2)));
    a.overflow_count = sc.ovf_count.as<int>();
    a.overflow_list = sc.ovf_list.as<int2>();
    a.overflow_cap = (int)std::min<long long>(n_chunks, INT_MAX);
    // latency mode (a few small clouds): the general kernel alone - one launch, no overflow hand-over
    const bool latency_mode = cs.max_n <= SMALL_GRID_MAX && cs.n_total <= 65536 &&
                              !(getenv("GICP_SMALL_GRID") && atoi(getenv("GICP_SMALL_GRID")) == 0);
    const bool fast = a.k + 8 <= knn_list_cap<Real>() && !latency_mode;
    const size_t smem_g = 128 + (size_t)KNN_WARPS * KNN_WARP_SMEM;
    const size_t smem_h = 128 + (size_t)KNN_WARPS * KNN_HIST_WARP_SMEM;
    ProfScope prof(h, GICP_STAGE_KNN_COV, st);
#define KNN_LAUNCH(KC, GRID, FROM_LIST)                                                                      \
    do {                                                                                                     \
        CU(cudaFuncSetAttribute(knn_general_kernel<D, Real, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                (int)smem_g));                                                               \
        knn_general_kernel<D, Real, KC><<<GRID, KNN_THREADS, smem_g, st>>>(a, FROM_LIST);                    \
    } while (0)
    if (latency_mode && cs.max_n <= KNN_BRUTE_MAX && slice_b < 0 &&
        !(getenv("GICP_KNN_BRUTE") && atoi(getenv("GICP_KNN_BRUTE")) == 0)) {
        // tiny clouds: brute force from shared memory, one block per cloud, one launch
        const size_t smem_b = (size_t)cs.max_n * sizeof(PRec<Real>);
        if (a.k <= 6) knn_brute_kernel<D, Real, 6><<<cs.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        else if (a.k <= 20) knn_brute_kernel<D, Real, 20><<<cs.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        else knn_brute_kernel<D, Real, 32><<<cs.n_clouds, KNN_BRUTE_THREADS, smem_b, st>>>(a);
        h->launches += 1;
        CU(cudaGetLastError());
        return 0;
    }
    if (fast) {
        CU(cudaMemsetAsync(sc.ovf_count.p, 0, sizeof(int), st));
        CU(cudaFuncSetAttribute(knn_hist_kernel<D, Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
        CU(cudaFuncSetAttribute(knn_hist_kernel<D, Real>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        const size_t smem_l = (size_t)KNN_WARPS * KNN_LANE_WARP_SMEM;
        // two equally fast variants (measured): warp-cooperative with TMA-staged cell blocks (default) and
        // per-lane cell walks from L1 (GICP_KNN_LANE=1)
        const bool per_lane = getenv("GICP_KNN_LANE") && atoi(getenv("GICP_KNN_LANE")) != 0;
        if (per_lane) {
            CU(cudaFuncSetAttribute(knn_lane_kernel<D, Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l));
            CU(cudaFuncSetAttribute(knn_lane_kernel<D, Real>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            knn_lane_kernel<D, Real><<<grid, KNN_THREADS, smem_l, st>>>(a);
        } else {
            knn_hist_kernel<D, Real><<<grid, KNN_THREADS, smem_h, st>>>(a);
        }
        const dim3 lgrid(296, 1);
        if (a.k <= 6) KNN_LAUNCH(6, lgrid, 1);
        else if (a.k <= 20) KNN_LAUNCH(20, lgrid, 1);
        else KNN_LAUNCH(32, lgrid, 1);
        h->launches += 2;
    } else {
        if (a.k <= 6) KNN_LAUNCH(6, grid, 0);
        else if (a.k <= 20) KNN_LAUNCH(20, grid, 0);
        else KNN_LAUNCH(32, grid, 0);
        h->launches += 1;
    }
#undef KNN_LAUNCH
    CU(cudaGetLastError());
    return 0;
}

// per-warp TMA stages + the block's work list (one entry per point of the block)
inline size_t obj_smem(int ppt) {
    return 128 + (size_t)(OBJ_THREADS / 32) * OBJ_STAGE_BYTES + (size_t)OBJ_THREADS * ppt * sizeof(int);
}

// cell edges; never smaller than (search radius)/8 so that a lane's ball spans <= 17 cells per axis
double auto_knn_cell(const gicpContext* h) {
    const double r = h->prm.max_distance_nearest_neighbors;
    if (getenv("GICP_KNN_CELL") && atof(getenv("GICP_KNN_CELL")) > 0) return std::max(atof(getenv("GICP_KNN_CELL")), r / 8.0);   // A/B timing
    if (h->prm.knn_cell > 0) return std::max(h->prm.knn_cell, r / 8.0);
    return 0.25 * r;   // measured optimum of the cooperative fast path on the bench workload (r = 5 m -> 1.25 m cells)
}
double auto_nn_cell(const gicpContext* h) {
    const double r = h->prm.max_distance_correspondence;
    if (getenv("GICP_NN_CELL") && atof(getenv("GICP_NN_CELL")) > 0) return std::max(atof(getenv("GICP_NN_CELL")), r / 8.0);   // A/B timing
    if (h->prm.nn_cell > 0) return std::max(h->prm.nn_cell, r / 8.0);
    return 0.5 * r;
}

// true when set_cloud takes the latency path for these clouds (small_grid_kernel + one k-NN launch): that path
// touches only the side's own buffers, none of the handle's shared scratch (same conditions as build_grid / launch_knn)
bool latency_path(const gicpContext* h, const int64_t* off, int n_clouds) {
    if (getenv("GICP_SMALL_GRID") && atoi(getenv("GICP_SMALL_GRID")) == 0) return false;
    if (n_clouds <= 0 || off[0] != 0 || h->prm.max_cells_per_cloud > (1LL << 20)) return false;
    int64_t max_n = 0;
    for (int i = 1; i <= n_clouds; ++i) {
        if (off[i] < off[i - 1]) return false;
        max_n = std::max<int64_t>(max_n, off[i] - off[i - 1]);
    }
    return max_n <= SMALL_GRID_MAX && off[n_clouds] > 0 && off[n_clouds] <= 65536;
}

template <int D, typename Real>
int set_cloud(gicpContext* h, int which, const void* d_points, const int64_t* h_offsets, int n_clouds,
              cudaStream_t st, int scratch_slot) {
    SetupScratch& sc = h->scr[scratch_slot];
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    cs.ready = false;
    h->last_stream = st;
    if (n_clouds <= 0) return fail("n_clouds must be positive");
    if (n_clouds > 65535) return fail("at most 65535 clouds per batch (got %d)", n_clouds);
    cs.raw = d_points;
    cs.n_clouds = n_clouds;
    cs.offsets.assign(h_offsets, h_offsets + n_clouds + 1);
    cs.n_total = h_offsets[n_clouds] - h_offsets[0];
    if (h_offsets[0] != 0) return fail("offsets[0] must be 0");
    if (cs.n_total >= (1LL << 31) - 1024) return fail("more than 2^31 points in one batch");
    cs.max_n = 0;
    std::vector<int>& off32 = cs.off32;
    off32.resize(n_clouds + 1);
    for (int i = 0; i <= n_clouds; ++i) {
        off32[i] = (int)h_offsets[i];
        if (i && h_offsets[i] < h_offsets[i - 1]) return fail("offsets must be non-decreasing");
        if (i) cs.max_n = std::max<int>(cs.max_n, (int)(h_offsets[i] - h_offsets[i - 1]));
    }
    if (cs.n_total > 0 && !d_points) return fail("null point array");
    CU(cs.d_offsets.ensure(off32.size() * sizeof(int)));
    // one small cloud (the reference's own calls): the single-block grid build takes the point count as an argument
    // and the 12-byte upload with its copy-engine hop disappears from the latency path
    cs.inline_n = (n_clouds == 1 && latency_path(h, h_offsets, 1)) ? (int)cs.n_total : -1;
    // no stream synchronisation here: a copy from pageable memory is staged by the driver before the call returns,
    // and the staging vector lives in the handle
    if (cs.inline_n < 0)
        CU(cudaMemcpyAsync(cs.d_offsets.p, off32.data(), off32.size() * sizeof(int), cudaMemcpyHostToDevice, st));

    const double h_knn = auto_knn_cell(h);
    const double h_nn = auto_nn_cell(h);
    // one grid for both stages when the k-NN cell suits the correspondence search: not larger than twice the search's
    // own choice (d_max / 2) and not smaller than d_max / 8 (a lane's ball then spans <= 17 cells per axis).  Measured
    // on the bench workload (k-NN cell 1.25 m, search cell 1.0 m): K3a 14.97 vs 15.16 ms per 512 pairs - no loss.
    cs.shared = h_knn <= 2.0 * h_nn && h_knn >= h->prm.max_distance_correspondence / 8.0 &&
                !(getenv("GICP_SHARED_GRID") && atoi(getenv("GICP_SHARED_GRID")) == 0);
    if (build_grid<D, Real>(h, cs, cs.knn, h_knn, st, sc)) return 1;
    CU(cs.cov_knn.ensure((size_t)std::max<int64_t>(cs.n_total, 1) * ns_of(D) * sizeof(Real)));

    // covariances; in sharded mode every rank computes an equal slice (k-NN grid order) of BOTH clouds
    // and the slices are all-gathered: the correspondence stage walks the clouds in a different
    // (1-NN grid) order, so every rank needs every covariance
    int slice_b = -1, slice_e = -1;
    const bool sharded = h->comm && n_clouds == 1;
    int64_t per = 0;
    if (sharded) {
        const int64_t n = cs.n_total;
        per = (n + h->n_ranks - 1) / h->n_ranks;   // equal-sized slices are required by ncclAllGather
        slice_b = (int)std::min<int64_t>(n, per * h->rank);
        slice_e = (int)std::min<int64_t>(n, per * (h->rank + 1));
        CU(cs.cov_knn.ensure((size_t)per * h->n_ranks * ns_of(D) * sizeof(Real)));
    }
    // covariance model (ICP family): GICP estimates both sides; point-to-point uses C_src = 0, C_tgt = I;
    // point-to-plane uses C_src = 0 and the estimated target covariances
    const int model = h->prm.covariance_model;
    const bool constant = (model == GICP_POINT_TO_POINT) || (model == GICP_POINT_TO_PLANE && which == GICP_SOURCE);
    if (constant) {
        const Real diag = (model == GICP_POINT_TO_POINT && which == GICP_TARGET) ? Real(1) : Real(0);
        const size_t n = (size_t)std::max<int64_t>(cs.n_total, 1);
        fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_knn.as<Real>(), n, diag);
        h->launches += 1;
    } else if (launch_knn<D, Real>(h, cs, nullptr, nullptr, st, slice_b, slice_e, sc)) return 1;
    if (sharded && !constant) {
        const size_t bytes = (size_t)per * ns_of(D) * sizeof(Real);
        char* basep = cs.cov_knn.as<char>();
        int rc = g_nccl.AllGather(basep + bytes * h->rank, basep, bytes, NCCL_INT8, h->comm, st);
        if (rc) return fail("ncclAllGather failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    }
    if (!cs.shared) {   // second ordering for the correspondence stage + the covariances carried over to it
        if (build_grid<D, Real>(h, cs, cs.nn, h_nn, st, sc)) return 1;
        CU(cs.cov_nn.ensure((size_t)std::max<int64_t>(cs.n_total, 1) * ns_of(D) * sizeof(Real)));
        if (cs.n_total > 0) {
            const int bx = (cs.max_n + 255) / 256;
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
    const size_t n = (size_t)std::max<int64_t>(cs.n_total, 1);
    fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_knn.as<Real>(), n, Real(0));
    if (!cs.shared) fill_cov_kernel<D, Real><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cs.cov_nn.as<Real>(), n, Real(0));
    h->launches += cs.shared ? 1 : 2;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int objective_args(gicpContext* h, ObjArgs<Real>& a, int& blocks_per_pair, bool allow_slice) {
    CloudSet &S = h->src, &T = h->tgt;
    if (!S.ready || !T.ready) return fail("set source and target first");
    if (S.n_clouds != T.n_clouds) return fail("source has %d clouds, target %d", S.n_clouds, T.n_clouds);
    a.src_meta = S.nng().meta.as<CloudMeta>();
    a.src_spts = S.nng().spts.as<PRec<Real>>();
    a.src_cov = S.covnn().as<Real>();
    a.tgt_meta = T.nng().meta.as<CloudMeta>();
    a.tgt_cell_start = T.nng().cell_start.as<int>();
    a.tgt_lut = T.nng().lut.as<int>();
    a.tgt_spts = T.nng().spts.as<PRec<Real>>();
    a.tgt_cov = T.covnn().as<Real>();
    a.tgt_inv_perm = T.nng().inv_perm.as<int>();
    a.match = nullptr;
    a.use_prev = 0;
    CU(h->state.ensure((size_t)S.n_clouds * sizeof(PairState)));
    a.state = h->state.as<PairState>();
    a.T_override = nullptr;
    a.d_max = h->prm.max_distance_correspondence;
    a.out_idx = nullptr;
    a.out_dist = nullptr;
    a.out_W = nullptr;
    a.slice_begin = a.slice_end = -1;
    a.ignore_status = 0;
    a.track_max_cells = getenv("GICP_TRACK_CELLS") ? atoi(getenv("GICP_TRACK_CELLS")) : 1 << 30;
    a.centre_first = getenv("GICP_CENTRE_FIRST") ? atoi(getenv("GICP_CENTRE_FIRST")) : 1;
    a.shell_search = getenv("GICP_SHELL_SEARCH") ? atoi(getenv("GICP_SHELL_SEARCH")) : 1;
    a.active_list = nullptr;
    a.n_list = nullptr;
    int span = S.max_n;
    if (allow_slice && h->comm && S.n_clouds == 1) {
        a.slice_begin = (int)(S.n_total * h->rank / h->n_ranks);
        a.slice_end = (int)(S.n_total * (h->rank + 1) / h->n_ranks);
        span = a.slice_end - a.slice_begin;
    }
    // enough blocks to fill the machine, as many points per thread as that allows (<= OBJ_MAX_PPT)
    const long long total_pts = (long long)std::max(span, 1) * S.n_clouds;
    int ppt = (int)(total_pts / (148LL * 8 * OBJ_THREADS));
    // the accumulation's software pipeline has a fill bubble per thread (match index -> gathered record): longer
    // per-thread runs amortise it when the batch is large enough.  Measured per 1024 pairs of the bench workload:
    // 16 / 32 / 64 points per thread -> 9.66 / 9.16 / 9.31 ms (GICP_ACC_PPT: A/B timing)
    const int ppt_cap = (getenv("GICP_ACC_PPT") && atoi(getenv("GICP_ACC_PPT")) > 0) ? atoi(getenv("GICP_ACC_PPT")) : 2 * OBJ_MAX_PPT;
    ppt = std::max(1, std::min(ppt_cap, ppt));
    a.ppt = ppt;
    blocks_per_pair = std::max(1, (span + OBJ_THREADS * ppt - 1) / (OBJ_THREADS * ppt));
    a.blocks_per_pair = blocks_per_pair;
    CU(h->partial.ensure((size_t)S.n_clouds * blocks_per_pair * Dim<D>::NRED * sizeof(double)));
    CU(h->red.ensure((size_t)S.n_clouds * Dim<D>::NRED * sizeof(double)));
    a.partial = h->partial.as<double>();
    CU(h->prev_match.ensure((size_t)std::max<int64_t>(S.n_total, 1) * sizeof(int)));
    a.match = h->prev_match.as<int>();
    CU(h->slack.ensure((size_t)std::max<int64_t>(S.n_total, 1) * sizeof(float)));
    a.slack = nullptr;
    return 0;
}

template <int D, typename Real>
int ensure_state(gicpContext* h, const double* h_T0, double* d_T, double* d_T_hist, int* d_n_outer,
                 int* d_converged, cudaStream_t st) {
    const int np = h->src.n_clouds;
    CU(h->state.ensure((size_t)np * sizeof(PairState)));
    CU(h->n_active.ensure(sizeof(int)));
    const double* d_T0 = nullptr;
    if (h_T0) {
        const size_t bytes = (size_t)np * (D + 1) * (D + 1) * sizeof(double);
        CU(h->T_dev.ensure(bytes));
        CU(cudaMemcpyAsync(h->T_dev.p, h_T0, bytes, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
        d_T0 = h->T_dev.as<double>();
    }
    init_state_kernel<D><<<(np + 127) / 128, 128, 0, st>>>(h->state.as<PairState>(), d_T0, h->tgt.knn.bbox.as<double>(), np,
                                                           d_T, d_T_hist, h->prm.max_iterations, d_n_outer, d_converged,
                                                           h->n_active.as<int>());
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_register(gicpContext* h, const double* h_T0, double* d_T, int* d_n_outer, int* d_converged,
                double* d_loss_hist, double* d_T_hist, int* d_inliers, cudaStream_t st) {
    ObjArgs<Real> oa;
    int bpp = 1;
    if (objective_args<D, Real>(h, oa, bpp, true)) return 1;
    const int np = h->src.n_clouds;
    h->last_stream = st;
    // Small pairs (every source cloud fits one block): the whole outer loop in one launch (fused.cuh).  Not with a
    // communicator (the all-reduce sits between the stages) and not while per-stage timing is on.
    const bool fused = !(h->comm && np == 1) && !h->prof_on && h->src.max_n <= OBJ_THREADS * OBJ_MAX_PPT &&
                       !(getenv("GICP_FUSED_LOOP") && atoi(getenv("GICP_FUSED_LOOP")) == 0);
    // without a start transform the fused loop initialises its pair itself (state, match and slack arrays)
    const bool self_init = fused && !h_T0;
    if (self_init) {
        CU(h->state.ensure((size_t)np * sizeof(PairState)));
    } else {
        if (ensure_state<D, Real>(h, h_T0, d_T, d_T_hist, d_n_outer, d_converged, st)) return 1;
        // last iteration's match per source point (bounds the next search); -1 = none yet
        CU(cudaMemsetAsync(h->prev_match.p, 0xFF, (size_t)std::max<int64_t>(h->src.n_total, 1) * sizeof(int), st));
        CU(cudaMemsetAsync(h->slack.p, 0, (size_t)std::max<int64_t>(h->src.n_total, 1) * sizeof(float), st));
    }
    oa.use_prev = 1;
    oa.slack = (getenv("GICP_NO_SKIP") && atoi(getenv("GICP_NO_SKIP"))) ? nullptr : h->slack.as<float>();
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
    if (fused) {
        oa.ppt = std::max(1, (h->src.max_n + OBJ_THREADS - 1) / OBJ_THREADS);
        oa.blocks_per_pair = 1;
        sa.blocks_per_pair = 1;
        sa.n_active = nullptr;   // nobody polls
        const size_t smem = obj_smem(oa.ppt);
        CU(cudaFuncSetAttribute(register_loop_kernel<D, Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ProfScope prof(h, GICP_STAGE_CORRESPOND, st);
        register_loop_kernel<D, Real><<<np, OBJ_THREADS, smem, st>>>(oa, sa,
                                                                     self_init ? h->tgt.knn.bbox.as<double>() : nullptr);
        h->launches += 1;
        CU(cudaGetLastError());
        return 0;
    }
    const dim3 ogrid(bpp, np);
    // thousands of block partials per pair (one large pair): fold them 64 to 1 before the one-warp sum of K4
    const bool presum = bpp > 2 * PRESUM_SPAN;
    const int bpp2 = (bpp + PRESUM_SPAN - 1) / PRESUM_SPAN;
    if (presum) {
        CU(h->partial2.ensure((size_t)np * bpp2 * Dim<D>::NRED * sizeof(double)));
        sa.partial = h->partial2.as<double>();
        sa.blocks_per_pair = bpp2;
    }
    // the search runs on smaller blocks than the accumulation (its work per point is uneven: better balance and
    // a shorter tail), the accumulation keeps the longer per-thread pipeline
    ObjArgs<Real> oc = oa;
    {
        int split = getenv("GICP_CORR_SPLIT") ? atoi(getenv("GICP_CORR_SPLIT")) : 2;
        while (oa.ppt / split > OBJ_MAX_PPT / 2) split *= 2;   // the search keeps blocks of <= 8 points per thread
        while (split > 1 && oa.ppt % split) --split;
        oc.ppt = oa.ppt / std::max(split, 1);
    }
    const dim3 cgrid(bpp * (oa.ppt / oc.ppt), np);
    const int sgrid = (np + SOLVE_WARPS - 1) / SOLVE_WARPS;
    const bool sharded = h->comm && np == 1;
    // Progress polls (4 bytes each, the only host<->device traffic inside the loop).  A single-process registration
    // does not wait for them: the count of still-active pairs is copied to pinned memory after every iteration and
    // looked at (cudaEventQuery) before later iterations are launched, so the host runs a few iterations ahead and the
    // GPU never idles on a round trip; an iteration launched after everything converged is a no-op (every block
    // returns on the pair's status).  With a communicator every rank must issue the same all-reduces, so the sharded
    // mode keeps a blocking poll on a fixed schedule (all ranks see the same count: they solve bit-identical forms).
    constexpr int LOOK = 3;
    int issued = 0, checked = 0;
    // Large batches: after every iteration the still-active pairs are compacted into a list (one small block), and
    // the next launches cover only `known_active` slots of it - the latest polled count, an upper bound of the list's
    // length since the count only falls.  Without it every launch of the convergence tail starts tens of thousands
    // of blocks that return at once (4096 pairs: 131 k blocks per search launch).
    const bool use_list = !sharded && np >= 64 && !(getenv("GICP_ACTIVE_LIST") && atoi(getenv("GICP_ACTIVE_LIST")) == 0);
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
            correspond_kernel<D, Real><<<dim3(cgrid.x, gy), OBJ_THREADS, obj_smem(oc.ppt), st>>>(oc);
        }
        {
            ProfScope prof(h, GICP_STAGE_ACCUMULATE, st);
            accumulate_kernel<D, Real><<<dim3(ogrid.x, gy), OBJ_THREADS, 0, st>>>(oa);
        }
        {
            ProfScope prof(h, GICP_STAGE_SOLVE, st);
            if (presum) {
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
        if (!sharded || (it + 1) % 2 == 0) {
            const int slot = issued % gicpContext::NPOLL;
            CU(cudaMemcpyAsync(h->h_poll + slot, h->n_active.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(h->poll_ev[slot], st));
            ++issued;
        }
    }
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_stage(gicpContext* h, const double* h_T, int* d_idx, double* d_dist, double* d_W, double* h_out,
             cudaStream_t st) {
    ObjArgs<Real> oa;
    int bpp = 1;
    if (objective_args<D, Real>(h, oa, bpp, false)) return 1;
    const int np = h->src.n_clouds;
    if (!h_T) return fail("h_T is required");
    if (ensure_state<D, Real>(h, nullptr, nullptr, nullptr, nullptr, nullptr, st)) return 1;
    const size_t bytes = (size_t)np * (D + 1) * (D + 1) * sizeof(double);
    CU(h->T_dev.ensure(bytes));
    CU(cudaMemcpyAsync(h->T_dev.p, h_T, bytes, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    oa.T_override = h->T_dev.as<double>();
    oa.out_idx = d_idx;
    oa.out_dist = d_dist;
    oa.out_W = d_W;
    oa.ignore_status = 1;
    // stage entry points always cover the whole source (no slicing), so their outputs are complete
    correspond_kernel<D, Real><<<dim3(bpp, np), OBJ_THREADS, obj_smem(oa.ppt), st>>>(oa);
    if (d_W || h_out) accumulate_kernel<D, Real><<<dim3(bpp, np), OBJ_THREADS, 0, st>>>(oa);
    h->launches += 2;
    if (h_out) {
        SolveArgs sa;
        memset(&sa, 0, sizeof sa);
        sa.partial = h->partial.as<double>();
        sa.blocks_per_pair = bpp;
        sa.n_pairs = np;
        sa.sum_out = h->red.as<double>();
        sa.state = h->state.as<PairState>();
        solve_kernel<D><<<(np + SOLVE_WARPS - 1) / SOLVE_WARPS, SOLVE_WARPS * 32, 0, st>>>(sa);
        h->launches += 1;
        CU(cudaMemcpyAsync(h_out, h->red.p, (size_t)np * Dim<D>::NRED * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_knn(gicpContext* h, int which, int* d_idx, double* d_dist, cudaStream_t st) {
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    if (!cs.ready) return fail("cloud not set");
    // re-runs K2 with the index outputs enabled (covariances are rewritten with identical values)
    return launch_knn<D, Real>(h, cs, d_idx, d_dist, st, -1, -1, h->scr[0]);
}

template <int D, typename Real>
int do_cov(gicpContext* h, int which, double* d_cov, cudaStream_t st) {
    CloudSet& cs = which == GICP_TARGET ? h->tgt : h->src;
    if (!cs.ready) return fail("cloud not set");
    if (cs.n_total == 0) return 0;
    const int bx = (cs.max_n + 255) / 256;
    export_cov_kernel<D, Real><<<dim3(bx, cs.n_clouds), 256, 0, st>>>(cs.knn.meta.as<CloudMeta>(),
                                                                      cs.knn.spts.as<PRec<Real>>(),
                                                                      cs.cov_knn.as<Real>(), d_cov);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

template <int D, typename Real>
int do_rotcov(gicpContext* h, const double* h_T, int n_T, double* d_out, cudaStream_t st) {
    CloudSet& cs = h->src;
    if (!cs.ready) return fail("source not set");
    if (n_T <= 0 || cs.n_total == 0) return 0;
    if (n_T > 65535) return fail("n_T too large");
    const size_t bytes = (size_t)n_T * cs.n_clouds * (D + 1) * (D + 1) * sizeof(double);
    CU(h->T_dev.ensure(bytes));
    CU(cudaMemcpyAsync(h->T_dev.p, h_T, bytes, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    const int bx = (cs.max_n + 255) / 256;
    rotated_cov_kernel<D, Real><<<dim3(bx, cs.n_clouds, n_T), 256, 0, st>>>(
        cs.knn.meta.as<CloudMeta>(), cs.knn.spts.as<PRec<Real>>(), cs.cov_knn.as<Real>(), h->T_dev.as<double>(),
        cs.n_clouds, (size_t)cs.n_total, d_out);
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
template <int D, typename Real>
int do_voxel(gicpContext* h, const void* d_points, const int64_t* h_off, int nc, double leaf, int min_points,
             void* d_out, int64_t* h_out_off, int* d_voxel_of, int* d_counts, cudaStream_t st) {
    VoxelScratch& v = h->vox;
    if (nc <= 0 || nc > 65535) return fail("n_clouds must be in [1, 65535] (got %d)", nc);
    if (h_off[0] != 0) return fail("offsets[0] must be 0");
    int max_n = 0;
    for (int i = 1; i <= nc; ++i) {
        if (h_off[i] < h_off[i - 1]) return fail("offsets must be non-decreasing");
        if (h_off[i] >= (1LL << 31) - 1024) return fail("more than 2^31 points in one batch");
        max_n = std::max<int>(max_n, (int)(h_off[i] - h_off[i - 1]));
    }
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
    voxel_centroid_kernel<D, Real><<<nb, 256, 0, st>>>(oa, pts, static_cast<Real*>(d_out));
    const int big_blocks = std::max(1, std::min(n / (VOX_SEQ_MAX + 1), 148 * 8));
    voxel_centroid_block_kernel<D, Real><<<big_blocks, VOX_THREADS, 0, st>>>(oa, pts, static_cast<Real*>(d_out));
    h->launches += 2;
    CU(cudaMemcpyAsync(v.h_out_off, v.out_off.p, (size_t)(nc + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    for (int i = 0; i <= nc; ++i) h_out_off[i] = v.h_out_off[i];
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
int gicpVersion(void) { return 101; }

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
    for (SetupScratch& sc : h->scr) sc.release();
    h->vox.release();
    DevBuf* bufs[] = {&h->state, &h->partial, &h->partial2, &h->red, &h->T_dev, &h->n_active, &h->prev_match, &h->slack,
                      &h->active_list};
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
    h->prm = *p;
    if (h->prm.inner_max_iterations <= 0) h->prm.inner_max_iterations = 50;
    h->src.ready = false;
    h->tgt.ready = false;
    return 0;
}

int gicpSetTarget(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_offsets) return fail("null offsets");
    return DISPATCH(h, set_cloud, h, GICP_TARGET, d_points, h_offsets, n_clouds, (cudaStream_t)stream, 0);
}

int gicpSetSource(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_offsets) return fail("null offsets");
    return DISPATCH(h, set_cloud, h, GICP_SOURCE, d_points, h_offsets, n_clouds, (cudaStream_t)stream, 0);
}

int gicpSetPair(gicpHandle h, const void* d_target, const int64_t* h_target_offsets, const void* d_source,
                const int64_t* h_source_offsets, int32_t n_clouds, void* stream) {
    if (check(h)) return 1;
    if (!h_target_offsets || !h_source_offsets) return fail("null offsets");
    cudaStream_t st = (cudaStream_t)stream;
    // Side by side while one side alone cannot fill the GPU: the single-block set-ups of small clouds, and up to ~1 M
    // points per side (a 100k cloud's k-NN is one partial wave of blocks whose duration is its slowest chunk).  Each
    // side has its own scratch (scr[0] / scr[1]).  Larger sides saturate the device on their own: sequential.
    if (n_clouds <= 0) return fail("n_clouds must be positive");
    const int64_t side_max = getenv("GICP_PAIR_OVERLAP_MAX") ? atoll(getenv("GICP_PAIR_OVERLAP_MAX")) : (1LL << 20);
    const bool concurrent = !h->comm && !h->prof_on && h_target_offsets[n_clouds] <= side_max &&
                            h_source_offsets[n_clouds] <= side_max;
    if (!concurrent) {
        if (DISPATCH(h, set_cloud, h, GICP_TARGET, d_target, h_target_offsets, n_clouds, st, 0)) return 1;
        return DISPATCH(h, set_cloud, h, GICP_SOURCE, d_source, h_source_offsets, n_clouds, st, 0);
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
    const int rc_t = DISPATCH(h, set_cloud, h, GICP_TARGET, d_target, h_target_offsets, n_clouds, st, 0);
    const int rc_s = rc_t ? 1 : DISPATCH(h, set_cloud, h, GICP_SOURCE, d_source, h_source_offsets, n_clouds, h->side_stream, 1);
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
    if (h->prm.covariance_model != GICP_PLANE_TO_PLANE) return DISPATCH(h, zero_source_cov, h, h->last_stream);
    return 0;
}

int gicpRegister(gicpHandle h, const double* h_T0, double* d_T, int32_t* d_n_outer, int32_t* d_converged,
                 double* d_loss_hist, double* d_T_hist, int32_t* d_inliers, void* stream) {
    if (check(h)) return 1;
    if (!d_T || !d_n_outer || !d_converged) return fail("d_T, d_n_outer and d_converged are required");
    return DISPATCH(h, do_register, h, h_T0, d_T, d_n_outer, d_converged, d_loss_hist, d_T_hist, d_inliers,
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
    return DISPATCH(h, do_stage, h, h_T, d_idx, d_dist, d_W, (double*)nullptr, (cudaStream_t)stream);
}

int gicpNormalEquations(gicpHandle h, const double* h_T, double* h_out, void* stream) {
    if (check(h)) return 1;
    if (!h_out) return fail("h_out is required");
    return DISPATCH(h, do_stage, h, h_T, (int*)nullptr, (double*)nullptr, (double*)nullptr, h_out,
                    (cudaStream_t)stream);
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

int gicpProfileRead(gicpHandle h, double ms_out[GICP_N_STAGES], int64_t count_out[GICP_N_STAGES]) {
    if (check(h)) return 1;
    CU(cudaDeviceSynchronize());
    for (int i = 0; i < GICP_N_STAGES; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
    for (auto& r : h->prof_recs) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, r.a, r.b));
        ms_out[r.stage] += ms;
        count_out[r.stage] += 1;
    }
    h->prof_recs.clear();
    h->ev_used = 0;
    return 0;
}

}  // extern "C"

