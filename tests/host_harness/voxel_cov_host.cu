// Test infrastructure (not part of the product library): the per-voxel finish of gicpSetVoxelized (moments ->
// regularised covariance, generalized-icp_b200/csrc/voxel.cuh vox_cov_finish) and the voxelized set-up plan
// (generalized-icp_b200/csrc/plan.h plan_setup_voxelized) compiled for the HOST behind a flat C interface, so that
// tests/test_voxel_dist_host.py can check them without a GPU.
#include "../../generalized-icp_b200/csrc/plan.h"
#include "../../generalized-icp_b200/csrc/voxel.cuh"

using namespace gicp;

extern "C" {

// The device's per-voxel arithmetic on n points (row-major (n, dim)): the moments about the first point accumulated
// in row order, as voxel_centroid_kernel does, then vox_cov_finish.  C: dim*(dim+1)/2 entries (packed upper triangle).
int gicp_test_voxel_cov(int dim, const double* pts, int n, double lam_t, double lam_n, double* C) {
    double sd[3] = {0.0, 0.0, 0.0}, sq[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int r = 1; r < n; ++r) {
        double d[3];
        for (int c = 0; c < dim; ++c) {
            d[c] = pts[r * dim + c] - pts[c];
            sd[c] += d[c];
        }
        for (int i = 0, k = 0; i < dim; ++i)
            for (int j = i; j < dim; ++j, ++k) sq[k] += d[i] * d[j];
    }
    if (dim == 2) vox_cov_finish<2>(n, sd, sq, lam_t, lam_n, C);
    else vox_cov_finish<3>(n, sd, sq, lam_t, lam_n, C);
    return 0;
}

// The voxelized plan of a batch and, beside it, the raw plan of the same points: out = {error, cov, knn, knn_whole,
// shared, grid sizing equal to the raw plan's, raw cov, raw shared}; knn_cell = the voxelized side's one grid cell,
// raw_search_cell = the cell a raw side searches.  cov: 0 Zero, 1 Identity, 2 Knn, 3 Voxel; knn: 0 Brute, 1 General, 2 HistGeneral, 3 None (the enum orders of plan.h)
void gicp_test_plan_voxelized(const gicpParams* prm, const int64_t* off, int n_clouds, int which, int f32,
                              double* knn_cell, double* raw_search_cell, long long* out) {
    const Switches sw;
    const SetupPlan p = plan_setup_voxelized(*prm, sw, off, n_clouds, which, f32 != 0);
    const SetupPlan raw = plan_setup(*prm, sw, off, n_clouds, which, f32 != 0, Ranks{});
    out[0] = p.error != nullptr;
    out[1] = (int)p.cov;
    out[2] = (int)p.knn;
    out[3] = (int)p.knn_whole;
    out[4] = p.shared;
    out[5] = p.single_block == raw.single_block && p.budget == raw.budget && p.inline_n == raw.inline_n;
    out[6] = (int)raw.cov;
    out[7] = raw.shared;
    *knn_cell = p.knn_cell;
    *raw_search_cell = raw.shared ? raw.knn_cell : raw.nn_cell;   // the cell of CloudSet::nng() of a raw side
}

}  // extern "C"
