// Test infrastructure (not part of the product library): the warp-cooperative 3-D inner solver of
// generalized-icp_b200/csrc/solve.cuh compiled for the HOST, so that tests/test_solve3_host.py can check its minimiser
// without a GPU.  Its 32 lanes run as 32 threads over one SolveScratch<3>; the solver's warp barrier is a
// pthread barrier of 32.  Built by the test with nvcc into a temporary directory.
#include <pthread.h>

#include <thread>
#include <vector>

#include "../../generalized-icp_b200/csrc/solve.cuh"

static pthread_barrier_t g_barrier;
static void host_barrier() { pthread_barrier_wait(&g_barrier); }
void (*gicp::g_host_warp_sync)() = host_barrier;

// red: the 80-double reduced form of one pair (include/gicp_b200.h layout).  Hd is expanded exactly as solve_pair
// does, then inner_solve_warp<3> runs with max_it LM iterations.  out: dt[3], dR[3][3] row-major, dtheta, f.
extern "C" int gicp_test_solve3d(const double* red, int max_it, double* out) {
    using DD = gicp::Dim<3>;
    constexpr int DN2 = gicp::SolveScratch<3>::DN * gicp::SolveScratch<3>::DN;
    gicp::SolveScratch<3> sc;
    for (int e = 0; e < DN2; ++e) sc.Hd[e] = gicp::dense_H_entry<3>(red, e);
    pthread_barrier_init(&g_barrier, nullptr, 32);
    std::vector<std::thread> lanes;
    for (int lane = 0; lane < 32; ++lane)
        lanes.emplace_back([&, lane] { gicp::inner_solve_warp<3>(sc, red + DD::NH, red[DD::NQ], max_it, lane); });
    for (auto& t : lanes) t.join();
    pthread_barrier_destroy(&g_barrier);
    for (int i = 0; i < 3; ++i) {
        out[i] = sc.dt[i];
        for (int j = 0; j < 3; ++j) out[3 + 3 * i + j] = sc.dR[i][j];
    }
    out[12] = sc.dtheta;
    out[13] = sc.f;
    return 0;
}
