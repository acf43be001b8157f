// Test infrastructure (not part of the product library): the host-side plans of generalized-icp_b200/csrc/plan.h
// compiled for the HOST behind a flat C interface, so that tests/test_plan_host.py can check every path decision
// on batch shapes the GPU suite cannot afford.
#include "../../generalized-icp_b200/csrc/plan.h"

using namespace gicp;

extern "C" {

struct FlatSwitches {
    int no_skip, track_max_cells, shell_search, centre_first, corr_split, active_list, fused_loop, small_grid, knn_brute;
    long long pair_overlap_max;
};

struct FlatSetup {
    int error, n_clouds, max_n;
    long long n_total;
    double knn_cell, nn_cell;
    int shared;
    long long budget;
    int single_block, inline_n, cov, knn, knn_whole, kc, sharded, slice_begin, slice_end;
    long long slice_len;
};

struct FlatLoop {
    int slice_begin, slice_end, acc_ppt, bpp, search_ppt, search_bpp, fused, self_init, fused_ppt, presum, bpp2,
        active_list, sharded, poll_every;
};

static Switches unflat(const FlatSwitches& f) {
    Switches s;
    s.no_skip = f.no_skip != 0;
    s.track_max_cells = f.track_max_cells;
    s.shell_search = f.shell_search;
    s.centre_first = f.centre_first;
    s.corr_split = f.corr_split;
    s.active_list = f.active_list != 0;
    s.fused_loop = f.fused_loop != 0;
    s.small_grid = f.small_grid != 0;
    s.knn_brute = f.knn_brute != 0;
    s.pair_overlap_max = f.pair_overlap_max;
    return s;
}

static void flat(const SetupPlan& p, FlatSetup* o) {
    *o = FlatSetup{p.error != nullptr, p.n_clouds, p.max_n, (long long)p.n_total, p.knn_cell, p.nn_cell, p.shared,
                   p.budget, p.single_block, p.inline_n, (int)p.cov, (int)p.knn, (int)p.knn_whole, p.kc, p.sharded,
                   p.slice_begin, p.slice_end, (long long)p.slice_len};
}

void gicp_test_read_switches(FlatSwitches* o) {
    const Switches s = read_switches();
    *o = FlatSwitches{s.no_skip, s.track_max_cells, s.shell_search, s.centre_first, s.corr_split, s.active_list,
                      s.fused_loop, s.small_grid, s.knn_brute, (long long)s.pair_overlap_max};
}

// cov: 0 Zero, 1 Identity, 2 Knn; knn: 0 Brute, 1 General, 2 HistGeneral (the enum orders of plan.h)
void gicp_test_plan_setup(const gicpParams* prm, const FlatSwitches* sw, const int64_t* off, int n_clouds, int which,
                          int f32, int comm, int n_ranks, int rank, FlatSetup* out) {
    flat(plan_setup(*prm, unflat(*sw), off, n_clouds, which, f32 != 0, Ranks{comm != 0, n_ranks, rank}), out);
}

void gicp_test_plan_loop(const gicpParams* prm, const FlatSwitches* sw, const int64_t* off, int n_clouds, int comm,
                         int n_ranks, int rank, int sliced, int prof_on, int has_T0, FlatLoop* out) {
    const Switches s = unflat(*sw);
    const Ranks ranks{comm != 0, n_ranks, rank};
    const SetupPlan src = plan_setup(*prm, s, off, n_clouds, GICP_SOURCE, false, ranks);
    const LoopPlan p = plan_loop(s, src, sliced != 0, ranks, prof_on != 0, has_T0 != 0);
    *out = FlatLoop{p.slice_begin, p.slice_end, p.acc_ppt, p.bpp, p.search_ppt, p.search_bpp, p.fused, p.self_init,
                    p.fused_ppt, p.presum, p.bpp2, p.active_list, p.sharded, p.poll_every};
}

// the loop a registration of one batch takes with a robust kernel (robust) and an adaptive scale (adaptive):
// out = {fused, robust, adaptive, presum}
void gicp_test_plan_loop_kernel(const gicpParams* prm, const FlatSwitches* sw, const int64_t* off, int n_clouds,
                                int robust, int adaptive, int* out) {
    const Switches s = unflat(*sw);
    const Ranks ranks{false, 1, 0};
    const SetupPlan src = plan_setup(*prm, s, off, n_clouds, GICP_SOURCE, false, ranks);
    const LoopPlan p = plan_loop(s, src, true, ranks, false, false, robust != 0, adaptive != 0);
    out[0] = p.fused;
    out[1] = p.robust;
    out[2] = p.adaptive;
    out[3] = p.presum;
}

int gicp_test_pair_overlap(const FlatSwitches* sw, int comm, int prof_on, long long n_target, long long n_source) {
    return pair_overlap(unflat(*sw), Ranks{comm != 0, 1, 0}, prof_on != 0, n_target, n_source);
}

}  // extern "C"
