// Test infrastructure (not part of the product library): plan_pairs of generalized-icp_b200/csrc/plan.h compiled for
// the HOST behind a flat C interface, so that tests/test_pair_list_host.py can check the validation, the offsets and
// the loop plan of a pair list against the one-to-one batch it stands for.
#include <cstring>

#include "../../generalized-icp_b200/csrc/plan.h"

using namespace gicp;

extern "C" {

struct FlatLoop {
    int slice_begin, slice_end, acc_ppt, bpp, search_ppt, search_bpp, fused, self_init, fused_ppt, presum, bpp2,
        active_list, sharded, poll_every, robust, adaptive;
};

static void flat(const LoopPlan& p, FlatLoop* o) {
    *o = FlatLoop{p.slice_begin, p.slice_end, p.acc_ppt, p.bpp, p.search_ppt, p.search_bpp, p.fused, p.self_init,
                  p.fused_ppt, p.presum, p.bpp2, p.active_list, p.sharded, p.poll_every, p.robust, p.adaptive};
}

// src_off / tgt_off: NULL for a side that is not set up.  Returns 0 with the offsets (n_pairs + 1), the view
// (n_clouds, max_n, n_total) and the loop plan of the pair list, or 1 with the refusal's message in err.
int gicp_test_plan_pairs(int n_pairs, const int32_t* src_cloud, const int32_t* tgt_cloud, int source_set,
                         const int64_t* src_off, int n_src, const int64_t* tgt_off, int n_tgt, int comm, int has_T0,
                         int robust, int adaptive, int64_t* offsets, long long* view, FlatLoop* loop, char* err,
                         int err_len) {
    const PairPlan pp = plan_pairs(n_pairs, src_cloud, tgt_cloud, source_set, SetSizes{src_off, n_src},
                                   SetSizes{tgt_off, n_tgt}, comm != 0);
    if (pp.error) {
        strncpy(err, pp.error, err_len - 1);
        err[err_len - 1] = 0;
        return 1;
    }
    for (size_t i = 0; i < pp.offsets.size(); ++i) offsets[i] = pp.offsets[i];
    view[0] = pp.view.n_clouds;
    view[1] = pp.view.max_n;
    view[2] = pp.view.n_total;
    flat(plan_loop(Switches{}, pp.view, true, Ranks{}, false, has_T0 != 0, robust != 0, adaptive != 0), loop);
    return 0;
}

// the loop plan of the one-to-one batch whose sources have the offsets `off` (set up as gicpSetSource does)
void gicp_test_plan_loop_batch(const gicpParams* prm, const int64_t* off, int n_clouds, int f32, int has_T0, int robust,
                               int adaptive, FlatLoop* out) {
    const SetupPlan src = plan_setup(*prm, Switches{}, off, n_clouds, GICP_SOURCE, f32 != 0, Ranks{});
    flat(plan_loop(Switches{}, src, true, Ranks{}, false, has_T0 != 0, robust != 0, adaptive != 0), out);
}

}  // extern "C"
