// Test infrastructure (not part of the product library): the robust kernel weight of K3b / the fused loop,
// generalized-icp_b200/csrc/objective.cuh, compiled for the HOST, so that tests/test_robust_host.py can compare it bit
// for bit with the float64 formulas of tests/robust_oracle.py.
#include "../../generalized-icp_b200/csrc/objective.cuh"

extern "C" void gicp_test_robust_weight(long long n, int kind, const double* d, const double* c, double* w) {
    for (long long i = 0; i < n; ++i) w[i] = gicp::robust_weight(kind, d[i], c[i]);
}
