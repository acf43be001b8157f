// Test infrastructure (not part of the product library): the adaptive robust scale of the select (scale.cuh),
// generalized-icp_b200/csrc/objective.cuh, compiled for the HOST, so that tests/test_adaptive_host.py can compare it bit
// for bit with the float64 formula of tests/adaptive_oracle.py.
#include "../../generalized-icp_b200/csrc/objective.cuh"

extern "C" void gicp_test_adaptive_scale(long long n, const double* kappa, const double* m, const double* min_scale,
                                         double* c) {
    for (long long i = 0; i < n; ++i) c[i] = gicp::adaptive_scale(kappa[i], m[i], min_scale[i]);
}
