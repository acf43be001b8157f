// Test infrastructure (not part of the product library): the map of gicpEvaluate from a pair's reduced form to its
// quality row, H and b, generalized-icp_b200/csrc/quality.cuh, compiled for the HOST, so that
// tests/test_quality_host.py can compare it with the float64 restatement of tests/quality_oracle.py.
#include "../../generalized-icp_b200/csrc/quality.cuh"

extern "C" void gicp_test_quality(int dim, long long n_pairs, const double* red, const double* sum_d2, const int* n_src,
                                  double* q, double* H, double* b) {
    for (long long p = 0; p < n_pairs; ++p) {
        if (dim == 3)
            gicp::quality_from_reduced<3>(red + p * 80, sum_d2[p], n_src[p], q + p * 4, H + p * 36, b + p * 6);
        else
            gicp::quality_from_reduced<2>(red + p * 32, sum_d2[p], n_src[p], q + p * 4, H + p * 9, b + p * 3);
    }
}
