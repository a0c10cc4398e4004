// friedman_twin.cpp -- TEST-ONLY host build of splicedice_b200/csrc/sd_friedman_math.cuh.
// Lets the CPU test-suite check the kernel's Friedman arithmetic against exact oracles without a GPU.
// Not part of the product: nothing under splicedice_b200/ loads it.
#include <stdint.h>

#include "../../splicedice_b200/csrc/sd_friedman_math.cuh"

// Q and p of `rows` rows: sum_c D_c^2, n, k and T per row
extern "C" void friedman_twin(int64_t rows, const int64_t *sum_d2, const int64_t *n, const int64_t *k,
                              const int64_t *t, double *q, double *p)
{
    for (int64_t r = 0; r < rows; ++r) {
        q[r] = sd::friedman::q_stat(sum_d2[r], n[r], k[r], t[r]);
        p[r] = sd::friedman::p_value(k[r], q[r]);
    }
}
