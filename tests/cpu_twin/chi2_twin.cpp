// chi2_twin.cpp -- TEST-ONLY host build of splicedice_b200/csrc/sd_chi2_math.cuh.
// Lets the CPU test-suite check the kernel's per-table chi-squared arithmetic against scipy and
// mpmath without a GPU.  Not part of the product: nothing under splicedice_b200/ loads it.
#include <stdint.h>

#include "../../splicedice_b200/csrc/sd_chi2_math.cuh"

extern "C" void chi2_twin_batch(int64_t count, const int64_t *a, const int64_t *b, const int64_t *c, const int64_t *d,
                                double *out, int32_t *status)
{
    for (int64_t i = 0; i < count; ++i) {
        int s = 0;
        out[i] = sd::chi2::yates_p(a[i], b[i], c[i], d[i], &s);
        status[i] = s;
    }
}
