// kruskal_twin.cpp -- TEST-ONLY host build of splicedice_b200/csrc/sd_kruskal_math.cuh.
// Lets the CPU test-suite check the kernel's Kruskal-Wallis arithmetic against exact oracles without
// a GPU.  Not part of the product: nothing under splicedice_b200/ loads it.
#include <stdint.h>

#include "../../splicedice_b200/csrc/sd_kruskal_math.cuh"

// H of `rows` rows of k groups each: d / n_g [rows, k], n / t [rows]
extern "C" void kruskal_twin_h(int64_t rows, int32_t k, const int64_t *d, const int64_t *n_g, const int64_t *n,
                               const int64_t *t, double *out)
{
    for (int64_t r = 0; r < rows; ++r) {
        double s = 0.0;
        for (int32_t g = 0; g < k; ++g) s += sd::kruskal::group_term(d[r * k + g], n_g[r * k + g]);
        out[r] = sd::kruskal::h_stat(s, n[r], t[r]);
    }
}

extern "C" void kruskal_twin_sf(int64_t count, const int32_t *df, const double *h, double *out)
{
    for (int64_t i = 0; i < count; ++i) out[i] = sd::kruskal::chi2_sf(df[i], h[i]);
}
