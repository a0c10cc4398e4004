// sd_friedman_math.cuh -- per-row arithmetic of the Friedman test (K9, sd_friedman.cu).
//
// Exact statistic.  In a complete block (one subject's k cells, none NaN) a cell with lo cells of the
// block below it and hi cells at or below it has twice its average rank within the block = lo + hi + 1.
// Over the n complete blocks, per condition c
//     D_c = sum_b (lo + hi + 1) - n (k + 1) = 2 R_c - n (k + 1)
// is an exact integer (sum_c D_c = 0), and so is the tie term
//     T = sum over cells of ((hi - lo)^2 - 1) = sum over the blocks' tie runs of (t^3 - t).
// Then
//     Q = 3 (k - 1) * sum_c D_c^2 / (n (k^3 - k) - T),
// which is scipy.stats.friedmanchisquare's (12 / (n k (k + 1)) sum_c R_c^2 - 3 n (k + 1)) /
// (1 - T / (n k (k^2 - 1))) rewritten without its cancellation.  With 3 <= k <= 256 and n k <= 16,384
// the numerator is below 2^46 and the denominator below 2^31, so both convert to binary64 exactly and Q
// is one correctly rounded division: bit-identical to the exact fraction rounded to the nearest double.
// Q >= 0 always, and Q == 0 exactly when every D_c is 0.  n == 0 (no complete block) or every complete
// block tied throughout (the denominator 0) leaves Q undefined (NaN).
//
// p = chi2.sf(Q, k - 1) is sd::kruskal::chi2_sf of sd_kruskal_math.cuh, unchanged (df <= 255).
//
// The header compiles for the device (sd_friedman.cu) and, without nvcc, for the host: the host build
// exists only so tests/ can check this arithmetic on machines with no GPU.
#pragma once

#include <math.h>
#include <stdint.h>

#include "sd_kruskal_math.cuh"

#ifdef __CUDACC__
#define SD_FR_HD __host__ __device__ __forceinline__
#else
#define SD_FR_HD inline
#endif

namespace sd {
namespace friedman {

// Q from sum_c D_c^2, the complete-block count n, the condition count k and the tie term T; NaN when
// n == 0 or every complete block is tied throughout
SD_FR_HD double q_stat(int64_t sum_d2, int64_t n, int64_t k, int64_t t)
{
    const int64_t den = n * (k * k * k - k) - t;
    if (n <= 0 || den <= 0) return __builtin_nan("");
    return (double)(3 * (k - 1) * sum_d2) / (double)den;
}

// p = chi2.sf(Q, k - 1); NaN for NaN Q, 1 for Q == 0
SD_FR_HD double p_value(int64_t k, double q) { return sd::kruskal::chi2_sf((int)(k - 1), q); }

}  // namespace friedman
}  // namespace sd
