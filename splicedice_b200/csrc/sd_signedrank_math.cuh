// sd_signedrank_math.cuh -- per-row arithmetic of the Wilcoxon signed-rank test (K8, sd_signedrank.cu).
//
// Inputs per row: n (pairs with both cells defined), zeros (d == 0), c (nonzero, non-NaN d; inf - inf
// gives NaN and counts in n only), 2 R+ = sum of the doubled ranks lo + hi + 1 over d > 0 and the tie
// term T = sum over runs of (t^3 - t), all exact integers.  The doubled ranks of all c differences sum
// to c (c + 1).
//
// Method switch (scipy 1.18.1's method='auto'): the exact null distribution when n <= 50 without ties
// or zeros, else the sign-flip permutation test when n <= 13 (exhaustive, so deterministic), else the
// normal approximation.  The first two are one computation: over the 2^c sign patterns of the c doubled
// ranks, count the patterns whose 2 R+ is at most B = min(2 R+, c (c + 1) - 2 R+) (the distribution is
// symmetric) and p = min(1, count * 2^(1 - c)).  scipy sums dyadic pmf values exactly, so this p is
// bit-identical to its; zeros and NaN differences scale its enumeration by 2^k and cancel.  The count
// is at most 2^50, exact in uint64 and in binary64.
//
// Normal approximation: se = sqrt((c (c + 1) (2 c + 1) - T / 2) / 24), z = (R+ - c (c + 1) / 4) / se.
// Every intermediate before the division and the square root is an integer or a quarter-integer below
// 2^53, so z rounds exactly where scipy's expression does; p = erfc(|z| / sqrt 2) = scipy's 2 Phi(-|z|)
// to ~1e-15 relative.
//
// The header compiles for the device (sd_signedrank.cu) and, without nvcc, for the host: the host build
// exists only so tests/ can check this arithmetic on machines with no GPU.
#pragma once

#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SD_SR_HD __host__ __device__ __forceinline__
#else
#define SD_SR_HD inline
#endif

namespace sd {
namespace signedrank {

constexpr int kUntested = 0, kExact = 1, kNormal = 2;
constexpr int64_t kExactMaxN = 50, kPermutationMaxN = 13;

// 0 = untested, 1 = exact count, 2 = normal approximation
SD_SR_HD int method(int64_t n, int64_t c, int64_t zeros, int64_t ties)
{
    if (n == 0) return kUntested;
    if ((n <= kExactMaxN && ties == 0 && zeros == 0) || n <= kPermutationMaxN)
        return (n == 1 && zeros == 1) ? kUntested : kExact;        // scipy raises for one zero difference
    return c == 0 ? kUntested : kNormal;
}

// the bound of the exact count and twice W: min(2 R+, c (c + 1) - 2 R+)
SD_SR_HD int64_t twice_w(int64_t c, int64_t rp2) { return rp2 < c * (c + 1) - rp2 ? rp2 : c * (c + 1) - rp2; }

// p of the exact methods from the number of sign patterns with 2 R+ <= twice_w
SD_SR_HD double exact_p(uint64_t count, int64_t c) { return fmin(1.0, ldexp((double)count, (int)(1 - c))); }

// z of the normal approximation
SD_SR_HD double normal_z(int64_t c, int64_t rp2, int64_t ties)
{
    const double cd = (double)c;
    const double se = sqrt((cd * (cd + 1.0) * (2.0 * cd + 1.0) - (double)ties / 2.0) / 24.0);
    return ((double)rp2 / 2.0 - cd * (cd + 1.0) * 0.25) / se;
}

SD_SR_HD double normal_p(double z) { return erfc(fabs(z) * 0.70710678118654752440); }

// Sequential reference of the exact count: the number of subsets of the c doubled ranks r2[0, c)
// whose sum is <= bound (a 0/1 knapsack over counts[0, bound], which the caller provides).
SD_SR_HD uint64_t count_reference(const int64_t *r2, int64_t c, int64_t bound, uint64_t *counts)
{
    for (int64_t s = 0; s <= bound; ++s) counts[s] = s == 0;
    for (int64_t k = 0; k < c; ++k)
        for (int64_t s = bound; s >= r2[k]; --s) counts[s] += counts[s - r2[k]];
    uint64_t total = 0;
    for (int64_t s = 0; s <= bound; ++s) total += counts[s];
    return total;
}

}  // namespace signedrank
}  // namespace sd
