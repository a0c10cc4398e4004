// sd_chi2_math.cuh -- per-table arithmetic of the Yates-corrected chi-squared test of a 2x2 table.
//
// What scipy.stats.chi2_contingency(table)[1] computes with its default correction=True (scipy
// 1.18.1, stats/contingency.py; the call the reference's `pairwise --chi2` makes per table), for
// the table [[a, b], [c, d]] with margins r1 = a+b, r2 = c+d, c1 = a+c, c2 = b+d and N = r1+r2:
//   - every |observed - expected| of a 2x2 table equals |ad - bc| / N, and scipy clamps the Yates
//     step at min(0.5, |diff|), so
//         stat = max(|ad - bc| - N/2, 0)^2 * N / (r1 r2 c1 c2),   p = chi2.sf(stat, 1) = erfc(sqrt(stat / 2));
//     |ad - bc| <= N/2 gives exactly p = 1.  (Releases before the clamp -- gh-13875 -- subtracted a
//     flat 0.5; this follows the installed 1.18.1, as the Fisher tie rule does.)
//   - N > 0 with a zero margin: scipy raises ValueError at the first zero of `expected` in row-major
//     order, (0, 0) if r1 == 0 or c1 == 0, else (0, 1) if c2 == 0, else (1, 0) (r2 == 0).
//   - the all-zero table does not raise: expected is 0/0, p is NaN.
// 2|ad - bc| - N is formed exactly in 128-bit integers (a, b < 2^31 and c, d < 2^61: products up to
// 2^92), so the only roundings are the FP64 margin products, one sqrt and erfc: within 4e-13 of the
// exact value at every scale the inputs allow (tests/test_chi2_twin.py against mpmath).
//
// The header compiles for the device (sd_chi2.cu) and, without nvcc, for the host: the host build
// exists only so tests/ can check this arithmetic against scipy on machines with no GPU.
#pragma once

#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SD_CHI2_HD __host__ __device__ __forceinline__
#else
#define SD_CHI2_HD inline
#endif

namespace sd {
namespace chi2 {

// outcome of one table; the kRefused* codes are the tables scipy refuses
enum Status : int {
    kValue = 0,          // p in [0, 1]
    kAllZero = 1,        // N == 0: p is NaN, as scipy
    kRefused00 = 2,      // zero margin, scipy's message names (0, 0)
    kRefused01 = 3,      // ... (0, 1)
    kRefused10 = 4,      // ... (1, 0)
    kRefusedEntry = 5,   // an entry outside the domain: a or b outside [0, 2^31), c or d outside [0, 2^61)
};

constexpr int64_t kMaxInc = int64_t(1) << 31;
constexpr int64_t kMaxExc = int64_t(1) << 61;

SD_CHI2_HD bool refused(int status) { return status >= kRefused00; }

// exact (signed) 2|ad - bc| - N as a double: one rounding when it fits 64 bits, two beyond
SD_CHI2_HD double twice_excess(int64_t a, int64_t b, int64_t c, int64_t d, int64_t n)
{
    __int128 diff = (__int128)a * d - (__int128)b * c;
    if (diff < 0) diff = -diff;
    const __int128 x = 2 * diff - n;
    if (x >= -(__int128)INT64_MAX && x <= (__int128)INT64_MAX) return (double)(int64_t)x;
    // |x| < 2^94: the high word is exact in binary64, the low word rounds once, the sum once more
    const int64_t hi = (int64_t)(x >> 64);
    const uint64_t lo = (uint64_t)x;
    return (double)hi * 18446744073709551616.0 + (double)lo;
}

// p of [[a, b], [c, d]]; *status receives a Status.  Refused tables return NaN.
SD_CHI2_HD double yates_p(int64_t a, int64_t b, int64_t c, int64_t d, int *status)
{
    const double nan = __builtin_nan("");
    if (a < 0 || b < 0 || c < 0 || d < 0 || a >= kMaxInc || b >= kMaxInc || c >= kMaxExc || d >= kMaxExc) {
        *status = kRefusedEntry;
        return nan;
    }
    const int64_t r1 = a + b, r2 = c + d, c1 = a + c, c2 = b + d, n = r1 + r2;
    if (n == 0) {
        *status = kAllZero;
        return nan;
    }
    if (r1 == 0 || c1 == 0 || c2 == 0 || r2 == 0) {
        *status = (r1 == 0 || c1 == 0) ? kRefused00 : (c2 == 0 ? kRefused01 : kRefused10);
        return nan;
    }
    *status = kValue;
    const double x2 = twice_excess(a, b, c, d, n);
    if (x2 <= 0.0) return 1.0;
    // z = sqrt(stat) = (x2 / 2) * sqrt(N / (r1 r2) / (c1 c2)); every factor stays far from overflow
    const double z = 0.5 * x2 * sqrt((double)n / ((double)r1 * (double)r2) / ((double)c1 * (double)c2));
    return erfc(z * 0.70710678118654752440);
}

}  // namespace chi2
}  // namespace sd
