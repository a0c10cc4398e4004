// sd_kruskal_math.cuh -- per-row arithmetic of the Kruskal-Wallis H test (K7, sd_kruskal.cu).
//
// Exact statistic.  A cell whose tie run occupies sorted positions [lo, hi) has twice its average rank
// = lo + hi + 1, so per group D_g = sum (lo + hi + 1) - n_g (n + 1) = 2 R_g - n_g (n + 1) is an exact
// integer (|D_g| <= n^2 / 4 < 2^26.5 for n <= 16,384, so D_g^2 is exact in binary64), and so is the
// tie term T = sum over runs of (t^3 - t) = sum over cells of ((hi - lo)^2 - 1).  Then
//     H = 3 (n - 1) * sum_g (D_g^2 / n_g) / (n^3 - n - T),
// which is scipy.stats.kruskal's (12 / (n (n + 1)) sum R_g^2 / n_g - 3 (n + 1)) / (1 - T / (n^3 - n))
// rewritten (sum_g D_g = 0) without its cancellation: H >= 0 always, and H == 0 exactly when every
// group's mean rank is (n + 1) / 2.  All defined cells tied (n^3 - n == T) leaves H undefined (NaN).
//
// p-value.  p = Q((k - 1) / 2, H / 2), the chi-square survival function with k - 1 degrees of freedom:
//     integer a:      Q(a, x) = e^-x sum_{i < a} x^i / i!
//     half-integer a: Q(a, x) = erfc(sqrt x) + e^-x sum_{i = 1 .. a - 1/2} x^(i - 1/2) / Gamma(i + 1/2)
// Every term is positive.  The largest term is formed in log space (one exp, one log, one lgamma) and
// the others from it by the ratio recurrence, so nothing underflows while p is still representable
// (a recurrence started at e^-x is 0 for x > 745 while p can be ~1e-190 with large df).  H == 0 gives
// p == 1 exactly.  tests/test_kruskal_twin.py checks both against exact oracles.
//
// The header compiles for the device (sd_kruskal.cu) and, without nvcc, for the host: the host build
// exists only so tests/ can check this arithmetic on machines with no GPU.
#pragma once

#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SD_KW_HD __host__ __device__ __forceinline__
#else
#define SD_KW_HD inline
#endif

namespace sd {
namespace kruskal {

// D_g^2 / n_g, the group's share of sum_g (D_g^2 / n_g)
SD_KW_HD double group_term(int64_t d, int64_t n_g) { return (double)(d * d) / (double)n_g; }

// H from sum_g (D_g^2 / n_g), the defined-cell count n and the tie term T; NaN when every cell is tied
SD_KW_HD double h_stat(double sum_terms, int64_t n, int64_t t)
{
    const int64_t den = n * n * n - n - t;
    if (den <= 0) return __builtin_nan("");
    return 3.0 * (double)(n - 1) * sum_terms / (double)den;
}

// chi-square survival function with df = 1 .. 255 degrees of freedom at h >= 0
SD_KW_HD double chi2_sf(int df, double h)
{
    if (isnan(h)) return h;
    if (h <= 0.0) return 1.0;
    const double x = 0.5 * h;
    const double lx = log(x);
    if (df % 2 == 0) {
        // e^-x sum_{i < a} x^i / i!, t_i / t_{i-1} = x / i, largest at i = min(a - 1, floor(x))
        const int a = df / 2;
        const int top = (int)fmin((double)(a - 1), floor(x));
        const double big = exp(-x + top * lx - lgamma(top + 1.0));
        double s = 1.0, t = 1.0;
        for (int i = top; i > 0; --i) s += (t *= i / x);
        t = 1.0;
        for (int i = top + 1; i < a; ++i) s += (t *= x / i);
        return fmin(1.0, big * s);
    }
    // erfc(sqrt x) + e^-x sum_{i = 1 .. m} x^(i - 1/2) / Gamma(i + 1/2), m = a - 1/2 = (df - 1) / 2;
    // u_i / u_{i-1} = x / (i - 1/2), largest at i = clamp(floor(x + 1/2), 1, m)
    const int m = (df - 1) / 2;
    double q = erfc(sqrt(x));
    if (m > 0) {
        const int top = (int)fmax(1.0, fmin((double)m, floor(x + 0.5)));
        const double big = exp(-x + (top - 0.5) * lx - lgamma(top + 0.5));
        double s = 1.0, t = 1.0;
        for (int i = top; i > 1; --i) s += (t *= (i - 0.5) / x);
        t = 1.0;
        for (int i = top + 1; i <= m; ++i) s += (t *= x / (i - 0.5));
        q += big * s;
    }
    return fmin(1.0, q);
}

}  // namespace kruskal
}  // namespace sd
