// sd_ranksum.cu -- Wilcoxon rank-sum test per event between two sample groups (`compare_groups`).
//
// For row j of a PS matrix, x = the non-NaN cells of the group-1 columns and y = those of the group-2
// columns; the test is scipy.stats.ranksums(x, y, nan_policy='omit') (scipy 1.18.1): rank x U y with
// average ranks for ties, R1 = the rank sum of x,
//     z = (R1 - n1 (n + 1) / 2) / sqrt(n1 n2 (n + 1) / 12),   p = 2 Phi(-|z|) = erfc(|z| / sqrt 2),
// no tie and no continuity correction.
//
// Exactness.  Average ranks are half-integers, so 2 R1 is an integer: a value v of x whose tie run
// occupies sorted positions [lo, hi) has rank (lo + 1 + hi) / 2, and 2 R1 = sum over x of (lo + hi + 1).
// lo and hi are a lower / upper bound search of v's key in the sorted keys of x U y, summed in 64-bit
// integers, so D = 2 R1 - n1 (n + 1) is exact; z = (D / 2) / sqrt((double)(n1 n2 (n + 1)) / 12) then
// rounds exactly where scipy's float expression does (its rank sum of half-integers below 2^53 is
// exact too), and D == 0 gives z == 0 and p == 1 exactly.
//
// Keys, gather, sort and searches are the shared ones of sd_ranksort.cuh: -0.0 ties +0.0, float32 cells
// are widened to double first, so both input types share one kernel body, and +-inf are ordinary keys.
//
// Mapping: one CTA per row (rows blockIdx.x, + gridDim.x, ...; one resident wave).  Gather the group
// columns into shared memory with warp-aggregated slots, bitonic sort of the next power of two above
// the row's valid count, then the group-1 cells are read again (L1 / L2 hits) for the two searches.
// Means are float64 sums over the same gather.  Thread 0 stores n1, n2 and (mean1, mean2, z, p) with
// __stcs.  A column index outside [0, n_samples) is never dereferenced: the row gets n1 = n2 = -1 and
// NaN statistics.
#include <algorithm>

#include "sd_common.cuh"
#include "sd_ranksort.cuh"

namespace sd {
namespace ranksum {

constexpr int kMaxN = SD_RANKSUM_MAX_SAMPLES;
constexpr int kMaxThreads = 256;
constexpr int kMaxWarps = kMaxThreads / 32;

struct Params {
    int32_t n_samples;
    const void *ps;
    int64_t ld_ps;
    int32_t n1, n2;
    const int32_t *cols1, *cols2;
    int32_t *n_out;
    int64_t ld_n;
    double *stats_out;
    int64_t ld_stats;
    int64_t row_begin, row_end;
};

using ranksort::order_key;
using ranksort::search;

template <typename T>
__global__ void __launch_bounds__(kMaxThreads) ranksum_rows_kernel(const Params p)
{
    extern __shared__ uint64_t keys[];
    __shared__ int s_m, s_bad;
    __shared__ long long s_r1[kMaxWarps];
    __shared__ double s_sum1[kMaxWarps], s_sum2[kMaxWarps];
    __shared__ int s_c1[kMaxWarps];
    const int n = p.n1 + p.n2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t j = p.row_begin + blockIdx.x; j < p.row_end; j += gridDim.x) {
        const T *row = static_cast<const T *>(p.ps) + j * p.ld_ps;
        if (threadIdx.x == 0) {
            s_m = 0;
            s_bad = 0;
        }
        __syncthreads();
        // gather: keys of every non-NaN cell of either group, in any order
        double sum1 = 0.0, sum2 = 0.0;
        int c1 = 0;
        for (int base = 0; base < n; base += blockDim.x) {              // uniform trip count: whole warps
            const int i = base + threadIdx.x;
            bool valid = false;
            uint64_t key = 0;
            if (i < n) {
                const int col = i < p.n1 ? __ldg(p.cols1 + i) : __ldg(p.cols2 + (i - p.n1));
                if ((unsigned)col >= (unsigned)p.n_samples) {
                    s_bad = 1;
                } else {
                    const double v = (double)__ldg(row + col);
                    if (!isnan(v)) {
                        valid = true;
                        key = order_key(v);
                        if (i < p.n1) {
                            sum1 += v;
                            ++c1;
                        } else {
                            sum2 += v;
                        }
                    }
                }
            }
            SD_RANKSORT_APPEND(keys, &s_m, lane, valid, key);
        }
        __syncthreads();
        const int m = s_m;
        if (s_bad) {                                                    // uniform over the CTA
            if (threadIdx.x == 0) {
                const double nan = __longlong_as_double(0x7ff8000000000000ll);
                __stcs(p.n_out + j * p.ld_n, -1);
                __stcs(p.n_out + j * p.ld_n + 1, -1);
                for (int k = 0; k < 4; ++k) __stcs(p.stats_out + j * p.ld_stats + k, nan);
            }
            __syncthreads();
            continue;
        }
        ranksort::sort(keys, m);
        // 2 R1 = sum over the group-1 cells of (lo + hi + 1), lo / hi the bounds of the cell's tie run
        long long r1 = 0;
        for (int i = threadIdx.x; i < p.n1; i += blockDim.x) {
            const double v = (double)__ldg(row + __ldg(p.cols1 + i));
            if (!isnan(v)) {
                const uint64_t key = order_key(v);
                const int lo = search(keys, 0, m, key, false);
                const int hi = search(keys, lo, m, key, true);
                r1 += lo + hi + 1;
            }
        }
        for (int o = 16; o; o >>= 1) {
            r1 += __shfl_xor_sync(0xffffffffu, r1, o);
            sum1 += __shfl_xor_sync(0xffffffffu, sum1, o);
            sum2 += __shfl_xor_sync(0xffffffffu, sum2, o);
            c1 += __shfl_xor_sync(0xffffffffu, c1, o);
        }
        if (lane == 0) {
            s_r1[warp] = r1;
            s_sum1[warp] = sum1;
            s_sum2[warp] = sum2;
            s_c1[warp] = c1;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
                r1 += s_r1[w];
                sum1 += s_sum1[w];
                sum2 += s_sum2[w];
                c1 += s_c1[w];
            }
            const int c2 = m - c1;
            const double nan = __longlong_as_double(0x7ff8000000000000ll);
            double z = nan, pv = nan;
            if (c1 > 0 && c2 > 0) {
                const long long d = r1 - (long long)c1 * (m + 1);
                const double sigma = sqrt((double)((long long)c1 * c2 * (m + 1)) / 12.0);
                z = (0.5 * (double)d) / sigma;
                pv = erfc(fabs(z) * 0.70710678118654752440);
            }
            __stcs(p.n_out + j * p.ld_n, c1);
            __stcs(p.n_out + j * p.ld_n + 1, c2);
            double *st = p.stats_out + j * p.ld_stats;
            __stcs(st, c1 ? sum1 / c1 : nan);
            __stcs(st + 1, c2 ? sum2 / c2 : nan);
            __stcs(st + 2, z);
            __stcs(st + 3, pv);
        }
        __syncthreads();
    }
}

template <typename T>
static int launch(const Params &p, cudaStream_t stream)
{
    int npad = 1;
    while (npad < p.n1 + p.n2) npad <<= 1;
    const int threads = std::min(kMaxThreads, std::max(32, npad / 2));
    const size_t smem = (size_t)npad * sizeof(uint64_t);
    SD_CHECK_CUDA(cudaFuncSetAttribute(ranksum_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ranksum_rows_kernel<T>, threads, smem) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    SD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t rows = p.row_end - p.row_begin;
    const int64_t grid = std::min<int64_t>(rows, (int64_t)sms * per_sm);
    ranksum_rows_kernel<T><<<(unsigned)grid, threads, smem, stream>>>(p);
    return check_launch("ranksum_rows_kernel");
}

}  // namespace ranksum
}  // namespace sd

extern "C" {

int sd_ranksum_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                    int32_t n1, const int32_t *cols1, int32_t n2, const int32_t *cols2,
                    int64_t row_begin, int64_t row_end,
                    int32_t *n_out, int64_t ld_n, double *stats_out, int64_t ld_stats, void *stream)
{
    SD_REQUIRE(n_events >= 0 && n_samples >= 0, "sd_ranksum_rows: negative size");
    SD_REQUIRE(n1 >= 1 && n2 >= 1, "sd_ranksum_rows: each group needs at least one column");
    SD_REQUIRE((int64_t)n1 + n2 <= sd::ranksum::kMaxN, "sd_ranksum_rows: n1 + n2 = %lld exceeds %d samples",
               (long long)n1 + n2, sd::ranksum::kMaxN);
    SD_REQUIRE(dtype == SD_RANKSUM_F32 || dtype == SD_RANKSUM_F64, "sd_ranksum_rows: dtype must be SD_RANKSUM_F32 or SD_RANKSUM_F64");
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_events,
               "sd_ranksum_rows: row range outside [0, n_events)");
    if (row_begin == row_end) return SD_OK;
    SD_REQUIRE(ps && cols1 && cols2 && n_out && stats_out, "sd_ranksum_rows: null pointer");
    SD_REQUIRE(ld_ps >= n_samples && ld_n >= 2 && ld_stats >= 4, "sd_ranksum_rows: ld too small");
    sd::ranksum::Params p{};
    p.n_samples = n_samples;
    p.ps = ps; p.ld_ps = ld_ps;
    p.n1 = n1; p.n2 = n2; p.cols1 = cols1; p.cols2 = cols2;
    p.n_out = n_out; p.ld_n = ld_n; p.stats_out = stats_out; p.ld_stats = ld_stats;
    p.row_begin = row_begin; p.row_end = row_end;
    return dtype == SD_RANKSUM_F32 ? sd::ranksum::launch<float>(p, (cudaStream_t)stream)
                                   : sd::ranksum::launch<double>(p, (cudaStream_t)stream);
}

}  // extern "C"
