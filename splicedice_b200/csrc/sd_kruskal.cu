// sd_kruskal.cu -- Kruskal-Wallis H test per event across any number of sample groups
// (`compare_conditions`).
//
// For row j of a PS matrix, the non-NaN cells of the listed columns, each in the group its label names,
// are ranked together with average ranks; the test is scipy.stats.kruskal(*groups, nan_policy='omit')
// (scipy 1.18.1) with the exact integer form of sd_kruskal_math.cuh:
//     D_g = sum over the group's cells of (lo + hi + 1) - n_g (n + 1),   T = sum over cells of ((hi - lo)^2 - 1),
//     H = 3 (n - 1) sum_g (D_g^2 / n_g) / (n^3 - n - T),                 p = chi2.sf(H, k - 1),
// [lo, hi) a cell's tie run in the sorted keys.  Edge rules, and where scipy differs:
//   - a group with no defined cell in the row: H = p = NaN (scipy: NaN too);
//   - every defined cell tied (T = n^3 - n): H = p = NaN.  scipy's rounding gives NaN for most such
//     rows but +inf (p = 0) or -inf for some; p = 0 for identical values would top the BH list;
//   - balanced rank sums: H = 0 and p = 1 exactly (scipy can give a tiny negative H there, then p = NaN);
//   - -0.0 ties +0.0 and +-inf are ordinary values, as in K6 (the keys of sd_ranksort.cuh);
//   - per-group counts and means (float64 sums) are written for every row, also where H is NaN.
//
// Mapping: one CTA per row (rows blockIdx.x, + gridDim.x, ...; one resident wave), K6's gather and
// bitonic sort (sd_ranksort.cuh), then one rank pass over all gathered cells: the two tie-run searches
// per cell, and D_g, n_g and the sum per group plus T.  Lanes of a warp that share a label combine
// their terms in a shuffle tree (__match_any_sync peers) and the lowest lane adds them to the warp's
// own per-group slots in shared memory: no atomics, and one add per label and warp when the caller
// lists the columns group by group (ops.kruskal_rows does).  The slots are summed in warp order, so
// every output is deterministic.  A column outside [0, n_samples) or a label outside [0, k) is never
// dereferenced: the row gets n = -1 in every group and NaN means and statistics.
#include <algorithm>

#include "sd_common.cuh"
#include "sd_kruskal_math.cuh"
#include "sd_ranksort.cuh"

namespace sd {
namespace kruskal {

constexpr int kMaxN = SD_RANKSUM_MAX_SAMPLES;
constexpr int kMaxGroups = SD_KRUSKAL_MAX_GROUPS;
constexpr int kMaxThreads = 256;
constexpr int kMaxWarps = kMaxThreads / 32;

struct Params {
    int32_t n_samples;
    const void *ps;
    int64_t ld_ps;
    int32_t n_groups, n_cols, npad;
    const int32_t *cols, *group_of;
    int32_t *n_out;
    int64_t ld_n;
    double *mean_out;
    int64_t ld_mean;
    double *stats_out;
    int64_t ld_stats;
    int64_t row_begin, row_end;
};

// Sums d, v, c over the lanes of `peers` (this lane's label group) into its lowest lane, in a tree that
// depends on `peers` alone.  Every lane of the warp calls it.
__device__ __forceinline__ void reduce_peers(unsigned peers, int lane, long long &d, double &v, int &c)
{
    int rel = __popc(peers & ((1u << lane) - 1u));              // rank among the peers
    unsigned rest = peers & (0xfffffffeu << lane);               // peers above this lane still adding
    while (__any_sync(0xffffffffu, rest)) {
        const int next = __ffs(rest);                            // 1 + the next peer up, 0 if none
        const long long d2 = __shfl_sync(0xffffffffu, d, (next - 1) & 31);
        const double v2 = __shfl_sync(0xffffffffu, v, (next - 1) & 31);
        const int c2 = __shfl_sync(0xffffffffu, c, (next - 1) & 31);
        if (next) {
            d += d2;
            v += v2;
            c += c2;
        }
        rest &= ~__ballot_sync(0xffffffffu, rel & 1);            // odd ranks have handed theirs on
        rel >>= 1;
    }
}

template <typename T>
__global__ void __launch_bounds__(kMaxThreads) kruskal_rows_kernel(const Params p)
{
    extern __shared__ uint64_t keys[];
    __shared__ int s_m, s_bad;
    __shared__ double s_terms[kMaxWarps];
    __shared__ long long s_ties[kMaxWarps];
    __shared__ int s_empty[kMaxWarps];
    const int k = p.n_groups, n = p.n_cols;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    // per-warp, per-group partial sums behind the keys: D terms, value sums, counts
    long long *part_d = reinterpret_cast<long long *>(keys + p.npad);
    double *part_sum = reinterpret_cast<double *>(part_d + warps * k);
    int *part_n = reinterpret_cast<int *>(part_sum + warps * k);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int64_t j = p.row_begin + blockIdx.x; j < p.row_end; j += gridDim.x) {
        const T *row = static_cast<const T *>(p.ps) + j * p.ld_ps;
        if (threadIdx.x == 0) {
            s_m = 0;
            s_bad = 0;
        }
        for (int g = lane; g < k; g += 32) {
            part_d[warp * k + g] = 0;
            part_sum[warp * k + g] = 0.0;
            part_n[warp * k + g] = 0;
        }
        __syncthreads();
        // gather: keys of every non-NaN listed cell, in any order
        for (int base = 0; base < n; base += blockDim.x) {              // uniform trip count: whole warps
            const int i = base + threadIdx.x;
            bool valid = false;
            uint64_t key = 0;
            if (i < n) {
                const int col = __ldg(p.cols + i), g = __ldg(p.group_of + i);
                if ((unsigned)col >= (unsigned)p.n_samples || (unsigned)g >= (unsigned)k) {
                    s_bad = 1;
                } else {
                    const double v = (double)__ldg(row + col);
                    if (!isnan(v)) {
                        valid = true;
                        key = ranksort::order_key(v);
                    }
                }
            }
            SD_RANKSORT_APPEND(keys, &s_m, lane, valid, key);
        }
        __syncthreads();
        const int m = s_m;
        if (s_bad) {                                                    // uniform over the CTA
            for (int g = threadIdx.x; g < k; g += blockDim.x) {
                __stcs(p.n_out + j * p.ld_n + g, -1);
                __stcs(p.mean_out + j * p.ld_mean + g, nan);
            }
            if (threadIdx.x == 0) {
                __stcs(p.stats_out + j * p.ld_stats, nan);
                __stcs(p.stats_out + j * p.ld_stats + 1, nan);
            }
            __syncthreads();
            continue;
        }
        ranksort::sort(keys, m);
        // rank pass: every defined cell's tie run [lo, hi) gives lo + hi + 1 to its group and
        // (hi - lo)^2 - 1 to T
        long long ties = 0;
        for (int base = 0; base < n; base += blockDim.x) {
            const int i = base + threadIdx.x;
            int g = -1;
            long long d = 0;
            double v = 0.0;
            int c = 0;
            if (i < n) {
                g = __ldg(p.group_of + i);
                const double x = (double)__ldg(row + __ldg(p.cols + i));
                if (!isnan(x)) {
                    const uint64_t key = ranksort::order_key(x);
                    const int lo = ranksort::search(keys, 0, m, key, false);
                    const int hi = ranksort::search(keys, lo, m, key, true);
                    d = lo + hi + 1;
                    v = x;
                    c = 1;
                    ties += (long long)(hi - lo) * (hi - lo) - 1;
                }
            }
            const unsigned peers = __match_any_sync(0xffffffffu, g);
            reduce_peers(peers, lane, d, v, c);
            if (g >= 0 && lane == __ffs(peers) - 1) {
                part_d[warp * k + g] += d;
                part_sum[warp * k + g] += v;
                part_n[warp * k + g] += c;
            }
            __syncwarp();
        }
        __syncthreads();
        // per group: the warps' partials in warp order; counts and means; D_g^2 / n_g
        double terms = 0.0;
        int empty = 0;
        for (int g = threadIdx.x; g < k; g += blockDim.x) {
            long long d = 0;
            double s = 0.0;
            int c = 0;
            for (int w = 0; w < warps; ++w) {
                d += part_d[w * k + g];
                s += part_sum[w * k + g];
                c += part_n[w * k + g];
            }
            __stcs(p.n_out + j * p.ld_n + g, c);
            __stcs(p.mean_out + j * p.ld_mean + g, c ? s / c : nan);
            if (c)
                terms += group_term(d - (long long)c * (m + 1), c);
            else
                empty = 1;
        }
        for (int o = 16; o; o >>= 1) {
            terms += __shfl_xor_sync(0xffffffffu, terms, o);
            ties += __shfl_xor_sync(0xffffffffu, ties, o);
            empty |= __shfl_xor_sync(0xffffffffu, empty, o);
        }
        if (lane == 0) {
            s_terms[warp] = terms;
            s_ties[warp] = ties;
            s_empty[warp] = empty;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < warps; ++w) {
                terms += s_terms[w];
                ties += s_ties[w];
                empty |= s_empty[w];
            }
            const double h = empty ? nan : h_stat(terms, m, ties);
            __stcs(p.stats_out + j * p.ld_stats, h);
            __stcs(p.stats_out + j * p.ld_stats + 1, chi2_sf(k - 1, h));
        }
        __syncthreads();
    }
}

template <typename T>
static int launch(const Params &p, cudaStream_t stream)
{
    const int threads = std::min(kMaxThreads, std::max(32, p.npad / 2));
    const size_t smem = (size_t)p.npad * sizeof(uint64_t) +
                        (size_t)(threads / 32) * p.n_groups * (sizeof(long long) + sizeof(double) + sizeof(int));
    SD_CHECK_CUDA(cudaFuncSetAttribute(kruskal_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kruskal_rows_kernel<T>, threads, smem) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    SD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t rows = p.row_end - p.row_begin;
    const int64_t grid = std::min<int64_t>(rows, (int64_t)sms * per_sm);
    kruskal_rows_kernel<T><<<(unsigned)grid, threads, smem, stream>>>(p);
    return check_launch("kruskal_rows_kernel");
}

}  // namespace kruskal
}  // namespace sd

extern "C" {

int sd_kruskal_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                    int32_t n_groups, int32_t n_cols, const int32_t *cols, const int32_t *group_of,
                    int64_t row_begin, int64_t row_end,
                    int32_t *n_out, int64_t ld_n, double *mean_out, int64_t ld_mean,
                    double *stats_out, int64_t ld_stats, void *stream)
{
    SD_REQUIRE(n_events >= 0 && n_samples >= 0, "sd_kruskal_rows: negative size");
    SD_REQUIRE(n_groups >= 2 && n_groups <= sd::kruskal::kMaxGroups, "sd_kruskal_rows: n_groups = %d outside [2, %d]",
               (int)n_groups, sd::kruskal::kMaxGroups);
    SD_REQUIRE(n_cols >= 1 && n_cols <= sd::kruskal::kMaxN, "sd_kruskal_rows: n_cols = %d outside [1, %d]",
               (int)n_cols, sd::kruskal::kMaxN);
    SD_REQUIRE(dtype == SD_RANKSUM_F32 || dtype == SD_RANKSUM_F64,
               "sd_kruskal_rows: dtype must be SD_RANKSUM_F32 or SD_RANKSUM_F64");
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_events,
               "sd_kruskal_rows: row range outside [0, n_events)");
    if (row_begin == row_end) return SD_OK;
    SD_REQUIRE(ps && cols && group_of && n_out && mean_out && stats_out, "sd_kruskal_rows: null pointer");
    SD_REQUIRE(ld_ps >= n_samples && ld_n >= n_groups && ld_mean >= n_groups && ld_stats >= 2,
               "sd_kruskal_rows: ld too small");
    sd::kruskal::Params p{};
    p.n_samples = n_samples;
    p.ps = ps; p.ld_ps = ld_ps;
    p.n_groups = n_groups; p.n_cols = n_cols; p.cols = cols; p.group_of = group_of;
    p.npad = 1;
    while (p.npad < n_cols) p.npad <<= 1;
    p.n_out = n_out; p.ld_n = ld_n; p.mean_out = mean_out; p.ld_mean = ld_mean;
    p.stats_out = stats_out; p.ld_stats = ld_stats;
    p.row_begin = row_begin; p.row_end = row_end;
    return dtype == SD_RANKSUM_F32 ? sd::kruskal::launch<float>(p, (cudaStream_t)stream)
                                   : sd::kruskal::launch<double>(p, (cudaStream_t)stream);
}

}  // extern "C"
