// sd_signedrank.cu -- Wilcoxon signed-rank test per event between matched sample pairs (`compare_paired`).
//
// For row j of a PS matrix, pair i has cells x_i = ps[j, cols1[i]] and y_i = ps[j, cols2[i]]; the test is
// scipy.stats.wilcoxon(x, y, nan_policy='omit') (scipy 1.18.1 defaults) with the exact integer terms and
// the method switch of sd_signedrank_math.cuh.  Per row:
//   - n = pairs with both cells non-NaN; their float64 sums give mean1 and mean2;
//   - d = x - y in the input's precision (a float32 matrix subtracts in float32, as numpy's x - y does,
//     and only then widens: widening first would split ties the float32 difference makes);
//   - inf - inf = NaN counts in n and carries no rank; d == 0 (-0.0 too) is a zero, dropped from the
//     ranking; the other c differences are ranked by |d|, whose keys (sd_ranksort.cuh) order +inf last;
//   - a difference whose |d| occupies the tie run [lo, hi) of the sorted keys has doubled rank
//     lo + hi + 1, so 2 R+ (the sum over d > 0) and T = sum ((hi - lo)^2 - 1) are exact int64 sums.
//
// Mapping: one CTA per row (rows blockIdx.x, + gridDim.x, ...; one resident wave), as K6.  Gather the
// keys of every rankable |d| into shared memory (warp-aggregated slots) and count n, zeros and the two
// sums; bitonic sort; a second pass over the pairs (L1 / L2 hits) redoes the two searches per rankable d
// for 2 R+ and T.  Thread 0 reduces the warps' partials and picks the method.  For the exact method
// (c <= 50) the CTA counts the sign patterns in shared memory, a 0/1 knapsack over the c doubled ranks
// in ascending order, bins [0, B] with B = min(2 R+, c (c + 1) - 2 R+) <= 1,275, uint64 counts: per
// rank v the bins s in [v, reach] (reach = the largest sum the ranks so far can make, capped at B) take
// counts[s - v], in descending chunks of blockDim bins, each read before a barrier and written after
// it, so a chunk's writes never meet a read of the same rank.  When every doubled rank is even (always
// without ties) ranks and bound are halved first.  A column outside [0, n_samples) is never
// dereferenced: the row gets n = c = -1, method 0 and NaN statistics.
#include <algorithm>

#include "sd_common.cuh"
#include "sd_ranksort.cuh"
#include "sd_signedrank_math.cuh"

namespace sd {
namespace signedrank {

constexpr int kMaxPairs = SD_SIGNEDRANK_MAX_PAIRS;
constexpr int kMaxThreads = 256;
constexpr int kMaxWarps = kMaxThreads / 32;
constexpr int kMaxExact = (int)kExactMaxN;

struct Params {
    int32_t n_samples;
    const void *ps;
    int64_t ld_ps;
    int32_t n_pairs, npad;
    const int32_t *cols1, *cols2;
    int32_t *n_out;
    int64_t ld_n;
    double *stats_out;
    int64_t ld_stats;
    int64_t row_begin, row_end;
};

// the difference of pair i in the input's precision, widened to double
template <typename T>
__device__ __forceinline__ double difference(T x, T y)
{
    const T d = x - y;
    return (double)d;
}

template <typename T>
__global__ void __launch_bounds__(kMaxThreads) signedrank_rows_kernel(const Params p)
{
    extern __shared__ uint64_t keys[];                              // npad keys, then the exact counts
    uint64_t *counts = keys + p.npad;
    __shared__ int s_c, s_bad;
    __shared__ int s_item[kMaxExact];                               // doubled ranks in sorted order
    __shared__ int s_n[kMaxWarps], s_zeros[kMaxWarps], s_odd[kMaxWarps];
    __shared__ double s_sum1[kMaxWarps], s_sum2[kMaxWarps];
    __shared__ long long s_rp2[kMaxWarps], s_ties[kMaxWarps];
    __shared__ unsigned long long s_count[kMaxWarps];
    __shared__ int s_method, s_shift;
    __shared__ long long s_bound;
    const int P = p.n_pairs;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int64_t j = p.row_begin + blockIdx.x; j < p.row_end; j += gridDim.x) {
        const T *row = static_cast<const T *>(p.ps) + j * p.ld_ps;
        if (threadIdx.x == 0) {
            s_c = 0;
            s_bad = 0;
        }
        __syncthreads();
        // gather: keys of |d| for every nonzero, non-NaN difference, in any order
        int n = 0, zeros = 0;
        double sum1 = 0.0, sum2 = 0.0;
        for (int base = 0; base < P; base += blockDim.x) {              // uniform trip count: whole warps
            const int i = base + threadIdx.x;
            bool valid = false;
            uint64_t key = 0;
            if (i < P) {
                const int c1 = __ldg(p.cols1 + i), c2 = __ldg(p.cols2 + i);
                if ((unsigned)c1 >= (unsigned)p.n_samples || (unsigned)c2 >= (unsigned)p.n_samples) {
                    s_bad = 1;
                } else {
                    const T x = __ldg(row + c1), y = __ldg(row + c2);
                    if (!isnan(x) && !isnan(y)) {
                        ++n;
                        sum1 += (double)x;
                        sum2 += (double)y;
                        const double d = difference(x, y);
                        if (d == 0.0) {
                            ++zeros;
                        } else if (!isnan(d)) {
                            valid = true;
                            key = ranksort::order_key(fabs(d));
                        }
                    }
                }
            }
            SD_RANKSORT_APPEND(keys, &s_c, lane, valid, key);
        }
        __syncthreads();
        const int c = s_c;
        if (s_bad) {                                                    // uniform over the CTA
            if (threadIdx.x == 0) {
                __stcs(p.n_out + j * p.ld_n, -1);
                __stcs(p.n_out + j * p.ld_n + 1, -1);
                __stcs(p.n_out + j * p.ld_n + 2, kUntested);
                for (int k = 0; k < 4; ++k) __stcs(p.stats_out + j * p.ld_stats + k, nan);
            }
            __syncthreads();
            continue;
        }
        ranksort::sort(keys, c);
        // the doubled ranks in sorted order, for the exact count (c <= 50 there)
        if (c <= kMaxExact) {
            for (int t = threadIdx.x; t < c; t += blockDim.x) {
                const int lo = ranksort::search(keys, 0, c, keys[t], false);
                const int hi = ranksort::search(keys, lo, c, keys[t], true);
                s_item[t] = lo + hi + 1;
            }
        }
        // second pass: 2 R+ over d > 0 and T over every rankable d
        long long rp2 = 0, ties = 0;
        int odd = 0;
        for (int i = threadIdx.x; i < P; i += blockDim.x) {
            const T x = __ldg(row + __ldg(p.cols1 + i)), y = __ldg(row + __ldg(p.cols2 + i));
            if (isnan(x) || isnan(y)) continue;
            const double d = difference(x, y);
            if (d == 0.0 || isnan(d)) continue;
            const uint64_t key = ranksort::order_key(fabs(d));
            const int lo = ranksort::search(keys, 0, c, key, false);
            const int hi = ranksort::search(keys, lo, c, key, true);
            if (d > 0.0) rp2 += lo + hi + 1;
            ties += (long long)(hi - lo) * (hi - lo) - 1;
            odd |= (lo + hi + 1) & 1;
        }
        for (int o = 16; o; o >>= 1) {
            n += __shfl_xor_sync(0xffffffffu, n, o);
            zeros += __shfl_xor_sync(0xffffffffu, zeros, o);
            odd |= __shfl_xor_sync(0xffffffffu, odd, o);
            sum1 += __shfl_xor_sync(0xffffffffu, sum1, o);
            sum2 += __shfl_xor_sync(0xffffffffu, sum2, o);
            rp2 += __shfl_xor_sync(0xffffffffu, rp2, o);
            ties += __shfl_xor_sync(0xffffffffu, ties, o);
        }
        if (lane == 0) {
            s_n[warp] = n;
            s_zeros[warp] = zeros;
            s_odd[warp] = odd;
            s_sum1[warp] = sum1;
            s_sum2[warp] = sum2;
            s_rp2[warp] = rp2;
            s_ties[warp] = ties;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < warps; ++w) {
                n += s_n[w];
                zeros += s_zeros[w];
                odd |= s_odd[w];
                sum1 += s_sum1[w];
                sum2 += s_sum2[w];
                rp2 += s_rp2[w];
                ties += s_ties[w];
            }
            const int m = method(n, c, zeros, ties);
            const long long b = twice_w(c, rp2);
            double *st = p.stats_out + j * p.ld_stats;
            __stcs(p.n_out + j * p.ld_n, n);
            __stcs(p.n_out + j * p.ld_n + 1, c);
            __stcs(p.n_out + j * p.ld_n + 2, m);
            __stcs(st, n ? sum1 / n : nan);
            __stcs(st + 1, n ? sum2 / n : nan);
            __stcs(st + 2, m == kUntested ? nan : 0.5 * (double)b);
            if (m != kExact) __stcs(st + 3, m == kNormal ? normal_p(normal_z(c, rp2, ties)) : nan);
            s_method = m;
            s_shift = odd ? 0 : 1;
            s_bound = b >> (odd ? 0 : 1);
        }
        __syncthreads();
        if (s_method != kExact) continue;                               // uniform; the next row syncs first
        // exact: counts[s] = sign patterns whose (halved when all even) doubled-rank sum is s, s <= bound
        const int shift = s_shift, bound = (int)s_bound, threads = blockDim.x;
        for (int s = threadIdx.x; s <= bound; s += threads) counts[s] = s == 0;
        __syncthreads();
        int reach = 0;
        for (int k = 0; k < c; ++k) {
            const int v = s_item[k] >> shift;
            reach = min(bound, reach + v);
            for (int top = reach; top >= v; top -= threads) {          // uniform trip count
                const int s = top - (int)threadIdx.x;
                const uint64_t add = s >= v ? counts[s - v] : 0ull;
                __syncthreads();
                if (s >= v) counts[s] += add;
            }
            __syncthreads();
        }
        unsigned long long total = 0;
        for (int s = threadIdx.x; s <= bound; s += threads) total += counts[s];
        for (int o = 16; o; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
        if (lane == 0) s_count[warp] = total;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < warps; ++w) total += s_count[w];
            __stcs(p.stats_out + j * p.ld_stats + 3, exact_p(total, c));
        }
        __syncthreads();
    }
}

// bins of the exact count: B + 1 with B <= c (c + 1) / 2 and c <= min(n_pairs, 50)
static int exact_bins(int n_pairs)
{
    const int c = std::min(n_pairs, kMaxExact);
    return c * (c + 1) / 2 + 1;
}

template <typename T>
static int launch(const Params &p, cudaStream_t stream)
{
    const int threads = std::min(kMaxThreads, std::max(32, p.npad / 2));
    const size_t smem = ((size_t)p.npad + exact_bins(p.n_pairs)) * sizeof(uint64_t);
    SD_CHECK_CUDA(cudaFuncSetAttribute(signedrank_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, signedrank_rows_kernel<T>, threads, smem) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    SD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t rows = p.row_end - p.row_begin;
    const int64_t grid = std::min<int64_t>(rows, (int64_t)sms * per_sm);
    signedrank_rows_kernel<T><<<(unsigned)grid, threads, smem, stream>>>(p);
    return check_launch("signedrank_rows_kernel");
}

}  // namespace signedrank
}  // namespace sd

extern "C" {

int sd_signedrank_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                       int32_t n_pairs, const int32_t *cols1, const int32_t *cols2,
                       int64_t row_begin, int64_t row_end,
                       int32_t *n_out, int64_t ld_n, double *stats_out, int64_t ld_stats, void *stream)
{
    SD_REQUIRE(n_events >= 0 && n_samples >= 0, "sd_signedrank_rows: negative size");
    SD_REQUIRE(n_pairs >= 1 && n_pairs <= sd::signedrank::kMaxPairs, "sd_signedrank_rows: n_pairs = %d outside [1, %d]",
               (int)n_pairs, sd::signedrank::kMaxPairs);
    SD_REQUIRE(dtype == SD_RANKSUM_F32 || dtype == SD_RANKSUM_F64,
               "sd_signedrank_rows: dtype must be SD_RANKSUM_F32 or SD_RANKSUM_F64");
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_events,
               "sd_signedrank_rows: row range outside [0, n_events)");
    if (row_begin == row_end) return SD_OK;
    SD_REQUIRE(ps && cols1 && cols2 && n_out && stats_out, "sd_signedrank_rows: null pointer");
    SD_REQUIRE(ld_ps >= n_samples && ld_n >= 3 && ld_stats >= 4, "sd_signedrank_rows: ld too small");
    sd::signedrank::Params p{};
    p.n_samples = n_samples;
    p.ps = ps; p.ld_ps = ld_ps;
    p.n_pairs = n_pairs; p.cols1 = cols1; p.cols2 = cols2;
    p.npad = 1;
    while (p.npad < n_pairs) p.npad <<= 1;
    p.n_out = n_out; p.ld_n = ld_n; p.stats_out = stats_out; p.ld_stats = ld_stats;
    p.row_begin = row_begin; p.row_end = row_end;
    return dtype == SD_RANKSUM_F32 ? sd::signedrank::launch<float>(p, (cudaStream_t)stream)
                                   : sd::signedrank::launch<double>(p, (cudaStream_t)stream);
}

}  // extern "C"
