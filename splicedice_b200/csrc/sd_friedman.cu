// sd_friedman.cu -- Friedman test per event across conditions measured on the same subjects
// (`compare_repeated`).
//
// For row j of a PS matrix, block (subject) b has one cell per condition c, ps[j, cols[c * n_blocks + b]];
// the test is scipy.stats.friedmanchisquare(*conditions, nan_policy='omit') (scipy 1.18.1) with the exact
// integer form of sd_friedman_math.cuh:
//     D_c = sum over complete blocks of (lo + hi + 1) - n (k + 1),   T = sum over cells of ((hi - lo)^2 - 1),
//     Q = 3 (k - 1) sum_c D_c^2 / (n (k^3 - k) - T),                 p = chi2.sf(Q, k - 1),
// lo / hi the cells of the same block below / at or below the cell.  Edge rules, and where scipy differs:
//   - a block with a NaN in any of its k cells is dropped; n = the complete blocks;
//   - n == 0: Q = p = NaN and NaN means (scipy: NaN too);
//   - every complete block tied throughout (the denominator 0): Q = p = NaN.  scipy's rounding gives NaN
//     for most such rows but +inf (p = 0) for some; p = 0 for identical values would top the BH list;
//   - every D_c == 0: Q = 0 and p = 1 exactly (scipy's rounding can give a tiny nonzero Q there);
//   - n == 1 is a valid test;
//   - cells are compared as the input type: IEEE order on float32 is the order of the float64-widened
//     values, -0.0 ties +0.0 and +-inf are ordinary values (the order of sd_ranksort.cuh's keys);
//   - the condition means are float64 sums over the complete blocks, reduced in a fixed order.
//
// Mapping: one CTA per row (rows blockIdx.x, + gridDim.x, ...; one resident wave); no sort.  The row's
// listed cells are staged once in shared memory in the column list's condition-major order, so a block's
// k cells sit n_blocks apart.  Each thread then takes cells: k compares against its block's cells (the
// lanes of a warp hold consecutive blocks of one condition, so they read consecutive words) give lo, hi
// and whether the block has a NaN; it stores lo + hi + 1 (0 in a dropped block) and adds its tie term.
// A warp per condition sums that condition's doubled ranks, counts and values in a shuffle tree and
// writes D_c^2 and the mean; warp 0 sums D_c^2 and the warps' tie terms, and lane 0 forms Q and p.  Every
// sum runs in a fixed order, so every output is deterministic.  The column list is checked once per CTA:
// a column outside [0, n_samples) is never dereferenced, and every row gets n = -1 and NaN means and
// statistics.
#include <algorithm>

#include "sd_common.cuh"
#include "sd_friedman_math.cuh"

namespace sd {
namespace friedman {

constexpr int kMaxCells = SD_RANKSUM_MAX_SAMPLES;
constexpr int kMaxConditions = SD_FRIEDMAN_MAX_CONDITIONS;
constexpr int kMaxThreads = 256;
constexpr int kMaxWarps = kMaxThreads / 32;
constexpr int kPre = 4;                    // cells per thread loaded a row ahead
// CTAs per SM the register allocation must allow: 5 (48 registers) for float32, which is latency-bound on
// its barriers and shuffle trees and gains from the extra CTA; the float64 build spills at 48, so 4 (64)
// for it
template <typename T>
constexpr int kMinBlocks = sizeof(T) == 4 ? 5 : 4;

struct Params {
    int32_t n_samples;
    const void *ps;
    int64_t ld_ps;
    int32_t k, n_blocks;
    int32_t step_b;                         // blockDim.x % n_blocks
    const int32_t *cols;
    int32_t *n_out;
    double *mean_out;
    int64_t ld_mean;
    double *stats_out;
    int64_t ld_stats;
    int64_t row_begin, row_end;
};

// the block of the cell blockDim.x after the one in block b
__device__ __forceinline__ int next_block(int b, int step, int nb)
{
    b += step;
    return b >= nb ? b - nb : b;
}

template <typename T>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks<T>) friedman_rows_kernel(const Params p)
{
    extern __shared__ uint64_t smem[];
    const int k = p.k, nb = p.n_blocks, cells = k * nb;
    long long *d2 = reinterpret_cast<long long *>(smem);             // D_c^2 per condition
    T *vals = reinterpret_cast<T *>(d2 + k);                          // the row's cells, condition-major
    int *rank2 = reinterpret_cast<int *>(vals + cells);               // lo + hi + 1; 0 in a dropped block
    int *hole = rank2 + cells;                                        // per block: the last row pass with a NaN
    __shared__ int s_ties[kMaxWarps];
    __shared__ int s_n, s_bad;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (threadIdx.x == 0) s_bad = 0;
    for (int b = threadIdx.x; b < nb; b += blockDim.x) hole[b] = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += blockDim.x)
        if ((unsigned)__ldg(p.cols + i) >= (unsigned)p.n_samples) s_bad = 1;
    __syncthreads();
    const bool bad = s_bad;
    const int b0 = threadIdx.x % nb;
    // the thread's first kPre cells of a row are loaded one row ahead, into registers, so that the next
    // row's reads are in flight while this row is ranked
    int col[kPre];
    T pre[kPre];
#pragma unroll
    for (int m = 0; m < kPre; ++m) {
        const int i = threadIdx.x + m * blockDim.x;
        col[m] = !bad && i < cells ? __ldg(p.cols + i) : -1;
    }
    const T *ps = static_cast<const T *>(p.ps);
    int64_t j = p.row_begin + blockIdx.x;
#pragma unroll
    for (int m = 0; m < kPre; ++m)
        if (col[m] >= 0 && j < p.row_end) pre[m] = __ldg(ps + j * p.ld_ps + col[m]);
    for (int pass = 0; j < p.row_end; j += gridDim.x, ++pass) {
        if (bad) {                                                    // uniform over the CTA
            for (int c = threadIdx.x; c < k; c += blockDim.x) __stcs(p.mean_out + j * p.ld_mean + c, nan);
            if (threadIdx.x == 0) {
                __stcs(p.n_out + j, -1);
                p.stats_out[j * p.ld_stats] = nan;
            }
            continue;
        }
        // stage: every listed cell once, and the blocks with a NaN stamped with this pass
        int b = b0;
#pragma unroll
        for (int m = 0; m < kPre; ++m) {
            if (col[m] >= 0) {
                vals[threadIdx.x + m * blockDim.x] = pre[m];
                if (isnan(pre[m])) hole[b] = pass;
            }
            b = next_block(b, p.step_b, nb);
        }
        const T *row = ps + j * p.ld_ps;
        for (int i = threadIdx.x + kPre * blockDim.x; i < cells; i += blockDim.x) {
            const T v = __ldg(row + __ldg(p.cols + i));
            vals[i] = v;
            if (isnan(v)) hole[b] = pass;
            b = next_block(b, p.step_b, nb);
        }
        __syncthreads();
        if (j + gridDim.x < p.row_end) {
#pragma unroll
            for (int m = 0; m < kPre; ++m)
                if (col[m] >= 0) pre[m] = __ldg(row + gridDim.x * p.ld_ps + col[m]);
        }
        // ranks within each complete block: k compares per cell against the cells n_blocks apart
        int ties = 0;
        b = b0;
        for (int i = threadIdx.x; i < cells; i += blockDim.x) {
            int r = 0;
            if (hole[b] != pass) {
                const T x = vals[i];
                const T *blk = vals + b;
                int lo = 0, hi = 0;
                for (int o = 0; o < k; ++o) {
                    const T y = blk[o * nb];
                    lo += y < x;
                    hi += y <= x;
                }
                r = lo + hi + 1;
                ties += (hi - lo) * (hi - lo) - 1;
            }
            rank2[i] = r;
            b = next_block(b, p.step_b, nb);
        }
        for (int o = 16; o; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
        if (lane == 0) s_ties[warp] = ties;
        __syncthreads();
        // per condition, one warp: doubled-rank sum, complete-block count and value sum in a shuffle tree
        for (int c = warp; c < k; c += warps) {
            const int *r = rank2 + c * nb;
            const T *v = vals + c * nb;
            int d = 0, cnt = 0;
            double s = 0.0;
            for (int bb = lane; bb < nb; bb += 32) {
                const int x = r[bb];
                if (x) {
                    d += x;
                    ++cnt;
                    s += (double)v[bb];
                }
            }
            for (int o = 16; o; o >>= 1) {
                d += __shfl_xor_sync(0xffffffffu, d, o);
                cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                s += __shfl_xor_sync(0xffffffffu, s, o);
            }
            if (lane == 0) {
                const long long dc = (long long)d - (long long)cnt * (k + 1);
                d2[c] = dc * dc;
                __stcs(p.mean_out + j * p.ld_mean + c, cnt ? s / cnt : nan);
                if (c == 0) s_n = cnt;
            }
        }
        __syncthreads();
        // warp 0: sum_c D_c^2 and T, then n and Q.  The other warps go on to the next row: its first
        // writes to what is read here (s_ties, d2, s_n) come after its staging barrier, which warp 0
        // reaches only when done.
        if (warp == 0) {
            long long sum = 0;
            int t = lane < warps ? s_ties[lane] : 0;
            for (int c = lane; c < k; c += 32) sum += d2[c];
            for (int o = 16; o; o >>= 1) {
                sum += __shfl_xor_sync(0xffffffffu, sum, o);
                t += __shfl_xor_sync(0xffffffffu, t, o);
            }
            if (lane == 0) {
                const int n = s_n;
                __stcs(p.n_out + j, n);
                p.stats_out[j * p.ld_stats] = q_stat(sum, n, k, t);
            }
        }
    }
    // epilogue: p of every row this CTA wrote, one row per thread, so the chi-square tail is not on the
    // row loop's critical path (the barrier makes the CTA's own Q stores visible to all its threads)
    __syncthreads();
    for (int64_t r = p.row_begin + blockIdx.x + (int64_t)threadIdx.x * gridDim.x; r < p.row_end;
         r += (int64_t)blockDim.x * gridDim.x) {
        const double q = p.stats_out[r * p.ld_stats];
        __stcs(p.stats_out + r * p.ld_stats + 1, p_value(k, q));
    }
}

template <typename T>
static int launch(Params p, cudaStream_t stream)
{
    const int cells = p.k * p.n_blocks;
    const int threads = std::min(kMaxThreads, (cells + 31) / 32 * 32);
    p.step_b = threads % p.n_blocks;
    const size_t smem = (size_t)p.k * sizeof(long long) + (size_t)cells * (sizeof(T) + sizeof(int)) +
                        (size_t)p.n_blocks * sizeof(int);
    SD_CHECK_CUDA(cudaFuncSetAttribute(friedman_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, friedman_rows_kernel<T>, threads, smem) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    SD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t rows = p.row_end - p.row_begin;
    const int64_t grid = std::min<int64_t>(rows, (int64_t)sms * per_sm);
    friedman_rows_kernel<T><<<(unsigned)grid, threads, smem, stream>>>(p);
    return check_launch("friedman_rows_kernel");
}

}  // namespace friedman
}  // namespace sd

extern "C" {

int sd_friedman_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                     int32_t n_conditions, int32_t n_blocks, const int32_t *cols,
                     int64_t row_begin, int64_t row_end,
                     int32_t *n_out, double *mean_out, int64_t ld_mean,
                     double *stats_out, int64_t ld_stats, void *stream)
{
    SD_REQUIRE(n_events >= 0 && n_samples >= 0, "sd_friedman_rows: negative size");
    SD_REQUIRE(n_conditions >= 3 && n_conditions <= sd::friedman::kMaxConditions,
               "sd_friedman_rows: n_conditions = %d outside [3, %d]", (int)n_conditions, sd::friedman::kMaxConditions);
    SD_REQUIRE(n_blocks >= 1 && (int64_t)n_blocks * n_conditions <= sd::friedman::kMaxCells,
               "sd_friedman_rows: n_blocks = %d (x %d conditions) outside [1, %d cells]", (int)n_blocks,
               (int)n_conditions, sd::friedman::kMaxCells);
    SD_REQUIRE(dtype == SD_RANKSUM_F32 || dtype == SD_RANKSUM_F64,
               "sd_friedman_rows: dtype must be SD_RANKSUM_F32 or SD_RANKSUM_F64");
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_events,
               "sd_friedman_rows: row range outside [0, n_events)");
    if (row_begin == row_end) return SD_OK;
    SD_REQUIRE(ps && cols && n_out && mean_out && stats_out, "sd_friedman_rows: null pointer");
    SD_REQUIRE(ld_ps >= n_samples && ld_mean >= n_conditions && ld_stats >= 2, "sd_friedman_rows: ld too small");
    sd::friedman::Params p{};
    p.n_samples = n_samples;
    p.ps = ps; p.ld_ps = ld_ps;
    p.k = n_conditions; p.n_blocks = n_blocks; p.cols = cols;
    p.n_out = n_out; p.mean_out = mean_out; p.ld_mean = ld_mean;
    p.stats_out = stats_out; p.ld_stats = ld_stats;
    p.row_begin = row_begin; p.row_end = row_end;
    return dtype == SD_RANKSUM_F32 ? sd::friedman::launch<float>(p, (cudaStream_t)stream)
                                   : sd::friedman::launch<double>(p, (cudaStream_t)stream);
}

}  // extern "C"
