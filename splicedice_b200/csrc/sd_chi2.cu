// sd_chi2.cu -- K3 chi-squared: Yates-corrected chi-squared p for every (junction, sample pair).
//
// Replaces the `--chi2` branch of the reference's pairwise loop (scipy.stats.chi2_contingency per
// table, pairwise_fisher.py:133-134,179); the per-table arithmetic is in sd_chi2_math.cuh.
//
// Mapping: blockIdx.x picks 256 consecutive pairs, so each thread loads its pair's two sample indices
// once and walks the rows blockIdx.y, blockIdx.y + gridDim.y, ...; a warp's stores of one row are 256
// contiguous bytes.  One table is a few integer products and ~120 FP64 / MUFU instructions (erfc and
// the divides) against an 8-byte store.  Tables scipy refuses get NaN, and the smallest refused
// j * n_pairs + k is lowered into *first_refused: a running minimum per thread, a CTA reduction and at
// most one atomicMin per CTA (zero-margin tables are common, so per-warp atomics would pile up on one
// address).
#include <algorithm>

#include "sd_chi2_math.cuh"
#include "sd_common.cuh"

namespace sd {

constexpr int kChi2Threads = 256;

struct Chi2Params {
    int32_t n_samples;
    const int32_t *inc;
    int64_t ld_inc;
    const int64_t *exc;
    int64_t ld_exc;
    int64_t n_pairs;
    const int32_t *pair_a, *pair_b;
    double *p_out;
    int64_t ld_p;
    int64_t row_begin, row_end;
    unsigned long long *first_refused;   // nullable
};

__global__ void __launch_bounds__(kChi2Threads) chi2_pairwise_kernel(const Chi2Params p)
{
    const int64_t k = (int64_t)blockIdx.x * kChi2Threads + threadIdx.x;
    unsigned long long first = ~0ull;
    if (k < p.n_pairs) {
        const int sa = __ldg(p.pair_a + k), sb = __ldg(p.pair_b + k);
        for (int64_t j = p.row_begin + blockIdx.y; j < p.row_end; j += gridDim.y) {
            const int32_t *inc = p.inc + j * p.ld_inc;
            const int64_t *exc = p.exc + j * p.ld_exc;
            int status;
            const double pv = chi2::yates_p(__ldg(inc + sa), __ldg(inc + sb), __ldg(exc + sa), __ldg(exc + sb), &status);
            // rows ascend, so the first refusal a thread meets is its minimum
            if (chi2::refused(status) && first == ~0ull) first = (unsigned long long)j * p.n_pairs + k;
            __stcs(p.p_out + j * p.ld_p + k, pv);
        }
    }
    if (p.first_refused == nullptr) return;                  // uniform over the CTA
    __shared__ unsigned long long s_min[kChi2Threads / 32];
    for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = first;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kChi2Threads / 32; ++w) first = min(first, s_min[w]);
        if (first != ~0ull) atomicMin(p.first_refused, first);
    }
}

static int launch_chi2_pairwise(const Chi2Params &p, cudaStream_t stream)
{
    const int64_t tiles = (p.n_pairs + kChi2Threads - 1) / kChi2Threads;
    int per_sm = 0, dev = 0, sms = kSMs;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, chi2_pairwise_kernel, kChi2Threads, 0) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    SD_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // one resident wave: every CTA walks the same number of rows (to within one)
    const int64_t rows = p.row_end - p.row_begin;
    const int64_t y = std::max<int64_t>(1, std::min<int64_t>({(int64_t)sms * per_sm / tiles, rows, 65535}));
    chi2_pairwise_kernel<<<dim3((unsigned)tiles, (unsigned)y), kChi2Threads, 0, stream>>>(p);
    return check_launch("chi2_pairwise_kernel");
}

}  // namespace sd

extern "C" {

int sd_chi2_pairwise(int64_t n_junctions, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                     const int64_t *exc, int64_t ld_exc, int64_t n_pairs, const int32_t *pair_a,
                     const int32_t *pair_b, double *p_out, int64_t ld_p, int64_t row_begin, int64_t row_end,
                     uint64_t *first_refused, void *stream)
{
    // the checks of the Fisher entry points (sd_fisher.cu: pairwise_params)
    SD_REQUIRE(n_junctions >= 0 && n_samples >= 0 && n_pairs >= 0, "sd_chi2_pairwise: negative size");
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_junctions,
               "sd_chi2_pairwise: row range outside [0, n_junctions)");
    if (row_begin == row_end || n_pairs == 0) return SD_OK;
    SD_REQUIRE(inc && exc && pair_a && pair_b && p_out, "sd_chi2_pairwise: null pointer");
    SD_REQUIRE(ld_inc >= n_samples && ld_exc >= n_samples && ld_p >= n_pairs, "sd_chi2_pairwise: ld too small");
    SD_REQUIRE(n_pairs <= (int64_t)INT32_MAX * sd::kChi2Threads, "sd_chi2_pairwise: too many pairs");
    sd::Chi2Params p{};
    p.n_samples = n_samples;
    p.inc = inc; p.ld_inc = ld_inc; p.exc = exc; p.ld_exc = ld_exc;
    p.n_pairs = n_pairs; p.pair_a = pair_a; p.pair_b = pair_b;
    p.p_out = p_out; p.ld_p = ld_p;
    p.row_begin = row_begin; p.row_end = row_end;
    p.first_refused = reinterpret_cast<unsigned long long *>(first_refused);
    return sd::launch_chi2_pairwise(p, (cudaStream_t)stream);
}

}  // extern "C"
