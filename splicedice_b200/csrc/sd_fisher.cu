// sd_fisher.cu -- K3: two-sided Fisher exact test for every (junction, sample pair).
//
// Replaces the hot loop of pairwise_fisher.run_with
// (/root/reference/splicedice/pairwise_fisher.py:154-180) and scipy.stats.fisher_exact's
// two-sided branch; the per-table arithmetic is in sd_fisher_math.cuh.
//
// Mapping: one table per lane.  Default (every table total below 2^30): the cost-binned kernel --
// one persistent 1,024-thread CTA per SM made of four independent 256-thread groups that share a
// single shared-memory copy of the double-double log-factorial table; a group takes up to 2,048
// pairs of one junction, stages the junction's inclusion / exclusion row in shared memory,
// counting-sorts the pairs by predicted tail length and hands out groups of 32 similar pairs to
// its warps.  64-bit totals: one warp per (junction, 32-pair tile) in pair order.
// Entries beyond the staged table prefix come from the global copy through L1/L2.  The kernel is
// FP64-pipe / issue bound: 7 FP64 instructions per summed tail term, no division or exp in the
// loop, cut and rescale tests on the exponent words with integer instructions.
#include <algorithm>
#include <chrono>
#include <mutex>
#include <vector>

#include "sd_common.cuh"
#include "sd_fisher_math.cuh"
#include "sd_hostpipe.h"
#include "sd_lgtable.h"
#include "sd_quant.cuh"

namespace sd {

// kMode 0: every index is inside the staged shared-memory prefix; 1: shared prefix + global
// table; 2: as 1, plus the double-double Stirling series (fisher::lgfact_stirling) beyond the
// table cap.

template <int kMode>
struct DeviceTable {
    uint32_t smem;           // shared-window address of the staged prefix (32-bit: plain LDS, no generic loads)
    const double2 *gmem;     // full table
    int64_t n_smem, n_gmem;
    __device__ __forceinline__ static double2 lds2(uint32_t addr)
    {
        double2 v;
        asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
        return v;
    }
    __device__ __forceinline__ static double lds1(uint32_t addr)
    {
        double v;
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
        return v;
    }
    template <class Int>
    __device__ __forceinline__ double2 load(Int k) const
    {
        if (kMode == 0) return lds2(smem + (uint32_t)k * 16u);
        if ((int64_t)k < n_smem) return lds2(smem + (uint32_t)k * 16u);
        if (kMode == 1 || (int64_t)k < n_gmem) return __ldg(gmem + k);
        const fisher::dd v = fisher::lgfact_stirling(*this, (double)k);
        return make_double2(v.hi, v.lo);
    }
    // entries the table is guaranteed to hold (k < 4096 <= n_gmem): no fallback branch
    __device__ __forceinline__ fisher::dd in_table(int32_t k) const
    {
        const double2 v = (int64_t)k < n_smem ? lds2(smem + (uint32_t)k * 16u) : __ldg(gmem + k);
        return fisher::dd_make(v.x, v.y);
    }
    template <class Int>
    __device__ __forceinline__ double hi(Int k) const
    {
        if (kMode == 0) return lds1(smem + (uint32_t)k * 16u);
        return load(k).x;
    }
    template <class Int>
    __device__ __forceinline__ fisher::dd get(Int k) const
    {
        const double2 v = load(k);
        return fisher::dd_make(v.x, v.y);
    }
};

constexpr int kFisherThreads = 256;
constexpr int kMaxDest = 16;

struct FisherParams {
    int64_t n_junctions;
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
    const double2 *table;
    int64_t table_entries;
    int32_t smem_entries;
    int64_t cell_bound;      // caller-promised (or measured) upper bound on inc + exc; entries outside [0, bound] give NaN
    bool binned;             // cost-binned kernel (every table total below 2^30)
    // Scatter form (sd_fisher_pairwise_scatter): the pairs are cut into n_dest contiguous column
    // blocks [dest_col[g], dest_col[g + 1]) and the p-value of (row j, pair k) goes straight to block
    // owner g's matrix, dest[g][(dest_row0 + j) * dest_ld[g] + (k - dest_col[g])] -- the owners may be
    // other GPUs (peer memory over NVLink), which turns the row-slab -> column-block exchange of the
    // per-pair Benjamini-Hochberg correction into the kernel's own stores.
    int32_t n_dest;          // 0: plain p_out
    int32_t stage_out;       // binned kernel: byte offset (from the dynamic shared memory base) of kSub x kBinChunk doubles
                             // in which a chunk's p-values are collected and then stored in pair order; 0 = store directly
    int32_t dest_col[kMaxDest + 1];
    double *dest[kMaxDest];
    int64_t dest_ld[kMaxDest];
    int64_t dest_row0;
};

__device__ __forceinline__ void store_p(const FisherParams &p, int64_t j, int64_t k, double pv)
{
    if (p.n_dest == 0) {
        __stcs(p.p_out + j * p.ld_p + k, pv);
        return;
    }
    int g = 0;
#pragma unroll 1
    while (g + 1 < p.n_dest && k >= p.dest_col[g + 1]) ++g;
    p.dest[g][(p.dest_row0 + j) * p.dest_ld[g] + (k - p.dest_col[g])] = pv;
}

__device__ __forceinline__ void stage_table(double2 *s_tab, const double2 *g_tab, int n)
{
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_tab[i] = __ldg(g_tab + i);
    __syncthreads();
}

// Pair-order kernel: tables whose totals reach 2^30 (64-bit arithmetic), which always extend
// beyond the device table (mode 2).
__global__ void __launch_bounds__(kFisherThreads, 3) fisher_pairwise_kernel(const FisherParams p)
{
    extern __shared__ __align__(16) double2 s_tab[];
    stage_table(s_tab, p.table, p.smem_entries);
    const DeviceTable<2> tab{smem_u32(s_tab), p.table, p.smem_entries, p.table_entries};

    const int lane = threadIdx.x & 31;
    const int64_t tiles_per_row = (p.n_pairs + 31) / 32;
    const int64_t n_items = (p.row_end - p.row_begin) * tiles_per_row;
    const int64_t warp0 = (int64_t)blockIdx.x * (kFisherThreads / 32) + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * (kFisherThreads / 32);
    // (row, tile) of the first item and the per-iteration advance, so the loop has no division
    int64_t j = p.row_begin + warp0 / tiles_per_row;
    int64_t t = warp0 % tiles_per_row;
    const int64_t dj = n_warps / tiles_per_row, dt = n_warps % tiles_per_row;
    for (int64_t item = warp0; item < n_items; item += n_warps) {
        const int64_t k = t * 32 + lane;
        if (k < p.n_pairs) {
            const int sa = __ldg(p.pair_a + k), sb = __ldg(p.pair_b + k);
            const int32_t *inc = p.inc + j * p.ld_inc;
            const int64_t *exc = p.exc + j * p.ld_exc;
            const int64_t a64 = __ldg(inc + sa), b64 = __ldg(inc + sb), c64 = __ldg(exc + sa), d64 = __ldg(exc + sb);
            double pv;
            if (a64 < 0 || b64 < 0 || c64 < 0 || d64 < 0 || a64 + c64 > p.cell_bound || b64 + d64 > p.cell_bound)
                pv = __longlong_as_double(0x7FF8000000000000ll);
            else
                pv = fisher::two_sided<int64_t>(tab, a64, b64, c64, d64);
            store_p(p, j, k, pv);
        }
        j += dj;
        t += dt;
        if (t >= tiles_per_row) { t -= tiles_per_row; ++j; }
    }
}

// ---- binned form: lanes of a warp get tables of similar cost -----------------------------------
// The tail sums dominate the work and their length varies several-fold between the pairs of one
// junction (it grows with the hypergeometric sigma and shrinks with the observed table's
// distance from the mode), so in the pair-order kernel a warp waits for its longest lane: 56 % lane
// occupancy in the tail loops.  Here a CTA takes up to 2,048 pairs of one junction, predicts the
// number of tail terms of each table in binary32,
//     terms ~ sigma * (sqrt(z^2 + 2 ln 2^48) - z),   z = |a - mode| / sigma
// (correlation 0.99 with the true count), counting-sorts the pairs by that key in shared memory
// and lets its warps pull groups of 32 consecutive pairs, longest first, from an atomic counter.
constexpr int kBinChunk = 2048;
constexpr int kBinBuckets = 64;

// Only the ORDER of the pairs depends on this key, so it uses the approximate SFU forms
// (MUFU.RCP / RSQ / LG2) throughout: ~45 instructions per pair.
__device__ __forceinline__ int cost_bucket(int a, int b, int c, int d)
{
    const float fa = (float)a, fb = (float)b, fc = (float)c, fd = (float)d;
    const float n1 = fa + fb, n2 = fc + fd, n = fa + fc, N = n1 + n2;
    if (n1 == 0.f || n2 == 0.f || n == 0.f || fb + fd == 0.f) return 0;
    const float rN = __fdividef(1.f, N);
    const float mode = floorf((n + 1.f) * (n1 + 1.f) * __fdividef(1.f, N + 2.f));
    const float var = fmaxf((n * rN) * (n1 * rN) * (n2 * (N - n)) * __fdividef(1.f, fmaxf(N - 1.f, 1.f)), 1e-6f);
    const float inv_sig = rsqrtf(var);
    const float z = fabsf(fa - mode) * inv_sig;
    const float t = fmaf(z, z, 1.3863f * (float)fisher::kCutBits);    // 2 ln 2^kCutBits
    const float terms = var * inv_sig * (t * rsqrtf(t) - z);
    return min(kBinBuckets - 1, 1 + (int)(6.0f * __log2f(1.0f + terms)));
}

// kSub independent groups of 256 threads share one CTA (and one copy of the staged table): each
// group walks its own items and synchronises on its own named barrier, so a 768-thread CTA
// behaves like three 256-thread CTAs that need a single table in shared memory.
__device__ __forceinline__ void group_sync(int group)
{
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(kFisherThreads) : "memory");
}

// kStaged: the junction's inclusion / exclusion row (n_samples <= kStageSamples) is copied to
// shared memory once per item as int32 pairs, cells outside [0, cell_bound] marked -1, so both
// passes over the pairs read it with 32-bit shared addressing instead of 64-bit global gathers.
constexpr int kStageSamples = 512;
struct GroupBins {
    uint16_t perm[kBinChunk], rank[kBinChunk];
    uint8_t key[kBinChunk];
    int hist[kBinBuckets], base[kBinBuckets], next, pad[3];
    int32_t cell[2][kStageSamples];
};
static_assert(sizeof(GroupBins) % 16 == 0, "GroupBins must keep 16-byte alignment between groups");

// kPre (needs kStaged): the per-sample halves of every table's log-factorial sums
// (fisher::SampleTerms: lg[inc] + lg[exc] and log C(inc + exc, inc), 32 bytes per sample) are
// computed once per (junction, sample) while the row is staged and kept in shared memory behind
// the GroupBins, so a table needs 9 compensated additions and 7 table look-ups instead of 16
// and 21.  Used whenever the staged table leaves room for kSub * n_samples of them.
template <int kMode, int kSub, bool kStaged, bool kPre>
__global__ void __launch_bounds__(kFisherThreads *kSub, 1) fisher_pairwise_binned_kernel(const FisherParams p)
{
    // dynamic shared memory: the staged table, one GroupBins per 256-thread group, the per-sample terms
    extern __shared__ __align__(16) double2 s_tab[];
    stage_table(s_tab, p.table, p.smem_entries);
    const DeviceTable<kMode> tab{smem_u32(s_tab), p.table, p.smem_entries, p.table_entries};

    const int group = (int)(threadIdx.x / kFisherThreads);
    const int tid = (int)(threadIdx.x % kFisherThreads), lane = tid & 31;
    GroupBins &bins = reinterpret_cast<GroupBins *>(s_tab + p.smem_entries)[group];
    fisher::SampleTerms *s_pre =
        reinterpret_cast<fisher::SampleTerms *>(reinterpret_cast<GroupBins *>(s_tab + p.smem_entries) + kSub) +
        (size_t)group * p.n_samples;
    // scatter form: a chunk's p-values are collected here and written out in pair order, so that a warp
    // stores 256 contiguous bytes per destination instead of 32 scattered doubles (which would cross
    // NVLink as 32 separate 8-byte writes)
    double *s_out = p.stage_out ? reinterpret_cast<double *>(reinterpret_cast<char *>(s_tab) + p.stage_out) + (size_t)group * kBinChunk
                                : nullptr;
    uint16_t *s_perm = bins.perm, *s_rank = bins.rank;
    uint8_t *s_key = bins.key;
    int *s_hist = bins.hist, *s_base = bins.base, *s_next = &bins.next;
    int32_t *s_inc = bins.cell[0], *s_exc = bins.cell[1];
    const int64_t chunks_per_row = (p.n_pairs + kBinChunk - 1) / kBinChunk;
    const int64_t n_items = (p.row_end - p.row_begin) * chunks_per_row;
    // the four cells of pair k of the current junction; a < 0 flags a cell outside the promise
    auto cells = [&](const int32_t *inc, const int64_t *exc, int64_t k, int &a, int &b, int &c, int &d) {
        const int sa = __ldg(p.pair_a + k), sb = __ldg(p.pair_b + k);
        if (kStaged) {
            a = s_inc[sa] | s_inc[sb]; b = s_inc[sb]; c = s_exc[sa]; d = s_exc[sb];
            if (a >= 0) a = s_inc[sa];
        } else {
            const int32_t ia = __ldg(inc + sa), ib = __ldg(inc + sb);
            const int64_t ea = __ldg(exc + sa), eb = __ldg(exc + sb);
            const bool bad = ia < 0 || ib < 0 || ea < 0 || eb < 0 || ia + ea > p.cell_bound || ib + eb > p.cell_bound;
            a = bad ? -1 : ia; b = ib; c = (int)ea; d = (int)eb;
        }
    };
    for (int64_t item = (int64_t)blockIdx.x * kSub + group; item < n_items; item += (int64_t)gridDim.x * kSub) {
        const int64_t j = p.row_begin + item / chunks_per_row;
        const int64_t k0 = (item % chunks_per_row) * kBinChunk;
        const int cnt = (int)min((int64_t)kBinChunk, p.n_pairs - k0);
        const int32_t *inc = p.inc + j * p.ld_inc;
        const int64_t *exc = p.exc + j * p.ld_exc;

        if (tid < kBinBuckets) s_hist[tid] = 0;
        if (tid == 0) *s_next = 0;
        if (kStaged) {
            for (int sm = tid; sm < p.n_samples; sm += kFisherThreads) {
                const int32_t ia = __ldg(inc + sm);
                const int64_t ea = __ldg(exc + sm);
                const bool bad = ia < 0 || ea < 0 || ia + ea > p.cell_bound;
                s_inc[sm] = bad ? -1 : ia;
                s_exc[sm] = bad ? -1 : (int32_t)ea;
                if (kPre && !bad) s_pre[sm] = fisher::sample_terms(tab, ia, (int32_t)ea);
            }
        }
        group_sync(group);
        // cost key of each pair and its rank inside the key's bucket
#pragma unroll 1
        for (int q = tid; q < cnt; q += kFisherThreads) {
            int a, b, c, d;
            cells(inc, exc, k0 + q, a, b, c, d);
            const int key = a < 0 ? 0 : cost_bucket(a, b, c, d);
            s_key[q] = (uint8_t)key;
            s_rank[q] = (uint16_t)atomicAdd(&s_hist[key], 1);
        }
        group_sync(group);
        if (tid < 32) {                         // descending key order: the costliest groups start first
            const int h1 = s_hist[kBinBuckets - 1 - 2 * tid], h2 = s_hist[kBinBuckets - 2 - 2 * tid];
            int incl = h1 + h2;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += up;
            }
            s_base[kBinBuckets - 1 - 2 * tid] = incl - h1 - h2;
            s_base[kBinBuckets - 2 - 2 * tid] = incl - h2;
        }
        group_sync(group);
#pragma unroll 1
        for (int q = tid; q < cnt; q += kFisherThreads) s_perm[s_base[s_key[q]] + s_rank[q]] = (uint16_t)q;
        group_sync(group);

        const int groups = (cnt + 31) / 32;
        for (;;) {
            int g = 0;
            if (lane == 0) g = atomicAdd(s_next, 1);
            g = __shfl_sync(0xffffffffu, g, 0);
            if (g >= groups) break;
            const int slot = g * 32 + lane;
            if (slot < cnt) {
                const int64_t k = k0 + s_perm[slot];
                int a, b, c, d;
                double pv;
                if (kPre) {
                    const int sa = __ldg(p.pair_a + k), sb = __ldg(p.pair_b + k);
                    a = s_inc[sa] | s_inc[sb]; b = s_inc[sb]; c = s_exc[sa]; d = s_exc[sb];
                    if (a < 0)
                        pv = __longlong_as_double(0x7FF8000000000000ll);  // outside the promised range: loud, not wrong
                    else
                        pv = fisher::two_sided_pre<int32_t>(tab, s_inc[sa], b, c, d, s_pre[sa], s_pre[sb]);
                } else {
                    cells(inc, exc, k, a, b, c, d);
                    if (a < 0)
                        pv = __longlong_as_double(0x7FF8000000000000ll);
                    else
                        pv = fisher::two_sided<int32_t>(tab, a, b, c, d);
                }
                if (s_out) s_out[s_perm[slot]] = pv;
                else store_p(p, j, k, pv);
            }
        }
        if (s_out) {
            group_sync(group);
            for (int q = tid; q < cnt; q += kFisherThreads) store_p(p, j, k0 + q, s_out[q]);
        }
        group_sync(group);                      // s_perm / s_hist / the staged row are rebuilt by the next item
    }
}

template <class Int, int kMode>
__global__ void __launch_bounds__(kFisherThreads, 2) fisher_tables_kernel(
    int64_t n, const int64_t *__restrict__ a, const int64_t *__restrict__ b,
    const int64_t *__restrict__ c, const int64_t *__restrict__ d, double *__restrict__ out,
    const double2 *table, int64_t table_entries, int32_t smem_entries)
{
    extern __shared__ __align__(16) double2 s_tab[];
    stage_table(s_tab, table, smem_entries);
    const DeviceTable<kMode> tab{smem_u32(s_tab), table, smem_entries, table_entries};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = fisher::two_sided<Int>(tab, (Int)a[i], (Int)b[i], (Int)c[i], (Int)d[i]);
}

// max over the row range of inc + exc (pairwise) or of a + b + c + d (tables); also flags
// negative entries (scipy raises ValueError on them, stats/_stats_py.py:5048-5049)
__global__ void __launch_bounds__(256) fisher_scan_pairwise(const FisherParams p, unsigned long long *max_out,
                                                            int *neg_out)
{
    const int64_t cells = (p.row_end - p.row_begin) * p.n_samples;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long m = 0;
    int neg = 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < cells; g += stride) {
        const int64_t j = p.row_begin + g / p.n_samples;
        const int s = (int)(g % p.n_samples);
        const int64_t a = p.inc[j * p.ld_inc + s], c = p.exc[j * p.ld_exc + s];
        if (a < 0 || c < 0) neg = 1;
        else m = max(m, (unsigned long long)(a + c));
    }
    for (int o = 16; o; o >>= 1) {
        m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        neg |= __shfl_xor_sync(0xffffffffu, neg, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (m) atomicMax(max_out, m);
        if (neg) atomicOr(neg_out, 1);
    }
}

__global__ void __launch_bounds__(256) fisher_scan_tables(int64_t n, const int64_t *a, const int64_t *b,
                                                          const int64_t *c, const int64_t *d,
                                                          unsigned long long *max_out, int *neg_out)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long m = 0;
    int neg = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (a[i] < 0 || b[i] < 0 || c[i] < 0 || d[i] < 0) neg = 1;
        else m = max(m, (unsigned long long)(a[i] + b[i] + c[i] + d[i]));
    }
    for (int o = 16; o; o >>= 1) {
        m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        neg |= __shfl_xor_sync(0xffffffffu, neg, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (m) atomicMax(max_out, m);
        if (neg) atomicOr(neg_out, 1);
    }
}

// ---- device copies of the table: one per device, grown on demand, never shrunk ----------
namespace {
constexpr int64_t kTableCap = int64_t(1) << 22;      // 4 Mi entries = 64 MB; beyond: fisher::lgfact_stirling
// totals that need 64-bit integers are always beyond the table: their kernels need table mode 2 only
static_assert(kTableCap < (int64_t(1) << 30), "64-bit totals must lie beyond the device table");
constexpr int kMaxDevices = 64;
std::mutex g_tab_mu;
double2 *g_tab_dev[kMaxDevices] = {};
int64_t g_tab_entries[kMaxDevices] = {};
}  // namespace

// Returns a device table with at least min(need, kTableCap) entries for the current device.
// Grows by reallocation; the old block is left allocated (kernels in flight may still read it)
// -- at most log2(cap) of them over the life of the process.
static int device_table(int64_t need, const double2 **table, int64_t *entries, cudaStream_t stream)
{
    int dev = 0;
    SD_CHECK_CUDA(cudaGetDevice(&dev));
    if (dev >= kMaxDevices) return fail(SD_ERR_UNSUPPORTED, "device ordinal %d too large", dev);
    need = std::min(std::max<int64_t>(need, 4096), kTableCap);
    std::lock_guard<std::mutex> lock(g_tab_mu);
    if (g_tab_entries[dev] < need) {
        int64_t n = 4096;
        while (n < need) n <<= 1;
        std::vector<double> host;
        lgtable_host(n, &host);
        double2 *d = nullptr;
        SD_CHECK_CUDA(cudaMalloc(&d, (size_t)n * sizeof(double2)));
        SD_CHECK_CUDA(cudaMemcpyAsync(d, host.data(), (size_t)n * sizeof(double2), cudaMemcpyHostToDevice, stream));
        SD_CHECK_CUDA(cudaStreamSynchronize(stream));    // `host` dies at scope exit
        g_tab_dev[dev] = d;
        g_tab_entries[dev] = n;
    }
    *table = g_tab_dev[dev];
    *entries = g_tab_entries[dev];
    return SD_OK;
}

constexpr int kSmemEntriesMax = 6144;      // 96 KB of double2: two CTAs per SM
constexpr int kSmemEntriesBinned = 10240;  // binned kernel: one CTA per SM, 160 KB of table + 60 KB of bins / staged rows

static int scan_result(unsigned long long *d_max, int *d_neg, cudaStream_t stream, int64_t *max_total,
                       const char *who)
{
    unsigned long long h_max = 0;
    int h_neg = 0;
    SD_CHECK_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof h_max, cudaMemcpyDeviceToHost, stream));
    SD_CHECK_CUDA(cudaMemcpyAsync(&h_neg, d_neg, sizeof h_neg, cudaMemcpyDeviceToHost, stream));
    SD_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (h_neg) return fail(SD_ERR_INVALID, "%s: all table entries must be non-negative", who);
    *max_total = (int64_t)h_max;
    return SD_OK;
}

static int fisher_grid(const void *kernel, size_t smem, int threads = kFisherThreads)
{
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    int dev = 0, sms = kSMs;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms * per_sm;
}

// table coverage of the largest table total: 0 inside the staged prefix, 1 inside the device
// table, 2 beyond it (Stirling series)
static int table_mode(int64_t max_total, int64_t smem_entries, int64_t table_entries)
{
    return max_total < smem_entries ? 0 : (max_total < table_entries ? 1 : 2);
}

// every table total fits 31 bits: the cost-binned kernel
template <int kMode>
struct BinnedLauncher {
    template <int kSub, bool kStaged>
    static int launch_binned(const FisherParams &p, cudaStream_t stream)
    {
        constexpr size_t kMaxSmem = kSmemEntriesBinned * sizeof(double2) + kSub * sizeof(GroupBins);
        const size_t base = (size_t)p.smem_entries * sizeof(double2) + kSub * sizeof(GroupBins);
        const size_t pre = (size_t)kSub * p.n_samples * sizeof(fisher::SampleTerms);
        const bool use_pre = kStaged && base + pre <= kMaxSmem && !getenv("SD_FISHER_NO_PRE");
        auto kernel = use_pre ? fisher_pairwise_binned_kernel<kMode, kSub, kStaged, kStaged>
                              : fisher_pairwise_binned_kernel<kMode, kSub, kStaged, false>;
        size_t smem = base + (use_pre ? pre : 0);
        FisherParams q = p;
        const size_t stage = (size_t)kSub * kBinChunk * sizeof(double);
        if (p.n_dest > 0 && smem + stage <= kMaxSmem) {          // scatter form with room to collect a chunk's outputs
            q.stage_out = (int32_t)smem;
            smem += stage;
        }
        SD_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
        const int64_t items = (p.row_end - p.row_begin) * ((p.n_pairs + kBinChunk - 1) / kBinChunk);
        int grid = fisher_grid((const void *)kernel, smem, kFisherThreads * kSub);
        grid = (int)std::min<int64_t>(grid, (items + kSub - 1) / kSub);
        kernel<<<grid, kFisherThreads * kSub, smem, stream>>>(q);
        return check_launch("fisher_pairwise_binned_kernel");
    }
    static int run(const FisherParams &p, cudaStream_t stream)
    {
        // 4 x 256 threads per SM when the whole table is staged (64 registers, no spills), 3 x 256 otherwise
        constexpr int kSub = kMode == 0 ? 4 : 3;
        return p.n_samples <= kStageSamples ? launch_binned<kSub, true>(p, stream)
                                            : launch_binned<kSub, false>(p, stream);
    }
};

static int launch_pair_order(const FisherParams &p, cudaStream_t stream)
{
    auto kernel = fisher_pairwise_kernel;
    const size_t smem = (size_t)p.smem_entries * sizeof(double2);
    SD_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(kSmemEntriesMax * sizeof(double2))));
    const int64_t items = (p.row_end - p.row_begin) * ((p.n_pairs + 31) / 32);
    int grid = fisher_grid((const void *)kernel, smem);
    grid = (int)std::min<int64_t>(grid, (items + kFisherThreads / 32 - 1) / (kFisherThreads / 32));
    kernel<<<grid, kFisherThreads, smem, stream>>>(p);
    return check_launch("fisher_pairwise_kernel");
}

template <class Int, int kMode>
static int launch_tables(int64_t n, const int64_t *a, const int64_t *b, const int64_t *c, const int64_t *d, double *out,
                         const double2 *table, int64_t entries, int32_t smem_entries, cudaStream_t stream)
{
    auto kernel = fisher_tables_kernel<Int, kMode>;
    const size_t smem = (size_t)smem_entries * sizeof(double2);
    SD_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(kSmemEntriesMax * sizeof(double2))));
    int grid = fisher_grid((const void *)kernel, smem);
    grid = (int)std::min<int64_t>(grid, (n + kFisherThreads - 1) / kFisherThreads);
    kernel<<<grid, kFisherThreads, smem, stream>>>(n, a, b, c, d, out, table, entries, smem_entries);
    return check_launch("fisher_tables_kernel");
}

// instantiation of fisher_tables_kernel for (largest table total, table coverage)
template <class... Args>
static int dispatch(int64_t max_total, int64_t smem_entries, int64_t table_entries, Args... args)
{
    if (max_total >= (int64_t(1) << 30)) return launch_tables<int64_t, 2>(args...);
    switch (table_mode(max_total, smem_entries, table_entries)) {
    case 0: return launch_tables<int32_t, 0>(args...);
    case 1: return launch_tables<int32_t, 1>(args...);
    default: return launch_tables<int32_t, 2>(args...);
    }
}

// max over rows [row_begin, row_end) of inc + exc (a table total is at most twice that);
// SD_ERR_INVALID on a negative entry.  Synchronises the stream.
int fisher_max_cell(const FisherParams &p, cudaStream_t stream, int64_t *max_cell)
{
    unsigned long long *d_max = nullptr;
    SD_CHECK_CUDA(cudaMallocAsync(&d_max, 16, stream));
    SD_CHECK_CUDA(cudaMemsetAsync(d_max, 0, 16, stream));
    int *d_neg = reinterpret_cast<int *>(d_max + 1);
    const int64_t cells = (p.row_end - p.row_begin) * p.n_samples;
    fisher_scan_pairwise<<<(int)std::min<int64_t>((cells + 255) / 256, kSMs * 8), 256, 0, stream>>>(p, d_max, d_neg);
    int rc = scan_result(d_max, d_neg, stream, max_cell, "sd_fisher_pairwise");
    cudaFreeAsync(d_max, stream);
    return rc;
}

// max_cell < 0: measure it first (one stream synchronisation)
int launch_fisher_pairwise(FisherParams p, cudaStream_t stream, int64_t max_cell)
{
    if (max_cell < 0)
        if (int rc = fisher_max_cell(p, stream, &max_cell)) return rc;
    const int64_t max_total = 2 * max_cell;
    p.cell_bound = max_cell;
    p.binned = max_total < (int64_t(1) << 30);
    if (int rc = device_table(max_total + 1, &p.table, &p.table_entries, stream)) return rc;
    p.smem_entries = (int32_t)std::min<int64_t>(std::min<int64_t>(max_total + 1, p.table_entries),
                                                p.binned ? kSmemEntriesBinned : kSmemEntriesMax);
    if (!p.binned) return launch_pair_order(p, stream);
    switch (table_mode(max_total, p.smem_entries, p.table_entries)) {
    case 0: return BinnedLauncher<0>::run(p, stream);
    case 1: return BinnedLauncher<1>::run(p, stream);
    default: return BinnedLauncher<2>::run(p, stream);
    }
}

// Checks and FisherParams fill shared by the device-pointer entry points (`who` names the entry point
// in the messages); *empty: no rows or no pairs, nothing to launch.
static int pairwise_params(const char *who, int64_t n_junctions, int32_t n_samples, const int32_t *inc,
                           int64_t ld_inc, const int64_t *exc, int64_t ld_exc, int64_t n_pairs, const int32_t *pair_a,
                           const int32_t *pair_b, int64_t row_begin, int64_t row_end, FisherParams *p, bool *empty)
{
    SD_REQUIRE(n_junctions >= 0 && n_samples >= 0 && n_pairs >= 0, "%s: negative size", who);
    SD_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n_junctions,
               "%s: row range outside [0, n_junctions)", who);
    *empty = row_begin == row_end || n_pairs == 0;
    if (*empty) return SD_OK;
    SD_REQUIRE(inc && exc && pair_a && pair_b, "%s: null pointer", who);
    SD_REQUIRE(ld_inc >= n_samples && ld_exc >= n_samples, "%s: ld too small", who);
    *p = FisherParams{};
    p->n_junctions = n_junctions; p->n_samples = n_samples;
    p->inc = inc; p->ld_inc = ld_inc; p->exc = exc; p->ld_exc = ld_exc;
    p->n_pairs = n_pairs; p->pair_a = pair_a; p->pair_b = pair_b;
    p->row_begin = row_begin; p->row_end = row_end;
    return SD_OK;
}

}  // namespace sd

extern "C" {

int sd_fisher_pairwise(int64_t n_junctions, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                       const int64_t *exc, int64_t ld_exc, int64_t n_pairs, const int32_t *pair_a,
                       const int32_t *pair_b, double *p_out, int64_t ld_p, int64_t row_begin,
                       int64_t row_end, void *stream)
{
    sd::FisherParams p;
    bool empty;
    if (int rc = sd::pairwise_params("sd_fisher_pairwise", n_junctions, n_samples, inc, ld_inc, exc, ld_exc, n_pairs,
                                     pair_a, pair_b, row_begin, row_end, &p, &empty))
        return rc;
    if (empty) return SD_OK;
    SD_REQUIRE(p_out, "sd_fisher_pairwise: null pointer");
    SD_REQUIRE(ld_p >= n_pairs, "sd_fisher_pairwise: ld too small");
    p.p_out = p_out; p.ld_p = ld_p;
    return sd::launch_fisher_pairwise(p, (cudaStream_t)stream, -1);
}

int sd_fisher_pairwise_bounded(int64_t n_junctions, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                               const int64_t *exc, int64_t ld_exc, int64_t n_pairs, const int32_t *pair_a,
                               const int32_t *pair_b, double *p_out, int64_t ld_p, int64_t row_begin,
                               int64_t row_end, int64_t max_cell_bound, void *stream)
{
    SD_REQUIRE(max_cell_bound >= 0 && max_cell_bound < (int64_t(1) << 61), "sd_fisher_pairwise_bounded: bad bound");
    sd::FisherParams p;
    bool empty;
    if (int rc = sd::pairwise_params("sd_fisher_pairwise_bounded", n_junctions, n_samples, inc, ld_inc, exc, ld_exc,
                                     n_pairs, pair_a, pair_b, row_begin, row_end, &p, &empty))
        return rc;
    if (empty) return SD_OK;
    SD_REQUIRE(p_out, "sd_fisher_pairwise_bounded: null pointer");
    SD_REQUIRE(ld_p >= n_pairs, "sd_fisher_pairwise_bounded: ld too small");
    p.p_out = p_out; p.ld_p = ld_p;
    return sd::launch_fisher_pairwise(p, (cudaStream_t)stream, max_cell_bound);
}

int sd_fisher_pairwise_scatter(int64_t n_junctions, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                               const int64_t *exc, int64_t ld_exc, int64_t n_pairs, const int32_t *pair_a,
                               const int32_t *pair_b, int32_t n_dest, double *const *dest, const int64_t *dest_col_begin,
                               const int64_t *dest_ld, int64_t dest_row_offset, int64_t row_begin, int64_t row_end,
                               int64_t max_cell_bound, void *stream)
{
    SD_REQUIRE(max_cell_bound >= 0 && max_cell_bound < (int64_t(1) << 61), "sd_fisher_pairwise_scatter: bad bound");
    SD_REQUIRE(n_dest >= 1 && n_dest <= sd::kMaxDest, "sd_fisher_pairwise_scatter: 1..%d destinations", sd::kMaxDest);
    SD_REQUIRE(n_pairs < (int64_t(1) << 31), "sd_fisher_pairwise_scatter: too many pairs");
    sd::FisherParams p;
    bool empty;
    if (int rc = sd::pairwise_params("sd_fisher_pairwise_scatter", n_junctions, n_samples, inc, ld_inc, exc, ld_exc,
                                     n_pairs, pair_a, pair_b, row_begin, row_end, &p, &empty))
        return rc;
    if (empty) return SD_OK;
    SD_REQUIRE(dest && dest_col_begin && dest_ld, "sd_fisher_pairwise_scatter: null pointer");
    SD_REQUIRE(dest_col_begin[0] == 0 && dest_col_begin[n_dest] == n_pairs,
               "sd_fisher_pairwise_scatter: the column blocks must cover [0, n_pairs)");
    p.n_dest = n_dest; p.dest_row0 = dest_row_offset;
    for (int g = 0; g < n_dest; ++g) {
        const int64_t width = dest_col_begin[g + 1] - dest_col_begin[g];
        SD_REQUIRE(width >= 0 && (width == 0 || (dest[g] && dest_ld[g] >= width)),
                   "sd_fisher_pairwise_scatter: destination %d: null pointer or ld below its %lld columns", g, (long long)width);
        p.dest[g] = dest[g]; p.dest_ld[g] = dest_ld[g]; p.dest_col[g] = (int32_t)dest_col_begin[g];
    }
    p.dest_col[n_dest] = (int32_t)n_pairs;
    return sd::launch_fisher_pairwise(p, (cudaStream_t)stream, max_cell_bound);
}

int sd_fisher_tables(int64_t n_tables, const int64_t *a, const int64_t *b, const int64_t *c,
                     const int64_t *d, double *p_out, void *stream_)
{
    SD_REQUIRE(n_tables >= 0, "sd_fisher_tables: negative size");
    if (n_tables == 0) return SD_OK;
    SD_REQUIRE(a && b && c && d && p_out, "sd_fisher_tables: null pointer");
    cudaStream_t stream = (cudaStream_t)stream_;
    unsigned long long *d_max = nullptr;
    SD_CHECK_CUDA(cudaMallocAsync(&d_max, 16, stream));
    SD_CHECK_CUDA(cudaMemsetAsync(d_max, 0, 16, stream));
    int *d_neg = reinterpret_cast<int *>(d_max + 1);
    sd::fisher_scan_tables<<<(int)std::min<int64_t>((n_tables + 255) / 256, sd::kSMs * 8), 256, 0, stream>>>(
        n_tables, a, b, c, d, d_max, d_neg);
    int64_t max_total = 0;
    int rc = sd::scan_result(d_max, d_neg, stream, &max_total, "sd_fisher_tables");
    cudaFreeAsync(d_max, stream);
    if (rc != SD_OK) return rc;
    const double2 *table = nullptr;
    int64_t entries = 0;
    if ((rc = sd::device_table(max_total + 1, &table, &entries, stream)) != SD_OK) return rc;
    const int32_t smem_entries =
        (int32_t)std::min<int64_t>(std::min<int64_t>(max_total + 1, entries), sd::kSmemEntriesMax);
    return sd::dispatch(max_total, (int64_t)smem_entries, entries, n_tables, a, b, c, d, p_out, table, entries,
                        smem_entries, stream);
}

}  // extern "C"

namespace sd {

// Host-buffer pipeline shared by sd_fisher_pairwise_host (exclusion counts given) and sd_pairwise_host
// (exclusion counts computed on the device from the inclusion counts and the cluster CSR): row blocks
// of p-values are computed on one stream and copied back on another, so the 8 B/test of D2H traffic
// -- the bound: 3.2 GB against 19 ms of FP64 work at 200,000 x 2,016 -- overlaps the kernels.  The
// first blocks are small so that the copy-back stream starts within a fraction of a millisecond.
static int pairwise_host_impl(const char *who, int device, int64_t J, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                              const int64_t *exc, int64_t ld_exc, const int32_t *row_ptr, const int32_t *col_idx,
                              int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b, double *p_out, int64_t ld_p)
{
    for (int64_t k = 0; k < n_pairs; ++k)
        if (!(pair_a[k] >= 0 && pair_a[k] < n_samples && pair_b[k] >= 0 && pair_b[k] < n_samples))
            return fail(SD_ERR_INVALID, "%s: pair %lld out of range", who, (long long)k);
    int64_t nnz = 0;
    if (!exc) {
        nnz = row_ptr[J];
        if (nnz < 0 || (nnz > 0 && !col_idx)) return fail(SD_ERR_INVALID, "%s: bad CSR", who);
        for (int64_t k = 0; k < nnz; ++k)
            if (col_idx[k] < 0 || col_idx[k] >= J)
                return fail(SD_ERR_INVALID, "%s: col_idx[%lld] = %d out of range", who, (long long)k, col_idx[k]);
    }
    const bool debug = getenv("SD_HOST_PIPE_DEBUG") != nullptr;
    using clk = std::chrono::steady_clock;
    const auto t_begin = clk::now();
    int prev_dev = 0;
    SD_CHECK_CUDA(cudaGetDevice(&prev_dev));
    SD_CHECK_CUDA(cudaSetDevice(device));
    // streams and device memory come from the per-device context the host-buffer calls share: they
    // live across calls, and the pool is private to the library (the process-wide default pool keeps
    // its settings)
    HostLease lease;
    if (int lrc = host_lease(device, &lease)) { cudaSetDevice(prev_dev); return lrc; }
    cudaStream_t s_k = lease.s_k, s_out = lease.s_out;
    int32_t *d_inc = nullptr, *d_pa = nullptr, *d_pb = nullptr, *d_rp = nullptr, *d_ci = nullptr;
    int64_t *d_exc = nullptr;
    double *d_p = nullptr;
    std::vector<cudaEvent_t> ev;
    int rc = SD_OK;
    // every exit path: drain both streams before the buffers go back to the pool
    auto cleanup = [&]() {
        cudaStreamSynchronize(s_out);
        cudaStreamSynchronize(s_k);
        for (auto e : ev) if (e) cudaEventDestroy(e);
        for (void *q : {(void *)d_inc, (void *)d_exc, (void *)d_pa, (void *)d_pb, (void *)d_p, (void *)d_rp, (void *)d_ci})
            if (q) cudaFreeAsync(q, s_k);
        cudaStreamSynchronize(s_k);
        cudaSetDevice(prev_dev);
    };
#define SD_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            rc = sd::fail(SD_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                          __LINE__);                                                              \
            cleanup();                                                                            \
            return rc;                                                                            \
        }                                                                                         \
    } while (0)
    // p-value blocks of ~64 MB, double buffered, after a ramp of 2, 8 and 32 MB
    // (tuning knob for experiments: SD_FISHER_HOST_BLOCK_MB)
    int64_t block_mb = 64;
    if (const char *env = getenv("SD_FISHER_HOST_BLOCK_MB")) block_mb = std::max<int64_t>(1, atoll(env));
    const int64_t full_rows = std::min<int64_t>(J, std::max<int64_t>(1, (block_mb << 20) / (n_pairs * 8)));
    std::vector<int64_t> cut{0};
    for (int64_t rows = std::max<int64_t>(1, full_rows / 32); cut.back() < J; rows = std::min(full_rows, rows * 4))
        cut.push_back(std::min(J, cut.back() + rows));
    const int64_t n_blocks = (int64_t)cut.size() - 1;
    const int64_t ldd = (n_samples + 3) & ~(int64_t)3;           // device leading dimension of the count matrices
    SD_TRY(cudaMallocFromPoolAsync(&d_inc, (size_t)J * ldd * 4, lease.pool, s_k));
    SD_TRY(cudaMallocFromPoolAsync(&d_exc, (size_t)J * ldd * 8, lease.pool, s_k));
    SD_TRY(cudaMallocFromPoolAsync(&d_pa, (size_t)n_pairs * 4, lease.pool, s_k));
    SD_TRY(cudaMallocFromPoolAsync(&d_pb, (size_t)n_pairs * 4, lease.pool, s_k));
    SD_TRY(cudaMallocFromPoolAsync(&d_p, (size_t)2 * full_rows * n_pairs * 8, lease.pool, s_k));
    if (ldd != n_samples) SD_TRY(cudaMemsetAsync(d_inc, 0, (size_t)J * ldd * 4, s_k));
    SD_TRY(cudaMemcpy2DAsync(d_inc, (size_t)ldd * 4, inc, (size_t)ld_inc * 4, (size_t)n_samples * 4, (size_t)J,
                             cudaMemcpyHostToDevice, s_k));
    if (exc) {
        SD_TRY(cudaMemcpy2DAsync(d_exc, (size_t)ldd * 8, exc, (size_t)ld_exc * 8, (size_t)n_samples * 8, (size_t)J,
                                 cudaMemcpyHostToDevice, s_k));
    } else {
        // exclusion counts on the device: 4 B per cell cross the link instead of 12
        SD_TRY(cudaMallocFromPoolAsync(&d_rp, (size_t)(J + 1) * 4, lease.pool, s_k));
        SD_TRY(cudaMallocFromPoolAsync(&d_ci, (size_t)std::max<int64_t>(nnz, 1) * 4, lease.pool, s_k));
        SD_TRY(cudaMemcpyAsync(d_rp, row_ptr, (size_t)(J + 1) * 4, cudaMemcpyHostToDevice, s_k));
        if (nnz) SD_TRY(cudaMemcpyAsync(d_ci, col_idx, (size_t)nnz * 4, cudaMemcpyHostToDevice, s_k));
        QuantParams q{};
        q.n_junctions = J; q.n_samples = n_samples;
        q.counts = d_inc; q.ld_counts = ldd;
        q.row_ptr = d_rp; q.col_idx = d_ci;
        q.exc = d_exc; q.ld_exc = ldd;
        q.row_begin = 0; q.row_end = J;
        rc = launch_quant(q, SD_QUANT_AUTO, s_k);
        if (rc != SD_OK) { cleanup(); return rc; }
    }
    SD_TRY(cudaMemcpyAsync(d_pa, pair_a, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s_k));
    SD_TRY(cudaMemcpyAsync(d_pb, pair_b, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s_k));
    int64_t max_cell = 0;
    {
        FisherParams all{};
        all.n_samples = n_samples; all.inc = d_inc; all.ld_inc = ldd; all.exc = d_exc; all.ld_exc = ldd;
        all.row_begin = 0; all.row_end = J;
        rc = fisher_max_cell(all, s_k, &max_cell);
        if (rc != SD_OK) { cleanup(); return rc; }
    }
    const auto t_scanned = clk::now();
    ev.resize((size_t)2 * n_blocks, nullptr);
    for (auto &e : ev) SD_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (int64_t b = 0; b < n_blocks; ++b) {
        const int64_t r0 = cut[b], r1 = cut[b + 1];
        double *buf = d_p + (b & 1) * full_rows * n_pairs;
        if (b >= 2) SD_TRY(cudaStreamWaitEvent(s_k, ev[2 * (b - 2) + 1], 0));   // buffer drained
        FisherParams p{};
        p.n_junctions = J; p.n_samples = n_samples;
        p.inc = d_inc; p.ld_inc = ldd; p.exc = d_exc; p.ld_exc = ldd;
        p.n_pairs = n_pairs; p.pair_a = d_pa; p.pair_b = d_pb;
        p.p_out = buf - r0 * n_pairs; p.ld_p = n_pairs; p.row_begin = r0; p.row_end = r1;
        rc = launch_fisher_pairwise(p, s_k, max_cell);
        if (rc != SD_OK) { cleanup(); return rc; }
        SD_TRY(cudaEventRecord(ev[2 * b], s_k));
        SD_TRY(cudaStreamWaitEvent(s_out, ev[2 * b], 0));
        if (ld_p == n_pairs)
            SD_TRY(cudaMemcpyAsync(p_out + r0 * ld_p, buf, (size_t)(r1 - r0) * n_pairs * 8, cudaMemcpyDeviceToHost, s_out));
        else
            SD_TRY(cudaMemcpy2DAsync(p_out + r0 * ld_p, (size_t)ld_p * 8, buf, (size_t)n_pairs * 8, (size_t)n_pairs * 8,
                                     (size_t)(r1 - r0), cudaMemcpyDeviceToHost, s_out));
        SD_TRY(cudaEventRecord(ev[2 * b + 1], s_out));
    }
    const auto t_enqueued = clk::now();
    SD_TRY(cudaStreamSynchronize(s_out));
#undef SD_TRY
    const auto t_done = clk::now();
    cleanup();
    if (debug) {
        auto ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "[%s] %lld blocks: upload + exclusions + max scan %.2f ms, enqueue %.2f ms, drain %.2f ms, cleanup %.2f ms\n",
                who, (long long)n_blocks, ms(t_begin, t_scanned), ms(t_scanned, t_enqueued), ms(t_enqueued, t_done),
                ms(t_done, clk::now()));
    }
    return SD_OK;
}

}  // namespace sd

extern "C" {

// Host-buffer form: inc / exc / pairs / p_out are HOST pointers.
int sd_fisher_pairwise_host(int device, int64_t n_junctions, int32_t n_samples, const int32_t *inc,
                            int64_t ld_inc, const int64_t *exc, int64_t ld_exc, int64_t n_pairs,
                            const int32_t *pair_a, const int32_t *pair_b, double *p_out, int64_t ld_p)
{
    SD_REQUIRE(n_junctions >= 0 && n_samples >= 0 && n_pairs >= 0, "sd_fisher_pairwise_host: negative size");
    if (n_junctions == 0 || n_pairs == 0) return SD_OK;
    SD_REQUIRE(inc && exc && pair_a && pair_b && p_out, "sd_fisher_pairwise_host: null pointer");
    SD_REQUIRE(ld_inc >= n_samples && ld_exc >= n_samples && ld_p >= n_pairs,
               "sd_fisher_pairwise_host: ld too small");
    return sd::pairwise_host_impl("sd_fisher_pairwise_host", device, n_junctions, n_samples, inc, ld_inc, exc, ld_exc, nullptr,
                                  nullptr, n_pairs, pair_a, pair_b, p_out, ld_p);
}

// The whole pairwise hot loop for host buffers (pairwise_fisher.py:154-180): inclusion counts and the
// cluster CSR in, p-values out; the exclusion counts never exist on the host.
int sd_pairwise_host(int device, int64_t n_junctions, int32_t n_samples, const int32_t *inc, int64_t ld_inc,
                     const int32_t *row_ptr, const int32_t *col_idx, int64_t n_pairs, const int32_t *pair_a,
                     const int32_t *pair_b, double *p_out, int64_t ld_p)
{
    SD_REQUIRE(n_junctions >= 0 && n_samples >= 0 && n_pairs >= 0, "sd_pairwise_host: negative size");
    if (n_junctions == 0 || n_pairs == 0) return SD_OK;
    SD_REQUIRE(inc && row_ptr && pair_a && pair_b && p_out, "sd_pairwise_host: null pointer");
    SD_REQUIRE(ld_inc >= n_samples && ld_p >= n_pairs, "sd_pairwise_host: ld too small");
    return sd::pairwise_host_impl("sd_pairwise_host", device, n_junctions, n_samples, inc, ld_inc, nullptr, 0, row_ptr, col_idx,
                                  n_pairs, pair_a, pair_b, p_out, ld_p);
}

}  // extern "C"
