// sd_cluster.cu -- K1: overlap adjacency ("clusters"), overlap components and output row order.
//
// Replaces SPLICEDICE.getClusters (/root/reference/splicedice/SPLICEDICE.py:230-255; twin
// counts_to_ps.determine_clusters, counts_to_ps.py:16-41) and the row index of SPLICEDICE.py:96.
//
// Closed form of the reference's sweep.  Sort by (chrom, strand, start, end) (:237); inside one
// (chrom, strand) segment junction i and a LATER junction k overlap iff end_i >= start_k (:250,
// closed interval), so the later neighbours of i are the contiguous run i+1 .. ub_i where ub_i
// is the last position whose start <= end_i (one binary search on the sorted keys).  Every i
// adds itself to the prior list of each k in that run: n_prior is a +1/-1 difference array
// followed by a prefix sum.  Overlap components are cut where the segmented running maximum of
// `end` over the earlier junctions of the segment falls below start_k (segmented max-scan).
// The reference's list for k holds its priors most recent first, then its laters ascending
// (:247-254); the priors come out of a radix sort of the (k, b) edge list on (k asc, b desc).
// All ids written to row_ptr / col_idx are OUTPUT rows (tuple order (chrom, start, end, strand)).
//
// The output row order needs no sort of its own (k_out_rank).  Device-wide sort / scan primitives
// are CUB's (one radix sort for the cluster order plus a fix-up of equal-key runs, one sort for the prior
// lists over 2 log2(n) bits, six scans); everything
// else is a kernel below.  One host synchronisation per call (nnz, component count, overflow check).
#include <cub/cub.cuh>

#include <algorithm>

#include "sd_common.cuh"

namespace sd {

namespace {

constexpr int kBlock = 256;
inline int grid_for(int64_t n) { return (int)std::min<int64_t>((n + kBlock - 1) / kBlock, (int64_t)kSMs * 64); }

#define SD_GRID_STRIDE(i, n)                                                         \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n);        \
         i += (int64_t)gridDim.x * blockDim.x)

// cluster-order key: chrom (25 bits) | strand (8 bits) | coordinate (31 bits)
__device__ __forceinline__ uint64_t seg_key(int32_t chrom, int32_t strand, int32_t coord)
{
    return ((uint64_t)(uint32_t)chrom << 39) | ((uint64_t)(uint32_t)(strand & 0xFF) << 31) | (uint64_t)(uint32_t)coord;
}

// bits of the build's flag word (workspace `misc`, read back once per attempt)
constexpr int32_t kFlagLongRun = 1;        // a run of equal keys is longer than kMaxRun: repeat with the two-pass sort
constexpr int32_t kFlagBadInput = 2;       // a field lies outside what seg_key can pack: the call is refused

__global__ void k_iota_end(int64_t n, const int32_t *end, uint32_t *key, int32_t *val)
{
    SD_GRID_STRIDE(i, n) { key[i] = (uint32_t)end[i]; val[i] = (int32_t)i; }
}
// (chrom, strand, start) key of every junction in input order.  Also the input check of the build:
// a junction that seg_key would alias onto another key (chrom >= 2^25 or negative, strand outside
// [0, 256), a negative start or end, whose bit 31 would land in the strand field) raises
// kFlagBadInput.  The build only runs a second attempt after this one was read back clean, so the
// second attempt's key kernel needs no check of its own.
__global__ void k_key_direct(int64_t n, const int32_t *chrom, const int32_t *strand, const int32_t *start,
                             const int32_t *end, uint64_t *key, int32_t *val, int32_t *flag)
{
    SD_GRID_STRIDE(i, n)
    {
        const int32_t c = chrom[i], s = strand[i], st = start[i];
        if ((uint32_t)c >= (1u << 25) || (uint32_t)s >= 256u || (st | end[i]) < 0) atomicOr(flag, kFlagBadInput);
        key[i] = seg_key(c, s, st);
        val[i] = (int32_t)i;
    }
}
// After ONE sort by (chrom, strand, start): junctions that share all three (a common donor site)
// form short runs that still have to be ordered by `end`.  The thread at the head of a run sorts
// it by insertion; a run longer than kMaxRun raises `flag` and the caller repeats the build with
// the two-pass sort (end first, then the 64-bit key).
constexpr int kMaxRun = 64;
__global__ void k_fix_ties(int64_t n, const uint64_t *key_sorted, int32_t *order, const int32_t *end, int32_t *flag)
{
    SD_GRID_STRIDE(i, n)
    {
        const uint64_t key = key_sorted[i];
        if ((i > 0 && key_sorted[i - 1] == key) || i + 1 >= n || key_sorted[i + 1] != key) continue;   // not the head of a run
        int64_t j = i + 2;
        while (j < n && j - i <= kMaxRun && key_sorted[j] == key) ++j;
        const int len = (int)(j - i);
        if (len > kMaxRun) { atomicOr(flag, kFlagLongRun); continue; }
        for (int a = 1; a < len; ++a) {
            const int32_t v = order[i + a];
            const int32_t e = end[v];
            int b = a - 1;
            while (b >= 0 && end[order[i + b]] > e) { order[i + b + 1] = order[i + b]; --b; }
            order[i + b + 1] = v;
        }
    }
}
__global__ void k_key_cluster(int64_t n, const int32_t *order, const int32_t *chrom, const int32_t *strand,
                              const int32_t *start, uint64_t *key)
{
    SD_GRID_STRIDE(i, n) { int32_t j = order[i]; key[i] = seg_key(chrom[j], strand[j], start[j]); }
}
// Output row (the rank under tuple order (chrom, start, end, strand), SPLICEDICE.py:96) of the
// junction at every cluster-order position, without another sort: cluster order is (chrom, strand,
// start, end), so inside one chromosome the output order is the merge of that chromosome's strand
// segments, each already sorted by (start, end).  The rank of a junction is the first position of
// its chromosome plus, for every strand segment of the chromosome, the number of its junctions
// that come before this one -- one binary search per segment (junctions are distinct, so the only
// ties are across strands and break on the strand rank).
// A chromosome or segment ends at the first key above its LAST possible key (all bits below the
// field set), not at the first key of the next chromosome or strand: for chrom 2^25 - 1 that key
// wraps to 0, and for strand 255 it carries into the chromosome field.  The segments then
// partition [c_lo, c_hi), and the only one whose strand equals this junction's is its own, so every
// rank lies in [c_lo, c_hi) whatever the keys hold.
constexpr uint64_t kBelowChrom = (uint64_t(1) << 39) - 1, kBelowStrand = (uint64_t(1) << 31) - 1;
__device__ __forceinline__ int64_t first_at_least(const uint64_t *key, int64_t lo, int64_t hi, uint64_t probe)
{
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key[mid] < probe) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ int64_t first_above(const uint64_t *key, int64_t lo, int64_t hi, uint64_t last)
{
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key[mid] <= last) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__global__ void k_out_rank(int64_t n, const int32_t *order, const uint64_t *key_sorted, const int32_t *end,
                           int32_t *out_row, int32_t *row_of_pos)
{
    SD_GRID_STRIDE(i, n)
    {
        const uint64_t key = key_sorted[i];
        const uint64_t chrom = key >> 39;
        const uint32_t strand = (uint32_t)(key >> 31) & 0xFFu, start = (uint32_t)key & 0x7FFFFFFFu;
        const int32_t j = order[i];
        const uint32_t my_end = (uint32_t)end[j];
        const int64_t c_lo = first_at_least(key_sorted, 0, i + 1, chrom << 39);
        const int64_t c_hi = first_above(key_sorted, i + 1, n, (chrom << 39) | kBelowChrom);
        int64_t rank = c_lo;
        for (int64_t pos = c_lo; pos < c_hi;) {
            const uint32_t s2 = (uint32_t)(key_sorted[pos] >> 31) & 0xFFu;
            const int64_t seg_end = first_above(key_sorted, pos + 1, c_hi, key_sorted[pos] | kBelowStrand);
            if (s2 == strand) {
                rank += i - pos;                                  // own segment: everything before this position
            } else {
                // first position of the segment that does not come before (start, my_end, strand)
                int64_t lo = pos, hi = seg_end;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    const uint32_t st = (uint32_t)key_sorted[mid] & 0x7FFFFFFFu;
                    bool before = st < start;
                    if (st == start) {
                        const uint32_t en = (uint32_t)end[order[mid]];
                        before = en < my_end || (en == my_end && s2 < strand);
                    }
                    if (before) lo = mid + 1; else hi = mid;
                }
                rank += lo - pos;
            }
            pos = seg_end;
        }
        out_row[j] = (int32_t)rank;
        row_of_pos[i] = (int32_t)rank;
    }
}

struct SegMax {
    int32_t head;   // a segment starts at or before this element (within the scanned span)
    int32_t val;
};
struct SegMaxOp {
    __device__ __forceinline__ SegMax operator()(const SegMax &a, const SegMax &b) const
    {
        SegMax r;
        r.head = a.head | b.head;
        r.val = b.head ? b.val : max(a.val, b.val);
        return r;
    }
};

// per position: later-neighbour run, segment heads, scan input, difference array
__global__ void k_sweep(int64_t n, const int32_t *order, const uint64_t *key_sorted, const int32_t *chrom,
                        const int32_t *strand, const int32_t *end, int32_t *n_later, int32_t *diff, SegMax *seg_in,
                        unsigned long long *edges)
{
    unsigned long long my_edges = 0;
    SD_GRID_STRIDE(i, n)
    {
        const int32_t j = order[i];
        const uint64_t probe = seg_key(chrom[j], strand[j], end[j]);
        // ub = (first position with key > probe) - 1
        int64_t lo = i + 1, hi = n;
        while (lo < hi) {
            int64_t mid = (lo + hi) >> 1;
            if (key_sorted[mid] <= probe) lo = mid + 1; else hi = mid;
        }
        const int32_t later = (int32_t)(lo - 1 - i);
        n_later[i] = later;
        my_edges += (unsigned long long)later;
        if (later > 0) {
            atomicAdd(diff + i + 1, 1);
            atomicAdd(diff + i + 1 + later, -1);
        }
        const bool head = i == 0 || (key_sorted[i] >> 31) != (key_sorted[i - 1] >> 31);
        seg_in[i].head = head ? 1 : 0;
        seg_in[i].val = end[j];
    }
    // 64-bit edge count of the whole build (the int32 CSR cannot hold more than 2^31 - 1 entries)
    for (int o = 16; o; o >>= 1) my_edges += __shfl_xor_sync(0xffffffffu, my_edges, o);
    if ((threadIdx.x & 31) == 0 && my_edges) atomicAdd(edges, my_edges);
}

// comp_head[k] = segment head, or the running max of `end` before k is below start_k; position 0 is
// left at 0 so that the inclusive count of heads is the 0-based component id
__global__ void k_comp_head(int64_t n, const uint64_t *key_sorted, const SegMax *seg_scan, int32_t *comp_head)
{
    SD_GRID_STRIDE(i, n)
    {
        const bool head = i == 0 || (key_sorted[i] >> 31) != (key_sorted[i - 1] >> 31);
        const int32_t start = (int32_t)(key_sorted[i] & 0x7FFFFFFFu);
        comp_head[i] = (i > 0 && (head || seg_scan[i - 1].val < start)) ? 1 : 0;
    }
}
__global__ void k_degree(int64_t n, const int32_t *row_of_pos, const int32_t *n_prior, const int32_t *n_later,
                         int32_t *deg_row)
{
    SD_GRID_STRIDE(i, n) deg_row[row_of_pos[i]] = n_prior[i] + n_later[i];
}
// edge (k, b), b < k: key = k in the high bits, (mask - b) in the low `shift` bits, so that one
// ascending sort over 2 * shift bits lists every k's priors most recent first
__global__ void k_edges(int64_t n, int shift, const int32_t *n_later, const int64_t *later_off, uint64_t *edge)
{
    const uint64_t mask = (uint64_t(1) << shift) - 1;
    SD_GRID_STRIDE(i, n)
    {
        const int32_t m = n_later[i];
        uint64_t *dst = edge + later_off[i];
        for (int32_t t = 0; t < m; ++t) dst[t] = ((uint64_t)(i + 1 + t) << shift) | (mask - (uint64_t)i);
    }
}
__global__ void k_fill(int64_t n, int shift, const int32_t *row_of_pos, const int32_t *row_ptr, const int32_t *n_prior,
                       const int32_t *n_later, const int64_t *prior_off, const uint64_t *edge_sorted,
                       int32_t *col_idx)
{
    const uint64_t mask = (uint64_t(1) << shift) - 1;
    SD_GRID_STRIDE(k, n)
    {
        int32_t *dst = col_idx + row_ptr[row_of_pos[k]];
        const int32_t np = n_prior[k], nl = n_later[k];
        const uint64_t *src = edge_sorted + prior_off[k];
        for (int32_t t = 0; t < np; ++t) dst[t] = row_of_pos[mask - (src[t] & mask)];
        for (int32_t t = 0; t < nl; ++t) dst[np + t] = row_of_pos[k + 1 + t];
    }
}
// int32 counts read as int64 by the offset scans (element n, one past the counts, reads as 0)
struct WidenCount {
    const int32_t *in;
    int64_t n;
    __device__ __forceinline__ int64_t operator()(int64_t i) const { return i < n ? (int64_t)in[i] : 0; }
};

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

// carve-up of the build workspace
struct BuildWs {
    size_t key_a, key_b, val_a, val_b, n_later, n_prior, diff, seg, deg_row, misc, cub, total;
    size_t cub_bytes;
};

int cub_bytes_build(int64_t n, size_t *out)
{
    size_t best = 0, b = 0;
    SD_CHECK_CUDA((cub::DeviceRadixSort::SortPairs<uint64_t, int32_t>(nullptr, b, nullptr, nullptr, nullptr, nullptr, (int)n)));
    best = std::max(best, b);
    SD_CHECK_CUDA((cub::DeviceRadixSort::SortPairs<uint32_t, int32_t>(nullptr, b, nullptr, nullptr, nullptr, nullptr, (int)n)));
    best = std::max(best, b);
    SD_CHECK_CUDA((cub::DeviceScan::InclusiveSum<const int32_t *, int32_t *>(nullptr, b, nullptr, nullptr, (int)(n + 1))));
    best = std::max(best, b);
    SD_CHECK_CUDA((cub::DeviceScan::ExclusiveSum<const int32_t *, int32_t *>(nullptr, b, nullptr, nullptr, (int)(n + 1))));
    best = std::max(best, b);
    SD_CHECK_CUDA((cub::DeviceScan::InclusiveScan<const SegMax *, SegMax *, SegMaxOp>(nullptr, b, nullptr, nullptr, SegMaxOp(), (int)n)));
    best = std::max(best, b);
    *out = best;
    return SD_OK;
}

int layout_build(int64_t n, BuildWs *w)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes); return o; };
    // persistent (read again by sd_cluster_fill)
    w->n_later = take((size_t)n * 4);
    w->n_prior = take((size_t)(n + 1) * 4);
    w->val_b = take((size_t)n * 4);          // row_of_pos copy lives in the caller's array; val_b is scratch
    // scratch
    w->key_a = take((size_t)n * 8);
    w->key_b = take((size_t)n * 8);
    w->val_a = take((size_t)n * 4);
    w->diff = take((size_t)(n + 1) * 4);
    w->seg = take((size_t)n * sizeof(SegMax) * 2);
    w->deg_row = take((size_t)(n + 1) * 4);
    w->misc = take(256);                      // [0] long-run flag (int32), [8] edge count (uint64)
    if (int rc = cub_bytes_build(n, &w->cub_bytes)) return rc;
    w->cub = take(w->cub_bytes);
    w->total = off;
    return SD_OK;
}

struct FillWs {
    size_t later_off, prior_off, edge_a, edge_b, cub, total;
    size_t cub_bytes;
};
int layout_fill(int64_t n, int64_t nnz, FillWs *w)
{
    const int64_t e = nnz / 2;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes); return o; };
    w->later_off = take((size_t)(n + 1) * 8);
    w->prior_off = take((size_t)(n + 1) * 8);
    w->edge_a = take((size_t)std::max<int64_t>(e, 1) * 8);
    w->edge_b = take((size_t)std::max<int64_t>(e, 1) * 8);
    size_t b1 = 0, b2 = 0;
    SD_CHECK_CUDA((cub::DeviceRadixSort::SortKeys<uint64_t>(nullptr, b1, nullptr, nullptr, (int)std::max<int64_t>(e, 1))));
    {
        cub::CountingInputIterator<int64_t> idx(0);
        cub::TransformInputIterator<int64_t, WidenCount, cub::CountingInputIterator<int64_t>> in(idx, WidenCount{nullptr, n});
        SD_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, b2, in, (int64_t *)nullptr, (int)(n + 1)));
    }
    w->cub_bytes = std::max(b1, b2);
    w->cub = take(w->cub_bytes);
    w->total = off;
    return SD_OK;
}

int bits_for(int64_t n)
{
    int b = 1;
    while (b < 32 && (int64_t(1) << b) < n) ++b;
    return b;
}

}  // namespace
}  // namespace sd

extern "C" {

size_t sd_cluster_workspace_bytes(int64_t n_junctions)
{
    if (n_junctions <= 0) return 256;
    sd::BuildWs w;
    if (sd::layout_build(n_junctions, &w) != SD_OK) return 0;
    return w.total;
}

size_t sd_cluster_fill_workspace_bytes(int64_t n_junctions, int64_t nnz)
{
    if (n_junctions <= 0) return 256;
    sd::FillWs w;
    if (sd::layout_fill(n_junctions, nnz, &w) != SD_OK) return 0;
    return w.total;
}

int sd_cluster_build(int64_t n, const int32_t *chrom_rank, const int32_t *strand_rank, const int32_t *start,
                     const int32_t *end, int32_t *cluster_order, int32_t *out_row, int32_t *row_of_pos,
                     int32_t *comp_id, int32_t *row_ptr, int64_t *nnz_host, int64_t *n_components_host,
                     void *workspace, size_t workspace_bytes, void *stream_)
{
    using namespace sd;
    SD_REQUIRE(n >= 0 && n < 0x7FFFFFFF, "sd_cluster_build: n_junctions out of range");
    SD_REQUIRE(nnz_host && n_components_host, "sd_cluster_build: null result pointer");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) {
        *nnz_host = 0; *n_components_host = 0;
        if (row_ptr) SD_CHECK_CUDA(cudaMemsetAsync(row_ptr, 0, 4, stream));
        return SD_OK;
    }
    SD_REQUIRE(chrom_rank && strand_rank && start && end && cluster_order && out_row && row_of_pos && comp_id &&
                   row_ptr && workspace,
               "sd_cluster_build: null pointer");
    BuildWs w;
    if (int rc = layout_build(n, &w)) return rc;
    if (workspace_bytes < w.total)
        return fail(SD_ERR_WORKSPACE, "sd_cluster_build: workspace %zu < %zu bytes", workspace_bytes, w.total);
    char *ws = static_cast<char *>(workspace);
    uint64_t *key_a = (uint64_t *)(ws + w.key_a), *key_b = (uint64_t *)(ws + w.key_b);
    int32_t *val_a = (int32_t *)(ws + w.val_a), *val_b = (int32_t *)(ws + w.val_b);
    int32_t *n_later = (int32_t *)(ws + w.n_later), *n_prior = (int32_t *)(ws + w.n_prior);
    int32_t *diff = (int32_t *)(ws + w.diff), *deg_row = (int32_t *)(ws + w.deg_row);
    SegMax *seg_in = (SegMax *)(ws + w.seg), *seg_out = seg_in + n;
    void *cub_ws = ws + w.cub;
    size_t cub_b = w.cub_bytes;
    const int g = grid_for(n);
    const int ni = (int)n;

    int32_t *d_flag = (int32_t *)(ws + w.misc);
    unsigned long long *d_edges = (unsigned long long *)(ws + w.misc + 8);
    unsigned long long h_edges = 0;
    int32_t h_nnz = 0, h_comp = 0, h_flag = 0;
    // First attempt: ONE radix sort by (chrom, strand, start) and a fix-up of the short runs that
    // share all three; a run longer than kMaxRun (seen at the final read-back) repeats the build
    // with the two-pass sort.
    for (int attempt = 0; attempt < 2; ++attempt) {
        SD_CHECK_CUDA(cudaMemsetAsync(ws + w.misc, 0, 16, stream));
        if (attempt == 0) {
            k_key_direct<<<g, kBlock, 0, stream>>>(n, chrom_rank, strand_rank, start, end, key_a, val_a, d_flag);
            SD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_b, key_a, key_b, val_a, cluster_order, ni, 0, 64, stream));
            k_fix_ties<<<g, kBlock, 0, stream>>>(n, key_b, cluster_order, end, d_flag);
        } else {
            // stable LSD sort, end then (chrom, strand, start)
            uint32_t *key32_a = (uint32_t *)key_a, *key32_b = (uint32_t *)key_b;
            k_iota_end<<<g, kBlock, 0, stream>>>(n, end, key32_a, val_a);
            SD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_b, key32_a, key32_b, val_a, val_b, ni, 0, 32, stream));
            k_key_cluster<<<g, kBlock, 0, stream>>>(n, val_b, chrom_rank, strand_rank, start, key_a);
            SD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_b, key_a, key_b, val_b, cluster_order, ni, 0, 64, stream));
        }
        // key_b = sorted (chrom, strand, start) keys
        // ---- output row order from the cluster order (merge ranks, no sort) --------------------
        k_out_rank<<<g, kBlock, 0, stream>>>(n, cluster_order, key_b, end, out_row, row_of_pos);

        // ---- sweep ----------------------------------------------------------------------------
        SD_CHECK_CUDA(cudaMemsetAsync(diff, 0, (size_t)(n + 1) * 4, stream));
        k_sweep<<<g, kBlock, 0, stream>>>(n, cluster_order, key_b, chrom_rank, strand_rank, end, n_later, diff, seg_in, d_edges);
        SD_CHECK_CUDA(cub::DeviceScan::InclusiveSum(cub_ws, cub_b, (const int32_t *)diff, n_prior, ni + 1, stream));
        SD_CHECK_CUDA(cub::DeviceScan::InclusiveScan(cub_ws, cub_b, (const SegMax *)seg_in, seg_out, SegMaxOp(), ni, stream));
        k_comp_head<<<g, kBlock, 0, stream>>>(n, key_b, seg_out, val_a);
        SD_CHECK_CUDA(cub::DeviceScan::InclusiveSum(cub_ws, cub_b, (const int32_t *)val_a, comp_id, ni, stream));

        // ---- CSR row pointer in output-row space -----------------------------------------------
        SD_CHECK_CUDA(cudaMemsetAsync(deg_row + n, 0, 4, stream));
        k_degree<<<g, kBlock, 0, stream>>>(n, row_of_pos, n_prior, n_later, deg_row);
        SD_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cub_b, (const int32_t *)deg_row, row_ptr, ni + 1, stream));
        if (int rc = check_launch("sd_cluster_build kernels")) return rc;

        // the call's single synchronisation: flag word, 64-bit edge count (an overflowing prefix
        // sum above only produces garbage that is never returned), nnz, component count.  Out-of-range
        // input runs the whole build on aliased keys; every write stays inside the caller's arrays
        // and the workspace (k_out_rank's ranks lie in [0, n)), and the call fails before any result.
        SD_CHECK_CUDA(cudaMemcpyAsync(&h_flag, d_flag, 4, cudaMemcpyDeviceToHost, stream));
        SD_CHECK_CUDA(cudaMemcpyAsync(&h_edges, d_edges, 8, cudaMemcpyDeviceToHost, stream));
        SD_CHECK_CUDA(cudaMemcpyAsync(&h_nnz, row_ptr + n, 4, cudaMemcpyDeviceToHost, stream));
        SD_CHECK_CUDA(cudaMemcpyAsync(&h_comp, comp_id + (n - 1), 4, cudaMemcpyDeviceToHost, stream));
        SD_CHECK_CUDA(cudaStreamSynchronize(stream));
        if (h_flag & kFlagBadInput)
            return fail(SD_ERR_INVALID, "sd_cluster_build: a junction has chrom_rank outside [0, 2^25), strand_rank "
                                        "outside [0, 256) or a negative start / end");
        if (!(h_flag & kFlagLongRun)) break;
    }
    if (2 * h_edges > 0x7FFFFFFFull)
        return fail(SD_ERR_OVERFLOW, "sd_cluster_build: %llu adjacency entries do not fit int32 indices", 2 * h_edges);
    *nnz_host = h_nnz;
    *n_components_host = (int64_t)h_comp + 1;            // comp_id is 0-based
    return SD_OK;
}

int sd_cluster_fill(int64_t n, int64_t nnz, const int32_t *row_of_pos, const int32_t *row_ptr, int32_t *col_idx,
                    void *build_workspace, size_t build_workspace_bytes, void *fill_workspace,
                    size_t fill_workspace_bytes, void *stream_)
{
    using namespace sd;
    SD_REQUIRE(n >= 0 && n < 0x7FFFFFFF && nnz >= 0 && nnz <= 0x7FFFFFFF && (nnz & 1) == 0,
               "sd_cluster_fill: bad sizes");
    if (n == 0 || nnz == 0) return SD_OK;
    SD_REQUIRE(row_of_pos && row_ptr && col_idx && build_workspace && fill_workspace, "sd_cluster_fill: null pointer");
    cudaStream_t stream = (cudaStream_t)stream_;
    BuildWs bw;
    if (int rc = layout_build(n, &bw)) return rc;
    FillWs fw;
    if (int rc = layout_fill(n, nnz, &fw)) return rc;
    if (build_workspace_bytes < bw.total || fill_workspace_bytes < fw.total)
        return fail(SD_ERR_WORKSPACE, "sd_cluster_fill: workspace too small (%zu < %zu or %zu < %zu)",
                    build_workspace_bytes, bw.total, fill_workspace_bytes, fw.total);
    char *b = static_cast<char *>(build_workspace), *f = static_cast<char *>(fill_workspace);
    const int32_t *n_later = (const int32_t *)(b + bw.n_later), *n_prior = (const int32_t *)(b + bw.n_prior);
    int64_t *later_off = (int64_t *)(f + fw.later_off), *prior_off = (int64_t *)(f + fw.prior_off);
    uint64_t *edge_a = (uint64_t *)(f + fw.edge_a), *edge_b = (uint64_t *)(f + fw.edge_b);
    void *cub_ws = f + fw.cub;
    size_t cub_b = fw.cub_bytes;
    const int g = grid_for(n);
    const int64_t e = nnz / 2;

    const int shift = bits_for(n + 1);
    {
        cub::CountingInputIterator<int64_t> idx(0);
        cub::TransformInputIterator<int64_t, WidenCount, cub::CountingInputIterator<int64_t>> later_in(idx, WidenCount{n_later, n});
        cub::TransformInputIterator<int64_t, WidenCount, cub::CountingInputIterator<int64_t>> prior_in(idx, WidenCount{n_prior, n});
        SD_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cub_b, later_in, later_off, (int)(n + 1), stream));
        SD_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cub_b, prior_in, prior_off, (int)(n + 1), stream));
    }
    k_edges<<<g, kBlock, 0, stream>>>(n, shift, n_later, later_off, edge_a);
    SD_CHECK_CUDA(cub::DeviceRadixSort::SortKeys(cub_ws, cub_b, edge_a, edge_b, (int)e, 0, 2 * shift, stream));
    k_fill<<<g, kBlock, 0, stream>>>(n, shift, row_of_pos, row_ptr, n_prior, n_later, prior_off, edge_b, col_idx);
    return check_launch("sd_cluster_fill kernels");
}

}  // extern "C"
