/* splicedice_b200.h -- C-ABI of the B200-native SpliceDICE hot path.
 *
 * One shared library, `libsplicedice_b200.so`, built from splicedice_b200/csrc/ with
 *   nvcc -gencode arch=compute_100a,code=sm_100a
 * Plain pointers and sizes only; no C++/torch types cross this boundary, so the
 * reference (a pure-Python package) binds it with ctypes -- see INTEGRATION.md.
 *
 * The reference has no FFI of its own: its hot path is a set of Python methods.
 * Each entry point below names the reference code it replaces (paths relative to
 * /root/reference/splicedice/).
 *
 * Conventions
 *   - `*_dev` / unsuffixed compute entry points take DEVICE pointers owned by the
 *     caller; the library never frees or retains them.  `*_host` entry points take
 *     HOST pointers and do their own (pipelined) transfers.
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = default stream).  Calls
 *     are asynchronous on that stream unless stated otherwise.
 *   - Matrices are row-major [row = junction][col = sample] with a leading dimension
 *     `ld_*` in ELEMENTS (>= n_samples); the 128-bit fast paths need the base pointer
 *     16-byte aligned and ld a multiple of 4, otherwise a scalar kernel runs.
 *   - Every function returns SD_OK (0) or an SD_ERR_* code; `sd_last_error()` gives the
 *     thread-local message.  No exceptions, no longjmp; re-entrant per stream.
 *   - There is NO CPU fallback: without a CUDA device the compute calls fail with
 *     SD_ERR_CUDA.
 */
#ifndef SPLICEDICE_B200_H
#define SPLICEDICE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SD_ABI_VERSION 1

#define SD_OK 0
#define SD_ERR_INVALID 1      /* bad argument (null pointer, negative size, ld < n_samples ...) */
#define SD_ERR_CUDA 2         /* CUDA runtime error; message carries cudaGetErrorString */
#define SD_ERR_WORKSPACE 3    /* workspace too small */
#define SD_ERR_OVERFLOW 4     /* adjacency does not fit int32 indices */
#define SD_ERR_UNSUPPORTED 5

/* ---- library ---------------------------------------------------------------- */
int sd_version(void);                       /* SD_ABI_VERSION of the built library */
const char *sd_last_error(void);            /* thread-local, never NULL */
/* SM count / compute capability / memory of `device`. */
int sd_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);

/* ---- K1: overlap adjacency ("clusters") + output row order --------------------
 * Replaces SPLICEDICE.getClusters (SPLICEDICE.py:230-255; twin
 * counts_to_ps.determine_clusters, counts_to_ps.py:16-41) and the row index of
 * SPLICEDICE.py:96.
 *
 * Input: J distinct junctions in any order as (chrom_rank, strand_rank, start, end);
 * the ranks are dense ranks of the chromosome / strand STRINGS under python's str
 * order (the host computes them: "chr10" < "chr2", "+" < "-").
 *
 * sd_cluster_build sorts by (chrom, strand, start, end) (:237), finds each junction's
 * later-neighbour run and prior count (closed-interval overlap, :250), the overlap
 * components (segmented running max of `end`), the output row of every junction
 * (tuple order (chrom, start, end, strand), :96) and the CSR row pointer in output-row
 * space.  It synchronises the stream to return nnz / n_components to the host.
 * sd_cluster_fill then writes col_idx[nnz] (columns are output rows; each list ordered
 * as the reference's: priors most-recent-first, then laters ascending, :247-254).  The
 * build workspace must be passed, untouched, to sd_cluster_fill together with a second
 * workspace sized by sd_cluster_fill_workspace_bytes(n_junctions, nnz).
 * Input domain: 0 <= start, end; 0 <= chrom_rank < 2^25; 0 <= strand_rank < 2^8.
 * sd_cluster_build checks it on the device and refuses a junction outside it with
 * SD_ERR_INVALID (reported at the call's read-back; the output arrays then hold
 * unspecified values and nothing outside them and the workspace is written).
 *
 *   cluster_order[pos] = input index of the junction at position pos of cluster order
 *   out_row[i]         = output row of input junction i
 *   row_of_pos[pos]    = output row of the junction at cluster position pos
 *   comp_id[pos]       = overlap-component id (non-decreasing in pos)
 *   row_ptr[J+1]       = CSR pointer over output rows
 * The *_workspace_bytes queries need a CUDA device (they return 0 and set sd_last_error()
 * without one).
 */
size_t sd_cluster_workspace_bytes(int64_t n_junctions);
size_t sd_cluster_fill_workspace_bytes(int64_t n_junctions, int64_t nnz);
int sd_cluster_build(int64_t n_junctions,
                     const int32_t *chrom_rank, const int32_t *strand_rank,
                     const int32_t *start, const int32_t *end,
                     int32_t *cluster_order, int32_t *out_row, int32_t *row_of_pos,
                     int32_t *comp_id, int32_t *row_ptr,
                     int64_t *nnz_host, int64_t *n_components_host,
                     void *workspace, size_t workspace_bytes, void *stream);
int sd_cluster_fill(int64_t n_junctions, int64_t nnz, const int32_t *row_of_pos,
                    const int32_t *row_ptr, int32_t *col_idx,
                    void *build_workspace, size_t build_workspace_bytes,
                    void *fill_workspace, size_t fill_workspace_bytes, void *stream);

/* ---- K2: exclusion aggregation fused with the PS divide -------------------------
 * Replaces SPLICEDICE.calculatePsi (SPLICEDICE.py:297-310) and the arithmetic of
 * counts_to_ps.writePsValues (counts_to_ps.py:62-68).
 *
 * For rows r in [row_begin, row_end):  exc[r,s] = sum_{c in adj(r)} counts[c,s]
 * (exact integer sum; duplicates in the list count twice, as the reference's loop),
 *   ps_f32[r,s] = (float)((double)inc / (double)(inc + exc))   -- calculatePsi's dtype chain
 *   ps_f64[r,s] = (double)inc / (double)(inc + exc)            -- counts_to_ps
 * 0/0 -> NaN; low_mask[r,s] != 0 -> ps_f32 = NaN (SPLICEDICE.py:307-309).
 * Any of ps_f32 / ps_f64 / exc_out may be NULL (at least one must be set); counts must
 * be non-negative.  `flags`: 0 = automatic kernel choice; see SD_QUANT_* below.
 */
#define SD_QUANT_AUTO 0u
#define SD_QUANT_GATHER 1u        /* direct gather kernel (any alignment) */
#define SD_QUANT_TILED 2u         /* TMA-staged shared-memory tile kernel (aligned inputs) */
#define SD_QUANT_VARIANT_MASK 0xFFu
/* bits 8..15: log2(rows per tile) override (tuning / tests) */
#define SD_QUANT_ROWS(n) (((uint32_t)(n) & 0xFFu) << 24)   /* wide kernel: n rows per tile, 8..128 (tuning / tests) */
#define SD_QUANT_VEC1 0x20000u           /* wide kernel: 128-column slabs (4 columns per lane) */
#define SD_QUANT_VEC2 0x40000u           /* wide kernel: 256-column slabs (8 columns per lane) */
#define SD_QUANT_NARROW_TILES 0x10000u   /* force the narrow-matrix tile kernel for any n_samples (tests) */
#define SD_QUANT_GENERAL 0x80000u        /* wide kernel: the general epilogue even for a single output (tests) */
int sd_quant_ps(int64_t n_junctions, int32_t n_samples,
                const int32_t *counts, int64_t ld_counts,
                const int32_t *row_ptr, const int32_t *col_idx,
                const uint8_t *low_mask, int64_t ld_mask,
                float *ps_f32, int64_t ld_ps32,
                double *ps_f64, int64_t ld_ps64,
                int64_t *exc_out, int64_t ld_exc,
                int64_t row_begin, int64_t row_end,
                uint32_t flags, void *stream);

/* Name, template arguments, tile shape and grid of the kernel the calling thread's last
 * sd_quant_ps / sd_ir_ratio call launched (diagnostics: bench.py reports it as roofline.kernel).
 * Thread-local storage owned by the library; "" before the first launch. */
const char *sd_quant_last_launch(void);

/* Host-buffer form of the PS path (the call a ctypes user makes): counts / ps are HOST
 * pointers (pinned memory gives full PCIe rate), row_ptr / col_idx are HOST pointers.
 * Transfers and the kernel are pipelined over row blocks on streams the library keeps per
 * device; row blocks whose counts are all below 65,536 cross the link as uint16 (narrowed by
 * host threads into pinned staging, widened on the device) -- results do not depend on it.  The
 * call returns when ps_f32 is complete; concurrent calls on one device are serialised.  Device
 * buffers come from a pool private to the library and stay cached between calls
 * (sd_host_pipeline_trim releases them).  `device` is the CUDA device ordinal.
 * Environment (experiments): SD_QUANT_HOST_BLOCK_MB, SD_QUANT_HOST_U16=0, SD_HOST_THREADS. */
int sd_quant_ps_host(int device, int64_t n_junctions, int32_t n_samples,
                     const int32_t *counts, int64_t ld_counts,
                     const int32_t *row_ptr, const int32_t *col_idx,
                     const uint8_t *low_mask, int64_t ld_mask,
                     float *ps_f32, int64_t ld_ps32);

/* Releases the device memory and pinned staging the host-buffer calls keep cached for `device`. */
int sd_host_pipeline_trim(int device);

/* ---- K3: pairwise two-sided Fisher exact test ------------------------------------
 * Replaces the hot loop of pairwise_fisher.run_with (pairwise_fisher.py:154-180) and
 * scipy.stats.fisher_exact's two-sided branch (scipy 1.18.1, stats/_stats_py.py:5042-5108).
 * For rows j in [row_begin, row_end) and pairs k < n_pairs:
 *   p_out[j, k] = two-sided p of [[inc[j,a_k], inc[j,b_k]], [exc[j,a_k], exc[j,b_k]]]
 * Tables with a zero margin give 1.0.  Entries must be non-negative (SD_ERR_INVALID otherwise,
 * as scipy raises ValueError).  The calls synchronise the stream once (a max-reduction over the
 * inputs sizes the log-factorial table, which is built on the host in binary128 the first time
 * a size is needed and cached per device for the life of the process -- the library's only
 * process-wide state, read-only once built).
 */
int sd_fisher_pairwise(int64_t n_junctions, int32_t n_samples,
                       const int32_t *inc, int64_t ld_inc,
                       const int64_t *exc, int64_t ld_exc,
                       int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                       double *p_out, int64_t ld_p,
                       int64_t row_begin, int64_t row_end, void *stream);
/* Fully asynchronous form: the caller promises 0 <= inc[j,s] + exc[j,s] <= max_cell_bound for every
 * cell of the row range (a host that filled the matrices knows it), so no reduction and no
 * stream synchronisation is needed (the table upload synchronises only the first time a larger
 * table is required).  A table with an entry outside the promise yields NaN, never a wrong p. */
int sd_fisher_pairwise_bounded(int64_t n_junctions, int32_t n_samples,
                               const int32_t *inc, int64_t ld_inc,
                               const int64_t *exc, int64_t ld_exc,
                               int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                               double *p_out, int64_t ld_p,
                               int64_t row_begin, int64_t row_end, int64_t max_cell_bound, void *stream);
/* Host-buffer form (the call a ctypes user makes): every pointer is a HOST pointer; row blocks
 * of p-values are computed on one stream while the previous block is copied back on another.
 * Returns when p_out is complete. */
int sd_fisher_pairwise_host(int device, int64_t n_junctions, int32_t n_samples,
                            const int32_t *inc, int64_t ld_inc,
                            const int64_t *exc, int64_t ld_exc,
                            int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                            double *p_out, int64_t ld_p);
/* The whole hot loop of pairwise_fisher.run_with (pairwise_fisher.py:154-180) for HOST buffers:
 * inclusion counts and the cluster CSR (np.isin set semantics are the caller's: one entry per
 * distinct partner) in, p-values out.  The exclusion counts are summed on the device (the kernel of
 * sd_quant_ps), so 4 bytes per cell cross the link instead of 12, then the same pipeline as
 * sd_fisher_pairwise_host runs.  Every pointer is a HOST pointer. */
int sd_pairwise_host(int device, int64_t n_junctions, int32_t n_samples,
                     const int32_t *inc, int64_t ld_inc,
                     const int32_t *row_ptr, const int32_t *col_idx,
                     int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                     double *p_out, int64_t ld_p);
/* Scatter form of the bounded call, for the multi-GPU pairwise path: the pairs are cut into n_dest
 * contiguous column blocks [dest_col_begin[g], dest_col_begin[g + 1]) and the p-value of (row j,
 * pair k) is stored straight into block owner g's matrix,
 *   dest[g][(dest_row_offset + j) * dest_ld[g] + (k - dest_col_begin[g])].
 * dest[g] are DEVICE pointers that may belong to other GPUs (peer memory, e.g. CUDA IPC mappings
 * over NVLink): the row-slab -> column-block exchange that the per-pair Benjamini-Hochberg
 * correction needs (pairwise_fisher.py:186-191 across GPUs) then happens inside the Fisher kernel's
 * own stores instead of a separate all-to-all.  dest / dest_col_begin / dest_ld are HOST arrays
 * (n_dest <= 16 entries, dest_col_begin has n_dest + 1).  Asynchronous on `stream`; the caller
 * orders the peers (e.g. a barrier) before anybody reads the column blocks. */
int sd_fisher_pairwise_scatter(int64_t n_junctions, int32_t n_samples,
                               const int32_t *inc, int64_t ld_inc,
                               const int64_t *exc, int64_t ld_exc,
                               int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                               int32_t n_dest, double *const *dest, const int64_t *dest_col_begin,
                               const int64_t *dest_ld, int64_t dest_row_offset,
                               int64_t row_begin, int64_t row_end,
                               int64_t max_cell_bound, void *stream);
/* Peer-memory plumbing for that scatter (one process per GPU): allocate a device buffer and export
 * it as a CUDA IPC handle (64 opaque bytes to hand to the other ranks, e.g. through
 * torch.distributed.all_gather_object); map a peer's handle into this process (a device pointer
 * valid on the caller's current device, NVLink peer access enabled by the mapping). */
int sd_peer_alloc(size_t bytes, void **ptr, unsigned char *handle64);
int sd_peer_free(void *ptr);
int sd_peer_open(const unsigned char *handle64, void **ptr);
int sd_peer_close(void *ptr);
/* The way back: rows [row_begin[g], row_begin[g + 1]) of the dense DEVICE matrix src[n_rows, width]
 * go to dest[g] (row owner g's matrix, possibly peer memory) at rows 0.., columns dest_col0.. --
 * one kernel, 256-byte contiguous stores.  dest / row_begin / dest_ld are HOST arrays. */
int sd_peer_scatter_rows(const double *src, int64_t n_rows, int64_t width, int32_t n_dest, double *const *dest,
                         const int64_t *row_begin, const int64_t *dest_ld, int64_t dest_col0, void *stream);

/* Element-wise form: p[i] for tables (a[i], b[i], c[i], d[i]) = [[a, b], [c, d]]. */
int sd_fisher_tables(int64_t n_tables, const int64_t *a, const int64_t *b,
                     const int64_t *c, const int64_t *d, double *p_out, void *stream);

/* ---- K3 chi-squared: pairwise Yates-corrected chi-squared test ------------------------------
 * Replaces the `--chi2` branch of the same loop: scipy.stats.chi2_contingency(table)[1] with its
 * default correction=True (scipy 1.18.1, stats/contingency.py; pairwise_fisher.py:133-134,179).
 * For rows j in [row_begin, row_end) and pairs k < n_pairs, on the same tables as sd_fisher_pairwise:
 *   p_out[j, k] = erfc(sqrt(stat / 2)),  stat = max(|ad - bc| - N/2, 0)^2 N / (r1 r2 c1 c2)
 * (p = 1 exactly where |ad - bc| <= N/2), NaN for the all-zero table (as scipy).  Tables scipy refuses
 * -- a zero margin with N > 0, or an entry outside inc in [0, 2^31), exc in [0, 2^61) -- give NaN, and
 * if first_refused (a DEVICE pointer, may be NULL) is set, *first_refused is lowered to the smallest
 * j * n_pairs + k among them (j the absolute row); the caller initialises it to UINT64_MAX.  Fully
 * asynchronous on `stream`: no scan, no synchronisation. */
int sd_chi2_pairwise(int64_t n_junctions, int32_t n_samples,
                     const int32_t *inc, int64_t ld_inc,
                     const int64_t *exc, int64_t ld_exc,
                     int64_t n_pairs, const int32_t *pair_a, const int32_t *pair_b,
                     double *p_out, int64_t ld_p,
                     int64_t row_begin, int64_t row_end,
                     uint64_t *first_refused, void *stream);

/* ---- Benjamini-Hochberg adjustment of the p-value matrix (device) ---------------------------
 * Replaces the multiple-test correction of pairwise_fisher.run_with (pairwise_fisher.py:182-191):
 * statsmodels multipletests(method="fdr_bh")[1] applied to every column ("pairwise", the CLI
 * default; SD_BH_COLUMNS) or to the flattened matrix ("all"; SD_BH_ALL).  For the n values of a
 * segment sorted ascending,  adj_(k) = min(1, min_{m >= k} p_(m) / (m / n))  with both divisions
 * in IEEE binary64, so results are bit-identical to the numpy restatement of statsmodels'
 * fdrcorrection (oracle/oracle_np.py; statsmodels itself is not installable here -- the
 * restatement is pinned to scipy.stats.false_discovery_control within 2 ulp, tests/test_bh_pin.py).
 * p / out: DEVICE matrices [n_rows, n_cols] (out may alias p); at most 2^31 - 1 values per call
 * (SD_ERR_UNSUPPORTED beyond: column blocks are independent, split them).  Scratch comes from a
 * caller-provided device workspace (~33 bytes per value).  SD_BH_ALL is asynchronous on `stream`;
 * SD_BH_COLUMNS with 8,192..524,288 rows runs a per-column sample sort and synchronises `stream`
 * once before returning (it reads back one flag that says whether the sampled splitters produced
 * a bucket too large to sort on chip; if so the call repeats with the global radix sort).
 */
#define SD_BH_COLUMNS 0
#define SD_BH_ALL 1
size_t sd_bh_workspace_bytes(int64_t n_rows, int64_t n_cols, int mode);
int sd_bh_adjust(int64_t n_rows, int64_t n_cols, const double *p, int64_t ld_p,
                 double *out, int64_t ld_out, int mode,
                 void *workspace, size_t workspace_bytes, void *stream);

/* ---- K6: Wilcoxon rank-sum test per event between two sample groups (compare_groups) ------------
 * For rows j in [row_begin, row_end) of the PS matrix ps[n_events, n_samples] (float32 or float64 by
 * `dtype`; NaN = undefined cell): x = the non-NaN cells of columns cols1[0, n1), y = those of
 * cols2[0, n2) (DEVICE int32 lists; the caller keeps the groups disjoint), and
 *   n_out[j * ld_n + 0, 1]            = |x|, |y|
 *   stats_out[j * ld_stats + 0 .. 3]  = mean(x), mean(y), z, p
 * with z, p = scipy.stats.ranksums(x, y, nan_policy='omit') (scipy 1.18.1): average ranks for ties, no
 * tie or continuity correction, p = erfc(|z| / sqrt 2).  2 R1 - n1 (n + 1) is exact in 64-bit
 * integers, so balanced rank sums give z == 0 and p == 1 exactly.  -0.0 ties +0.0; +-inf are ordinary
 * values; means are float64 sums.  An empty x or y gives NaN z, p and NaN for that group's mean.
 * n1, n2 >= 1 and n1 + n2 <= SD_RANKSUM_MAX_SAMPLES (the sort runs in shared memory).  A column index
 * outside [0, n_samples) is never read: the rows get n = -1 and NaN statistics.  One asynchronous
 * launch on `stream`, no synchronisation.
 */
#define SD_RANKSUM_F32 0
#define SD_RANKSUM_F64 1
#define SD_RANKSUM_MAX_SAMPLES 16384
int sd_ranksum_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                    int32_t n1, const int32_t *cols1, int32_t n2, const int32_t *cols2,
                    int64_t row_begin, int64_t row_end,
                    int32_t *n_out, int64_t ld_n, double *stats_out, int64_t ld_stats, void *stream);

/* ---- K7: Kruskal-Wallis H test per event across sample groups (compare_conditions) ---------------
 * For rows j in [row_begin, row_end) of ps (as K6): the non-NaN cells of columns cols[0, n_cols), the
 * cell of cols[i] in group group_of[i] (DEVICE int32 lists; columns listed once), ranked together with
 * average ranks, and
 *   n_out[j * ld_n + g]              = defined cells of group g, g < n_groups
 *   mean_out[j * ld_mean + g]        = their mean (float64 sum; NaN for an empty group)
 *   stats_out[j * ld_stats + 0, 1]   = H, p
 * with H, p = scipy.stats.kruskal(*groups, nan_policy='omit') (scipy 1.18.1) computed without its
 * cancellation: H = 3 (n - 1) sum_g (D_g^2 / n_g) / (n^3 - n - T), D_g = 2 R_g - n_g (n + 1) and the tie
 * term T exact in 64-bit integers, p = chi2.sf(H, n_groups - 1).  H >= 0, and balanced rank sums give
 * H == 0 and p == 1 exactly.  An empty group, or every defined cell tied, gives H = p = NaN (scipy gives
 * NaN for the first, NaN or +-inf for the second).  -0.0 ties +0.0; +-inf are ordinary values.
 * 2 <= n_groups <= SD_KRUSKAL_MAX_GROUPS, 1 <= n_cols <= SD_RANKSUM_MAX_SAMPLES.  A column outside
 * [0, n_samples) or a label outside [0, n_groups) is never dereferenced: the rows get n = -1 in every
 * group and NaN means and statistics.  One asynchronous launch on `stream`, no synchronisation.
 */
#define SD_KRUSKAL_MAX_GROUPS 256
int sd_kruskal_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                    int32_t n_groups, int32_t n_cols, const int32_t *cols, const int32_t *group_of,
                    int64_t row_begin, int64_t row_end,
                    int32_t *n_out, int64_t ld_n, double *mean_out, int64_t ld_mean,
                    double *stats_out, int64_t ld_stats, void *stream);

/* ---- K8: Wilcoxon signed-rank test per event between matched sample pairs (compare_paired) -------
 * For rows j in [row_begin, row_end) of ps (as K6): pair i has cells x_i = ps[j, cols1[i]] and
 * y_i = ps[j, cols2[i]] (DEVICE int32 lists of n_pairs columns each; no column listed twice), and
 *   n_out[j * ld_n + 0 .. 2]          = n, c, method
 *   stats_out[j * ld_stats + 0 .. 3]  = mean1, mean2, W, p
 * with W, p = scipy.stats.wilcoxon(x, y, nan_policy='omit') (scipy 1.18.1 defaults: zero_method
 * 'wilcox', no continuity correction, two-sided, method 'auto').  n = pairs with both cells non-NaN
 * (a pair with a NaN cell is dropped); d_i = x_i - y_i is subtracted in the input's precision and then
 * widened; inf - inf counts in n but carries no rank; zeros (-0.0 included) are dropped; c = the
 * remaining differences, ranked by |d| with average ranks.  2 R+ and the tie term are exact in 64-bit
 * integers and W = min(R+, R-).  method 1 (n <= 50 without ties or zeros, or n <= 13): p is the exact
 * sign-flip distribution of the c doubled ranks counted in 64-bit integers, bit-identical to scipy;
 * method 2 (otherwise): the normal approximation with tie correction, z bit-identical to scipy and
 * p = erfc(|z| / sqrt 2).  method 0 (untested: n = 0, n = 1 with a zero difference, or method 2 with
 * c = 0): W = p = NaN.  mean1 / mean2 are float64 means of x and y over the n pairs (NaN for n = 0).
 * 1 <= n_pairs <= SD_SIGNEDRANK_MAX_PAIRS (the sort runs in shared memory).  A column outside
 * [0, n_samples) is never read: the rows get n = c = -1, method 0 and NaN statistics.  One asynchronous
 * launch on `stream`, no synchronisation.
 */
#define SD_SIGNEDRANK_MAX_PAIRS 8192
int sd_signedrank_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                       int32_t n_pairs, const int32_t *cols1, const int32_t *cols2,
                       int64_t row_begin, int64_t row_end,
                       int32_t *n_out, int64_t ld_n, double *stats_out, int64_t ld_stats, void *stream);

/* ---- K9: Friedman test per event across conditions measured on the same subjects (compare_repeated) --
 * For rows j in [row_begin, row_end) of ps (as K6): block (subject) b < n_blocks has one cell per
 * condition c < n_conditions, ps[j, cols[c * n_blocks + b]] (a DEVICE int32 list, condition-major; no
 * column listed twice), and
 *   n_out[j]                         = n, the complete blocks (no NaN in any of their k cells)
 *   mean_out[j * ld_mean + c]        = the mean of condition c over those blocks (float64 sum)
 *   stats_out[j * ld_stats + 0, 1]   = Q, p
 * with Q, p = scipy.stats.friedmanchisquare(*conditions, nan_policy='omit') (scipy 1.18.1) computed
 * without its cancellation: cells ranked within their block with average ranks, D_c = 2 R_c - n (k + 1)
 * and the tie term T exact integers, Q = 3 (k - 1) sum_c D_c^2 / (n (k^3 - k) - T) in one correctly
 * rounded division, p = chi2.sf(Q, k - 1).  Every D_c == 0 gives Q == 0 and p == 1 exactly.  n == 0 (NaN
 * means too), or every complete block tied throughout, gives Q = p = NaN (scipy gives NaN for the first,
 * NaN or +inf for the second).  -0.0 ties +0.0; +-inf are ordinary values.  3 <= n_conditions <=
 * SD_FRIEDMAN_MAX_CONDITIONS, n_blocks >= 1, n_blocks * n_conditions <= SD_RANKSUM_MAX_SAMPLES.  A column
 * outside [0, n_samples) is never read: the rows get n = -1 and NaN means and statistics.  One
 * asynchronous launch on `stream`, no synchronisation.
 */
#define SD_FRIEDMAN_MAX_CONDITIONS 256   /* chi2_sf handles df <= 255 */
int sd_friedman_rows(int64_t n_events, int32_t n_samples, const void *ps, int64_t ld_ps, int dtype,
                     int32_t n_conditions, int32_t n_blocks, const int32_t *cols,
                     int64_t row_begin, int64_t row_end,
                     int32_t *n_out, double *mean_out, int64_t ld_mean,
                     double *stats_out, int64_t ld_stats, void *stream);

/* ---- K4: intron-retention ratio ----------------------------------------------------
 * Replaces the arithmetic of ir_table.calculateIR (ir_table.py:118-132):
 *   ir[r,s] = median[r,s] / (median[r,s] + inc[r,s] + sum_{c in adj(r)} inc[c,s]),  x/0 -> NaN
 * (row_ptr == NULL: single-junction form, -s).  sd_rsd5: rsd[i] = std(cov[i,0:5]) / mean(cov[i,0:5])
 * with numpy's population std.
 */
int sd_ir_ratio(int64_t n_junctions, int32_t n_samples,
                const double *median, int64_t ld_median,
                const int32_t *counts, int64_t ld_counts,
                const int32_t *row_ptr, const int32_t *col_idx,
                double *ir_out, int64_t ld_ir,
                int64_t row_begin, int64_t row_end, void *stream);
int sd_rsd5(int64_t n, const double *cov5, double *rsd_out, void *stream);

/* ---- host-side text output (no CUDA) ---------------------------------------------------
 * Replaces the per-cell f-strings of the reference's writers: SPLICEDICE.writeInclusions /
 * writeAllpsi (SPLICEDICE.py:332-353, f'{x:.0f}' / f'{x:.3f}') and counts_to_ps.writePsValues
 * (counts_to_ps.py:69, f"{x:0.3f}").  Formats `rows` rows of a HOST matrix as
 * "name<TAB>v<TAB>...<TAB>v\n" (names == NULL: values only), byte-identical to the python
 * formatting (exact round-half-even; "nan" for any NaN), on `n_threads` host threads (<= 0: all).
 * kind 0: float32 as %.3f, 1: float64 as %.3f, 2: int32 as a decimal integer, 3: float64 as
 * python's str()/repr() (shortest round-trip digits; pairwise_fisher.py:200 writes str(p)).
 * names / name_off[rows + 1]: concatenated row names and their offsets.
 * *written receives the byte count; SD_ERR_WORKSPACE (with *written = bytes needed) if cap is
 * too small.
 */
int sd_host_format_rows(int kind, const void *matrix, int64_t rows, int32_t cols, int64_t ld,
                        const char *names, const int64_t *name_off, char *out, size_t cap,
                        size_t *written, int n_threads);
/* Same formatting, without the final compaction: every thread leaves its rows' text in its own
 * slice of `out`; segment k is out[seg_off[k], seg_off[k] + seg_len[k]) for k < *n_segments
 * (<= max_segments), to be written in order.  SD_ERR_WORKSPACE with *needed set if cap is too
 * small.  The file writers stream ~64 MB row chunks through one reusable buffer this way. */
int sd_host_format_rows_segments(int kind, const void *matrix, int64_t rows, int32_t cols, int64_t ld,
                                 const char *names, const int64_t *name_off, char *out, size_t cap,
                                 int64_t *seg_off, int64_t *seg_len, int32_t max_segments,
                                 int32_t *n_segments, size_t *needed, int n_threads);

/* Table reader for "header\nname<TAB>v<TAB>...\n" files (the reference parses them one python
 * float per cell: counts_to_ps.py:43-51, pairwise_fisher.py:46-61, ir_table.py:72-80).
 * sd_host_table_open maps the file and reports its shape; sd_host_table_read fills the raw
 * header line, the row names (concatenated, with offsets) and a float64 [rows, cols] matrix on
 * n_threads threads; ragged rows / non-numeric fields fail with SD_ERR_INVALID.
 */
void *sd_host_table_open(const char *path, int64_t *rows, int32_t *cols, int64_t *header_bytes,
                         int64_t *name_bytes);
void sd_host_table_close(void *handle);
int sd_host_table_read(void *handle, char *header, char *names, int64_t *name_off, double *values,
                       int64_t ld, int32_t n_threads);

/* ---- host-side sample-file ingest for quant (no CUDA) ------------------------------------
 * Replaces the per-line python passes SPLICEDICE.getAllJunctions (SPLICEDICE.py:147-228) and
 * SPLICEDICE.getJunctionCounts (SPLICEDICE.py:257-295): memory-mapped files, several threads,
 * hash-table union / lookup, the reference's admission rules per file type.
 * File types: 0 = STAR SJ.out.tab, 1 = bam_to_junc_bed BED (tagged name field), 2 = plain BED or
 * leafcutter; any other value = opened and ignored (.bam / unknown suffix).
 * A malformed line fails the call with SD_ERR_INVALID and "path:line: reason".
 */
typedef struct sd_quant_filter {
    int32_t max_length, min_length, min_overhang, min_unique;   /* --maxLength --minLength --minOverhang --minUnique */
    int32_t no_multimap, low_coverage_nan;                      /* --noMultimap --lowCoverageNan */
    uint32_t motif_mask;                                        /* bit m: STAR motif code m admitted (--filter) */
    uint32_t reserved;
    double min_entropy;                                         /* --minEntropy */
} sd_quant_filter;
void *sd_ingest_create(void);
void sd_ingest_destroy(void *handle);
int sd_ingest_collect(void *handle, int32_t n_files, const char *const *paths, const int32_t *types,
                      const sd_quant_filter *filter, int32_t n_threads);
int64_t sd_ingest_junction_count(void *handle);
int32_t sd_ingest_chrom_count(void *handle);
const char *sd_ingest_chrom_name(void *handle, int32_t id);
int sd_ingest_export(void *handle, int32_t *chrom_id, int32_t *left, int32_t *right, int8_t *strand);
int sd_ingest_index(void *handle, int64_t n, const char *const *chrom_names, const int32_t *chrom_of,
                    const int32_t *left, const int32_t *right, const int8_t *strand, const int32_t *row);
int sd_ingest_counts(void *handle, int32_t n_files, const char *const *paths, const int32_t *types,
                     const int32_t *samples, const sd_quant_filter *filter, int32_t *counts,
                     int64_t ld_counts, uint8_t *low_mask, int64_t ld_mask, int32_t n_threads);

/* ---- synthetic inputs + probes (bench / tests) --------------------------------------
 * sd_synth_counts: the counter-based generator of splicedice_b200/synth.py:counts_host,
 * bit for bit.  out[r - row0, c] for r in [row0, row0 + n_rows), c < n_cols.
 * sd_probe_fp64: sustained FP64 FMA rate (GFLOP/s) of the device behind `stream`.
 * sd_probe_copy: device-to-device copy bandwidth (GB/s, read + write bytes).
 */
int sd_synth_counts(uint64_t seed, int64_t row0, int64_t n_rows, int32_t n_cols,
                    int64_t logical_cols, uint32_t scale,
                    int32_t *out, int64_t ld_out, void *stream);
int sd_probe_fp64(double *gflops_out, void *stream);
int sd_probe_copy(int64_t bytes, double *gbs_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SPLICEDICE_B200_H */
