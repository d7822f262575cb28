/*
 * illico_b200.h -- C ABI of the B200-native asymptotic Wilcoxon rank-sum (Mann-Whitney U) hot path.
 *
 * This is the drop-in boundary for the ONE path this repository accelerates: the six batch
 * "dispatcher" kernels of remydubois/illico and the primitives under them (SURVEY.md section 8).
 * Plain `extern "C"`, plain pointers and sizes, no torch / Python types.  Every buffer is owned by
 * the caller (device pointers unless stated otherwise); the library allocates nothing persistent.
 * All functions return 0 on success, non-zero on failure; `illico_last_error()` gives the message
 * (thread-local).  All work is enqueued on the caller's `stream` (a `cudaStream_t` passed as void*).
 * Re-entrant per (device, stream).
 *
 * Reference interface each entry point replaces (paths relative to the reference repo):
 *
 *   illico_stage_dense_f32   chunk_and_fortranize            illico/utils/math.py:247-278
 *                            (+ the per-group row gathers of  illico/ovo/dense_ovo.py:111-123)
 *   illico_stage_csr_f32     csr_get_contig_cols_into_csc     illico/utils/sparse/csr.py:199-257
 *                            csr_get_contig_cols_into_csr     illico/utils/sparse/csr.py:144-196
 *                            csr_get_rows_into_csc            illico/utils/sparse/csr.py:103-141
 *   illico_stage_csc_f32     csc_get_cols                     illico/utils/sparse/csc.py:99-136
 *                            csc_get_contig_cols_into_csr     illico/utils/sparse/csc.py:139-183
 *   illico_rank_ovr          dense_ovr_mwu_kernel_over_contiguous_col_chunk  illico/ovr/dense_ovr.py:15-80
 *                            sparse_ovr_mwu_kernel            illico/ovr/sparse_ovr.py:23-97
 *                            _accumulate_group_ranksums_from_argsort         illico/utils/ranking.py:7-49
 *   illico_rank_ovo          dense_ovo_mwu_kernel(+wrapper)   illico/ovo/dense_ovo.py:15-137
 *                            single_/multi_group_sparse_ovo_mwu_kernel       illico/ovo/sparse_ovo.py:22-158
 *                            rank_sum_and_ties_from_sorted    illico/utils/ranking.py:52-158
 *   (both rank kernels)      compute_pval                     illico/utils/math.py:64-118
 *                            dense_/csc_/csr_fold_change, fold_change_from_summed_expr
 *                                                             illico/utils/math.py:168-221,
 *                                                             illico/utils/sparse/csc.py:186-211, csr.py:261-286
 *   illico_check_csr_sorted  check_indices_sorted_per_parcel  illico/utils/ranking.py:245-273
 *   illico_recode_*          the dtype specialisations of the numba kernels (float64 input)   illico/ovr/dense_ovr.py:46-53
 *   illico_csr_shard_*       csr_get_contig_cols_into_csr, across GPUs                        illico/utils/sparse/csr.py:144-196
 *   illico_{ovr,ovo}_{dense,csc,csr}_f32   the six dispatchers registered in
 *                            illico/utils/registry.py:193-202 (call site illico/asymptotic_wilcoxon.py:59-67)
 *
 * Data model.  A gene batch is first STAGED into a group-segmented, gene-major list of its
 * non-zero values (zeros are one analytic tie block, for dense input too), then RANKED:
 *
 *   plan      : cells permuted to group-contiguous order; each group is cut into segments of at most
 *               `seg_max` cells; segment s owns slot [seg_base[s], seg_base[s+1]) of every gene's
 *               slot space (capacity `slot_cap` floats per gene).
 *   ir_vals   : float  [n_genes_batch, slot_cap]   non-zero values of (gene, segment), compacted at
 *                                                  the start of the segment's slot
 *   ir_cnt    : uint32 [n_genes_batch, n_segments] how many values each (gene, segment) slot holds
 *   results   : double [n_groups, result_gene_stride/3 .., 3] = (p_value, statistic, fold_change),
 *               the layout of the reference's `results[G, N, 3]` (asymptotic_wilcoxon.py:210, 241-244).
 *
 * The dense and CSR dispatchers (illico_{ovr,ovo}_{dense,csr}_f32) take a shorter road when the batch is count-like
 * (at most 12 distinct non-zero values per gene): ONE pass over the input writes each group's histogram over the
 * gene's value table into the 24 bytes its result will occupy, and an epilogue turns it into (p, U, fold change) in
 * place -- no staged lists, no rank kernel (illico_b200/csrc/fused.cu; same statistics bit for bit).  Genes that
 * do not qualify are listed ON THE DEVICE and finished by the stage + rank kernels above, through the same buffers.
 *
 * Every entry point only ENQUEUES work on `stream` and returns: no dispatcher synchronises the stream or reads anything
 * back (illico_check_csr_sorted is the one call whose answer is a host value).  Calls on different streams with different
 * illico_batch_buffers_t run concurrently; `workspace` must be illico_rank_workspace_bytes() large.
 */
#ifndef ILLICO_B200_H
#define ILLICO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ILLICO_ABI_VERSION 3

enum illico_alternative { ILLICO_TWO_SIDED = 0, ILLICO_LESS = 1, ILLICO_GREATER = 2 };

/* tie-sum accumulation order of the reference kernels (SURVEY.md appendix A.4) */
enum illico_tie_order {
    ILLICO_TIES_DENSE = 0, /* zero block at its sorted position (dense kernels, utils/ranking.py:31-47) */
    ILLICO_TIES_SPARSE = 1 /* non-zero runs first, zero block last (ovr/sparse_ovr.py:83, ovo/sparse_ovo.py:85) */
};

/* Group plan: the device-side form of the reference's GroupContainer (illico/utils/groups.py:6-15). */
typedef struct illico_plan {
    int32_t n_cells;
    int32_t n_groups;
    int32_t n_segments;
    int32_t ref_group;          /* -1 = one-versus-rest (groups.py:55-57) */
    int32_t max_group_size;
    int32_t ref_group_size;     /* cells of the reference group (0 for one-versus-rest) */
    int32_t ref_seg_begin;      /* segments [ref_seg_begin, ref_seg_end) belong to the reference group */
    int32_t ref_seg_end;
    int32_t slot_cap;           /* floats per gene in ir_vals (= seg_base[n_segments]) */
    int32_t max_target_group_size; /* largest group other than the reference group (= max_group_size without one) */
    const int32_t* perm;        /* [n_cells]     perm[pos] = cell (row) index, groups contiguous, stable */
    const int32_t* cell_seg;    /* [n_cells]     segment of each cell (row -> segment) */
    const int32_t* seg_pos;     /* [n_segments+1] positions (into perm) covered by each segment.  Every segment must
                                   have fewer than 65536 cells (seg_pos[s+1] - seg_pos[s] <= 65535): the staging kernels'
                                   count tiles, the one-versus-rest table bins and the fused CSR pass's control
                                   histogram count a segment's cells in 16 bits.  Not checked here. */
    const int32_t* seg_base;    /* [n_segments+1] slot offset of each segment inside a gene's slot space */
    const int32_t* seg_group;   /* [n_segments]  owning group */
    const int32_t* group_seg;   /* [n_groups+1]  segments of each group */
    const int32_t* group_size;  /* [n_groups]    cells per group (GroupContainer.counts) */
} illico_plan_t;

typedef struct illico_flags {
    int32_t is_log1p;       /* fold change on expm1(x) (utils/math.py:212) */
    int32_t use_continuity; /* 0.5 continuity correction (utils/math.py:100-114) */
    int32_t tie_correct;    /* 0 -> tie sum := 0 in the p-value (ovr/dense_ovr.py:70) */
    int32_t alternative;    /* enum illico_alternative */
    int32_t tie_order;      /* enum illico_tie_order */
    int32_t n_cols_hint;    /* unused (kept so that the layout stays as in ABI version 3); pass 0 */
    /* Optional [n_groups, n_genes_batch] float64 expression sums (device).  When set, the fold change uses them
     * instead of sums of the staged values: the host stages ORDER-PRESERVING float32 codes of values that
     * float32 cannot hold (float64 / large integers), which keeps U, ties and p exact. */
    const double* group_sums;
    /* Optional signed effect score of every test (device, NULL = not written): (mu - U) / sigma with mu = n_r n_t / 2 and
     * the sigma of the p-value (tie-corrected iff tie_correct; no continuity correction, whatever the alternative) --
     * positive when the group ranks above the reference / rest; 0 where the tie correction is <= 1e-9 (p = 1) and on the
     * one-versus-reference control row.  Points at element [group 0, first gene of the batch], like `results`;
     * score_group_stride = doubles between consecutive groups. */
    double* scores;
    int64_t score_group_stride;
} illico_flags_t;

/* Optional per-test debug outputs for bit-exact parity checks (any pointer may be NULL). */
typedef struct illico_debug {
    int64_t* u2;       /* [n_groups, n_genes_batch]  2*U as an exact integer */
    double* tie_sum;   /* OVR: [n_genes_batch]; OVO: [n_groups, n_genes_batch]  f64 tie sum fed to the p-value */
    int64_t* tie_exact;/* same shape as tie_sum: exact integer sum of t^3 - t */
} illico_debug_t;

int illico_abi_version(void);
const char* illico_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t illico_launch_count(void);
/* >= 0 when the last dispatcher call of this thread enqueued a fused pass (fused.cu), -1 when it took the general stage +
 * rank path (per-kernel durations: illico_profile_report) */
double illico_last_fused_ms(void);
/* with ILLICO_PROFILE=1: every kernel this library launches is bracketed by CUDA events on the launching stream.  This
 * call waits for the recorded launches, writes one line "kernel_name\ttotal_ms\tlaunches\n" per kernel (in first-launch
 * order) into `out` (at most cap - 1 bytes + NUL), forgets them, and returns the full text length.  bench.py's roofline. */
int64_t illico_profile_report(char* out, int64_t cap);

/* ---- column shards in, result slabs out -------------------------------------------------------------
 * Strided asynchronous copy (cudaMemcpy2DAsync) on `stream`: kind 1 = host to device, 2 = device to host, 3 = device to
 * device (the two sides may be on different GPUs: how the shards' slabs of a ranking run meet on one GPU).  The host side
 * should be page-locked for the copy to be asynchronous.  This is how a GPU receives its gene shard X[:, lb:ub] of a
 * C-order host matrix (height = n_cells rows of width_bytes = 4 (ub - lb), spitch = 4 n_genes) and how it delivers its
 * slab results[:, lb:ub, :] into the one host array of the reference's layout (illico/asymptotic_wilcoxon.py:210,
 * 241-244: the reference's threads write their batches into the same array). */
int illico_memcpy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                          int kind, void* stream);

/* ---- staging: input formats -> group-segmented non-zero lists ------------------------------- */

/* X: row-major [n_cells, ld] float32 on the device; genes [gene_lb, gene_lb + n_genes_batch). */
int illico_stage_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                           const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, void* stream);

/* CSR (rows = cells): data/indices [nnz], indptr [n_cells+1] (int64).  Row indices must be sorted
 * (illico/asymptotic_wilcoxon.py:185-193).  Needs illico_stage_csr_workspace_bytes() of device scratch (may be
 * the rank workspace: the rank kernels run after staging on the same stream). */
size_t illico_stage_csr_workspace_bytes(const illico_plan_t* plan, int32_t n_genes_batch);
int illico_stage_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr,
                         int32_t gene_lb, int32_t n_genes_batch, const illico_plan_t* plan,
                         float* ir_vals, uint32_t* ir_cnt, void* workspace, size_t workspace_bytes, void* stream);

/* CSC (columns = genes): data/indices [nnz], indptr [n_genes+1] (int64); columns gene_lb..
 * ir_cnt must be zeroed by the caller (illico_zero_counts). */
int illico_stage_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr,
                         int32_t gene_lb, int32_t n_genes_batch, const illico_plan_t* plan,
                         float* ir_vals, uint32_t* ir_cnt, void* stream);

int illico_zero_counts(uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan, void* stream);

/* returns 1 if every row's indices ascend, 0 if not, <0 on error; result read back synchronously */
int illico_check_csr_sorted(const int32_t* indices, const int64_t* indptr, int64_t n_rows, int32_t* d_flag,
                            void* stream);

/* ---- ranking + fused epilogue ------------------------------------------------------------- */

/* bytes of device scratch the rank kernels need for this plan (pass >= this many to illico_rank_*) */
size_t illico_rank_workspace_bytes(const illico_plan_t* plan, int32_t n_genes_batch);

/* results: pointer to element [group 0, first gene of the batch, 0]; result_group_stride in doubles
 * between consecutive groups (= 3 * total genes of the final array). */
int illico_rank_ovr(const float* ir_vals, const uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan,
                    const illico_flags_t* flags, double* results, int64_t result_group_stride,
                    void* workspace, size_t workspace_bytes, const illico_debug_t* dbg, void* stream);

int illico_rank_ovo(const float* ir_vals, const uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan,
                    const illico_flags_t* flags, double* results, int64_t result_group_stride,
                    void* workspace, size_t workspace_bytes, const illico_debug_t* dbg, void* stream);

/* ---- the six dispatchers (stage + rank in one call), reference registry.py:193-202 ---------- */

typedef struct illico_batch_buffers {
    float* ir_vals;          /* [n_genes_batch * plan->slot_cap] */
    uint32_t* ir_cnt;        /* [n_genes_batch * plan->n_segments] */
    void* workspace;         /* illico_rank_workspace_bytes() */
    size_t workspace_bytes;
} illico_batch_buffers_t;

int illico_ovr_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                         const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                         double* results, int64_t result_group_stride, const illico_debug_t* dbg, void* stream);
int illico_ovo_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                         const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                         double* results, int64_t result_group_stride, const illico_debug_t* dbg, void* stream);
int illico_ovr_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                       int32_t n_genes_batch, const illico_plan_t* plan, const illico_flags_t* flags,
                       const illico_batch_buffers_t* buf, double* results, int64_t result_group_stride,
                       const illico_debug_t* dbg, void* stream);
int illico_ovo_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                       int32_t n_genes_batch, const illico_plan_t* plan, const illico_flags_t* flags,
                       const illico_batch_buffers_t* buf, double* results, int64_t result_group_stride,
                       const illico_debug_t* dbg, void* stream);
int illico_ovr_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                       int32_t n_genes_batch, const illico_plan_t* plan, const illico_flags_t* flags,
                       const illico_batch_buffers_t* buf, double* results, int64_t result_group_stride,
                       const illico_debug_t* dbg, void* stream);
int illico_ovo_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                       int32_t n_genes_batch, const illico_plan_t* plan, const illico_flags_t* flags,
                       const illico_batch_buffers_t* buf, double* results, int64_t result_group_stride,
                       const illico_debug_t* dbg, void* stream);

/* ---- input dtypes (SURVEY.md section 8b) ----------------------------------------------------------------------------
 * The dispatchers above take float32 values.  The reference ranks whatever dtype the matrix has (numba specialises its
 * kernels per dtype, illico/ovr/dense_ovr.py:46-53); here every real dtype that float32 holds exactly (integer counts,
 * float16, ...) is converted on upload, and ILLICO_DTYPE_F64 -- values float32 cannot hold -- goes through the recode
 * entry points: per gene, the values become order-preserving float32 codes (the signed rank among the gene's distinct
 * values: zero -> 0, negatives < 0 < positives, equal values equal -- ranks, U and tie sums only depend on that) in the
 * input's own layout, and the fold change's float64 group sums (illico/utils/math.py:168-221) are computed from the
 * original values into `group_sums` [n_groups, n_genes_batch], to be passed on in illico_flags_t::group_sums.  The
 * ordinary dispatcher is then called on the codes.  cell_group: [n_cells] group of every cell (GroupContainer
 * .encoded_groups).  Hand-written kernels (64-bit LSD radix sort per gene, csrc/recode.cu); workspace from
 * illico_recode_workspace_bytes(total_keys, n_genes_batch) with total_keys = n_cells * n_genes_batch (dense, CSR) or the
 * batch's stored values (CSC). */
enum illico_dtype {
    ILLICO_DTYPE_F32 = 0, ILLICO_DTYPE_F64 = 1, ILLICO_DTYPE_F16 = 2, ILLICO_DTYPE_I8 = 3, ILLICO_DTYPE_U8 = 4,
    ILLICO_DTYPE_I16 = 5, ILLICO_DTYPE_I32 = 6, ILLICO_DTYPE_I64 = 7
};
/* Conversion on upload: `count` values of `dtype` -> dst_f32 (optional) and / or dst_f64 (optional); *inexact (device int,
 * zeroed by this call) is set when float32 changes some value -- such a matrix keeps its float64 copy and goes through
 * the recode entry points, nothing is ever rounded (rounding would create ties that are not in the data). */
int illico_convert_values(const void* src, int32_t dtype, int64_t count, float* dst_f32, double* dst_f64, int32_t* inexact,
                          void* stream);
size_t illico_recode_workspace_bytes(int64_t total_keys, int32_t n_genes_batch);
/* X: row-major [n_cells, ld] of `dtype`; codes: row-major [n_cells, n_genes_batch] */
int illico_recode_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch, int64_t n_cells,
                        const int32_t* cell_group, int32_t n_groups, int32_t is_log1p, float* codes, double* group_sums,
                        void* workspace, size_t workspace_bytes, void* stream);
/* codes: parallel to `data` (the whole array; only the batch's entries are written) */
int illico_recode_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                      int32_t n_genes_batch, int64_t batch_nnz, const int32_t* cell_group, int32_t n_groups, int32_t is_log1p,
                      float* codes, double* group_sums, void* workspace, size_t workspace_bytes, void* stream);
int illico_recode_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int64_t n_cells,
                      int32_t gene_lb, int32_t n_genes_batch, const int32_t* cell_group, int32_t n_groups, int32_t is_log1p,
                      float* codes, double* group_sums, void* workspace, size_t workspace_bytes, void* stream);

/* ---- rows -> genes repartition of a CSR matrix across GPUs (SURVEY.md section 8e) -------------------------------------
 * Replaces, across GPUs, csr_get_contig_cols_into_csr (illico/utils/sparse/csr.py:144-196): every GPU holds a block of
 * ROWS [row0, row0 + n_rows) of the CSR matrix (indptr rebased to the block: indptr[0] = 0) and cuts it into n_shards
 * (<= 32) column ranges bounds[j] <= column < bounds[j + 1] (device array of n_shards + 1 ascending column indices).
 *   illico_csr_shard_count    cnt[j * n_rows + r] = entries of row r in shard j; totals[j] += their sum (zero it first).
 *   illico_csr_shard_scatter  writes row r's piece for shard j at out_data[j][out_pos[j * n_rows + r] ...] /
 *                             out_indices[j][...] (column index rebased to the shard) and its count at
 *                             out_row_cnt[j][row0 + r].  The out_* arrays (host arrays of n_shards device pointers) may live
 *                             on OTHER GPUs with peer access enabled (illico_enable_peer_access): the kernel's stores are
 *                             the exchange.  out_pos = the shard's running offset: entries of earlier row blocks + the
 *                             exclusive scan of cnt over this block's rows.
 * The owner of shard j then has its genes as a CSR matrix over all rows: data / indices as written, indptr = the scan of its
 * row counts. */
int illico_enable_peer_access(int32_t device, int32_t peer_device);
int illico_csr_shard_count(const int32_t* indices, const int64_t* indptr, int64_t n_rows, const int32_t* bounds,
                           int32_t n_shards, int32_t* cnt, uint64_t* totals, void* stream);
int illico_csr_shard_scatter(const float* data, const int32_t* indices, const int64_t* indptr, int64_t n_rows, int64_t row0,
                             const int32_t* bounds, int32_t n_shards, const int32_t* cnt, const int64_t* out_pos,
                             float* const* out_data, int32_t* const* out_indices, int32_t* const* out_row_cnt, void* stream);

/* ---- packed upload of a dense float32 matrix (host input; replaces the zero-copy InRAMDataHandler.fetch of
 * illico/utils/registry.py:97-100 at the device boundary) ---------------------------------------------------------------
 * A dense expression matrix is mostly zeros and its upload is the end-to-end time.  The host threads that stage row chunks
 * squeeze them (csrc/hostpack.c: plain C, AVX-512 / AVX2 / scalar code chosen at run time) into
 *   mask [n_rows][(n_cols + 31) / 32] uint32 (bit k of word w: element 32 w + k is non-zero), row_off [n_rows + 1] uint32
 *   (position of each row's first value), vals: the non-zero values row by row (capacity vals_cap floats, 16 of them slack);
 * the packed chunk crosses PCIe and the device call rebuilds the dense rows in HBM (every element written once, zeros
 * included).  All pointers of the host call are HOST pointers; it returns the number of values, or -1 when they do not fit
 * (the caller then sends the chunk as it is).  The isa call returns 2 / 1 / 0 = AVX-512 / AVX2 / scalar. */
long illico_host_pack_rows_f32(const float* src, long row_stride, long n_rows, long n_cols, uint32_t* mask, uint32_t* row_off,
                               float* vals, long vals_cap);
int illico_host_pack_isa(void);
int illico_unpack_rows_f32(const uint32_t* mask, const uint32_t* row_off, const float* vals, int64_t n_rows, int32_t n_cols,
                           float* dst, int64_t dst_ld, void* stream);

/* ---- next to the path (SURVEY.md section 8f.4) and a test hook ------------------------------------------- */

/* Benjamini-Hochberg adjusted p-values over the genes of each group (statsmodels multipletests(method="fdr_bh") /
 * scanpy `pvals_adj`): p_values[g * group_stride + j * gene_stride] -> p_adj[g * n_genes + j].  Reads the p-value plane
 * of the results array in place with group_stride = 3 * n_genes, gene_stride = 3. */
size_t illico_bh_workspace_bytes(int32_t n_groups, int32_t n_genes);
int illico_bh_adjust(const double* p_values, int64_t group_stride, int64_t gene_stride, int32_t n_groups, int32_t n_genes,
                     double* p_adj, void* workspace, size_t workspace_bytes, void* stream);

/* Per-group ranking of the genes (scanpy rank_genes_groups' order): group g's n_genes scores
 * scores[g * score_group_stride + j] sorted descending (by_abs != 0: by |score|), ties by gene index ascending, NaN after
 * every number, -0.0 equal to +0.0.  The first k (1 <= k <= n_genes) gene indices go to out_gene [n_groups, k] (int32) and
 * their records (score, p_value, statistic, fold_change, p_adj) to out_rec [n_groups, k, 5] (float64), gathered from the
 * score plane, results[g * result_group_stride + 3 j ..] and p_adj[g * n_genes + j] (NULL: NaN).  Stable LSD radix sort,
 * one CTA per group; workspace from illico_top_genes_workspace_bytes. */
size_t illico_top_genes_workspace_bytes(int32_t n_groups, int32_t n_genes);
int illico_top_genes(const double* scores, int64_t score_group_stride, const double* results, int64_t result_group_stride,
                     const double* p_adj, int32_t n_groups, int32_t n_genes, int32_t k, int32_t by_abs, int32_t* out_gene,
                     double* out_rec, void* workspace, size_t workspace_bytes, void* stream);

/* illico_top_genes with scanpy's marker filter (filter_rank_genes_groups) applied before the selection.  A gene is kept
 * when every GIVEN criterion holds: pct_group >= min_in_group, pct_ref <= max_out_group, fold_change >= fc_min or
 * fold_change <= fc_max (pass NaN for a criterion that is not given; fc_max is the host's 1 / fc_min for a by-|fold change|
 * filter, NaN otherwise).  A NaN meeting a given criterion fails it.  Kept genes come first in illico_top_genes' order,
 * dropped genes after all of them; the first min(k, kept[g]) are written, the rest of the row gets gene -1 and an all-NaN
 * record.  Records are [n_groups, k, 7] = (score, p_value, statistic, fold_change, p_adj, pct_group, pct_ref), each NaN where
 * its plane is NULL; pct_group / pct_ref are [n_groups, n_genes] like p_adj (illico_nonzero_fractions) and must be given
 * with their bound.  kept [n_groups] (NULL: not written) = genes of the group that pass.  The BH p_adj is the caller's:
 * over all genes, as scanpy adjusts before it filters.  Workspace: illico_top_genes_workspace_bytes. */
int illico_top_genes_filtered(const double* scores, int64_t score_group_stride, const double* results, int64_t result_group_stride,
                              const double* p_adj, const double* pct_group, const double* pct_ref, int32_t n_groups, int32_t n_genes,
                              int32_t k, int32_t by_abs, double min_in_group, double max_out_group, double fc_min, double fc_max,
                              int32_t* out_gene, double* out_rec, int32_t* kept, void* workspace, size_t workspace_bytes,
                              void* stream);

/* ---- cells that express a gene (scanpy rank_genes_groups(pts=True): pct_nz_group / pct_nz_reference) -------------------
 * counts[g * count_group_stride + j] (int32) = cells of group g whose value in gene gene_lb + j satisfies x != 0: -0.0 and
 * explicitly stored zeros do not count, NaN does.  Every element of the batch's [n_groups, n_genes_batch] plane is written
 * (the caller zeroes nothing).  `dtype` is ILLICO_DTYPE_F32 or ILLICO_DTYPE_F64 (a recoded batch is counted on its original
 * float64 values, not on the codes); any other dtype is an error.  The inputs are those of the staging calls: dense rows of
 * any `ld` (no alignment needed), CSR rows with sorted indices, CSC columns gene_lb.. .  Rows are walked through the plan
 * (perm / segments; CSC: group of a row = seg_group[cell_seg[row]]).  A read-only pass of its own over the batch, run only
 * when asked for (csrc/counts.cu). */
int illico_count_nonzero_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                               const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride, void* stream);
int illico_count_nonzero_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride,
                             void* stream);
int illico_count_nonzero_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride,
                             void* stream);
/* The gathered count plane counts [n_groups, >= n_genes] -> pct_group / pct_ref [n_groups, n_genes] float64, one IEEE
 * division each:  pct_group[g, j] = count[g, j] / n_g;  one-versus-reference (ref_group >= 0): pct_ref[g, j] =
 * count[ref, j] / n_ref on every row, the reference's own included;  one-versus-rest (ref_group < 0): pct_ref[g, j] =
 * (total_j - count[g, j]) / (n_cells - n_g), total_j the exact sum over the groups (0 / 0 = NaN with a single group).
 * group_size: device [n_groups]; n_cells = their sum. */
int illico_nonzero_fractions(const int32_t* counts, int64_t count_group_stride, const int32_t* group_size, int32_t n_groups,
                             int32_t n_genes, int32_t ref_group, int64_t n_cells, double* pct_group, double* pct_ref, void* stream);

/* ---- Welch's t-test (scanpy rank_genes_groups(method="t-test" | "t-test_overestim_var")) -----------------------------------
 * illico_group_moments_*: the count kernels' walks with float64 accumulators.  For group g and gene gene_lb + j:
 * sums[g * group_stride + j] = sum of x, sumsq[..] = sum of x * x (x widened to float64 first, then squared), and with
 * is_log1p fsums[..] = sum of expm1(x) (the fold change's values; fsums is not touched otherwise and may be NULL).  counts
 * (may be NULL) receives illico_count_nonzero_*'s plane in the same launch, counts[g * count_group_stride + j].  Every element of the
 * [n_groups, n_genes_batch] planes is written.  A group with one plan segment stores its sums; one with several adds its
 * segments' sums (exact for integer data, any order).  dtype ILLICO_DTYPE_F32 or ILLICO_DTYPE_F64: float64 input is read as
 * it is, no recoding.  Inputs as for illico_count_nonzero_* (csrc/counts.cu). */
int illico_group_moments_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                               const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq, double* fsums,
                               int32_t* counts, int64_t count_group_stride, int64_t group_stride, void* stream);
int illico_group_moments_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq,
                             double* fsums, int32_t* counts, int64_t count_group_stride, int64_t group_stride,
                             void* stream);
int illico_group_moments_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq,
                             double* fsums, int32_t* counts, int64_t count_group_stride, int64_t group_stride,
                             void* stream);
/* The moment planes of a batch of n_genes genes -> results[g * result_group_stride + 3 j ..] = (p, t, fold_change) and, when
 * scores is not NULL, scores[g * score_group_stride + j] = t with NaN -> 0.  One thread per gene (csrc/ttest.cu):
 *   mean = S1 / n;  var = S2 / n - mean * mean;  if n != 1: var *= n / (n - 1)        (scanpy 1.10 _get_mean_var, dense)
 *   comparison sample: group ref_group (>= 0), or all other cells (< 0: the gene's sums over the groups in a fixed order,
 *   minus the group's; n_cells - n_g cells)
 *   vn = sqrt(var)**2 / n;  df = (vn1 + vn2)**2 / (vn1**2 / (n1 - 1) + vn2**2 / (n2 - 1)), NaN -> 1;
 *   t = (mean1 - mean2) / sqrt(vn1 + vn2)                   (scipy 1.18 _unequal_var_ttest_denom, _ttest_ind_from_stats)
 *   p = 2 stdtr(df, -|t|) | stdtr(df, -t) (greater) | stdtr(df, t) (less), NaN -> 1          (scipy _get_pvalue; scanpy)
 * with n2 = the group's own size for overestim_var != 0 ("t-test_overestim_var"; the comparison variance still comes from
 * its own cells).  The fold change is the Wilcoxon kernels' expression on fsums (sums when fsums is NULL): OVO
 * (sum_g * (1 / n_g)) * (1 / (sum_r / n_r)), OVR (sum_g * (1 / n_g)) / ((total - sum_g) / (n_cells - n_g)), inf where the
 * comparison mean is 0.  The reference group's row is (1, 0, fold change of the control with itself), score 0.
 * group_size: device [n_groups].  Two launches: t, df and the fold change (CTA = 32 genes x 16 group lanes), then p. */
int illico_welch_ttest(const double* sums, const double* sumsq, const double* fsums, int64_t group_stride, const int32_t* group_size,
                       int32_t n_groups, int32_t n_genes, int32_t ref_group, int64_t n_cells, int32_t overestim_var,
                       int32_t alternative, double* results, int64_t result_group_stride, double* scores, int64_t score_group_stride,
                       void* stream);
/* The t-test's p-value on arrays (device pointers): out[i] = 2 stdtr(df[i], -|t[i]|) (ILLICO_TWO_SIDED), stdtr(df[i], -t[i])
 * (ILLICO_GREATER) or stdtr(df[i], t[i]) (ILLICO_LESS), stdtr the Student t CDF (scipy.special.stdtr), without the NaN -> 1
 * replacement: the known-answer hook of the device code. */
int illico_student_t_batch(const double* df, const double* t, int64_t n, int32_t alternative, double* out, void* stream);

/* The device epilogue's compute_pval (illico/utils/math.py:64-118) on arrays of arguments (device pointers): lets the
 * known-answer vectors of the reference's primitive be checked against the GPU code itself. */
int illico_compute_pval_batch(const int64_t* n_ref, const int64_t* n_tgt, const int64_t* n, const double* tie_sum,
                              const double* U, const double* mu, const double* contin_corr, const int32_t* alternative,
                              double* out, int64_t count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ILLICO_B200_H */
