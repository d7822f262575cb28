// extras.cu -- consumers next to the hot path (SURVEY.md section 8f.4) and a test hook for the fused epilogue.
//
//   illico_bh_adjust           Benjamini-Hochberg adjusted p-values over the genes of each group: what scanpy reports as
//                              `pvals_adj` next to the statistic users compare illico with
//                              (reference tests/test_asymptotic_wilcoxon.py:30-60).  Same operation order as
//                              statsmodels' multipletests(method="fdr_bh"): p_sorted / (k / N), reverse running minimum,
//                              clipped at 1.
//   illico_top_genes           ranks the genes of each group by score (stable radix sort of order-preserving keys carrying
//                              the gene index) and gathers the first k genes' records: scanpy's rank_genes_groups order.
//   illico_top_genes_filtered  the same ranking with scanpy's filter_rank_genes_groups criteria applied first (dropped genes
//                              sort after every kept one) and the expressing-cell fractions in the record.
//   illico_bonferroni_adjust   Bonferroni adjusted p-values, min(p * n_genes, 1) (scanpy's corr_method="bonferroni").
//   illico_top_genes_columns   illico_top_genes' ranking written column-major in scanpy's record layout ([k, groups]
//                              planes of gene index, float32 score / log fold change, float64 p / p_adj).
//   illico_filter_marker_pairs scanpy's filter_rank_genes_groups criteria on the listed (rank, group) pairs of a stored
//                              result: a uint8 keep mask [k, groups], from device planes or from planes taken from `uns`.
//   illico_compute_pval_batch  evaluates the epilogue's compute_pval (epilogue.cuh; reference illico/utils/math.py:64-118)
//                              on arrays of arguments, so the known-answer vectors of tests/golden/primitives.npz can be
//                              checked against the device code itself.
#include "common.cuh"
#include "epilogue.cuh"
#include "sort.cuh"

namespace illico {

namespace {

constexpr int BH_THREADS = 512;
constexpr int BH_NW = BH_THREADS / 32;

// One CTA per group (grid-strided).  keys: the group's p-values as u64 (non-negative doubles order like their bits).
// A group with a NaN p-value (one-versus-rest with a single group: sigma = 0) gets NaN for every gene, as in statsmodels,
// where the NaN sorts last and the reverse running minimum carries it to every rank.
__global__ void __launch_bounds__(BH_THREADS) bh_adjust_kernel(const double* __restrict__ p, long long group_stride,
                                                               long long gene_stride, int G, int N, double* __restrict__ padj,
                                                               unsigned long long* __restrict__ slab) {
    __shared__ uint32_t hist[BH_NW * 256];
    __shared__ uint32_t aux[RADIX_AUX_WORDS];
    __shared__ double wmin[BH_NW];
    __shared__ int has_nan;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    unsigned long long* A = slab + (long long)blockIdx.x * 2 * N;
    unsigned long long* B = A + N;
    for (int g = blockIdx.x; g < G; g += gridDim.x) {
        const double* pg = p + (long long)g * group_stride;
        if (tid == 0) has_nan = 0;
        __syncthreads();
        for (int j = tid; j < N; j += BH_THREADS) {
            double v = pg[(long long)j * gene_stride];
            if (v != v) has_nan = 1;
            if (!(v >= 0.0)) v = 0.0;                                   // (negative p-values never come out of compute_pval)
            A[j] = (unsigned long long)__double_as_longlong(v);
        }
        __syncthreads();
        if (has_nan) {
            for (int j = tid; j < N; j += BH_THREADS) padj[(long long)g * N + j] = NAN;
            __syncthreads();                                             // (every thread has read has_nan before it is reset)
            continue;
        }
        unsigned long long* S = block_radix_sort_t<unsigned long long>(A, B, N, hist, aux);
        double* M = reinterpret_cast<double*>(S == A ? B : A);          // suffix minima of p_(k) / (k / N)
        // reverse running minimum: thread t owns the contiguous ranks [lo, hi) counted from the END of the order
        const int per = (N + BH_THREADS - 1) / BH_THREADS;
        const int hi = N - tid * per, lo = max(0, hi - per);            // ranks (0-based) [lo, hi)
        double local = INFINITY;
        for (int k = hi - 1; k >= lo; --k) {
            const double raw = __ddiv_rn(__longlong_as_double((long long)S[k]), __ddiv_rn((double)(k + 1), (double)N));
            local = fmin(local, raw);
            M[k] = local;
        }
        // exclusive scan (min) over threads in order of increasing tid = decreasing rank
        double incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl = fmin(incl, t);
        }
        if (lane == 31) wmin[w] = incl;
        __syncthreads();
        double before = INFINITY;                                        // minimum over all threads with smaller tid
        for (int ww = 0; ww < w; ++ww) before = fmin(before, wmin[ww]);
        const double up = __shfl_up_sync(FULL, incl, 1);
        if (lane > 0) before = fmin(before, up);
        for (int k = hi - 1; k >= lo; --k) M[k] = fmin(1.0, fmin(M[k], before));
        __syncthreads();
        // every gene takes the value at the rank of the LAST element tied with it
        for (int j = tid; j < N; j += BH_THREADS) {
            double v = pg[(long long)j * gene_stride];
            if (!(v >= 0.0)) v = 0.0;                                   // (the group holds no NaN: see has_nan)
            const unsigned long long key = (unsigned long long)__double_as_longlong(v);
            int a = 0, b = N;
            while (a < b) { const int mid = (a + b) >> 1; if (S[mid] <= key) a = mid + 1; else b = mid; }
            padj[(long long)g * N + j] = M[a - 1];
        }
        __syncthreads();
    }
}

// A thread per test: p * n_genes clipped at 1, NaN kept (np.minimum(p * n_genes, 1.0))
__global__ void __launch_bounds__(256) bonferroni_kernel(const double* __restrict__ p, long long group_stride, long long gene_stride,
                                                         int G, int N, double* __restrict__ padj) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= (long long)G * N) return;
    const int g = (int)(i / N), j = (int)(i - (long long)g * N);
    const double v = __dmul_rn(p[(long long)g * group_stride + (long long)j * gene_stride], (double)N);
    padj[i] = (v > 1.0) ? 1.0 : v;
}

// Per-group ranking (illico_top_genes, illico_top_genes_filtered): one CTA per group (grid-strided), like bh_adjust_kernel.
// The key of gene j is the order-preserving u64 image of its score, complemented so that an ascending sort puts the largest
// score first.  NaN keys come after every number (~0 - 1: no number's key is above -inf's 0xFFF0...0) and the keys of
// genes the filter drops after those (~0).  The gene indices ride along as the payload: they go in ascending, and the sort
// is stable, so equal scores stay in index order.
__device__ __forceinline__ unsigned long long score_key_desc(double x, int by_abs) {
    if (x != x) return ~0ull - 1;
    if (by_abs) x = fabs(x);
    if (x == 0.0) x = 0.0;                                              // -0.0 sorts as +0.0
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    const unsigned long long asc = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    return ~asc;
}

// The marker filter and the optional fraction planes of illico_top_genes_filtered.  A NaN bound is a criterion not given;
// illico_top_genes passes no planes, NaN bounds and rec_w = 5.
struct TopFilter {
    const double* pct_group;
    const double* pct_ref;
    double min_in, max_out, fc_lo, fc_hi;
    int* kept;
    int rec_w;
};

// The column-major outputs of illico_top_genes_columns: output column c is group rows[c] (rows NULL: group c), rank r of
// it goes to element r * n_cols + c of each plane; lfc (NULL: NaN) is read at g * lfc_stride + j.
struct TopColumns {
    const int32_t* rows;
    int n_cols;
    const double* lfc;
    long long lfc_stride;
    float* score;
    float* lfc_out;
    double* p;
    double* p_adj;
};

// COLS = false: records [G, k, rec_w] (illico_top_genes, illico_top_genes_filtered); COLS = true: TopColumns' planes, no
// filter.  The keys and the sort are the same.
template <bool COLS>
__global__ void __launch_bounds__(BH_THREADS) top_genes_kernel(const double* __restrict__ score, long long score_stride,
                                                               const double* __restrict__ res, long long res_stride,
                                                               const double* __restrict__ padj, int G, int N, int k, int by_abs,
                                                               TopFilter F, int* __restrict__ out_gene, double* __restrict__ out_rec,
                                                               unsigned long long* __restrict__ slab, TopColumns O) {
    __shared__ uint32_t hist[BH_NW * 256];
    __shared__ uint32_t aux[RADIX_AUX_WORDS];
    __shared__ int n_kept;
    const int tid = threadIdx.x;
    unsigned long long* A = slab + (long long)blockIdx.x * 3 * N;
    unsigned long long* B = A + N;
    uint32_t* IA = reinterpret_cast<uint32_t*>(B + N);
    uint32_t* IB = IA + N;
    const bool by_in = F.min_in == F.min_in, by_out = F.max_out == F.max_out, by_fc = F.fc_lo == F.fc_lo || F.fc_hi == F.fc_hi;
    const int n_out = COLS ? O.n_cols : G;
    for (int oc = blockIdx.x; oc < n_out; oc += gridDim.x) {
        const int g = (COLS && O.rows) ? O.rows[oc] : oc;
        const double* sg = score + (long long)g * score_stride;
        const double* rg = res + (long long)g * res_stride;
        const long long plane = (long long)g * N;
        if (tid == 0) n_kept = 0;
        __syncthreads();
        int mine = 0;
        for (int j = tid; j < N; j += BH_THREADS) {
            bool keep = true;                                           // a NaN fails every criterion it meets
            if (by_in) keep = F.pct_group[plane + j] >= F.min_in;
            if (by_out) keep = keep && F.pct_ref[plane + j] <= F.max_out;
            if (by_fc) {
                const double fc = rg[3 * (long long)j + 2];
                keep = keep && (fc >= F.fc_lo || fc <= F.fc_hi);
            }
            A[j] = keep ? score_key_desc(sg[j], by_abs) : ~0ull;
            IA[j] = (uint32_t)j;
            mine += keep;
        }
        if (mine) atomicAdd(&n_kept, mine);
        __syncthreads();
        const unsigned long long* S = block_radix_sort_t<unsigned long long, uint32_t>(A, B, N, hist, aux, IA, IB);
        const uint32_t* idx = (S == A) ? IA : IB;
        const int m = min(k, n_kept);
        if constexpr (COLS) {
            for (int r = tid; r < k; r += BH_THREADS) {                // (no filter: every gene is kept, m == k)
                const long long o = (long long)r * O.n_cols + oc;
                const int j = (int)idx[r];
                out_gene[o] = j;
                O.score[o] = (float)sg[j];
                O.lfc_out[o] = O.lfc ? (float)O.lfc[(long long)g * O.lfc_stride + j] : NAN;
                O.p[o] = rg[3 * (long long)j];
                O.p_adj[o] = padj ? padj[plane + j] : NAN;
            }
        } else {
            for (int r = tid; r < k; r += BH_THREADS) {
                const long long o = (long long)g * k + r;
                double* rec = out_rec + o * F.rec_w;
                if (r >= m) {                                           // fewer than k genes kept
                    out_gene[o] = -1;
                    for (int f = 0; f < F.rec_w; ++f) rec[f] = NAN;
                    continue;
                }
                const int j = (int)idx[r];
                out_gene[o] = j;
                rec[0] = sg[j];
                rec[1] = rg[3 * (long long)j];
                rec[2] = rg[3 * (long long)j + 1];
                rec[3] = rg[3 * (long long)j + 2];
                rec[4] = padj ? padj[plane + j] : NAN;
                if (F.rec_w == 7) {
                    rec[5] = F.pct_group ? F.pct_group[plane + j] : NAN;
                    rec[6] = F.pct_ref ? F.pct_ref[plane + j] : NAN;
                }
            }
        }
        if (tid == 0 && F.kept) F.kept[g] = n_kept;
        __syncthreads();
    }
}

// One source of a filter_marker_pairs quantity (ILLICO_PAIRS_*): a float64 [groups, plane_stride] plane read at (group row,
// gene), or a [k, n_cols] float64 / float32 plane read at the pair itself.
struct PairSource {
    const void* p;
    int kind;
};

// v > bound (above) or v < bound, |v| first with absval; a float32 source is compared with the bound rounded to float32
// (numpy's comparison of a float32 array with a Python float), a float64 one in float64.  NaN fails either way.
__device__ __forceinline__ bool pair_passes(PairSource s, long long at_plane, long long at_pair, double bound, bool above,
                                            bool absval) {
    if (s.kind == ILLICO_PAIRS_F32) {
        float v = static_cast<const float*>(s.p)[at_pair];
        if (absval) v = fabsf(v);
        const float b = __double2float_rn(bound);
        return above ? v > b : v < b;
    }
    double v = static_cast<const double*>(s.p)[s.kind == ILLICO_PAIRS_PLANE ? at_plane : at_pair];
    if (absval) v = fabs(v);
    return above ? v > bound : v < bound;
}

// A thread per pair i = r * n_cols + c: gene[i] (-1: never kept) of output column c, whose group row is rows[c].
__global__ void __launch_bounds__(256) filter_marker_pairs_kernel(const int32_t* __restrict__ gene, const int32_t* __restrict__ rows,
                                                                  long long n_pairs, int n_cols, long long plane_stride,
                                                                  PairSource in, PairSource out, PairSource fc, double min_in,
                                                                  double max_out, double min_fc, int compare_abs,
                                                                  uint8_t* __restrict__ keep) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_pairs) return;
    const int j = gene[i];
    bool ok = j >= 0;
    if (ok) {
        const bool planes = in.kind == ILLICO_PAIRS_PLANE || out.kind == ILLICO_PAIRS_PLANE || fc.kind == ILLICO_PAIRS_PLANE;
        const long long at = planes ? (long long)rows[i % n_cols] * plane_stride + j : 0;
        ok = pair_passes(in, at, i, min_in, true, false) && pair_passes(out, at, i, max_out, false, false) &&
             pair_passes(fc, at, i, min_fc, true, compare_abs != 0);
    }
    keep[i] = ok ? 1 : 0;
}

__global__ void compute_pval_batch_kernel(const long long* n_ref, const long long* n_tgt, const long long* n, const double* tie,
                                          const double* U, const double* mu, const double* cc, const int* alt, double* out,
                                          long long count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = compute_pval(n_ref[i], n_tgt[i], n[i], tie[i], U[i], mu[i], cc[i], alt[i]);
}

// ---- packed upload: rebuilds dense float32 rows from (bit mask, values) -- see csrc/hostpack.c
// Warp per row.  The lanes fetch 32 mask words at a time (coalesced), then word by word: lane k is element k of the
// word, its value sits at the row's running offset + the number of set bits below it; one coalesced 128-byte store per
// word, zeros included (the destination is written exactly once, nothing has to be cleared first).
__global__ void __launch_bounds__(256) unpack_rows_kernel(const uint32_t* __restrict__ mask, const uint32_t* __restrict__ row_off,
                                                          const float* __restrict__ vals, long long n_rows, int n_cols,
                                                          float* __restrict__ dst, long long ld) {
    const int lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int W = (n_cols + 31) >> 5;
    for (long long r = warp; r < n_rows; r += nwarps) {
        const uint32_t* m = mask + r * W;
        uint32_t base = row_off[r];
        float* out = dst + r * ld;
        for (int w0 = 0; w0 < W; w0 += 32) {
            const uint32_t mine = (w0 + lane < W) ? m[w0 + lane] : 0u;
            const int nw = min(32, W - w0);
            for (int k = 0; k < nw; ++k) {
                const uint32_t word = __shfl_sync(FULL, mine, k);
                const int c = ((w0 + k) << 5) + lane;
                float v = 0.0f;
                if ((word >> lane) & 1u) v = __ldcs(vals + base + __popc(word & below));
                if (c < n_cols) out[c] = v;
                base += __popc(word);
            }
        }
    }
}

}  // namespace
}  // namespace illico

using namespace illico;

extern "C" {

size_t illico_bh_workspace_bytes(int32_t n_groups, int32_t n_genes) {
    long long ctas = n_groups < 148 * 2 ? n_groups : 148 * 2;
    if (ctas < 1) ctas = 1;
    return (size_t)ctas * 2 * (size_t)(n_genes > 0 ? n_genes : 1) * sizeof(unsigned long long) + 256;
}

int illico_bh_adjust(const double* p_values, int64_t group_stride, int64_t gene_stride, int32_t n_groups, int32_t n_genes,
                     double* p_adj, void* workspace, size_t workspace_bytes, void* stream) {
    if (!p_values || !p_adj || !workspace) { set_error("illico_bh_adjust: NULL argument"); return 1; }
    if (n_groups <= 0 || n_genes <= 0) return 0;
    if (workspace_bytes < illico_bh_workspace_bytes(n_groups, n_genes)) { set_error("illico_bh_adjust: workspace too small"); return 1; }
    const int ctas = n_groups < 148 * 2 ? n_groups : 148 * 2;
    unsigned long long* slab =
        reinterpret_cast<unsigned long long*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("bh_adjust_kernel", st,
                  bh_adjust_kernel<<<ctas, BH_THREADS, 0, st>>>(p_values, group_stride, gene_stride, n_groups, n_genes, p_adj, slab));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

size_t illico_top_genes_workspace_bytes(int32_t n_groups, int32_t n_genes) {
    long long ctas = n_groups < 148 * 2 ? n_groups : 148 * 2;
    if (ctas < 1) ctas = 1;
    // per CTA: two u64 key buffers and two u32 index buffers of n_genes
    return (size_t)ctas * 3 * (size_t)(n_genes > 0 ? n_genes : 1) * sizeof(unsigned long long) + 256;
}

static int launch_top_genes(const char* who, const double* scores, int64_t score_group_stride, const double* results,
                            int64_t result_group_stride, const double* p_adj, int32_t n_groups, int32_t n_genes, int32_t k,
                            int32_t by_abs, const TopFilter& F, int32_t* out_gene, double* out_rec, void* workspace,
                            size_t workspace_bytes, void* stream) {
    if (!scores || !results || !out_gene || !out_rec || !workspace) { set_error("%s: NULL argument", who); return 1; }
    if (n_groups <= 0 || n_genes <= 0) return 0;
    if (k < 1 || k > n_genes) { set_error("%s: k = %d outside [1, %d]", who, k, n_genes); return 1; }
    if (workspace_bytes < illico_top_genes_workspace_bytes(n_groups, n_genes)) {
        set_error("%s: workspace too small", who);
        return 1;
    }
    const int ctas = n_groups < 148 * 2 ? n_groups : 148 * 2;
    unsigned long long* slab =
        reinterpret_cast<unsigned long long*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("top_genes_kernel", st,
                  top_genes_kernel<false><<<ctas, BH_THREADS, 0, st>>>(scores, score_group_stride, results, result_group_stride,
                                                                       p_adj, n_groups, n_genes, k, by_abs ? 1 : 0, F, out_gene, out_rec,
                                                                       slab, TopColumns{}));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_top_genes(const double* scores, int64_t score_group_stride, const double* results, int64_t result_group_stride,
                     const double* p_adj, int32_t n_groups, int32_t n_genes, int32_t k, int32_t by_abs, int32_t* out_gene,
                     double* out_rec, void* workspace, size_t workspace_bytes, void* stream) {
    const TopFilter F{nullptr, nullptr, NAN, NAN, NAN, NAN, nullptr, 5};
    return launch_top_genes("illico_top_genes", scores, score_group_stride, results, result_group_stride, p_adj, n_groups, n_genes,
                            k, by_abs, F, out_gene, out_rec, workspace, workspace_bytes, stream);
}

int illico_top_genes_filtered(const double* scores, int64_t score_group_stride, const double* results, int64_t result_group_stride,
                              const double* p_adj, const double* pct_group, const double* pct_ref, int32_t n_groups, int32_t n_genes,
                              int32_t k, int32_t by_abs, double min_in_group, double max_out_group, double fc_min, double fc_max,
                              int32_t* out_gene, double* out_rec, int32_t* kept, void* workspace, size_t workspace_bytes,
                              void* stream) {
    if ((min_in_group == min_in_group && !pct_group) || (max_out_group == max_out_group && !pct_ref)) {
        set_error("illico_top_genes_filtered: a fraction bound is given without its plane");
        return 1;
    }
    const TopFilter F{pct_group, pct_ref, min_in_group, max_out_group, fc_min, fc_max, kept, 7};
    return launch_top_genes("illico_top_genes_filtered", scores, score_group_stride, results, result_group_stride, p_adj, n_groups,
                            n_genes, k, by_abs, F, out_gene, out_rec, workspace, workspace_bytes, stream);
}

int illico_bonferroni_adjust(const double* p_values, int64_t group_stride, int64_t gene_stride, int32_t n_groups, int32_t n_genes,
                             double* p_adj, void* stream) {
    if (!p_values || !p_adj) { set_error("illico_bonferroni_adjust: NULL argument"); return 1; }
    if (n_groups <= 0 || n_genes <= 0) return 0;
    const long long tests = (long long)n_groups * n_genes;
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("bonferroni_kernel", st,
                  bonferroni_kernel<<<(unsigned)((tests + 255) / 256), 256, 0, st>>>(p_values, group_stride, gene_stride, n_groups,
                                                                                   n_genes, p_adj));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_top_genes_columns(const double* scores, int64_t score_group_stride, const double* results, int64_t result_group_stride,
                             const double* p_adj, const double* lfc, int64_t lfc_group_stride, int32_t n_groups, int32_t n_genes,
                             const int32_t* group_rows, int32_t n_cols, int32_t k, int32_t by_abs, int32_t* out_gene, float* out_score,
                             float* out_lfc, double* out_p, double* out_p_adj, void* workspace, size_t workspace_bytes, void* stream) {
    const char* who = "illico_top_genes_columns";
    if (!scores || !results || !out_gene || !out_score || !out_lfc || !out_p || !out_p_adj || !workspace) {
        set_error("%s: NULL argument", who);
        return 1;
    }
    if (n_groups <= 0 || n_genes <= 0 || n_cols <= 0) return 0;
    if (k < 1 || k > n_genes) { set_error("%s: k = %d outside [1, %d]", who, k, n_genes); return 1; }
    if ((!group_rows && n_cols > n_groups) || (lfc && lfc_group_stride < n_genes)) {
        set_error("%s: n_cols > n_groups without group_rows, or lfc_group_stride < n_genes", who);
        return 1;
    }
    if (workspace_bytes < illico_top_genes_workspace_bytes(n_cols, n_genes)) { set_error("%s: workspace too small", who); return 1; }
    const int ctas = n_cols < 148 * 2 ? n_cols : 148 * 2;
    unsigned long long* slab =
        reinterpret_cast<unsigned long long*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    const TopFilter F{nullptr, nullptr, NAN, NAN, NAN, NAN, nullptr, 0};
    const TopColumns O{group_rows, n_cols, lfc, lfc_group_stride, out_score, out_lfc, out_p, out_p_adj};
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("top_genes_columns_kernel", st,
                  top_genes_kernel<true><<<ctas, BH_THREADS, 0, st>>>(scores, score_group_stride, results, result_group_stride, p_adj,
                                                                      n_groups, n_genes, k, by_abs ? 1 : 0, F, out_gene, nullptr,
                                                                      slab, O));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_filter_marker_pairs(const int32_t* gene, const int32_t* group_rows, int32_t k, int32_t n_cols, int64_t plane_stride,
                               const void* pct_in, int32_t pct_in_kind, const void* pct_out, int32_t pct_out_kind,
                               const void* fold_change, int32_t fold_change_kind, double min_in_group_fraction,
                               double max_out_group_fraction, double min_fold_change, int32_t compare_abs, uint8_t* keep,
                               void* stream) {
    const char* who = "illico_filter_marker_pairs";
    if (k <= 0 || n_cols <= 0) return 0;
    const int kinds[3] = {pct_in_kind, pct_out_kind, fold_change_kind};
    bool planes = false;
    for (int q = 0; q < 3; ++q) {
        if (kinds[q] < ILLICO_PAIRS_PLANE || kinds[q] > ILLICO_PAIRS_F32) { set_error("%s: unknown source kind %d", who, kinds[q]); return 1; }
        planes = planes || kinds[q] == ILLICO_PAIRS_PLANE;
    }
    if (!gene || !keep || !pct_in || !pct_out || !fold_change || (planes && (!group_rows || plane_stride < 1))) {
        set_error("%s: NULL argument, or a plane source without group_rows / plane_stride", who);
        return 1;
    }
    const long long n_pairs = (long long)k * n_cols;
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("filter_marker_pairs_kernel", st,
                  filter_marker_pairs_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(
                      gene, group_rows, n_pairs, n_cols, (long long)plane_stride, PairSource{pct_in, pct_in_kind},
                      PairSource{pct_out, pct_out_kind}, PairSource{fold_change, fold_change_kind}, min_in_group_fraction,
                      max_out_group_fraction, min_fold_change, compare_abs ? 1 : 0, keep));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_compute_pval_batch(const int64_t* n_ref, const int64_t* n_tgt, const int64_t* n, const double* tie_sum,
                              const double* U, const double* mu, const double* contin_corr, const int32_t* alternative,
                              double* out, int64_t count, void* stream) {
    if (count <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("compute_pval_batch_kernel", st,
                  compute_pval_batch_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(
                      (const long long*)n_ref, (const long long*)n_tgt, (const long long*)n, tie_sum, U, mu, contin_corr, alternative,
                      out, (long long)count));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_unpack_rows_f32(const uint32_t* mask, const uint32_t* row_off, const float* vals, int64_t n_rows, int32_t n_cols, float* dst,
                           int64_t dst_ld, void* stream) {
    if (n_rows <= 0 || n_cols <= 0) return 0;
    if (!mask || !row_off || !vals || !dst || dst_ld < n_cols) { set_error("illico_unpack_rows_f32: bad argument"); return 1; }
    long long blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ILLICO_LAUNCH("unpack_rows_kernel", (cudaStream_t)stream,
                  unpack_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(mask, row_off, vals, n_rows, n_cols, dst, dst_ld));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
