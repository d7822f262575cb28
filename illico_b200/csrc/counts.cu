// counts.cu -- how many cells of each group express each gene, and the fractions scanpy reports next to its markers
// (rank_genes_groups(pts=True): `pct_nz_group` / `pct_nz_reference`).
//
//   illico_count_nonzero_{dense,csr,csc}  counts[g * count_group_stride + j] = cells of group g whose value in gene
//                                         gene_lb + j satisfies x != 0 (so -0.0 and stored zeros do not count, NaN does:
//                                         what the staging kernels and hostpack.c keep as a non-zero).  float32 or float64
//                                         values; every element of the batch's [G, n_genes_batch] plane is written.
//   illico_nonzero_fractions              the gathered count plane -> pct_group / pct_ref, one IEEE division each.
//   illico_group_moments_{dense,csr,csc}  the same walks with f64 accumulators (MOMENTS): per (group, gene) S1 = sum x,
//                                         S2 = sum x*x (x widened to f64, then squared) and, for log1p data,
//                                         Sf = sum expm1(x); optionally the count plane in the same launch.  What the
//                                         t-test (ttest.cu) needs from the matrix.
//   illico_group_sums_{dense,csr,csc}     the same walks with one f64 accumulator (SUMS): S1 = sum x per (group, gene),
//                                         optionally the count plane in the same launch.  What scanpy's log fold change
//                                         needs from the matrix in a Wilcoxon run (ttest.cu: illico_log_fold_changes).
//
// A pass of its own, not part of the dispatchers: the five result writers would need a pointer in illico_flags_t (an ABI
// change), and the staging kernels, which also count per (gene, segment), write every non-zero value besides.  The pass
// only reads the batch once more and runs only when a caller asks for the counts.
#include "common.cuh"

namespace illico {

namespace {

constexpr int CNT_THREADS = 256;
constexpr int DENSE_UNROLL = 8;       // independent row loads in flight per thread
constexpr int CSR_TILE = 8192;        // genes per CTA: one u32 shared counter each (32 KB)
constexpr int CSR_UNROLL = 4;
constexpr int CSR_MOM_TILE = 1024;    // moments: genes per CTA, 3 f64 + 1 u32 shared accumulators each (28 KB)
constexpr int CSR_SUM_TILE = 4096;    // sums: genes per CTA, 1 f64 + 1 u32 shared accumulators each (48 KB)
constexpr int CSC_SMEM_GROUPS = 8192; // larger G: the CTA counts straight into its global column
constexpr int CSC_MOM_SMEM_GROUPS = 1536;   // moments: 3 f64 + 1 u32 per group in shared memory (42 KB)
constexpr int CSC_SUM_SMEM_GROUPS = 4096;   // sums: 1 f64 + 1 u32 per group in shared memory (48 KB)

// What a walk accumulates besides the counts: nothing (COUNT), S1 (SUMS) or S1, S2 and Sf (MOMENTS).
enum Mode { COUNT = 0, SUMS = 1, MOMENTS = 2 };
constexpr int FRAC_COLS = 32;         // fractions: genes per CTA (one warp row), FRAC_ROWS group lanes
constexpr int FRAC_ROWS = 32;

// Group g's count of gene j, from one plan segment: a group with one segment owns the element, the others add to the
// zeroed plane.
__device__ __forceinline__ void put_count(int* __restrict__ counts, long long cstride, const int32_t* __restrict__ group_seg,
                                          int g, int j, unsigned v) {
    int* out = counts + (long long)g * cstride + j;
    if (group_seg[g + 1] - group_seg[g] == 1) *out = (int)v;
    else if (v) atomicAdd(out, (int)v);
}

// The sum planes (the count-only instantiations take an empty one): s1 / s2 / sf [G, b] at stride ms, s2 and sf NULL in
// SUMS mode, sf NULL unless the data is log1p (the fold change then sums expm1(x) instead of x).  counts may be NULL
// unless the mode is COUNT.
struct Moments {
    double* s1;
    double* s2;
    double* sf;
    long long ms;
};

template <bool MOM>
__device__ __forceinline__ void add_moments(double d, double& s1, double& s2, double& sf, bool log1p) {
    s1 = __dadd_rn(s1, d);
    if (!MOM) return;
    s2 = __dadd_rn(s2, __dmul_rn(d, d));
    if (log1p && d != 0.0) sf = __dadd_rn(sf, expm1(d));
}

// put_count for the sums (S1 only unless MOM)
template <bool MOM>
__device__ __forceinline__ void put_moments(const Moments& mo, const int32_t* __restrict__ group_seg, int g, int j, double s1,
                                            double s2, double sf) {
    const long long o = (long long)g * mo.ms + j;
    if (group_seg[g + 1] - group_seg[g] == 1) {
        mo.s1[o] = s1;
        if (!MOM) return;
        mo.s2[o] = s2;
        if (mo.sf) mo.sf[o] = sf;
    } else {
        atomicAdd(mo.s1 + o, s1);
        if (!MOM) return;
        atomicAdd(mo.s2 + o, s2);
        if (mo.sf) atomicAdd(mo.sf + o, sf);
    }
}

// Dense: CTA = one plan segment x a tile of TW = 2^tw_log2 genes; thread (r, c) reads gene c of the tile in rows r, r + R, ..
// of the segment (R = 256 / TW), in perm order, and the R partial counts meet in shared memory.
template <typename T, int MODE>
__global__ void __launch_bounds__(CNT_THREADS) count_dense_kernel(const T* __restrict__ X, long long ld, int gene_lb, int b,
                                                                  int tw_log2, const int32_t* __restrict__ perm,
                                                                  const int32_t* __restrict__ seg_pos,
                                                                  const int32_t* __restrict__ seg_group,
                                                                  const int32_t* __restrict__ group_seg, int* __restrict__ counts,
                                                                  long long cstride, Moments mo) {
    constexpr bool ACC = MODE != COUNT, MOM = MODE == MOMENTS;
    __shared__ unsigned part[CNT_THREADS];
    __shared__ double mpart[MOM ? 3 * CNT_THREADS : ACC ? CNT_THREADS : 1];
    const bool log1p = MOM && mo.sf != nullptr;
    double s1 = 0.0, s2 = 0.0, sf = 0.0;
    const int s = blockIdx.x;
    const int c = threadIdx.x & ((1 << tw_log2) - 1), r = threadIdx.x >> tw_log2, R = CNT_THREADS >> tw_log2;
    const int j = (blockIdx.y << tw_log2) + c;
    const int p1 = seg_pos[s + 1];
    unsigned cnt = 0;
    if (j < b) {
        const T* col = X + gene_lb + j;
        int p = seg_pos[s] + r;
        for (; p + (DENSE_UNROLL - 1) * R < p1; p += DENSE_UNROLL * R) {
            T v[DENSE_UNROLL];
#pragma unroll
            for (int u = 0; u < DENSE_UNROLL; ++u) v[u] = col[(long long)perm[p + u * R] * ld];
#pragma unroll
            for (int u = 0; u < DENSE_UNROLL; ++u) {
                cnt += v[u] != T(0);
                if (ACC) add_moments<MOM>((double)v[u], s1, s2, sf, log1p);
            }
        }
        for (; p < p1; p += R) {
            const T v = col[(long long)perm[p] * ld];
            cnt += v != T(0);
            if (ACC) add_moments<MOM>((double)v, s1, s2, sf, log1p);
        }
    }
    part[threadIdx.x] = cnt;
    if (ACC) {
        mpart[threadIdx.x] = s1;
        if (MOM) { mpart[CNT_THREADS + threadIdx.x] = s2; mpart[2 * CNT_THREADS + threadIdx.x] = sf; }
    }
    __syncthreads();
    if (r == 0 && j < b) {
        for (int q = 1; q < R; ++q) cnt += part[(q << tw_log2) + c];
        if (!ACC || counts) put_count(counts, cstride, group_seg, seg_group[s], j, cnt);
        if (ACC) {
            for (int q = 1; q < R; ++q) {           // fixed order: row phase 0, 1, .. R - 1
                const int i = (q << tw_log2) + c;
                s1 = __dadd_rn(s1, mpart[i]);
                if (MOM) {
                    s2 = __dadd_rn(s2, mpart[CNT_THREADS + i]);
                    sf = __dadd_rn(sf, mpart[2 * CNT_THREADS + i]);
                }
            }
            put_moments<MOM>(mo, group_seg, seg_group[s], j, s1, s2, sf);
        }
    }
}

// first position in [a, e) whose column is >= col (indices ascend within a row); every lane computes the same answer
__device__ __forceinline__ long long col_lower_bound(const int32_t* __restrict__ indices, long long a, long long e, int col) {
    while (a < e) {
        const long long m = (a + e) >> 1;
        if (indices[m] < col) a = m + 1; else e = m;
    }
    return a;
}

// shared-memory sums of one stored value (CSR / CSC with sums): sums [1 or 3][stride], element i (any order: exact for
// integer data)
template <bool MOM>
__device__ __forceinline__ void shared_add_moments(double* ms, int stride, int i, double d, bool log1p) {
    atomicAdd(ms + i, d);
    if (!MOM) return;
    atomicAdd(ms + stride + i, __dmul_rn(d, d));
    if (log1p) atomicAdd(ms + 2 * stride + i, expm1(d));
}

// CSR: CTA = one plan segment x a tile of up to CSR_TILE genes (fused_csr_pass_kernel's decomposition), warp per row,
// one shared u32 counter per gene.  Rows whose columns reach outside the tile are cut to it by binary search.
template <typename T, int MODE>
__global__ void __launch_bounds__(CNT_THREADS) count_csr_kernel(const T* __restrict__ data, const int32_t* __restrict__ indices,
                                                                const long long* __restrict__ indptr, int gene_lb, int b,
                                                                const int32_t* __restrict__ perm, const int32_t* __restrict__ seg_pos,
                                                                const int32_t* __restrict__ seg_group,
                                                                const int32_t* __restrict__ group_seg, int* __restrict__ counts,
                                                                long long cstride, Moments mo) {
    constexpr bool ACC = MODE != COUNT, MOM = MODE == MOMENTS;
    extern __shared__ unsigned smem_cnt[];
    constexpr int TILE = MOM ? CSR_MOM_TILE : ACC ? CSR_SUM_TILE : CSR_TILE;
    constexpr int NACC = MOM ? 3 : 1;
    constexpr int UNR = MOM ? 2 : CSR_UNROLL;   // (MOM: four f64 loads in flight spill around expm1)
    // ACC: [NACC][TILE] f64 sums, then the counters
    double* ms = reinterpret_cast<double*>(smem_cnt);
    unsigned* tile_cnt = ACC ? reinterpret_cast<unsigned*>(ms + NACC * TILE) : smem_cnt;
    const bool log1p = MOM && mo.sf != nullptr;
    const int s = blockIdx.x, t0 = blockIdx.y * TILE, tn = min(TILE, b - t0);
    const int lo = gene_lb + t0, hi = lo + tn;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < tn; i += CNT_THREADS) {
        tile_cnt[i] = 0;
        if (MOM) ms[i] = ms[TILE + i] = ms[2 * TILE + i] = 0.0;
        else if (ACC) ms[i] = 0.0;
    }
    __syncthreads();
    const int p1 = seg_pos[s + 1];
    for (int p = seg_pos[s] + warp; p < p1; p += CNT_THREADS / 32) {
        const int row = perm[p];
        long long a = indptr[row], e = indptr[row + 1];
        if (a < e && indices[a] < lo) a = col_lower_bound(indices, a, e, lo);
        if (a < e && indices[e - 1] >= hi) e = col_lower_bound(indices, a, e, hi);
        long long q = a + lane;
        for (; q + (UNR - 1) * 32 < e; q += UNR * 32) {
            int col[UNR];
            T v[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) { col[u] = indices[q + u * 32]; v[u] = data[q + u * 32]; }
#pragma unroll
            for (int u = 0; u < UNR; ++u)
                if (v[u] != T(0)) {
                    atomicAdd(&tile_cnt[col[u] - lo], 1u);
                    if (ACC) shared_add_moments<MOM>(ms, TILE, col[u] - lo, (double)v[u], log1p);
                }
        }
        for (; q < e; q += 32) {
            const T v = data[q];
            if (v != T(0)) {
                atomicAdd(&tile_cnt[indices[q] - lo], 1u);
                if (ACC) shared_add_moments<MOM>(ms, TILE, indices[q] - lo, (double)v, log1p);
            }
        }
    }
    __syncthreads();
    const int g = seg_group[s];
    for (int i = threadIdx.x; i < tn; i += CNT_THREADS) {
        if (!ACC || counts) put_count(counts, cstride, group_seg, g, t0 + i, tile_cnt[i]);
        if (ACC) put_moments<MOM>(mo, group_seg, g, t0 + i, ms[i], MOM ? ms[TILE + i] : 0.0, MOM ? ms[2 * TILE + i] : 0.0);
    }
}

// CSC: CTA per gene column, group of a row = seg_group[cell_seg[row]].  SMEM: a shared histogram over the groups, written
// out once; otherwise the CTA zeroes its own column of the plane and adds to it.
template <typename T, bool SMEM, int MODE>
__global__ void __launch_bounds__(CNT_THREADS) count_csc_kernel(const T* __restrict__ data, const int32_t* __restrict__ indices,
                                                                const long long* __restrict__ indptr, int gene_lb, int G,
                                                                const int32_t* __restrict__ cell_seg,
                                                                const int32_t* __restrict__ seg_group, int* __restrict__ counts,
                                                                long long cstride, Moments mo) {
    constexpr bool ACC = MODE != COUNT, MOM = MODE == MOMENTS;
    extern __shared__ unsigned smem_hist[];
    // ACC and SMEM: [1 or 3][G] f64 sums, then the counters.  ACC without SMEM: the CTA zeroes its columns of the planes too.
    double* ms = reinterpret_cast<double*>(smem_hist);
    unsigned* hist = ACC ? reinterpret_cast<unsigned*>(ms + (MOM ? 3 : 1) * (long long)G) : smem_hist;
    const bool log1p = MOM && mo.sf != nullptr;
    const bool cnt_out = !ACC || counts;
    const int j = blockIdx.x;
    int* out = counts + j;
    for (int g = threadIdx.x; g < G; g += CNT_THREADS) {
        if (SMEM) {
            hist[g] = 0;
            if (MOM) ms[g] = ms[G + g] = ms[2 * G + g] = 0.0;
            else if (ACC) ms[g] = 0.0;
        } else {
            if (cnt_out) out[(long long)g * cstride] = 0;
            if (ACC) {
                const long long o = (long long)g * mo.ms + j;
                mo.s1[o] = 0.0;
                if (MOM) mo.s2[o] = 0.0;
                if (log1p) mo.sf[o] = 0.0;
            }
        }
    }
    __syncthreads();
    const long long a = indptr[gene_lb + j], e = indptr[gene_lb + j + 1];
    for (long long q = a + threadIdx.x; q < e; q += CNT_THREADS) {
        const T v = data[q];
        if (v != T(0)) {
            const int g = seg_group[cell_seg[indices[q]]];
            if (SMEM) {
                if (cnt_out) atomicAdd(&hist[g], 1u);
                if (ACC) shared_add_moments<MOM>(ms, G, g, (double)v, log1p);
            } else {
                if (cnt_out) atomicAdd(out + (long long)g * cstride, 1);
                if (ACC) {
                    const double d = (double)v;
                    const long long o = (long long)g * mo.ms + j;
                    atomicAdd(mo.s1 + o, d);
                    if (MOM) atomicAdd(mo.s2 + o, __dmul_rn(d, d));
                    if (log1p) atomicAdd(mo.sf + o, expm1(d));
                }
            }
        }
    }
    if (SMEM) {
        __syncthreads();
        for (int g = threadIdx.x; g < G; g += CNT_THREADS) {
            if (cnt_out) out[(long long)g * cstride] = (int)hist[g];
            if (ACC) {
                const long long o = (long long)g * mo.ms + j;
                mo.s1[o] = ms[g];
                if (MOM) mo.s2[o] = ms[G + g];
                if (log1p) mo.sf[o] = ms[2 * G + g];
            }
        }
    }
}

// CTA = FRAC_COLS genes x FRAC_ROWS group lanes.  One-versus-rest first sums every group's count of the gene (exact, int64).
__global__ void __launch_bounds__(FRAC_COLS * FRAC_ROWS) nonzero_fractions_kernel(const int* __restrict__ counts, long long cstride,
                                                                                  const int32_t* __restrict__ group_size, int G, int N,
                                                                                  int ref, long long n_cells,
                                                                                  double* __restrict__ pct_group,
                                                                                  double* __restrict__ pct_ref) {
    __shared__ long long part[FRAC_ROWS][FRAC_COLS + 1];
    const int c = threadIdx.x % FRAC_COLS, r = threadIdx.x / FRAC_COLS;
    const int j = blockIdx.x * FRAC_COLS + c;
    const bool in = j < N;
    long long total = 0;
    if (ref < 0) {
        if (in)
            for (int g = r; g < G; g += FRAC_ROWS) total += counts[(long long)g * cstride + j];
        part[r][c] = total;
        __syncthreads();
        total = 0;
        for (int q = 0; q < FRAC_ROWS; ++q) total += part[q][c];
    }
    if (!in) return;
    const double ref_frac = ref >= 0 ? __ddiv_rn((double)counts[(long long)ref * cstride + j], (double)group_size[ref]) : 0.0;
    for (int g = r; g < G; g += FRAC_ROWS) {
        const int cnt = counts[(long long)g * cstride + j];
        const int ng = group_size[g];
        const long long o = (long long)g * N + j;
        pct_group[o] = __ddiv_rn((double)cnt, (double)ng);
        pct_ref[o] = ref >= 0 ? ref_frac : __ddiv_rn((double)(total - cnt), (double)(n_cells - ng));
    }
}

int check_plan_dtype(const char* who, int32_t dtype, const illico_plan_t* plan) {
    if (!plan || !plan->perm || !plan->cell_seg || !plan->seg_pos || !plan->seg_group || !plan->group_seg || plan->n_groups <= 0 ||
        plan->n_segments < plan->n_groups) {
        set_error("%s: invalid plan", who);
        return 1;
    }
    if (dtype != ILLICO_DTYPE_F32 && dtype != ILLICO_DTYPE_F64) {
        set_error("%s: dtype %d is neither ILLICO_DTYPE_F32 nor ILLICO_DTYPE_F64", who, dtype);
        return 1;
    }
    return 0;
}

int check_count_args(const char* who, int32_t dtype, const illico_plan_t* plan, const int* counts, int64_t cstride, int32_t b) {
    if (check_plan_dtype(who, dtype, plan)) return 1;
    if (!counts || cstride < b) { set_error("%s: counts NULL or count_group_stride < n_genes_batch", who); return 1; }
    return 0;
}

int check_moment_args(const char* who, int32_t dtype, const illico_plan_t* plan, int32_t is_log1p, const double* sums,
                      const double* sumsq, const double* fsums, int64_t stride, const int* counts, int64_t cstride, int32_t b) {
    if (check_plan_dtype(who, dtype, plan)) return 1;
    if (!sums || !sumsq || (is_log1p && !fsums) || stride < b || (counts && cstride < b)) {
        set_error("%s: sums / sumsq NULL, fsums NULL with is_log1p, or a group stride < n_genes_batch", who);
        return 1;
    }
    return 0;
}

int check_sum_args(const char* who, int32_t dtype, const illico_plan_t* plan, const double* sums, int64_t stride, const int* counts,
                   int64_t cstride, int32_t b) {
    if (check_plan_dtype(who, dtype, plan)) return 1;
    if (!sums || stride < b || (counts && cstride < b)) {
        set_error("%s: sums NULL or a group stride < n_genes_batch", who);
        return 1;
    }
    return 0;
}

// Zeroes what the launch adds to: the count plane, and the sum planes of groups with several segments (a group with
// one segment stores its sums; when every group has one, nothing of the sum planes is cleared).
template <int MODE>
int clear_planes(const illico_plan_t* plan, int* counts, int64_t cstride, const Moments& mo, int b, cudaStream_t st) {
    if (counts)
        ILLICO_CUDA_OK(cudaMemset2DAsync(counts, (size_t)cstride * sizeof(int), 0, (size_t)b * sizeof(int), (size_t)plan->n_groups, st));
    if (MODE != COUNT && plan->n_segments > plan->n_groups)
        for (double* q : {mo.s1, mo.s2, mo.sf})
            if (q)
                ILLICO_CUDA_OK(cudaMemset2DAsync(q, (size_t)mo.ms * sizeof(double), 0, (size_t)b * sizeof(double),
                                                 (size_t)plan->n_groups, st));
    return 0;
}

// kernel names by mode, for the launch profile
constexpr const char* DENSE_NAMES[] = {"count_dense_kernel", "sums_dense_kernel", "moments_dense_kernel"};
constexpr const char* CSR_NAMES[] = {"count_csr_kernel", "sums_csr_kernel", "moments_csr_kernel"};
constexpr const char* CSC_NAMES[] = {"count_csc_kernel", "sums_csc_kernel", "moments_csc_kernel"};
constexpr const char* CSC_GLOBAL_NAMES[] = {"count_csc_global_kernel", "sums_csc_global_kernel", "moments_csc_global_kernel"};

template <int MODE>
int launch_dense(const char* who, const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int b, const illico_plan_t* plan,
                 int* counts, int64_t cstride, const Moments& mo, void* stream) {
    if (b <= 0) return 0;
    if (!X || gene_lb < 0 || ld < (int64_t)gene_lb + b) { set_error("%s: bad X / ld / gene range", who); return 1; }
    int tw_log2 = 5;
    while (tw_log2 < 8 && (1 << tw_log2) < b) ++tw_log2;
    const long long tiles = ((long long)b + (1 << tw_log2) - 1) >> tw_log2;
    if (tiles > 65535) { set_error("%s: %d genes in one batch", who, b); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    if (clear_planes<MODE>(plan, counts, cstride, mo, b, st)) return 1;
    const dim3 grid((unsigned)plan->n_segments, (unsigned)tiles);
    const char* name = DENSE_NAMES[MODE];
    if (dtype == ILLICO_DTYPE_F32)
        ILLICO_LAUNCH(name, st,
                      (count_dense_kernel<float, MODE><<<grid, CNT_THREADS, 0, st>>>((const float*)X, ld, gene_lb, b, tw_log2, plan->perm,
                                                                                     plan->seg_pos, plan->seg_group, plan->group_seg,
                                                                                     counts, cstride, mo)));
    else
        ILLICO_LAUNCH(name, st,
                      (count_dense_kernel<double, MODE><<<grid, CNT_THREADS, 0, st>>>((const double*)X, ld, gene_lb, b, tw_log2, plan->perm,
                                                                                      plan->seg_pos, plan->seg_group, plan->group_seg,
                                                                                      counts, cstride, mo)));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

template <int MODE>
int launch_csr(const char* who, const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
               int b, const illico_plan_t* plan, int* counts, int64_t cstride, const Moments& mo, void* stream) {
    if (b <= 0) return 0;
    if (!indptr || gene_lb < 0) { set_error("%s: bad indptr / gene range", who); return 1; }
    constexpr int TILE = MODE == MOMENTS ? CSR_MOM_TILE : MODE == SUMS ? CSR_SUM_TILE : CSR_TILE;
    constexpr size_t ACC_BYTES = (MODE == MOMENTS ? 3 : MODE == SUMS ? 1 : 0) * (size_t)TILE * sizeof(double);
    const long long tiles = ((long long)b + TILE - 1) / TILE;
    if (tiles > 65535) { set_error("%s: %d genes in one batch", who, b); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    if (clear_planes<MODE>(plan, counts, cstride, mo, b, st)) return 1;
    const dim3 grid((unsigned)plan->n_segments, (unsigned)tiles);
    const size_t smem = (size_t)(b < TILE ? b : TILE) * sizeof(unsigned) + ACC_BYTES;
    const long long* ip = (const long long*)indptr;
    const char* name = CSR_NAMES[MODE];
    if (dtype == ILLICO_DTYPE_F32)
        ILLICO_LAUNCH(name, st,
                      (count_csr_kernel<float, MODE><<<grid, CNT_THREADS, smem, st>>>((const float*)data, indices, ip, gene_lb, b, plan->perm,
                                                                                      plan->seg_pos, plan->seg_group, plan->group_seg, counts,
                                                                                      cstride, mo)));
    else
        ILLICO_LAUNCH(name, st,
                      (count_csr_kernel<double, MODE><<<grid, CNT_THREADS, smem, st>>>((const double*)data, indices, ip, gene_lb, b,
                                                                                       plan->perm, plan->seg_pos, plan->seg_group,
                                                                                       plan->group_seg, counts, cstride, mo)));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename T, int MODE>
void launch_csc_typed(const void* data, const int32_t* indices, const long long* ip, int32_t gene_lb, int b, int G,
                      const illico_plan_t* plan, int* counts, int64_t cstride, const Moments& mo, cudaStream_t st) {
    const int smem_groups = MODE == MOMENTS ? CSC_MOM_SMEM_GROUPS : MODE == SUMS ? CSC_SUM_SMEM_GROUPS : CSC_SMEM_GROUPS;
    if (G <= smem_groups) {
        const size_t smem = (size_t)G * (sizeof(unsigned) + (MODE == MOMENTS ? 3 : MODE == SUMS ? 1 : 0) * sizeof(double));
        ILLICO_LAUNCH(CSC_NAMES[MODE], st,
                      (count_csc_kernel<T, true, MODE><<<b, CNT_THREADS, smem, st>>>((const T*)data, indices, ip, gene_lb, G,
                                                                                     plan->cell_seg, plan->seg_group, counts, cstride, mo)));
    } else {
        ILLICO_LAUNCH(CSC_GLOBAL_NAMES[MODE], st,
                      (count_csc_kernel<T, false, MODE><<<b, CNT_THREADS, 0, st>>>((const T*)data, indices, ip, gene_lb, G,
                                                                                   plan->cell_seg, plan->seg_group, counts, cstride, mo)));
    }
}

template <int MODE>
int launch_csc(const char* who, const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
               int b, const illico_plan_t* plan, int* counts, int64_t cstride, const Moments& mo, void* stream) {
    if (b <= 0) return 0;
    if (!indptr || gene_lb < 0) { set_error("%s: bad indptr / gene range", who); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    const int G = plan->n_groups;
    const long long* ip = (const long long*)indptr;
    if (dtype == ILLICO_DTYPE_F32) launch_csc_typed<float, MODE>(data, indices, ip, gene_lb, b, G, plan, counts, cstride, mo, st);
    else launch_csc_typed<double, MODE>(data, indices, ip, gene_lb, b, G, plan, counts, cstride, mo, st);
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace
}  // namespace illico

using namespace illico;

extern "C" {

int illico_count_nonzero_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                               const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride, void* stream) {
    if (check_count_args("illico_count_nonzero_dense", dtype, plan, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_dense<COUNT>("illico_count_nonzero_dense", X, dtype, ld, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                               Moments{}, stream);
}

int illico_count_nonzero_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride,
                             void* stream) {
    if (check_count_args("illico_count_nonzero_csr", dtype, plan, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_csr<COUNT>("illico_count_nonzero_csr", data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts,
                             count_group_stride, Moments{}, stream);
}

int illico_count_nonzero_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t* counts, int64_t count_group_stride,
                             void* stream) {
    if (check_count_args("illico_count_nonzero_csc", dtype, plan, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_csc<COUNT>("illico_count_nonzero_csc", data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts,
                             count_group_stride, Moments{}, stream);
}

int illico_group_moments_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                               const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq, double* fsums,
                               int32_t* counts, int64_t count_group_stride, int64_t group_stride, void* stream) {
    const char* who = "illico_group_moments_dense";
    if (check_moment_args(who, dtype, plan, is_log1p, sums, sumsq, fsums, group_stride, counts, count_group_stride, n_genes_batch))
        return 1;
    return launch_dense<MOMENTS>(who, X, dtype, ld, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                              Moments{sums, sumsq, is_log1p ? fsums : nullptr, group_stride}, stream);
}

int illico_group_moments_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq,
                             double* fsums, int32_t* counts, int64_t count_group_stride, int64_t group_stride,
                             void* stream) {
    const char* who = "illico_group_moments_csr";
    if (check_moment_args(who, dtype, plan, is_log1p, sums, sumsq, fsums, group_stride, counts, count_group_stride, n_genes_batch))
        return 1;
    return launch_csr<MOMENTS>(who, data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                            Moments{sums, sumsq, is_log1p ? fsums : nullptr, group_stride}, stream);
}

int illico_group_moments_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                             int32_t n_genes_batch, const illico_plan_t* plan, int32_t is_log1p, double* sums, double* sumsq,
                             double* fsums, int32_t* counts, int64_t count_group_stride, int64_t group_stride,
                             void* stream) {
    const char* who = "illico_group_moments_csc";
    if (check_moment_args(who, dtype, plan, is_log1p, sums, sumsq, fsums, group_stride, counts, count_group_stride, n_genes_batch))
        return 1;
    return launch_csc<MOMENTS>(who, data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                            Moments{sums, sumsq, is_log1p ? fsums : nullptr, group_stride}, stream);
}

int illico_group_sums_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t n_genes_batch,
                            const illico_plan_t* plan, double* sums, int32_t* counts, int64_t count_group_stride,
                            int64_t group_stride, void* stream) {
    const char* who = "illico_group_sums_dense";
    if (check_sum_args(who, dtype, plan, sums, group_stride, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_dense<SUMS>(who, X, dtype, ld, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                              Moments{sums, nullptr, nullptr, group_stride}, stream);
}

int illico_group_sums_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                          int32_t n_genes_batch, const illico_plan_t* plan, double* sums, int32_t* counts,
                          int64_t count_group_stride, int64_t group_stride, void* stream) {
    const char* who = "illico_group_sums_csr";
    if (check_sum_args(who, dtype, plan, sums, group_stride, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_csr<SUMS>(who, data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                            Moments{sums, nullptr, nullptr, group_stride}, stream);
}

int illico_group_sums_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                          int32_t n_genes_batch, const illico_plan_t* plan, double* sums, int32_t* counts,
                          int64_t count_group_stride, int64_t group_stride, void* stream) {
    const char* who = "illico_group_sums_csc";
    if (check_sum_args(who, dtype, plan, sums, group_stride, counts, count_group_stride, n_genes_batch)) return 1;
    return launch_csc<SUMS>(who, data, dtype, indices, indptr, gene_lb, n_genes_batch, plan, counts, count_group_stride,
                            Moments{sums, nullptr, nullptr, group_stride}, stream);
}

int illico_nonzero_fractions(const int32_t* counts, int64_t count_group_stride, const int32_t* group_size, int32_t n_groups,
                             int32_t n_genes, int32_t ref_group, int64_t n_cells, double* pct_group, double* pct_ref, void* stream) {
    if (!counts || !group_size || !pct_group || !pct_ref) { set_error("illico_nonzero_fractions: NULL argument"); return 1; }
    if (n_groups <= 0 || n_genes <= 0) return 0;
    if (count_group_stride < n_genes || ref_group >= n_groups) {
        set_error("illico_nonzero_fractions: count_group_stride < n_genes or ref_group out of range");
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned ctas = (unsigned)(((long long)n_genes + FRAC_COLS - 1) / FRAC_COLS);
    ILLICO_LAUNCH("nonzero_fractions_kernel", st,
                  nonzero_fractions_kernel<<<ctas, FRAC_COLS * FRAC_ROWS, 0, st>>>(counts, count_group_stride, group_size, n_groups,
                                                                                  n_genes, ref_group < 0 ? -1 : ref_group,
                                                                                  (long long)n_cells, pct_group, pct_ref));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
