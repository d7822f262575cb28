// rank_ovo.cu -- one-versus-reference Mann-Whitney U on group-segmented non-zero lists (sm_100a).
//
// Replaces illico/ovo/dense_ovo.py:15-137, illico/ovo/sparse_ovo.py:22-158 and the merge
// illico/utils/ranking.py:52-158.  The reference re-walks the whole sorted control column for every
// perturbation (G x n_ref steps per gene).  Here the control's non-zero values are sorted ONCE per gene
// into shared memory and every perturbation value is ranked against it by binary search:
//
//     2U_g = sum_{v in g} ( 2 #{ref > v} + #{ref == v} )                      (SURVEY.md appendix A.2)
//     T_g  = T_ref + sum_{distinct v in g} [ (a+b)^3 - (a+b) - (a^3 - a) ] + (Z^3 - Z)
//
// with a / b the multiplicity of v in the control / the perturbation and Z the number of zeros of the
// pair (zeros are never stored: they are one analytic tie block, for dense input too).  Everything is
// exact integer arithmetic; the f64 epilogue follows illico/utils/math.py:95-118 operation by operation.
//
// One CTA per gene (persistent; genes are handed out by an atomic counter, so that a few expensive genes do not
// leave their CTAs behind).  Per gene, in order of preference:
//   table path   the control has at most DT_CAP distinct values (raw counts, also dense high-count genes): one THREAD
//                per group, private histogram over the control's values (two 16-bit bins per shared-memory word), no
//                sort, no search;
//   stream tier  any other gene, groups of at most STREAM_MAX non-zeros: one THREAD per group streams its values once:
//                each is ranked against the control by one binary search and contributes 2 #{ref > v} + a and the tie
//                terms of its run on the spot (a private 32-slot hash counts the occurrences of a value inside the
//                group; the per-element terms telescope to the per-run formulas above) -- no sort;
//   warp tier    one WARP per group (bitonic sort in shared memory, runs, binary searches), up to WARP_CAP non-zeros;
//   block tier   larger groups one at a time by the whole CTA (radix sort in the CTA's global slab).
#include "common.cuh"
#include "epilogue.cuh"
#include "sort.cuh"

namespace illico {

constexpr int WARP_CAP = 1024;     // keys per warp buffer in the warp tier
constexpr int GROUP_CHUNK = 1024;  // groups handled per sweep (bounds the per-chunk lists)
constexpr int DT_CAP = 64;         // distinct control values for the table path
constexpr int DT_HASH = 256;       // slots of the value -> table-index hash (load factor <= 1/4)
constexpr int NE_CAP = 4;          // table path: distinct values of a group that the control does not have
constexpr int ST_CAP = 1024;       // distinct control values kept in the shared-memory search table
constexpr int STREAM_MAX = 28;     // stream tier: most non-zeros per group (16 buckets x 2 slots of the occurrence hash)
constexpr int STREAM_SLOTS = 32;
constexpr int MBINS = 64;          // groups of a chunk are handed to the threads in order of their non-zero count (bins)
constexpr int HCAP = 4096;         // slots of the hash that finds the distinct values of a large control
constexpr int REF_CAP = 1536;      // control keys sorted in shared memory (larger controls: the CTA's global slab)
constexpr int GCN = 5;             // per-group constants of the p-value (see ovo_group_consts_kernel)
constexpr int OVO_THREADS = 256;   // threads per CTA of ovo_kernel
constexpr int OVO_MIN_CTAS = 3;    // CTAs per SM it is compiled for

struct OvoParams {
    const float* ir_vals;
    const uint32_t* ir_cnt;
    int n_genes;
    illico_plan_t plan;
    illico_flags_t flags;
    double* results;
    long long gstride;
    uint32_t* slab;          // global scratch, slab_words per CTA
    long long slab_words;
    int scratch_words;       // shared scratch (control ping-pong partner, later the tier buffers)
    int* gene_counter;       // next gene to hand out (zeroed before the launch)
    const int* n_genes_dev;  // optional: number of genes decided on the device (a hand-back list), else n_genes
    const int* gene_map;     // optional: staged gene j is column gene_map[j] of the results / debug / group-sum arrays
    int n_cols;              // width of the debug / group-sum arrays (= n_genes unless gene_map is set)
    const double* gc;        // [GCN][Gs] per-group constants (ovo_group_consts_kernel)
    int Gs;
    long long* dbg_u2;
    double* dbg_tie;
    long long* dbg_tie_exact;
};

// Sorted shared-memory array of n >= 1 keys, described once per gene: p = largest power of two <= n.
struct SortedS {
    uint32_t base;   // shared address
    int n, p;
};
__device__ __forceinline__ SortedS sorted_s(uint32_t base, int n) {
    SortedS a;
    // (n = 0: p = 1, so that the first probe's address -- which the compiler may load ahead of the n > 0 test, lds_ro
    // being a plain asm -- stays inside the array; `base` must be a valid shared address even then)
    a.base = base; a.n = n; a.p = (n > 0) ? (1 << (31 - __clz(n))) : 1;
    return a;
}

struct RefInfo {
    const uint32_t* keys;  // sorted non-zero control keys (NULL when only the table below was built)
    uint32_t keys_s;       // their shared-memory address, 0 when they live in the CTA's global slab
    int nnz;               // how many
    int npos;              // control values > 0
    int zeros;             // control zeros
    long long n_ref;
    unsigned long long tie;  // sum over control non-zero runs of a^3 - a
    double sum;              // sum of f(x) over the control
    double mean;             // sum / n_ref
    double inv_mean;
    // search table (st_n >= 0): the control's distinct keys ascending and the position of each one's first
    // occurrence in the sorted control (st_lo[st_n] = nnz), in shared memory.  A rank then costs a binary search over
    // <= 1024 shared-memory entries whatever the size of the control.
    uint32_t st_key_s, st_lo_s;   // shared-memory addresses
    int st_n;
    SortedS st, ks;        // search descriptors of the table / of the keys when they are in shared memory
    // bucket index over the search table (bk_T >= 0): the key range [kmin, kmax] is cut into <= 1023 equal buckets,
    // bk[b] = first table entry of bucket b or later; a search reads its bucket's bounds and halves at most bk_T times
    // (bk_T from the fullest bucket: uniform trip count, 2-4 for spread-out values instead of 10-11 over the table)
    uint32_t bk_s, kmin;
    int bk_shift, bk_last, bk_T;
};

template <bool LOG1P>
__device__ __forceinline__ double fc_val(float v) {
    if (LOG1P) return expm1((double)v);
    return (double)v;
}

// shared-memory loads through 32-bit shared addresses.  lds_ro: tables that are constant while they are read (the
// compiler may schedule these freely, which is what lets several searches overlap); lds_u32: private, read-modify-write
// data (ordered with the stores)
__device__ __forceinline__ uint32_t lds_ro(uint32_t a) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
// NK lower bounds at once (UPPER: upper bounds): NK independent dependent-load chains in flight per thread.  The trip
// count only depends on n, so a warp stays converged.  First probe at p - 1 moves the window to [n - p, n) when the answer
// lies beyond p; the window then halves p -> 1 (the answer stays inside [start, start + width]).
template <int NK, bool UPPER>
__device__ __forceinline__ void bound_shared(const SortedS& A, const uint32_t (&key)[NK], int (&out)[NK]) {
    if (A.n <= 0) {
#pragma unroll
        for (int e = 0; e < NK; ++e) out[e] = 0;
        return;
    }
    uint32_t a[NK];
    const uint32_t first = A.base + (uint32_t)(A.p - 1) * 4u, jump = (uint32_t)(A.n - A.p) * 4u;
#pragma unroll
    for (int e = 0; e < NK; ++e) {
        const uint32_t k = lds_ro(first);
        a[e] = A.base + ((UPPER ? (k <= key[e]) : (k < key[e])) ? jump : 0u);
    }
    for (uint32_t step = (uint32_t)A.p * 2u; step >= 4u; step >>= 1) {   // byte steps: p/2 ... 1 elements
        uint32_t k[NK];
#pragma unroll
        for (int e = 0; e < NK; ++e) k[e] = lds_ro(a[e] + step - 4u);
#pragma unroll
        for (int e = 0; e < NK; ++e) a[e] += (UPPER ? (k[e] <= key[e]) : (k[e] < key[e])) ? step : 0u;
    }
#pragma unroll
    for (int e = 0; e < NK; ++e) {
        const uint32_t k = lds_ro(a[e]);
        out[e] = (int)((a[e] - A.base) >> 2) + ((UPPER ? (k <= key[e]) : (k < key[e])) ? 1 : 0);
    }
}
__device__ __forceinline__ int lb_shared(uint32_t base_s, int n, uint32_t key) {
    const uint32_t k1[1] = {key};
    int o[1];
    bound_shared<1, false>(sorted_s(base_s, n), k1, o);
    return o[0];
}

// position of NK keys in the sorted control: [lo, hi) = the key's run (empty when the control does not have the value)
// NK lower bounds in the search table through the bucket index
template <int NK>
__device__ __forceinline__ void bound_bucket(const RefInfo& R, const uint32_t (&key)[NK], int (&out)[NK]) {
    uint32_t lo[NK], len[NK];
#pragma unroll
    for (int e = 0; e < NK; ++e) {
        const uint32_t kk = max(key[e], R.kmin);
        const uint32_t bq = min((kk - R.kmin) >> R.bk_shift, (uint32_t)R.bk_last);
        const uint32_t a = R.bk_s + bq * 2u;
        uint32_t i0, i1;
        asm("ld.shared.u16 %0, [%1];" : "=r"(i0) : "r"(a));
        asm("ld.shared.u16 %0, [%1+2];" : "=r"(i1) : "r"(a));
        lo[e] = i0;
        len[e] = i1 - i0;
    }
    for (int s = 0; s < R.bk_T; ++s) {
        uint32_t k[NK];
#pragma unroll
        for (int e = 0; e < NK; ++e) k[e] = lds_ro(R.st_key_s + (lo[e] + (len[e] >> 1)) * 4u);
#pragma unroll
        for (int e = 0; e < NK; ++e) {
            const uint32_t half = len[e] >> 1;
            const bool right = len[e] != 0u && k[e] < key[e];
            lo[e] = right ? lo[e] + half + 1u : lo[e];
            len[e] = right ? len[e] - half - 1u : half;
        }
    }
#pragma unroll
    for (int e = 0; e < NK; ++e) out[e] = (int)lo[e];
}

template <int NK>
__device__ __forceinline__ void rank_pos_n(const RefInfo& R, const uint32_t (&key)[NK], int (&lo)[NK], int (&hi)[NK]) {
    if (R.st_n >= 0) {
        int t[NK];
        if (R.bk_T >= 0) bound_bucket<NK>(R, key, t);
        else bound_shared<NK, false>(R.st, key, t);
#pragma unroll
        for (int e = 0; e < NK; ++e) {
            lo[e] = (int)lds_ro(R.st_lo_s + (uint32_t)t[e] * 4u);
            const bool eq = t[e] < R.st_n && lds_ro(R.st_key_s + (uint32_t)t[e] * 4u) == key[e];
            hi[e] = eq ? (int)lds_ro(R.st_lo_s + (uint32_t)(t[e] + 1) * 4u) : lo[e];
        }
    } else if (R.keys_s) {
        bound_shared<NK, false>(R.ks, key, lo);
        bool any_eq = false;
#pragma unroll
        for (int e = 0; e < NK; ++e) {
            hi[e] = lo[e];
            any_eq |= lo[e] < R.nnz && lds_ro(R.keys_s + (uint32_t)lo[e] * 4u) == key[e];
        }
        if (any_eq) bound_shared<NK, true>(R.ks, key, hi);
    } else {
#pragma unroll
        for (int e = 0; e < NK; ++e) {
            lo[e] = lower_bound_u32(R.keys, R.nnz, key[e]);
            hi[e] = lo[e];
            if (lo[e] < R.nnz && R.keys[lo[e]] == key[e]) hi[e] = upper_bound_u32(R.keys, R.nnz, key[e]);
        }
    }
}
__device__ __forceinline__ void rank_pos(const RefInfo& R, uint32_t key, int& lo, int& hi) {
    const uint32_t k1[1] = {key};
    int l[1], h[1];
    rank_pos_n<1>(R, k1, l, h);
    lo = l[0]; hi = h[0];
}

// contribution of one distinct perturbation value (key, multiplicity b)
__device__ __forceinline__ void rank_value(const RefInfo& R, uint32_t key, uint32_t b, unsigned long long& u2,
                                           unsigned long long& tie) {
    int lo, hi;
    rank_pos(R, key, lo, hi);
    const uint32_t a = (uint32_t)(hi - lo);
    const uint32_t gt = (uint32_t)(R.nnz - hi) + ((key < KEY_ZERO) ? (uint32_t)R.zeros : 0u);
    u2 += (unsigned long long)b * (unsigned long long)(2u * gt + a);             // 2 gt + a <= 2 n_ref < 2^32
    // (a+b)^3 - (a+b) - (a^3 - a) = b (3 a (a + b) + b^2 - 1)
    if (a | (b - 1u)) tie += (unsigned long long)b * (3ull * a * ((unsigned long long)a + b) + (unsigned long long)b * b - 1ull);
}

// The reference's sequential f64 tie accumulation for ONE pair (illico/utils/ranking.py:52-158 for the dense
// kernels: merged runs ascending, only t > 1 added, the zero block at its sorted position;
// illico/ovo/sparse_ovo.py:85 for the sparse ones: non-zero runs, then Z^3 - Z last).  Only needed when the
// exact sum reaches 2^53 (pairs of more than 208 063 cells); one thread walks both sorted key lists.
__device__ __noinline__ double ordered_pair_tie(const uint32_t* A, int nA, const uint32_t* B, int strideB, int nB,
                                                long long Z, bool sparse_order) {
    int i = 0, jx = 0;
    double acc = 0.0;
    bool zero_done = sparse_order || Z == 0;
    while (i < nA || jx < nB) {
        const uint32_t ka = (i < nA) ? A[i] : 0xffffffffu, kb = (jx < nB) ? B[(long long)jx * strideB] : 0xffffffffu;
        const uint32_t k = min(ka, kb);
        if (!zero_done && k > KEY_ZERO) {
            if (Z > 1) acc += (double)cube_minus(Z);
            zero_done = true;
        }
        long long t = 0;
        while (i < nA && A[i] == k) { ++i; ++t; }
        while (jx < nB && B[(long long)jx * strideB] == k) { ++jx; ++t; }
        if (t > 1) acc += (double)cube_minus(t);
    }
    if (!zero_done && Z > 1) acc += (double)cube_minus(Z);
    if (sparse_order) acc += (double)cube_minus(Z);
    return acc;
}

template <bool SCORE>
__device__ __forceinline__ void finalize_group(const OvoParams& P, const RefInfo& R, int j, int g, long long m,
                                               unsigned long long u2, unsigned long long tie_nz, double sum,
                                               const uint32_t* gkeys = nullptr, int gstride = 1) {
    const long long n_t = P.plan.group_size[g];
    const long long z_t = n_t - m;
    const int jo = P.gene_map ? P.gene_map[j] : j;
    if (P.flags.group_sums) sum = P.flags.group_sums[(long long)g * P.n_cols + jo];
    const long long Z = (long long)R.zeros + z_t;
    u2 += (unsigned long long)(z_t * (2ll * R.npos + R.zeros));
    const unsigned long long tie_exact = R.tie + tie_nz + (unsigned long long)cube_minus(Z);
    // Every partial sum of the reference's sequential f64 accumulation is an exact integer while the
    // total stays below 2^53 (pairs of up to 208 063 cells), so the exact sum converts without rounding;
    // above it the accumulation is replayed in the reference's order.
    double tie = (double)tie_exact;
    if (tie >= TWO53 && gkeys != nullptr)
        tie = ordered_pair_tie(R.keys, R.nnz, gkeys, gstride, (int)m, Z, P.flags.tie_order == ILLICO_TIES_SPARSE);
    const double U = (double)u2 * 0.5;
    const double cc = P.flags.use_continuity ? 0.5 : 0.0;
    // per-group constants of compute_pval (illico/utils/math.py:95-103) from the table: same operations, once per group
    const double* gc = P.gc + g;
    const double tie_corr = __dsub_rn(1.0, __ddiv_rn(P.flags.tie_correct ? tie : 0.0, gc[3 * P.Gs]));
    const double p = pval_core(gc[1 * P.Gs], gc[0], gc[2 * P.Gs], tie_corr, U, cc, P.flags.alternative);
    if (SCORE) P.flags.scores[(long long)g * P.flags.score_group_stride + jo] = score_core(gc[0], gc[2 * P.Gs], tie_corr, U);
    const double fc = (R.mean == 0.0) ? INFINITY : (sum * gc[4 * P.Gs]) * R.inv_mean;
    double* o = P.results + (long long)g * P.gstride + (long long)jo * 3;
    o[0] = p; o[1] = U; o[2] = fc;
    const long long di = (long long)g * P.n_cols + jo;
    if (P.dbg_u2) P.dbg_u2[di] = (long long)u2;
    if (P.dbg_tie) P.dbg_tie[di] = tie;
    if (P.dbg_tie_exact) P.dbg_tie_exact[di] = (long long)tie_exact;
}

// Everything in compute_pval that depends on the group sizes only: [0] mu = n_r n_t / 2, [1] float(n_r n_t),
// [2] float(n_r n_t (n_r + n_t + 1)) / 12, [3] float(n (n-1) (n+1)) with n = n_r + n_t, [4] 1 / n_t.
__global__ void __launch_bounds__(256) ovo_group_consts_kernel(const illico_plan_t pl, double* gc, int Gs) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pl.n_groups) return;
    const long long n_t = pl.group_size[g], n_r = pl.group_size[pl.ref_group], nn = n_r + n_t;
    gc[0 * Gs + g] = (double)(n_r * n_t) / 2.0;
    gc[1 * Gs + g] = (double)(n_r * n_t);
    gc[2 * Gs + g] = __ddiv_rn((double)(n_r * n_t * (n_r + n_t + 1)), 12.0);
    gc[3 * Gs + g] = (double)(nn * (nn - 1) * (nn + 1));
    gc[4 * Gs + g] = 1.0 / (double)n_t;
}

// SCORE: also writes the score plane (illico_flags_t::scores), in an instantiation of its own
template <bool LOG1P, bool SCORE>
__global__ void __launch_bounds__(OVO_THREADS, OVO_MIN_CTAS) ovo_kernel(const OvoParams P) {
    constexpr int NT = OVO_THREADS;
    constexpr int OVO_NW = OVO_THREADS / 32;
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const illico_plan_t& pl = P.plan;
    const int S = pl.n_segments, G = pl.n_groups, ref = pl.ref_group;

    // ---- shared carve-up
    uint32_t* refA = smem;                                  // [REF_CAP]
    uint32_t* scratch = refA + REF_CAP;                     // [scratch_words] (>= REF_CAP, >= 2 * HCAP)
    uint32_t* hist = scratch + P.scratch_words;             // [OVO_NW * 256]
    uint32_t* aux = hist + OVO_NW * 256;                    // [RADIX_AUX_WORDS]
    uint16_t* mlist = (uint16_t*)(aux + RADIX_AUX_WORDS);   // [GROUP_CHUNK] groups left to the warp tier (index inside the chunk; bit 15: passed on to the block tier)
    uint16_t* bkidx = mlist + GROUP_CHUNK;                  // [GROUP_CHUNK] bucket index of the search table (RefInfo::bk_s)
    uint16_t* order = bkidx + GROUP_CHUNK;                  // [GROUP_CHUNK] the chunk's groups by non-zero count
    uint16_t* marr = order + GROUP_CHUNK;                   // [GROUP_CHUNK] non-zero count of each group (capped)
    int* counters = (int*)(marr + GROUP_CHUNK);             // [8] rotating {medium, big} list counters, [6] scratch, [7] next gene
    int* mh = counters + 8;                                 // [MBINS] histogram / cursors of the non-zero counts
    double* redd = (double*)(mh + MBINS);                   // [32]
    unsigned long long* redu = (unsigned long long*)(redd + 32);  // [32]
    double* dval = (double*)(redu + 32);                    // [DT_CAP]   f(x) of each distinct control value
    uint32_t* dwt = (uint32_t*)(dval + DT_CAP);             // [DT_CAP]   2 #{ref > v} + a
    uint32_t* dmult = dwt + DT_CAP;                         // [DT_CAP]   a = multiplicity in the control
    uint2* hkv = (uint2*)(dmult + DT_CAP);                  // [DT_HASH]  open-addressed {float bits, table index}
    uint32_t* st_key = (uint32_t*)(hkv + DT_HASH);          // [ST_CAP]   search table: distinct control keys, ascending
    int* st_lo = (int*)(st_key + ST_CAP);                   // [ST_CAP+1] first position of each

    uint32_t* slab = P.slab + (long long)blockIdx.x * P.slab_words;
    const int maxg = pl.max_group_size;
    uint32_t* gA = slab;            // block-tier group buffers (global)
    uint32_t* gB = slab + maxg;
    __shared__ int mmax3[3];
    __shared__ int ref_nnz_s;  // the control's non-zeros (thread 0's prefix over its segments)
    // control segments whose offsets hist[] holds at a time (+1 entry: the start of the next chunk)
    constexpr int REF_SEG_CHUNK = OVO_NW * 256 - 1;

    const int ref_s0 = pl.group_seg[ref], ref_s1 = pl.group_seg[ref + 1];
    if (tid < 8) counters[tid] = 0;
    if (tid < 3) mmax3[tid] = 0;
    int cc = 0;  // chunk counter: chunk c uses counter set c % 3 and clears set (c + 1) % 3 for the next chunk
    const int n_genes = P.n_genes_dev ? *P.n_genes_dev : P.n_genes;
    const uint32_t hkv_s = (uint32_t)__cvta_generic_to_shared(hkv);
    const long long n_ref_cells = pl.group_size[ref];
    // pairs above 208 063 cells replay the reference's ordered tie sum from the SORTED control: no hashing then
    const bool may_hash = n_ref_cells + (long long)pl.max_target_group_size <= 208063;
    __syncthreads();

    for (;;) {
        if (tid == 0) counters[7] = atomicAdd(P.gene_counter, 1);
        __syncthreads();
        const int j = counters[7];
        if (j >= n_genes) break;
        const uint32_t* cnt = P.ir_cnt + (long long)j * S;
        const float* vals = P.ir_vals + (long long)j * pl.slot_cap;

        // ================= phase 1: the control, once per gene =================
        // offsets of the control's segments: serial prefix by thread 0 into hist[] (free now).  hist[] holds the offsets
        // of the first REF_SEG_CHUNK segments and the start of the next one; the sort path refills it for the others.
        if (tid == 0) {
            uint32_t acc = 0;
            for (int s = ref_s0; s < ref_s1; ++s) {
                if (s - ref_s0 <= REF_SEG_CHUNK) hist[s - ref_s0] = acc;
                acc += cnt[s];
            }
            if (ref_s1 - ref_s0 <= REF_SEG_CHUNK) hist[ref_s1 - ref_s0] = acc;
            ref_nnz_s = (int)acc;
            counters[6] = 0;
        }
        __syncthreads();
        const int nref_nz = ref_nnz_s;
        const bool ref_smem = nref_nz <= REF_CAP;
        RefInfo R;
        R.nnz = nref_nz;
        R.n_ref = n_ref_cells;
        R.zeros = (int)(R.n_ref - nref_nz);
        R.st_key_s = (uint32_t)__cvta_generic_to_shared(st_key);
        R.st_lo_s = (uint32_t)__cvta_generic_to_shared(st_lo);
        R.st_n = -1;
        R.st = sorted_s(R.st_key_s, 0);
        R.keys = nullptr; R.keys_s = 0u;
        R.ks = sorted_s(R.st_key_s, 0);
        double rsum = 0.0;
        int D = 0;
        bool hashed = false;
        if (!ref_smem && may_hash) {
            // ---- a large control (a dense gene).  Count data has a handful of distinct values whatever the size: find
            // them with a shared-memory hash (value -> multiplicity) instead of sorting 10k keys through the global slab.
            uint32_t* hk = scratch;
            uint32_t* hc = scratch + HCAP;
            for (int i = tid; i < 2 * HCAP; i += OVO_THREADS) scratch[i] = 0u;
            __syncthreads();
            for (int s = ref_s0 + w; s < ref_s1; s += OVO_NW) {
                const int c = (int)cnt[s];
                const float* src = vals + pl.seg_base[s];
                for (int i = lane; i < c; i += 32) {
                    const float v = src[i];
                    rsum += fc_val<LOG1P>(v);
                    uint32_t key = f2key(v);
                    if (key == 0u) key = 1u;
                    if (*(volatile int*)&counters[6] > ST_CAP) continue;      // not count-like: the sort path takes over
                    uint32_t h = (key * 2654435761u) >> 20;
                    for (;;) {
                        const uint32_t prev = atomicCAS(&hk[h], 0u, key);
                        if (prev == 0u) atomicAdd(&counters[6], 1);
                        if (prev == 0u || prev == key) { atomicAdd(&hc[h], 1u); break; }
                        h = (h + 1) & (HCAP - 1);
                    }
                }
            }
            __syncthreads();
            D = counters[6];
            __syncthreads();
            if (D <= ST_CAP) {
                // distinct (key, multiplicity) pairs -> sorted by key -> first positions by an exclusive scan
                if (tid == 0) counters[6] = 0;
                __syncthreads();
                for (int t = tid; t < HCAP; t += OVO_THREADS)
                    if (hk[t] != 0u) {
                        const int idx = atomicAdd(&counters[6], 1);
                        st_key[idx] = hk[t];
                        st_lo[idx] = (int)hc[t];
                    }
                const int Pd = max(2, next_pow2(D));
                for (int i = D + tid; i < Pd; i += OVO_THREADS) { st_key[i] = 0xffffffffu; st_lo[i] = 0; }
                __syncthreads();
                block_bitonic_sort_pairs(st_key, (uint32_t*)st_lo, Pd);
                // exclusive prefix of the multiplicities: ST_CAP / OVO_THREADS consecutive entries per thread
                constexpr int PER = (ST_CAP + OVO_THREADS - 1) / OVO_THREADS;
                uint32_t cv[PER], loc = 0;
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int i = tid * PER + q;
                    cv[q] = (i < D) ? (uint32_t)st_lo[i] : 0u;
                    loc += cv[q];
                }
                const uint32_t incl = warp_incl_scan(loc, lane);
                if (lane == 31) aux[w] = incl;
                __syncthreads();
                uint32_t basev = incl - loc;
                for (int ww = 0; ww < w; ++ww) basev += aux[ww];
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int i = tid * PER + q;
                    if (i < D) st_lo[i] = (int)basev;
                    basev += cv[q];
                }
                if (tid == 0) st_lo[D] = nref_nz;
                __syncthreads();
                hashed = true;
                R.st_n = D;
                R.st = sorted_s(R.st_key_s, D);
            } else {
                rsum = 0.0;   // recomputed by the sort path below
            }
        }
        if (!hashed) {
            // ---- sort path: control keys in shared memory when they fit, else in this CTA's global slab
            uint32_t* rA = ref_smem ? refA : slab + 2ll * maxg;
            uint32_t* rB = ref_smem ? scratch : slab + 3ll * maxg;
            for (int c0 = ref_s0; c0 < ref_s1; c0 += REF_SEG_CHUNK) {
                const int c1 = min(ref_s1, c0 + REF_SEG_CHUNK);
                if (c0 > ref_s0) {   // (CTA-uniform) offsets of the next chunk, from the start hist[REF_SEG_CHUNK] left
                    __syncthreads();
                    if (tid == 0) {
                        uint32_t acc = hist[REF_SEG_CHUNK];
                        for (int s = c0; s < c1; ++s) { hist[s - c0] = acc; acc += cnt[s]; }
                        hist[c1 - c0] = acc;
                    }
                    __syncthreads();
                }
                for (int s = c0 + w; s < c1; s += OVO_NW) {
                    const uint32_t off = hist[s - c0];
                    const int c = (int)cnt[s];
                    const float* src = vals + pl.seg_base[s];
                    for (int i = lane; i < c; i += 32) {
                        const float v = src[i];
                        uint32_t key = f2key(v);
                        if (key == 0u) key = 1u;
                        rA[off + i] = key;
                        rsum += fc_val<LOG1P>(v);
                    }
                }
            }
            __syncthreads();
            const uint32_t* rk = block_radix_sort(rA, rB, nref_nz, hist, aux);
            if (rk != rA) {  // keep the sorted keys in rA: rB is recycled as tier scratch
                for (int i = tid; i < nref_nz; i += OVO_THREADS) rA[i] = rB[i];
                __syncthreads();
            }
            R.keys = rA;
            R.keys_s = ref_smem ? (uint32_t)__cvta_generic_to_shared(rA) : 0u;
            R.ks = sorted_s(ref_smem ? R.keys_s : R.st_key_s, ref_smem ? nref_nz : 0);
            // distinct control values: how many, then (when they fit) the ordered search table
            int heads = 0;
            for (int i = tid; i < nref_nz; i += OVO_THREADS) heads += (i == 0 || rA[i - 1] != rA[i]) ? 1 : 0;
            D = (int)block_sum<unsigned long long>((unsigned long long)heads, redu);
            if (D <= ST_CAP) {
                // ordered compaction of the run starts of rA: chunks of OVO_THREADS elements, ballot + warp totals
                int base = 0;
                for (int i0 = 0; i0 < nref_nz; i0 += OVO_THREADS) {
                    const int i = i0 + tid;
                    const bool head = i < nref_nz && (i == 0 || rA[i - 1] != rA[i]);
                    const unsigned bal = __ballot_sync(FULL, head);
                    if (lane == 0) hist[w] = (uint32_t)__popc(bal);
                    __syncthreads();
                    int before = 0, total = 0;
                    for (int ww = 0; ww < OVO_NW; ++ww) { const int c = (int)hist[ww]; if (ww < w) before += c; total += c; }
                    if (head) {
                        const int slot = base + before + __popc(bal & ((1u << lane) - 1u));
                        st_key[slot] = rA[i];
                        st_lo[slot] = i;
                    }
                    base += total;
                    __syncthreads();
                }
                if (tid == 0) st_lo[D] = nref_nz;
                R.st_n = D;
                R.st = sorted_s(R.st_key_s, D);
                __syncthreads();
            }
        }
        // ---- bucket index of the search table
        R.bk_s = (uint32_t)__cvta_generic_to_shared(bkidx);
        R.bk_T = -1; R.kmin = 0u; R.bk_shift = 0; R.bk_last = 0;
        if (R.st_n > 1) {
            const uint32_t kmin = st_key[0], span = st_key[D - 1] - kmin;
            int shift = max(0, 22 - __clz(span));                         // span >> shift < 1024
            if ((span >> shift) > (uint32_t)(GROUP_CHUNK - 2)) ++shift;   // ... and at most GROUP_CHUNK - 1 buckets
            const int NB = (int)(span >> shift) + 1;
            if (tid == 0) counters[6] = 0;
            __syncthreads();
            for (int i = tid; i < D; i += OVO_THREADS) {
                const int bi = (int)((st_key[i] - kmin) >> shift);
                const int bp = i ? (int)((st_key[i - 1] - kmin) >> shift) : -1;
                for (int bb = bp + 1; bb <= bi; ++bb) bkidx[bb] = (uint16_t)i;
                if (i == D - 1) for (int bb = bi + 1; bb <= NB; ++bb) bkidx[bb] = (uint16_t)D;
            }
            __syncthreads();
            int occ = 0;
            for (int bb = tid; bb < NB; bb += OVO_THREADS) occ = max(occ, (int)bkidx[bb + 1] - (int)bkidx[bb]);
            if (occ) atomicMax(&counters[6], occ);
            __syncthreads();
            R.kmin = kmin; R.bk_shift = shift; R.bk_last = NB - 1;
            R.bk_T = 32 - __clz(counters[6]);                             // halvings that empty a range of that many entries
            __syncthreads();
        }
        rsum = block_sum<double>(rsum, redd);
        R.sum = P.flags.group_sums ? P.flags.group_sums[(long long)ref * P.n_cols + (P.gene_map ? P.gene_map[j] : j)] : rsum;
        R.mean = R.sum / (double)R.n_ref;
        R.inv_mean = 1.0 / R.mean;
        unsigned long long tsum = 0;
        if (R.st_n >= 0) {
            for (int a = tid; a < D; a += OVO_THREADS) tsum += (unsigned long long)cube_minus((long long)(st_lo[a + 1] - st_lo[a]));
            R.npos = nref_nz - st_lo[lb_shared(R.st_key_s, D, KEY_ZERO + 1u)];
        } else {
            const uint32_t* rA = R.keys;
            for (int i = tid; i < nref_nz; i += OVO_THREADS) {
                const uint32_t k = rA[i];
                if (i == 0 || rA[i - 1] != k) tsum += (unsigned long long)cube_minus((long long)(upper_bound_u32(rA, nref_nz, k) - i));
            }
            R.npos = nref_nz - upper_bound_u32(rA, nref_nz, KEY_ZERO);
        }
        R.tie = block_sum<unsigned long long>(tsum, redu);
        // ---- table path set-up: value -> table index hash, per-entry weights and f(value)
        const bool table = D <= DT_CAP;
        if (table) {
            for (int a = tid; a < DT_HASH; a += OVO_THREADS) hkv[a] = make_uint2(0u, 0u);  // +0.0f is never staged
            __syncthreads();
            for (int a = tid; a < D; a += OVO_THREADS) {
                const float v = key2f(st_key[a]);
                dval[a] = fc_val<LOG1P>(v);
                const uint32_t mult = (uint32_t)(st_lo[a + 1] - st_lo[a]);
                const uint32_t gt = (uint32_t)(nref_nz - st_lo[a + 1]) + ((st_key[a] < KEY_ZERO) ? (uint32_t)R.zeros : 0u);
                dwt[a] = 2u * gt + mult;
                dmult[a] = mult;
                const uint32_t bits = __float_as_uint(v);
                uint32_t h = (bits * 2654435761u) >> 24;
                while (atomicCAS(&hkv[h].x, 0u, bits) != 0u) h = (h + 1) & (DT_HASH - 1);
                hkv[h].y = (uint32_t)a;
            }
        }
        __syncthreads();

        // ================= phase 2: perturbations, in chunks of GROUP_CHUNK groups =================
        for (int g0 = 0; g0 < G; g0 += GROUP_CHUNK) {
            const int g1 = min(G, g0 + GROUP_CHUNK), ng = g1 - g0;
            int* cnt_m = counters + 2 * (cc % 3);      // [0] medium list length, [1] big list length
            int* m_max = mmax3 + (cc % 3);             // largest non-zero count among the chunk's warp-tier groups
            if (tid == 0) { const int nx = (cc + 1) % 3; counters[2 * nx] = 0; counters[2 * nx + 1] = 0; mmax3[nx] = 0; }
            ++cc;
            // ---- the chunk's groups in order of their non-zero count (counting sort over MBINS bins): the 32 groups a
            // warp works on at a time then have about the same length, so its lanes finish together
            for (int i = tid; i < MBINS; i += OVO_THREADS) mh[i] = 0;
            __syncthreads();
            for (int i = tid; i < ng; i += OVO_THREADS) {
                const int g = g0 + i;
                int m = 0;
                for (int s = pl.group_seg[g]; s < pl.group_seg[g + 1]; ++s) m += (int)cnt[s];
                marr[i] = (uint16_t)min(m, 65535);
                atomicAdd(&mh[min(m, MBINS - 1)], 1);
            }
            __syncthreads();
            if (w == 0) {   // exclusive scan of the MBINS counts
                const int c0 = mh[2 * lane], c1 = mh[2 * lane + 1];
                const uint32_t incl = warp_incl_scan((uint32_t)(c0 + c1), lane);
                mh[2 * lane] = (int)incl - c0 - c1;
                mh[2 * lane + 1] = (int)incl - c1;
            }
            __syncthreads();
            for (int i = tid; i < ng; i += OVO_THREADS) order[atomicAdd(&mh[min((int)marr[i], MBINS - 1)], 1)] = (uint16_t)i;
            __syncthreads();
            // ---- one thread per group
            for (int i = tid; i < ng; i += OVO_THREADS) {
                const int gi = order[i], g = g0 + gi;
                if (g == ref) {
                    // control row: the sparse kernels' convention (ovo/sparse_ovo.py:140-143); fold change of the
                    // control against itself (utils/math.py:191-192)
                    const int jo = P.gene_map ? P.gene_map[j] : j;
                    double* o = P.results + (long long)g * P.gstride + (long long)jo * 3;
                    o[0] = 1.0; o[1] = -1.0; o[2] = (R.mean == 0.0) ? INFINITY : R.mean / R.mean;
                    if (SCORE) P.flags.scores[(long long)g * P.flags.score_group_stride + jo] = 0.0;
                    const long long di = (long long)g * P.n_cols + jo;
                    if (P.dbg_u2) P.dbg_u2[di] = -2;
                    if (P.dbg_tie) P.dbg_tie[di] = 0.0;
                    if (P.dbg_tie_exact) P.dbg_tie_exact[di] = 0;
                    continue;
                }
                const int s0 = pl.group_seg[g], s1 = pl.group_seg[g + 1];
                int m = marr[gi];
                if (m == 65535) { m = 0; for (int s = s0; s < s1; ++s) m += (int)cnt[s]; }
                const bool big_pair = R.n_ref + (long long)pl.group_size[g] > 208063;  // tie sum may pass 2^53
                bool done = false;
                if (table && !big_pair && pl.group_size[g] < 65536) {
                    // ---- table path: private histogram over the control's distinct values, two 16-bit bins per word
                    // (word q of the thread at scratch[q * NT + tid]: conflict-free whatever the values are)
                    uint32_t* bins = scratch + tid;
                    uint32_t* ex = scratch + (DT_CAP / 2) * NT + tid;   // values the control lacks: (bits, count) pairs
                    const int nwords = (D + 1) >> 1;
                    for (int q = 0; q < nwords; ++q) bins[q * NT] = 0u;
                    bool ok = true;
                    int ne = 0;
                    const uint32_t bins_s = (uint32_t)__cvta_generic_to_shared(bins);
                    // one stored value: hash probe (one 64-bit shared load on a hit) + bump of the private bin
                    auto bump = [&](float v) {
                        const uint32_t bits = __float_as_uint(v);
                        uint32_t h = (bits * 2654435761u) >> 24;
                        uint32_t k, t;
                        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(k), "=r"(t) : "r"(hkv_s + h * 8u));
                        if (k != bits) {  // collision chain, or a value the control does not have (rare)
                            while (k != bits && k != 0u) {
                                h = (h + 1) & (DT_HASH - 1);
                                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(k), "=r"(t) : "r"(hkv_s + h * 8u));
                            }
                            if (k == 0u) {
                                int x = 0;
                                while (x < ne && ex[(2 * x) * NT] != bits) ++x;
                                if (x < ne) ex[(2 * x + 1) * NT] += 1;
                                else if (ne < NE_CAP) {
                                    ex[(2 * ne) * NT] = bits;
                                    ex[(2 * ne + 1) * NT] = 1;
                                    ++ne;
                                } else ok = false;
                                return;
                            }
                        }
                        const uint32_t addr = bins_s + (t >> 1) * (NT * 4u);
                        uint32_t r;
                        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr) : "memory");
                        asm volatile("st.shared.u32 [%0], %1;" :: "r"(addr), "r"(r + (1u << ((t & 1u) << 4))) : "memory");
                    };
                    for (int s = s0; s < s1 && ok; ++s) {
                        const int c = (int)cnt[s];
                        const float4* src4 = reinterpret_cast<const float4*>(vals + pl.seg_base[s]);  // 32-byte aligned, padded slot
                        const int n4 = (c + 3) >> 2;
                        // two 16-byte loads (one 32-byte sector) in flight ahead of the values being counted
                        float4 q0 = (n4 > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
                        float4 q1 = (n4 > 1) ? src4[1] : make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int i4 = 0; i4 < n4; i4 += 2) {
                            const float4 a4 = q0, b4 = q1;
                            if (i4 + 2 < n4) q0 = src4[i4 + 2];
                            if (i4 + 3 < n4) q1 = src4[i4 + 3];
                            const float q[8] = {a4.x, a4.y, a4.z, a4.w, b4.x, b4.y, b4.z, b4.w};
                            const int left = c - 4 * i4;
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (e < left) bump(q[e]);
                        }
                    }
                    if (ok) {
                        unsigned long long u2 = 0, tie = 0;
                        double sum = 0.0;
                        for (int q = 0; q < nwords; ++q) {
                            const uint32_t wd = bins[q * NT];
                            if (wd == 0u) continue;
#pragma unroll
                            for (int hsel = 0; hsel < 2; ++hsel) {
                                const uint32_t bq = hsel ? (wd >> 16) : (wd & 0xffffu);
                                if (bq) {
                                    // b (2 gt + a)  and  (a+b)^3 - (a+b) - (a^3 - a) = b (3 a (a + b) + b^2 - 1)
                                    const int t = 2 * q + hsel;
                                    const uint32_t a = dmult[t];
                                    u2 += (unsigned long long)bq * (unsigned long long)dwt[t];
                                    tie += (unsigned long long)bq * (3ull * a * ((unsigned long long)a + bq) + (unsigned long long)bq * bq - 1ull);
                                    sum += (double)bq * dval[t];
                                }
                            }
                        }
                        for (int x = 0; x < ne; ++x) {  // absent from the control: a = 0, position by binary search
                            const float v = __uint_as_float(ex[(2 * x) * NT]);
                            const uint32_t bq = ex[(2 * x + 1) * NT];
                            rank_value(R, f2key(v), bq, u2, tie);
                            sum += (double)bq * fc_val<LOG1P>(v);
                        }
                        finalize_group<SCORE>(P, R, j, g, m, u2, tie, sum);
                        done = true;
                    }
                } else if (!table && !big_pair && m <= STREAM_MAX) {
                    // ---- stream tier: every value is ranked on arrival.  The k-th occurrence of a value inside the group
                    // (a = its multiplicity in the control) adds 2 gt + a to 2U and (a+k)^3 - (a+k) - ((a+k-1)^3 - (a+k-1)) =
                    // 3 (a+k) (a+k-1) to the tie term -- the sums telescope to the per-run formulas, so no sort is needed;
                    // k comes from a private hash of 16 buckets x 2 key slots (slot q of the thread at
                    // scratch[q * NT + tid]) with the occurrence count of slot q in byte q of the words behind them
                    // (log-normalised counts repeat values often: small integer counts over integer library sizes).
                    uint32_t* hs = scratch + tid;
                    const uint32_t hs_s = (uint32_t)__cvta_generic_to_shared(hs);
                    const uint32_t hc_s = hs_s + STREAM_SLOTS * (NT * 4u);
#pragma unroll
                    for (int q = 0; q < STREAM_SLOTS + STREAM_SLOTS / 4; ++q) hs[q * NT] = 0u;
                    unsigned long long u2 = 0, tie = 0;
                    double sum = 0.0;
                    // four values at a time: their searches are independent load chains and overlap; the occurrence hash
                    // is updated one value after the other
                    auto take4 = [&](const float4 q4, int nv) {
                        const float q[4] = {q4.x, q4.y, q4.z, q4.w};
                        uint32_t key[4];
                        int lo[4], hi[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            key[e] = (e < nv) ? f2key(q[e]) : 0xffffffffu;
                            if (key[e] == 0u) key[e] = 1u;                         // (only a NaN payload maps to 0)
                        }
                        rank_pos_n<4>(R, key, lo, hi);
                        // occurrence hash: the four buckets are probed together (eight loads in flight); a value is then
                        // resolved against what it loaded unless an earlier value of this quadruple wrote to its bucket.
                        // The count byte of a slot is only touched from the second occurrence on (0 = seen once).
                        uint32_t bk[4], k0[4], k1[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            bk[e] = (key[e] * 2654435761u) >> 28;
                            const uint32_t a0 = hs_s + (2u * bk[e]) * (NT * 4u);
                            k0[e] = lds_u32(a0);
                            k1[e] = lds_u32(a0 + NT * 4u);
                        }
                        uint32_t dirty = 0u;                                      // buckets written by this quadruple
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            if (e < nv) {
                                const uint32_t a = (uint32_t)(hi[e] - lo[e]);
                                const uint32_t gt = (uint32_t)(R.nnz - hi[e]) + ((key[e] < KEY_ZERO) ? (uint32_t)R.zeros : 0u);
                                u2 += (unsigned long long)(2u * gt + a);
                                sum += fc_val<LOG1P>(q[e]);
                                uint32_t bkt = bk[e], c0 = k0[e], c1 = k1[e], k = 1u;
                                bool fresh = ((dirty >> bkt) & 1u) == 0u;
                                for (;;) {
                                    const uint32_t a0 = hs_s + (2u * bkt) * (NT * 4u), a1 = a0 + NT * 4u;
                                    if (!fresh) { c0 = lds_u32(a0); c1 = lds_u32(a1); }
                                    const bool hit0 = c0 == key[e], hit1 = c1 == key[e];
                                    if (hit0 || hit1) {                                   // seen before: k-th occurrence
                                        const uint32_t slot = 2u * bkt + (hit0 ? 0u : 1u);
                                        const uint32_t ca = hc_s + (slot >> 2) * (NT * 4u) + (slot & 3u);
                                        uint32_t cnt8;
                                        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(cnt8) : "r"(ca) : "memory");
                                        k = cnt8 + 2u;
                                        asm volatile("st.shared.u8 [%0], %1;" :: "r"(ca), "r"(cnt8 + 1u) : "memory");
                                        break;
                                    }
                                    if (c0 == 0u || c1 == 0u) {
                                        asm volatile("st.shared.u32 [%0], %1;" :: "r"(c0 == 0u ? a0 : a1), "r"(key[e]) : "memory");
                                        dirty |= 1u << bkt;
                                        break;
                                    }
                                    bkt = (bkt + 1u) & 15u;                               // bucket full of other values
                                    fresh = false;
                                }
                                const unsigned long long t = (unsigned long long)a + k;
                                if (t > 1ull) tie += 3ull * t * (t - 1ull);
                            }
                        }
                    };
                    for (int s = s0; s < s1; ++s) {
                        const int c = (int)cnt[s];
                        const float4* src4 = reinterpret_cast<const float4*>(vals + pl.seg_base[s]);
                        float4 nxt = (c > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int i4 = 0; 4 * i4 < c; ++i4) {
                            const float4 q4 = nxt;
                            if (4 * i4 + 4 < c) nxt = src4[i4 + 1];
                            take4(q4, min(4, c - 4 * i4));
                        }
                    }
                    finalize_group<SCORE>(P, R, j, g, m, u2, tie, sum);
                    done = true;
                }
                if (!done) {  // a whole warp (or the CTA) ranks this group by sorting it
                    mlist[atomicAdd(&cnt_m[0], 1)] = (uint16_t)gi;
                    atomicMax(m_max, m);
                }
            }
            __syncthreads();
            // ---- warp tier (usually empty: then this barrier is the only one of the chunk)
            const int nm = cnt_m[0];
            if (nm == 0) continue;
            // warp-tier buffers: 512 keys each when every group of the chunk fits (more warps then own one)
            const int wcap = (*m_max <= WARP_CAP / 2) ? WARP_CAP / 2 : WARP_CAP;
            const int nwb = min(OVO_NW, P.scratch_words / wcap);
            for (int e = w; e < nm && w < nwb; e += nwb) {
                const int g = g0 + mlist[e];
                const int s0 = pl.group_seg[g], s1 = pl.group_seg[g + 1];
                int m = 0;
                for (int s = s0; s < s1; ++s) m += (int)cnt[s];
                if (m > WARP_CAP || (R.keys == nullptr && R.n_ref + (long long)pl.group_size[g] > 208063)) {
                    if (lane == 0) { mlist[e] = (uint16_t)((g - g0) | 0x8000); atomicAdd(&cnt_m[1], 1); }
                    continue;
                }
                uint32_t* buf = scratch + w * wcap;
                int k = 0;
                for (int s = s0; s < s1; ++s) {
                    const int c = (int)cnt[s];
                    const float* src = vals + pl.seg_base[s];
                    for (int i = lane; i < c; i += 32) { uint32_t key = f2key(src[i]); buf[k + i] = key ? key : 1u; }
                    k += c;
                }
                const int Pw = next_pow2(m);
                for (int i = m + lane; i < Pw; i += 32) buf[i] = 0xffffffffu;
                __syncwarp();
                warp_bitonic_sort(buf, Pw, lane);
                unsigned long long u2 = 0, tie = 0;
                double sum = 0.0;
                for (int i = lane; i < m; i += 32) {
                    const uint32_t key = buf[i];
                    sum += fc_val<LOG1P>(key2f(key));
                    if (i == 0 || buf[i - 1] != key) {
                        const uint32_t b = (i + 1 < m && buf[i + 1] == key) ? (uint32_t)(upper_bound_u32(buf, m, key) - i) : 1u;
                        rank_value(R, key, b, u2, tie);
                    }
                }
                u2 = warp_sum_u64(u2);
                tie = warp_sum_u64(tie);
                sum = warp_sum_f64(sum);
                if (lane == 0) finalize_group<SCORE>(P, R, j, g, m, u2, tie, sum, buf, 1);
                __syncwarp();
            }
            __syncthreads();
            // ---- block tier: one group at a time, sorted in the CTA's global slab
            const int nb = cnt_m[1];
            for (int e = 0; e < nm && nb > 0; ++e) {
                const int me = mlist[e];
                if (!(me & 0x8000)) continue;                             // (CTA-uniform)
                const int g = g0 + (me & 0x7fff);
                const int s0 = pl.group_seg[g], s1 = pl.group_seg[g + 1];
                int m = 0;
                for (int s = s0; s < s1; ++s) {
                    const int c = (int)cnt[s];
                    const float* src = vals + pl.seg_base[s];
                    for (int i = tid; i < c; i += OVO_THREADS) { uint32_t key = f2key(src[i]); gA[m + i] = key ? key : 1u; }
                    m += c;
                }
                __syncthreads();
                const uint32_t* gk = block_radix_sort(gA, gB, m, hist, aux);
                unsigned long long u2 = 0, tie = 0;
                double sum = 0.0;
                for (int i = tid; i < m; i += OVO_THREADS) {
                    const uint32_t key = gk[i];
                    sum += fc_val<LOG1P>(key2f(key));
                    if (i == 0 || gk[i - 1] != key) {
                        const uint32_t b = (i + 1 < m && gk[i + 1] == key) ? (uint32_t)(upper_bound_u32(gk, m, key) - i) : 1u;
                        rank_value(R, key, b, u2, tie);
                    }
                }
                u2 = block_sum<unsigned long long>(u2, redu);
                tie = block_sum<unsigned long long>(tie, redu);
                sum = block_sum<double>(sum, redd);
                if (tid == 0) finalize_group<SCORE>(P, R, j, g, m, u2, tie, sum, gk, 1);
                __syncthreads();
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// workspace: [gene counter | per-group constants | per-CTA slabs]
static size_t ovo_head_bytes(const illico_plan_t* plan) {
    const size_t Gs = (size_t)((plan->n_groups + 63) & ~63);
    return 256 + Gs * GCN * sizeof(double);
}
size_t ovo_workspace_bytes(const illico_plan_t* plan, int n_ctas) {
    return ovo_head_bytes(plan) + (size_t)n_ctas * 4 * (size_t)plan->max_group_size * sizeof(uint32_t);
}

template <bool LOG1P, bool SCORE>
static int launch_ovo_t(OvoParams& P, const illico_plan_t* plan, void* workspace, size_t workspace_bytes, int sms,
                        int max_smem, cudaStream_t stream) {
    constexpr int NT = OVO_THREADS, NW = NT / 32;
    // shared memory: control buffer + scratch + fixed part.  Genes whose control has more non-zeros than REF_CAP
    // keep the control in the CTA's global slab.
    const size_t fixed = (size_t)(NW * 256 + RADIX_AUX_WORDS + 2 * GROUP_CHUNK + 8 + MBINS) * 4 + 32 * 8 * 2 + DT_CAP * 16 + DT_HASH * 8 +
                         (2 * ST_CAP + 1) * 4 + 64;
    int scratch_words = (DT_CAP / 2 + 2 * NE_CAP) * NT;              // table path: bins + extras per thread
    if (scratch_words < (STREAM_SLOTS + STREAM_SLOTS / 4) * NT) scratch_words = (STREAM_SLOTS + STREAM_SLOTS / 4) * NT;
    if (scratch_words < 2 * HCAP) scratch_words = 2 * HCAP;          // distinct-value hash of a large control
    if (scratch_words < 2 * WARP_CAP) scratch_words = 2 * WARP_CAP;  // at least two warp-tier buffers
    const size_t need = fixed + (size_t)(REF_CAP + scratch_words) * 4;
    if (need > (size_t)max_smem) { set_error("ovo_kernel needs %zu bytes of shared memory", need); return 1; }
    P.scratch_words = scratch_words;
    auto kern = ovo_kernel<LOG1P, SCORE>;
    ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    int occ = 0;
    ILLICO_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, need));
    if (occ < 1) { set_error("ovo_kernel does not fit: %zu bytes of shared memory", need); return 1; }
    int grid = sms * occ;
    if (grid > P.n_genes) grid = P.n_genes;
    const size_t head = ovo_head_bytes(plan);
    if (workspace_bytes < head) { set_error("rank workspace too small: %zu bytes", workspace_bytes); return 1; }
    const size_t slab_words = 4 * (size_t)plan->max_group_size;
    if ((size_t)grid * slab_words * 4 > workspace_bytes - head) {
        grid = (int)((workspace_bytes - head) / (slab_words * 4));
        if (grid < 1) { set_error("rank workspace too small: %zu bytes", workspace_bytes); return 1; }
    }
    char* ws = reinterpret_cast<char*>(workspace);
    P.gene_counter = reinterpret_cast<int*>(ws);
    P.Gs = (plan->n_groups + 63) & ~63;
    double* gc = reinterpret_cast<double*>(ws + 256);
    P.gc = gc;
    P.slab = reinterpret_cast<uint32_t*>(ws + head); P.slab_words = (long long)slab_words;
    ILLICO_CUDA_OK(cudaMemsetAsync(P.gene_counter, 0, sizeof(int), stream));
    ILLICO_LAUNCH("ovo_group_consts_kernel", stream,
                  ovo_group_consts_kernel<<<(plan->n_groups + 255) / 256, 256, 0, stream>>>(*plan, gc, P.Gs));
    ILLICO_LAUNCH("ovo_kernel", stream, kern<<<grid, NT, need, stream>>>(P));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

// n_genes_dev / gene_map: see OvoParams (both may be NULL)
int launch_ovo_mapped(const float* ir_vals, const uint32_t* ir_cnt, int n_genes, const int* n_genes_dev, const int* gene_map, int n_cols,
                      const illico_plan_t* plan, const illico_flags_t* flags, double* results, long long gstride,
                      void* workspace, size_t workspace_bytes, const illico_debug_t* dbg, cudaStream_t stream) {
    if (n_genes <= 0) return 0;
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
        const size_t adj = 256 - (reinterpret_cast<uintptr_t>(workspace) & 255);
        if (workspace_bytes <= adj) { set_error("rank workspace too small"); return 1; }
        workspace = reinterpret_cast<char*>(workspace) + adj;
        workspace_bytes -= adj;
    }
    int dev = 0, sms = 0, max_smem = 0;
    ILLICO_CUDA_OK(cudaGetDevice(&dev));
    ILLICO_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    ILLICO_CUDA_OK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));

    OvoParams P;
    P.ir_vals = ir_vals; P.ir_cnt = ir_cnt; P.n_genes = n_genes; P.plan = *plan; P.flags = *flags;
    P.results = results; P.gstride = gstride;
    P.n_genes_dev = n_genes_dev; P.gene_map = gene_map; P.n_cols = n_cols;
    P.dbg_u2 = dbg ? (long long*)dbg->u2 : nullptr; P.dbg_tie = dbg ? dbg->tie_sum : nullptr;
    P.dbg_tie_exact = dbg ? (long long*)dbg->tie_exact : nullptr;
    const int v = (flags->is_log1p ? 1 : 0) | (flags->scores ? 2 : 0);
    if (v == 0) return launch_ovo_t<false, false>(P, plan, workspace, workspace_bytes, sms, max_smem, stream);
    if (v == 1) return launch_ovo_t<true, false>(P, plan, workspace, workspace_bytes, sms, max_smem, stream);
    if (v == 2) return launch_ovo_t<false, true>(P, plan, workspace, workspace_bytes, sms, max_smem, stream);
    return launch_ovo_t<true, true>(P, plan, workspace, workspace_bytes, sms, max_smem, stream);
}

int launch_ovo(const float* ir_vals, const uint32_t* ir_cnt, int n_genes, const illico_plan_t* plan,
               const illico_flags_t* flags, double* results, long long gstride, void* workspace,
               size_t workspace_bytes, const illico_debug_t* dbg, cudaStream_t stream) {
    return launch_ovo_mapped(ir_vals, ir_cnt, n_genes, nullptr, nullptr, n_genes, plan, flags, results, gstride, workspace, workspace_bytes,
                             dbg, stream);
}

}  // namespace illico
