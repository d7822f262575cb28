// rank_ovr.cu -- one-versus-rest Mann-Whitney U on group-segmented non-zero lists (sm_100a).
//
// Replaces illico/ovr/dense_ovr.py:15-80, illico/ovr/sparse_ovr.py:23-97 and
// illico/utils/ranking.py:7-49.  The reference argsorts every gene column and scatters mid-ranks into
// per-group sums.  Here labels never move: per gene the kernel builds a RANK ORACLE over the column's
// non-zero values and every group looks its values up in it:
//
//   path H (few distinct values, e.g. raw counts): shared-memory hash table value -> multiplicity, its
//           <= 2048 distinct values sorted and prefix-summed; lookup = one hash probe.
//   path S (continuous data): keys-only block radix sort (shared memory when the column fits, else the
//           CTA's global slab); lookup = lower/upper bound.
//
// A run of equal values at sorted positions [lo, hi) has doubled mid-rank r2 = lo + hi + 1 (an integer,
// SURVEY.md appendix A.1).  Zeros are not stored: with n0 zeros and n_neg negative values, positives
// are shifted by n0 and the zero block has r2 = 2 n_neg + n0 + 1 (appendix A.3, extended to negatives).
// 2R_g, 2U_g and the tie terms are exact integers; the tie sum is accumulated in the reference's order
// when it exceeds 2^53 (appendix A.4).
#include "common.cuh"
#include "epilogue.cuh"
#include "sort.cuh"

namespace illico {

constexpr int OVR_THREADS = 512;
constexpr int OVR_NW = OVR_THREADS / 32;
constexpr int HASH_CAP = 4096;
constexpr int MAX_DISTINCT = 2048;
constexpr uint32_t HASH_EMPTY = 0u;
constexpr int T_THREADS = 128;  // table kernel: threads per CTA (one gene at a time, ~8 CTAs per SM)
constexpr int T_SLOTS = 32;     // slots of the small value table (also the bins of a segment histogram)
constexpr int T_CAP = 20;       // most distinct values the table kernel takes
constexpr int T_WORDS = T_SLOTS / 2;  // two 16-bit bins per 32-bit word
constexpr int T_MULTI = 256;    // multi-segment groups handed to whole warps per gene (more are ranked inline)
constexpr int T_REC_WORDS = T_SLOTS / 4;  // segment record: one 8-bit bin per table slot = 32 bytes (one sector)

struct OvrParams {
    const float* ir_vals;
    const uint32_t* ir_cnt;
    int n_genes;
    illico_plan_t plan;
    illico_flags_t flags;
    double* results;
    long long gstride;
    unsigned long long* slab;  // global scratch, slab_qwords (8-byte words) per CTA
    long long slab_qwords;
    int sort_cap;              // keys per shared-memory sort buffer (path S): HASH_CAP
    long long* dbg_u2;
    double* dbg_tie;
    long long* dbg_tie_exact;
    const int* n_genes_dev;    // optional: number of genes decided on the device (a hand-back list), else n_genes
    const int* gene_map;       // optional: staged gene j is column gene_map[j] of the results / debug / group-sum arrays
    int n_cols;                // width of the debug / group-sum arrays (= n_genes unless gene_map is set)
    int* todo;        // genes the table kernel could not take (NULL: the general kernel ranks every gene)
    int* todo_count;
    uint4* table_rec;          // table kernel: per-CTA [n_segments][2] segment records (NULL: second pass re-reads the values)
    long long table_rec_stride;  // uint4 per CTA
};

__device__ __forceinline__ uint32_t hash_slot(uint32_t key) { return (key * 2654435761u) >> 20; }  // 12 bits

__device__ __forceinline__ void hash_insert(uint32_t* hkeys, uint32_t* hvals, int* ndist, int* overflow, uint32_t key,
                                            uint32_t c, int max_distinct) {
    if (*(volatile int*)ndist >= max_distinct) { *overflow = 1; return; }
    uint32_t h = hash_slot(key);
    for (;;) {
        uint32_t prev = atomicCAS(&hkeys[h], HASH_EMPTY, key);
        if (prev == HASH_EMPTY) atomicAdd(ndist, 1);
        if (prev == HASH_EMPTY || prev == key) { atomicAdd(&hvals[h], c); return; }
        h = (h + 1) & (HASH_CAP - 1);
    }
}
__device__ __forceinline__ uint32_t hash_find(const uint32_t* hkeys, uint32_t key) {
    uint32_t h = hash_slot(key);
    while (hkeys[h] != key) h = (h + 1) & (HASH_CAP - 1);
    return h;
}

// n0^3 - n0 the way the sparse reference kernel forms it: n0 is a float64 (ovr/sparse_ovr.py:49,83)
__device__ __forceinline__ double zero_block_term_f64(long long n0) {
    double x = (double)n0;
    double c = __dmul_rn(__dmul_rn(x, x), x);
    return __dsub_rn(c, x);
}

// SCORE: also writes the score plane (illico_flags_t::scores), in an instantiation of its own
template <bool SCORE>
__global__ void __launch_bounds__(OVR_THREADS, 2) ovr_kernel(const OvrParams P) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, lane = tid & 31;
    const illico_plan_t& pl = P.plan;
    const int S = pl.n_segments, G = pl.n_groups;
    const long long n = pl.n_cells;

    // ---- shared carve-up: region0 = hash table (path H) or sort ping-pong (path S)
    const int region0_words = max(2 * HASH_CAP, 2 * P.sort_cap);
    uint32_t* hkeys = smem;
    uint32_t* hvals = smem + HASH_CAP;
    uint32_t* sortA = smem;
    uint32_t* sortB = smem + P.sort_cap;
    uint32_t* hist = smem + region0_words;        // [OVR_NW*256] path S;  path H: dkeys | dcnt
    uint32_t* dkeys = hist;                       // [MAX_DISTINCT]
    uint32_t* dcnt = hist + MAX_DISTINCT;         // [MAX_DISTINCT]
    uint32_t* aux = hist + OVR_NW * 256;          // [RADIX_AUX_WORDS]
    int* sc = (int*)(aux + RADIX_AUX_WORDS);      // [8] scalars
    double* redd = (double*)(sc + 8);             // [32]
    unsigned long long* redu = (unsigned long long*)(redd + 32);  // [32]
    double* tie_slot = (double*)(redu + 32);      // [1]

    unsigned long long* slab = P.slab + (long long)blockIdx.x * P.slab_qwords;
    unsigned long long* seg_r2 = slab;                       // [S]
    double* seg_sum = (double*)(slab + S);                   // [S]
    uint32_t* gsortA = (uint32_t*)(slab + 2ll * S);          // [n_cells]
    uint32_t* gsortB = gsortA + ((n + 1) & ~1ll);            // [n_cells]

    const double cc = P.flags.use_continuity ? 0.5 : 0.0;

    const int n_work = P.todo ? *P.todo_count : (P.n_genes_dev ? *P.n_genes_dev : P.n_genes);
    for (int wi = blockIdx.x; wi < n_work; wi += gridDim.x) {
        const int j = P.todo ? P.todo[wi] : wi;
        const int jo = P.gene_map ? P.gene_map[j] : j;   // column of the results / side arrays
        const uint32_t* cnt = P.ir_cnt + (long long)j * S;
        const float* vals = P.ir_vals + (long long)j * pl.slot_cap;

        long long nnz = 0, n0 = 0, n_neg = 0;
        unsigned long long tie_nz_exact = 0;
        bool path_s = false, bk_on = false;
        uint32_t bk_kmin = 0;
        int bk_shift = 0, bk_last = 0;
        const uint32_t* sk = nullptr;  // sorted keys (path S)
        {
        // ================= phase A: value -> multiplicity hash (path H attempt) =================
        for (int i = tid; i < 2 * HASH_CAP; i += OVR_THREADS) smem[i] = 0;
        if (tid < 8) sc[tid] = 0;  // [0] ndist [1] overflow [2] cursor [3] dn
        __syncthreads();
        unsigned long long my_nnz = 0;
        for (int s0 = 0; s0 < S; s0 += OVR_THREADS) {
            const int s = s0 + tid;
            const int c = (s < S) ? (int)cnt[s] : 0;
            my_nnz += c;
            const float* src = vals + ((s < S) ? pl.seg_base[s] : 0);
            // continuous data overflows the table within the first segments: from then on only the counts are needed
            // (warp-uniform decision: the loop below votes)
            if (__any_sync(FULL, *(volatile int*)&sc[1] != 0)) continue;
            int maxc = c;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) maxc = max(maxc, __shfl_xor_sync(FULL, maxc, o));
            const float4* src4 = reinterpret_cast<const float4*>(src);  // slots are 32-byte aligned and padded
            float4 nxt = (c > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < maxc; i += 4) {
                const float4 q4 = nxt;
                if (i + 4 < c) nxt = src4[(i >> 2) + 1];
                const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const bool act = i + e < c;
                    uint32_t key = act ? f2key(q[e]) : HASH_EMPTY;
                    if (act && key == HASH_EMPTY) key = 1u;  // only a NaN payload maps here
                    const unsigned peers = __match_any_sync(FULL, key);
                    if (act && lane == __ffs(peers) - 1 && !*(volatile int*)&sc[1])
                        hash_insert(hkeys, hvals, &sc[0], &sc[1], key, __popc(peers), MAX_DISTINCT);
                }
            }
        }
        nnz = (long long)block_sum<unsigned long long>(my_nnz, redu);  // syncs
        n0 = n - nnz;
        path_s = sc[1] != 0 || sc[0] > MAX_DISTINCT;
        __syncthreads();

        if (!path_s) {
            // ---- distinct values: compact, sort, prefix
            for (int t = tid; t < HASH_CAP; t += OVR_THREADS)
                if (hkeys[t] != HASH_EMPTY) {
                    int idx = atomicAdd(&sc[3], 1);
                    dkeys[idx] = hkeys[t];
                    dcnt[idx] = hvals[t];
                }
            __syncthreads();
            const int D = sc[3];
            const int Pd = max(2, next_pow2(D));
            for (int i = D + tid; i < Pd; i += OVR_THREADS) { dkeys[i] = 0xffffffffu; dcnt[i] = 0; }
            __syncthreads();
            block_bitonic_sort_pairs(dkeys, dcnt, Pd);
            // exclusive prefix of dcnt: 4 consecutive entries per thread (MAX_DISTINCT = 4 * OVR_THREADS)
            uint32_t c4[4], loc = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int i = tid * 4 + q;
                c4[q] = (i < D) ? dcnt[i] : 0;
                loc += c4[q];
            }
            uint32_t incl = warp_incl_scan(loc, lane);
            if (lane == 31) aux[tid >> 5] = incl;
            __syncthreads();
            uint32_t base = incl - loc;
            for (int ww = 0; ww < (tid >> 5); ++ww) base += aux[ww];
            unsigned long long t_exact = 0, negs = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int i = tid * 4 + q;
                if (i < D) {
                    const uint32_t key = dkeys[i];
                    const uint32_t lo = base, hi = base + c4[q];
                    unsigned long long r2 = (unsigned long long)lo + hi + 1;
                    if (key > KEY_ZERO) r2 += 2ull * (unsigned long long)n0;
                    hvals[hash_find(hkeys, key)] = (uint32_t)r2;  // table now maps value -> doubled mid-rank
                    t_exact += (unsigned long long)cube_minus((long long)c4[q]);
                    if (key < KEY_ZERO) negs += c4[q];
                }
                base += c4[q];
            }
            tie_nz_exact = block_sum<unsigned long long>(t_exact, redu);
            n_neg = (long long)block_sum<unsigned long long>(negs, redu);
            // ---- ordered f64 accumulation when the exact sum may not be representable
            const unsigned long long zterm = (unsigned long long)cube_minus(n0);
            const bool sparse_order = P.flags.tie_order == ILLICO_TIES_SPARSE;
            const bool need_walk = sparse_order ? ((double)tie_nz_exact >= TWO53)
                                                : ((double)tie_nz_exact + (double)zterm >= TWO53);
            if (tid == 0) {
                double acc;
                if (!need_walk) {
                    acc = sparse_order ? (double)tie_nz_exact : (double)(tie_nz_exact + zterm);
                } else {
                    acc = 0.0;
                    bool zero_done = sparse_order || n0 == 0;
                    for (int i = 0; i < D; ++i) {
                        if (!zero_done && dkeys[i] > KEY_ZERO) { acc += (double)(long long)zterm; zero_done = true; }
                        acc += (double)cube_minus((long long)dcnt[i]);
                    }
                    if (!zero_done) acc += (double)(long long)zterm;
                }
                if (sparse_order) acc = __dadd_rn(acc, zero_block_term_f64(n0));
                *tie_slot = acc;
            }
            __syncthreads();
        } else {
            {
            // ---- path S: gather keys, sort, scan runs
            const bool in_smem = nnz <= P.sort_cap;
            uint32_t* A = in_smem ? sortA : gsortA;
            uint32_t* B = in_smem ? sortB : gsortB;
            for (int s = tid; s < S; s += OVR_THREADS) {
                const int c = (int)cnt[s];
                if (c == 0) continue;
                const float* src = vals + pl.seg_base[s];
                const int at = atomicAdd(&sc[2], c);
                for (int i = 0; i < c; ++i) A[at + i] = f2key(src[i]);
            }
            __syncthreads();
            sk = block_radix_sort(A, B, (int)nnz, hist, aux);
            n_neg = lower_bound_u32(sk, (int)nnz, KEY_ZERO);
            // ---- bucket index of the sorted keys (they sit in the global slab: region0 is free): the key range is cut
            // into equal buckets, bk[b] = first position of bucket b or later, so a rank reads its bucket's bounds from
            // shared memory and halves a few times in L2 instead of 15 times
            bk_on = !in_smem && nnz > 1 && nnz < 65536;
            if (bk_on) {
                uint16_t* bk = reinterpret_cast<uint16_t*>(smem);
                const int cap = 4 * HASH_CAP - 2;                                   // u16 entries in region0, one spare
                const uint32_t kmin = sk[0], span = sk[nnz - 1] - kmin;
                int shift = 0;
                while ((span >> shift) > (uint32_t)(cap - 2)) ++shift;
                const int NB = (int)(span >> shift) + 1;
                for (int i = tid; i < (int)nnz; i += OVR_THREADS) {
                    const int bi = (int)((sk[i] - kmin) >> shift);
                    const int bp = i ? (int)((sk[i - 1] - kmin) >> shift) : -1;
                    for (int bb = bp + 1; bb <= bi; ++bb) bk[bb] = (uint16_t)i;
                    if (i == (int)nnz - 1) for (int bb = bi + 1; bb <= NB; ++bb) bk[bb] = (uint16_t)nnz;
                }
                bk_kmin = kmin; bk_shift = shift; bk_last = NB - 1;
                __syncthreads();
            }
            unsigned long long t_exact = 0;
            for (int i = tid; i < (int)nnz; i += OVR_THREADS) {
                const uint32_t k = sk[i];
                if ((i == 0 || sk[i - 1] != k) && i + 1 < (int)nnz && sk[i + 1] == k)      // (a run of one adds nothing)
                    t_exact += (unsigned long long)cube_minus(upper_bound_u32(sk, (int)nnz, k) - i);
            }
            tie_nz_exact = block_sum<unsigned long long>(t_exact, redu);
            const unsigned long long zterm = (unsigned long long)cube_minus(n0);
            const bool sparse_order = P.flags.tie_order == ILLICO_TIES_SPARSE;
            const bool need_walk = sparse_order ? ((double)tie_nz_exact >= TWO53)
                                                : ((double)tie_nz_exact + (double)zterm >= TWO53);
            // The reference adds the runs' terms one by one in ascending value order (the zero block where the values cross
            // zero, or last for the sparse kernels): once the partial sum passes 2^53 that order decides the bits.  Only runs
            // of two or more equal values contribute, so their terms are compacted, in order, into the sort's free buffer
            // by the whole CTA and one thread adds up that (for continuous data empty) list -- not the 30 000 sorted keys.
            int n_terms = 0, n_terms_neg = 0;
            if (need_walk && tie_nz_exact != 0) {
                unsigned long long* terms = reinterpret_cast<unsigned long long*>(const_cast<uint32_t*>(sk == A ? B : A));
                const int w = tid >> 5;
                const unsigned lt = (1u << lane) - 1u;
                for (int i0 = 0; i0 < (int)nnz; i0 += OVR_THREADS) {
                    const int i = i0 + tid;
                    bool head = false;
                    uint32_t k = 0;
                    if (i < (int)nnz) {
                        k = sk[i];
                        head = (i == 0 || sk[i - 1] != k) && i + 1 < (int)nnz && sk[i + 1] == k;
                    }
                    const unsigned bal = __ballot_sync(FULL, head), bal_neg = __ballot_sync(FULL, head && i < (int)n_neg);
                    if (lane == 0) { hist[w] = (uint32_t)__popc(bal); hist[OVR_NW + w] = (uint32_t)__popc(bal_neg); }
                    __syncthreads();
                    int before = 0, total = 0, total_neg = 0;
                    for (int ww = 0; ww < OVR_NW; ++ww) {
                        const int c = (int)hist[ww];
                        if (ww < w) before += c;
                        total += c;
                        total_neg += (int)hist[OVR_NW + ww];
                    }
                    if (head) terms[n_terms + before + __popc(bal & lt)] = (unsigned long long)cube_minus((long long)(upper_bound_u32(sk, (int)nnz, k) - i));
                    n_terms += total;
                    n_terms_neg += total_neg;
                    __syncthreads();
                }
            }
            if (tid == 0) {
                double acc;
                if (!need_walk) {
                    acc = sparse_order ? (double)tie_nz_exact : (double)(tie_nz_exact + zterm);
                } else {
                    const unsigned long long* terms = reinterpret_cast<const unsigned long long*>(sk == A ? B : A);
                    acc = 0.0;
                    bool zero_done = sparse_order || n0 == 0;
                    for (int t = 0; t < n_terms_neg; ++t) acc += (double)(long long)terms[t];
                    if (!zero_done && (long long)n_neg < nnz) { acc += (double)(long long)zterm; zero_done = true; }   // a positive value follows
                    for (int t = n_terms_neg; t < n_terms; ++t) acc += (double)(long long)terms[t];
                    if (!zero_done) acc += (double)(long long)zterm;
                }
                if (sparse_order) acc = __dadd_rn(acc, zero_block_term_f64(n0));
                *tie_slot = acc;
            }
            __syncthreads();
            }
        }
        }
        const double tie = *tie_slot;
        const unsigned long long r2_zero = 2ull * (unsigned long long)n_neg + (unsigned long long)n0 + 1ull;

        // ================= phase B: per-segment doubled rank sums and expression sums =================
        for (int s = tid; s < S; s += OVR_THREADS) {
            const int c = (int)cnt[s];
            const float* src = vals + pl.seg_base[s];
            unsigned long long acc = 0;
            double sum = 0.0;
            const float4* src4 = reinterpret_cast<const float4*>(src);
            float4 nxt = (c > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < c; i += 4) {
                const float4 q4 = nxt;
                if (i + 4 < c) nxt = src4[(i >> 2) + 1];
                const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (i + e < c) {
                        const float v = q[e];
                        uint32_t key = f2key(v);
                        if (key == HASH_EMPTY) key = 1u;
                        if (!path_s) {
                            acc += hvals[hash_find(hkeys, key)];
                        } else {
                            int lo, hi;
                            if (bk_on) {
                                const uint16_t* bk = reinterpret_cast<const uint16_t*>(smem);
                                const uint32_t bq = min((key - bk_kmin) >> bk_shift, (uint32_t)bk_last);   // (key is one of the sorted keys)
                                lo = bk[bq];
                                int e = bk[bq + 1];
                                while (lo < e) { const int mid = (lo + e) >> 1; if (sk[mid] < key) lo = mid + 1; else e = mid; }
                            } else {
                                lo = lower_bound_u32(sk, (int)nnz, key);
                            }
                            // the run of the key: continuous values are alone in theirs
                            hi = lo + 1;
                            if (hi < (int)nnz && sk[hi] == key) hi = upper_bound_u32(sk, (int)nnz, key);
                            acc += (unsigned long long)lo + hi + 1 + ((key > KEY_ZERO) ? 2ull * (unsigned long long)n0 : 0ull);
                        }
                        sum += fc_value(v, P.flags.is_log1p);
                    }
                }
            }
            seg_r2[s] = acc;
            seg_sum[s] = sum;
        }
        __syncthreads();

        // ================= phase C: per-group U and p; expression sums parked in the fold-change slot ============
        double my_total = 0.0;
        for (int g = tid; g < G; g += OVR_THREADS) {
            unsigned long long R2 = 0;
            double sum = 0.0;
            long long nnz_g = 0;
            for (int s = pl.group_seg[g]; s < pl.group_seg[g + 1]; ++s) { R2 += seg_r2[s]; sum += seg_sum[s]; nnz_g += cnt[s]; }
            if (P.flags.group_sums) sum = P.flags.group_sums[(long long)g * P.n_cols + jo];
            const long long n_t = pl.group_size[g], n_r = n - n_t;
            R2 += (unsigned long long)(n_t - nnz_g) * r2_zero;
            const long long u2 = 2 * n_r * n_t + n_t * (n_t + 1) - (long long)R2;
            const double U = (double)u2 / 2.0;
            const double mu = (double)(n_r * n_t) / 2.0;
            const double p = compute_pval(n_r, n_t, n, P.flags.tie_correct ? tie : 0.0, U, mu, cc, P.flags.alternative);
            if (SCORE)
                P.flags.scores[(long long)g * P.flags.score_group_stride + jo] = compute_score(n_r, n_t, n, P.flags.tie_correct ? tie : 0.0, U, mu);
            double* o = P.results + (long long)g * P.gstride + (long long)jo * 3;
            o[0] = p; o[1] = U; o[2] = sum;
            my_total += sum;
            if (P.dbg_u2) P.dbg_u2[(long long)g * P.n_cols + jo] = u2;
        }
        const double total = block_sum<double>(my_total, redd);
        // ================= phase D: fold change (illico/utils/math.py:168-193, one-versus-rest branch) ============
        for (int g = tid; g < G; g += OVR_THREADS) {
            double* o = P.results + (long long)g * P.gstride + (long long)jo * 3;
            const double sum = o[2];
            const long long n_t = pl.group_size[g];
            const double mu_t = sum * (1.0 / (double)n_t);   // (the fused epilogue's form: every path gives the same bits)
            const double mu_r = (total - sum) / (double)(n - n_t);
            o[2] = (mu_r == 0.0) ? INFINITY : mu_t / mu_r;
        }
        if (tid == 0) {
            if (P.dbg_tie) P.dbg_tie[jo] = tie;
            if (P.dbg_tie_exact) P.dbg_tie_exact[jo] = (long long)(tie_nz_exact + (unsigned long long)cube_minus(n0));
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------
// Table kernel: genes with a handful of distinct non-zero values (raw counts).  Small CTAs, little shared
// memory, so ~8 genes are in flight per SM and the dependent global loads of one gene overlap with the work
// of the others.  Per gene:
//   pass 1  one thread per segment: every value is looked up in a 32-slot shared table (unseen values are
//           inserted) and bumps an 8-bit bin of the segment's histogram.  The finished histogram (32 bytes, one
//           sector) goes to the CTA's record area in global memory -- it is re-read a moment later, normally from
//           L2 -- and is added to the thread's 16-bit column accumulators;
//   finish  thread 0 sorts the <= 20 values, turns multiplicities into doubled mid-ranks, tie sum, totals;
//   pass 2  one thread per group: sum over the group's segment histograms of count x doubled mid-rank and
//           count x expression value -> 2U, p, fold change.  The staged values are read ONCE.
// A segment with more than 255 stored values could overflow an 8-bit bin: such a gene keeps 16-bit bins only
// and its second pass re-reads the values (the round-1 two-pass scheme).  A gene with more distinct values is
// appended to `todo` for the general kernel.
template <bool SCORE>
__global__ void __launch_bounds__(T_THREADS, 8) ovr_table_kernel(const OvrParams P) {
    __shared__ uint32_t tkey[T_SLOTS];      // raw float bits, 0 = empty
    __shared__ uint32_t gcount[T_SLOTS];    // multiplicity in the whole column
    __shared__ uint32_t r2slot[T_SLOTS];    // doubled mid-rank of the slot's value
    __shared__ double fcslot[T_SLOTS];      // f(x) of the slot's value
    __shared__ uint32_t bins[T_WORDS][T_THREADS];      // 16-bit column accumulators: word 2q+r = slots 4q+r, 4q+r+2
    __shared__ uint32_t seg8[T_REC_WORDS][T_THREADS];  // 8-bit bins of the segment in progress: word q = slots 4q..4q+3
    __shared__ unsigned long long redu[8];
    __shared__ double redd[4];
    __shared__ int sc[4];
    __shared__ int multi[T_MULTI];          // groups with several segments (e.g. the rest-of-cells sized clusters)
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const illico_plan_t& pl = P.plan;
    const int S = pl.n_segments, G = pl.n_groups;
    const long long n = pl.n_cells;
    const double cc = P.flags.use_continuity ? 0.5 : 0.0;
    uint4* rec = P.table_rec ? P.table_rec + (long long)blockIdx.x * P.table_rec_stride : nullptr;

    const int n_genes = P.n_genes_dev ? *P.n_genes_dev : P.n_genes;
    for (int j = blockIdx.x; j < n_genes; j += gridDim.x) {
        const int jo = P.gene_map ? P.gene_map[j] : j;   // column of the results / side arrays
        const uint32_t* cnt = P.ir_cnt + (long long)j * S;
        const float* vals = P.ir_vals + (long long)j * pl.slot_cap;
        __syncthreads();
        if (tid < T_SLOTS) { tkey[tid] = 0u; gcount[tid] = 0u; }
        if (tid < 4) sc[tid] = 0;  // [0] distinct [1] overflow [2] multi-segment groups [3] gene has a wide segment
        __syncthreads();
        // ================= pass 1 =================
        unsigned long long my_nnz = 0;
        uint32_t since_flush = 0;
        auto flush_bins = [&]() {
#pragma unroll 4
            for (int a = 0; a < T_WORDS; ++a) {
                const uint32_t w2 = bins[a][tid];
                const int lo_slot = 4 * (a >> 1) + (a & 1);
                if (w2 & 0xffffu) atomicAdd(&gcount[lo_slot], w2 & 0xffffu);
                if (w2 >> 16) atomicAdd(&gcount[lo_slot + 2], w2 >> 16);
                bins[a][tid] = 0u;
            }
            since_flush = 0;
        };
#pragma unroll
        for (int a = 0; a < T_WORDS; ++a) bins[a][tid] = 0u;
#pragma unroll
        for (int q = 0; q < T_REC_WORDS; ++q) seg8[q][tid] = 0u;
        bool ok = true;
        for (int s = tid; s < S && ok; s += T_THREADS) {
            if (*(volatile int*)&sc[1]) break;
            const int c = (int)cnt[s];
            if (since_flush + (uint32_t)c > 60000u) flush_bins();
            since_flush += (uint32_t)c;
            my_nnz += c;
            const bool narrow = rec != nullptr && c <= 255;   // 8-bit bins cannot overflow
            if (!narrow) sc[3] = 1;
            const float4* src4 = reinterpret_cast<const float4*>(vals + pl.seg_base[s]);  // 32-byte aligned, padded slot
            float4 nxt = (c > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < c && ok; i += 4) {
                const float4 q4 = nxt;
                if (i + 4 < c) nxt = src4[(i >> 2) + 1];
                const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (i + e < c && ok) {
                        const uint32_t bits = __float_as_uint(q[e]);
                        uint32_t h = (bits * 2654435761u) >> 27;
                        int probes = 0;
                        for (;;) {
                            uint32_t kk = *(volatile uint32_t*)&tkey[h];
                            if (kk == 0u) {
                                kk = atomicCAS(&tkey[h], 0u, bits);
                                if (kk == 0u) {
                                    if (atomicAdd(&sc[0], 1) >= T_CAP) { sc[1] = 1; ok = false; }
                                    break;
                                }
                            }
                            if (kk == bits) break;
                            h = (h + 1) & (T_SLOTS - 1);
                            if (++probes > T_SLOTS) { sc[1] = 1; ok = false; break; }
                        }
                        if (ok) {
                            if (narrow) seg8[h >> 2][tid] += 1u << ((h & 3u) << 3);
                            else bins[((h >> 2) << 1) | (h & 1u)][tid] += 1u << ((h & 2u) << 3);
                        }
                    }
                }
            }
            if (narrow && ok) {
                uint32_t r[T_REC_WORDS];
#pragma unroll
                for (int q = 0; q < T_REC_WORDS; ++q) {
                    r[q] = seg8[q][tid];
                    if (r[q]) {
                        seg8[q][tid] = 0u;
                        bins[2 * q][tid] += r[q] & 0x00ff00ffu;
                        bins[2 * q + 1][tid] += (r[q] >> 8) & 0x00ff00ffu;
                    }
                }
                __stcg(rec + 2 * (long long)s, make_uint4(r[0], r[1], r[2], r[3]));
                __stcg(rec + 2 * (long long)s + 1, make_uint4(r[4], r[5], r[6], r[7]));
            }
        }
        if (ok) flush_bins();
        // block sum of my_nnz
        my_nnz = warp_sum_u64(my_nnz);
        if (lane == 0) redu[w] = my_nnz;
        __syncthreads();
        if (sc[1]) {  // too many distinct values: leave the gene to the general kernel
            if (tid == 0) P.todo[atomicAdd(P.todo_count, 1)] = j;
            continue;
        }
        const bool from_records = sc[3] == 0;   // every segment left a histogram record
        const long long nnz = (long long)(redu[0] + redu[1] + redu[2] + redu[3]);
        const long long n0 = n - nnz;
        // ================= finish the table (thread 0; <= 20 entries) =================
        if (tid == 0) {
            uint32_t skey[T_CAP + 1], sslot[T_CAP + 1];
            int D = 0;
            for (int q = 0; q < T_SLOTS; ++q)
                if (tkey[q] != 0u) {  // insertion sort by order-preserving key
                    const uint32_t k = f2key(__uint_as_float(tkey[q]));
                    int a = D - 1;
                    while (a >= 0 && skey[a] > k) { skey[a + 1] = skey[a]; sslot[a + 1] = sslot[a]; --a; }
                    skey[a + 1] = k; sslot[a + 1] = (uint32_t)q;
                    ++D;
                }
            unsigned long long lo = 0, t_exact = 0, negs = 0;
            double total = 0.0;
            for (int a = 0; a < D; ++a) {
                const uint32_t q = sslot[a], cq = gcount[q];
                unsigned long long r2 = 2ull * lo + cq + 1ull;   // lo + hi + 1 with hi = lo + cq
                if (skey[a] > KEY_ZERO) r2 += 2ull * (unsigned long long)n0;
                r2slot[q] = (uint32_t)r2;
                const double f = fc_value(__uint_as_float(tkey[q]), P.flags.is_log1p);
                fcslot[q] = f;
                total += (double)cq * f;
                t_exact += (unsigned long long)cube_minus((long long)cq);
                if (skey[a] < KEY_ZERO) negs += cq;
                lo += cq;
            }
            const unsigned long long zterm = (unsigned long long)cube_minus(n0);
            const bool sparse_order = P.flags.tie_order == ILLICO_TIES_SPARSE;
            const bool need_walk = sparse_order ? ((double)t_exact >= TWO53) : ((double)t_exact + (double)zterm >= TWO53);
            double acc;
            if (!need_walk) {
                acc = sparse_order ? (double)t_exact : (double)(t_exact + zterm);
            } else {  // the reference's sequential f64 accumulation, in its order (SURVEY.md appendix A.4)
                acc = 0.0;
                bool zero_done = sparse_order || n0 == 0;
                for (int a = 0; a < D; ++a) {
                    if (!zero_done && skey[a] > KEY_ZERO) { acc += (double)(long long)zterm; zero_done = true; }
                    acc += (double)cube_minus((long long)gcount[sslot[a]]);
                }
                if (!zero_done) acc += (double)(long long)zterm;
            }
            if (sparse_order) acc = __dadd_rn(acc, zero_block_term_f64(n0));
            redd[0] = acc;
            redd[1] = total;
            redu[4] = t_exact;
            redu[5] = negs;
        }
        __syncthreads();
        const double tie = redd[0], total = redd[1];
        const unsigned long long r2_zero = 2ull * redu[5] + (unsigned long long)n0 + 1ull;
        // ================= pass 2: one thread per single-segment group, one warp per multi-segment group =========
        auto rank_values = [&](int s, unsigned long long& R2, double& sum, long long& nnz_g) {
            const int c = (int)cnt[s];
            nnz_g += c;
            const float4* src4 = reinterpret_cast<const float4*>(vals + pl.seg_base[s]);
            float4 nxt = (c > 0) ? src4[0] : make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < c; i += 4) {
                const float4 q4 = nxt;
                if (i + 4 < c) nxt = src4[(i >> 2) + 1];
                const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (i + e < c) {
                        const uint32_t bits = __float_as_uint(q[e]);
                        uint32_t h = (bits * 2654435761u) >> 27;
                        while (tkey[h] != bits) h = (h + 1) & (T_SLOTS - 1);
                        R2 += r2slot[h];
                        sum += fcslot[h];
                    }
                }
            }
        };
        auto rank_record = [&](int s, unsigned long long& R2, double& sum, long long& nnz_g) {
            const uint4 ra = __ldcg(rec + 2 * (long long)s), rb = __ldcg(rec + 2 * (long long)s + 1);
            const uint32_t r[T_REC_WORDS] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
            for (int q = 0; q < T_REC_WORDS; ++q) {
                uint32_t x = r[q];
                while (x) {  // the non-empty bins of this word (a segment holds a few distinct values)
                    const int byte = (__ffs(x) - 1) >> 3;
                    const uint32_t bq = (x >> (byte << 3)) & 0xffu;
                    x &= ~(0xffu << (byte << 3));
                    const int h = 4 * q + byte;
                    R2 += (unsigned long long)bq * r2slot[h];
                    sum += (double)bq * fcslot[h];
                    nnz_g += bq;
                }
            }
        };
        auto rank_segment = [&](int s, unsigned long long& R2, double& sum, long long& nnz_g) {
            if (from_records) rank_record(s, R2, sum, nnz_g); else rank_values(s, R2, sum, nnz_g);
        };
        auto finish_group = [&](int g, unsigned long long R2, double sum, long long nnz_g) {
            const long long n_t = pl.group_size[g], n_r = n - n_t;
            R2 += (unsigned long long)(n_t - nnz_g) * r2_zero;
            const long long u2 = 2 * n_r * n_t + n_t * (n_t + 1) - (long long)R2;
            const double U = (double)u2 / 2.0;
            const double mu = (double)(n_r * n_t) / 2.0;
            const double p = compute_pval(n_r, n_t, n, P.flags.tie_correct ? tie : 0.0, U, mu, cc, P.flags.alternative);
            if (SCORE)
                P.flags.scores[(long long)g * P.flags.score_group_stride + jo] = compute_score(n_r, n_t, n, P.flags.tie_correct ? tie : 0.0, U, mu);
            const double mu_t = sum * (1.0 / (double)n_t);   // (the fused epilogue's form: every path gives the same bits)
            // exactly zero when the group holds every non-zero of the gene (see fused_epilogue_kernel); 0 / 0 = NaN, as in
            // ovr_kernel and the oracle, when it holds every cell (a single group: there is no rest)
            const double mu_r = (n_t == n) ? NAN : (nnz_g == nnz) ? 0.0 : (total - sum) / (double)(n - n_t);
            double* o = P.results + (long long)g * P.gstride + (long long)jo * 3;
            o[0] = p; o[1] = U; o[2] = (mu_r == 0.0) ? INFINITY : mu_t / mu_r;
            if (P.dbg_u2) P.dbg_u2[(long long)g * P.n_cols + jo] = u2;
        };
        for (int g = tid; g < G; g += T_THREADS) {
            const int s0 = pl.group_seg[g], s1 = pl.group_seg[g + 1];
            if (s1 - s0 > 1) {  // big group: leave it to a whole warp (one lane per segment)
                const int slot = atomicAdd(&sc[2], 1);
                if (slot < T_MULTI) { multi[slot] = g; continue; }
            }
            unsigned long long R2 = 0;
            double sum = 0.0;
            long long nnz_g = 0;
            for (int s = s0; s < s1; ++s) rank_segment(s, R2, sum, nnz_g);
            finish_group(g, R2, sum, nnz_g);
        }
        __syncthreads();
        const int n_multi = min(sc[2], T_MULTI);
        for (int m = w; m < n_multi; m += T_THREADS / 32) {
            const int g = multi[m];
            unsigned long long R2 = 0;
            double sum = 0.0;
            long long nnz_g = 0;
            for (int s = pl.group_seg[g] + lane; s < pl.group_seg[g + 1]; s += 32) rank_segment(s, R2, sum, nnz_g);
            R2 = warp_sum_u64(R2);
            sum = warp_sum_f64(sum);
            nnz_g = (long long)warp_sum_u64((unsigned long long)nnz_g);
            if (lane == 0) finish_group(g, R2, sum, nnz_g);
        }
        if (tid == 0) {
            if (P.dbg_tie) P.dbg_tie[jo] = tie;
            if (P.dbg_tie_exact) P.dbg_tie_exact[jo] = (long long)(redu[4] + (unsigned long long)cube_minus(n0));
        }
    }
}

size_t ovr_table_rec_bytes(const illico_plan_t* plan) { return (size_t)plan->n_segments * 32; }  // per table-kernel CTA
constexpr int T_MAX_CTAS_PER_SM = 8;

size_t ovr_slab_qwords(const illico_plan_t* plan) {
    return 2 * (size_t)plan->n_segments + (size_t)((plan->n_cells + 1) & ~1) + 2;
}

int launch_ovr_mapped(const float* ir_vals, const uint32_t* ir_cnt, int n_genes, const int* n_genes_dev, const int* gene_map, int n_cols,
                      const illico_plan_t* plan, const illico_flags_t* flags, double* results, long long gstride, void* workspace,
                      size_t workspace_bytes, const illico_debug_t* dbg, cudaStream_t stream);

int launch_ovr(const float* ir_vals, const uint32_t* ir_cnt, int n_genes, const illico_plan_t* plan,
               const illico_flags_t* flags, double* results, long long gstride, void* workspace,
               size_t workspace_bytes, const illico_debug_t* dbg, cudaStream_t stream) {
    return launch_ovr_mapped(ir_vals, ir_cnt, n_genes, nullptr, nullptr, n_genes, plan, flags, results, gstride, workspace, workspace_bytes,
                             dbg, stream);
}

// n_genes: how many genes the staged lists can hold at most (sizes the grids); n_genes_dev / gene_map / n_cols: see OvrParams
int launch_ovr_mapped(const float* ir_vals, const uint32_t* ir_cnt, int n_genes, const int* n_genes_dev, const int* gene_map, int n_cols,
                      const illico_plan_t* plan, const illico_flags_t* flags, double* results, long long gstride, void* workspace,
                      size_t workspace_bytes, const illico_debug_t* dbg, cudaStream_t stream) {
    if (n_genes <= 0) return 0;
    int dev = 0, sms = 0;
    ILLICO_CUDA_OK(cudaGetDevice(&dev));
    ILLICO_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));

    OvrParams P;
    P.ir_vals = ir_vals; P.ir_cnt = ir_cnt; P.n_genes = n_genes; P.plan = *plan; P.flags = *flags;
    P.results = results; P.gstride = gstride;
    P.n_genes_dev = n_genes_dev; P.gene_map = gene_map; P.n_cols = n_cols;
    P.dbg_u2 = dbg ? (long long*)dbg->u2 : nullptr; P.dbg_tie = dbg ? dbg->tie_sum : nullptr;
    P.dbg_tie_exact = dbg ? (long long*)dbg->tie_exact : nullptr;

    // Fixed part: histogram / distinct table 16 KB + scalars.  Path S sorts in shared memory only up to HASH_CAP keys
    // (the hash table's footprint); what is not carved out stays L1 cache for the scattered reads of the group slots.
    const size_t fixed = (size_t)(OVR_NW * 256 + RADIX_AUX_WORDS + 8) * 4 + 32 * 8 * 2 + 8 + 64;
    P.sort_cap = HASH_CAP;
    const size_t need = fixed + (size_t)2 * HASH_CAP * 4;

    auto kern = flags->scores ? ovr_kernel<true> : ovr_kernel<false>;
    auto tkern = flags->scores ? ovr_table_kernel<true> : ovr_table_kernel<false>;
    ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    int occ = 0;
    ILLICO_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, OVR_THREADS, need));
    if (occ < 1) { set_error("ovr_kernel does not fit: %zu bytes of shared memory", need); return 1; }
    int grid = sms * occ;
    if (grid > n_genes) grid = n_genes;
    const size_t slab_q = ovr_slab_qwords(plan);
    // workspace head: the list of genes left to the general kernel
    const size_t head = (((size_t)n_genes + 64) * sizeof(int) + 255) & ~(size_t)255;
    if (workspace_bytes < head + slab_q * 8) { set_error("rank workspace too small: %zu bytes", workspace_bytes); return 1; }
    int* todo_count = reinterpret_cast<int*>(workspace);
    int* todo = todo_count + 16;
    workspace = reinterpret_cast<char*>(workspace) + head;
    workspace_bytes -= head;
    if ((size_t)grid * slab_q * 8 > workspace_bytes) {
        grid = (int)(workspace_bytes / (slab_q * 8));
        if (grid < 1) { set_error("rank workspace too small: %zu bytes", workspace_bytes); return 1; }
    }
    P.slab = (unsigned long long*)workspace; P.slab_qwords = (long long)slab_q;
    P.table_rec = nullptr; P.table_rec_stride = 0;
    if (flags->group_sums == nullptr) {
        P.todo = todo; P.todo_count = todo_count;
        ILLICO_CUDA_OK(cudaMemsetAsync(todo_count, 0, sizeof(int), stream));
        int tocc = 0;
        ILLICO_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tocc, tkern, T_THREADS, 0));
        if (tocc > T_MAX_CTAS_PER_SM) tocc = T_MAX_CTAS_PER_SM;
        int tgrid = sms * (tocc > 0 ? tocc : 1);
        if (tgrid > n_genes) tgrid = n_genes;
        // segment-record area of the table kernel: behind the general kernel's slabs (both kernels may be resident)
        const size_t slabs = ((size_t)grid * slab_q * 8 + 255) & ~(size_t)255;
        const size_t rec_cta = ovr_table_rec_bytes(plan);
        if (workspace_bytes >= slabs + (size_t)tgrid * rec_cta) {
            P.table_rec = reinterpret_cast<uint4*>(reinterpret_cast<char*>(workspace) + slabs);
            P.table_rec_stride = (long long)(rec_cta / 16);
        }
        ILLICO_LAUNCH("ovr_table_kernel", stream, tkern<<<tgrid, T_THREADS, 0, stream>>>(P));
        ILLICO_CUDA_OK(cudaGetLastError());
    } else {
        P.todo = nullptr; P.todo_count = nullptr;
    }
    ILLICO_LAUNCH("ovr_kernel", stream, kern<<<grid, OVR_THREADS, need, stream>>>(P));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace illico
