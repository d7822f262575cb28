// fused.cu -- dense one-versus-reference and one-versus-rest in ONE pass over the matrix, without staged
// non-zero lists (sm_100a).
//
// Replaces, for genes with few distinct values (raw counts, log1p of counts), the pair stage_dense + rank kernel, i.e.
// illico/ovo/dense_ovo.py:15-137 and illico/ovr/dense_ovr.py:15-80 with illico/utils/ranking.py:7-158 and
// illico/utils/math.py:64-118,168-221.
//
// Why: writing the staged lists (1.2 GB of scattered 32-byte sectors at the K562 shape) costs the staging kernel a
// quarter of its time although it is a ninth of its bytes, and the rank kernels read them back with 2-3x sector
// amplification.  When a gene has at most 12 distinct non-zero values, all a test needs from a group is its histogram
// over those values -- 12 x u16 = the 24 bytes the result occupies anyway:
//
//   OVO  2U_g = sum_t b_t (2 #{ref > v_t} + a_t) + z_g (2 npos + Z_ref),   a_t / b_t = multiplicity in control / g
//        T_g  = T_ref + sum_t [(a_t + b_t)^3 - (a_t + b_t) - (a_t^3 - a_t)] + (Z^3 - Z)
//   OVR  2R_g = sum_t b_t r2_t + z_g r2_zero,   r2_t = doubled mid-rank of v_t among all cells (from sum_g b_t)
//
// Steps (all on the caller's stream):
//   1. a few segments are staged alone (stage_dense_tma.cu) -- the control group for OVO, a 16k-cell sample for OVR --
//      and `fused_ctab_kernel` turns them into a per-gene table: distinct values ascending + multiplicities;
//   2. `fused_pass_kernel` streams the rows through a TMA ring (one producer warp issuing bulk copies, as in
//      stage_dense_tma.cu); lane = gene; non-zeros are compacted into a lane-private shared column (no divergence per
//      element) and, at the end of each group, looked up in the lane's copy of the table and counted.  Values the
//      table lacks claim a free slot of the gene's GLOBAL table with atomicCAS, so every CTA indexes a gene's values
//      the same way.  The group's histogram is written where its result will be;
//   3. a per-gene kernel turns the table into per-slot weights (OVO: 2 #{ref > v} + a; OVR: doubled mid-ranks, tie sum
//      in the reference's accumulation order), and an epilogue kernel turns each 24-byte histogram into
//      (p, U, fold change) in place, in the reference's f64 operation order (epilogue.cuh).
//   4. (round 2) one-versus-reference on raw counts: genes with up to DW = 64 distinct integer values take the WIDE table
//      instead (fused_wide_pass_kernel: counters indexed by the value, folded against the control at the end of each
//      group); which pass owns which gene is decided per tile of 256 genes by fused_mode_kernel.
// Genes that fit neither table (continuous values, negative values, NaN) are flagged, listed ON THE DEVICE after the
// epilogue (fused_list_kernel) and go through the general stage + rank path -- gene by gene when they are few, the whole
// batch when they are many; nothing is read back to the host, every launch is enqueued unconditionally and the kernels
// that find nothing to do leave at once.
#include "common.cuh"
#include "epilogue.cuh"
#include "tma.cuh"

#include <stdlib.h>

namespace illico {

// general path (stage.cu, rank_ovo.cu, rank_ovr.cu) for the genes the fused path hands back
int launch_stage_dense_list(const float* X, long long ld, int gene_lb, const int* list, const int* n_list_dev, const int* mode_dev,
                            int want_mode, const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, cudaStream_t stream);
int launch_stage_dense_tma_if(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                              uint32_t* ir_cnt, int seg_lo, int seg_hi, cudaStream_t stream, int segs_per_cta_req,
                              const int* mode_dev, int want_mode);
int launch_stage_csr_if(const float*, const int32_t*, const long long*, int, int, const illico_plan_t*, float*, uint32_t*, void*, size_t,
                        const int*, int, cudaStream_t);
int launch_stage_csr_list(const float*, const int32_t*, const long long*, int, int, const int*, const int*, int, int,
                          const illico_plan_t*, float*, uint32_t*, cudaStream_t);
int launch_ovo_mapped(const float*, const uint32_t*, int, const int*, const int*, int, const illico_plan_t*, const illico_flags_t*, double*,
                      long long, void*, size_t, const illico_debug_t*, cudaStream_t);
int launch_ovr_mapped(const float*, const uint32_t*, int, const int*, const int*, int, const illico_plan_t*, const illico_flags_t*, double*,
                      long long, void*, size_t, const illico_debug_t*, cudaStream_t);
bool stage_dense_tma_ok(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan);
int launch_stage_dense_tma(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                           uint32_t* ir_cnt, int seg_lo, int seg_hi, cudaStream_t stream, int segs_per_cta = 0);

namespace {

constexpr int FUSED_WARPS = 8;
constexpr int FUSED_LANES = FUSED_WARPS * 32;      // genes per CTA (lane = gene)
constexpr int FUSED_THREADS = FUSED_LANES + 32;    // + one producer warp
constexpr int DCAP = 12;                           // table slots per gene = u16 counters in a 24-byte record
constexpr long long PAIR_MAX = 208063;             // above it an OVO pair's tie sum can pass 2^53 (ordered replay needed)

// Per-gene tables, structure-of-arrays over the batch's genes (lane = gene accesses are coalesced).
struct Gtab {
    float* key;                // [DCAP][bs]  slot values (> 0; 0 = free slot); the staged sample's values come first, ascending
    uint32_t* mult;            // [DCAP][bs]  OVO: multiplicity in the control; OVR: multiplicity among all cells
    uint32_t* wgt;             // [DCAP][bs]  OVO: 2 #{ref > v} + a; OVR: doubled mid-rank
    double* fval;              // [DCAP][bs]  f(value) for the fold change
    uint32_t* nnz;             // [bs]        OVO: control non-zeros; OVR: doubled mid-rank of the zero block
    unsigned long long* tie;   // [bs]        OVO: sum over control runs of a^3 - a; OVR: f64 bits of the gene's tie correction
    double* sum;               // [bs]        OVO: sum of f(x) over the control; OVR: over all cells
    int* n_bad;                // [16]        control block: [0] genes flagged so far, [1] length of `list`, [2] hand-back mode
    int* list;                 // [bs]        the genes handed back to the general path (built on the device after the pass)
    int* cmap;                 // [bs]        CSR hand-back: position of a gene in `list`, -1 when it is not on it
    unsigned char* bad;        // [bs]        1 = the gene takes the general path
    unsigned char* cls;        // [bs]        what the table step found: CLS_NARROW | CLS_IDENT | CLS_WANTS_WIDE
    unsigned char* mode;       // [bs]        0 = 12-slot histogram records (fused_pass_kernel), 1 = wide table (fused_wide_pass_kernel)
    uint32_t* wm;              // [DW/2][bs]  wide table: multiplicity of the integer values 2 q + 1 | 2 q + 2 (16 bits each) in the control
    double* gc;                // [GC_N][Gs]  per-group constants of the p-value (fused_group_kernel)
    int Gs;                    //             groups, padded to a multiple of 64
};
constexpr int DW = 64;                                // wide table: integer counts 1 .. DW, indexed by value
constexpr int CLS_NARROW = 1, CLS_IDENT = 2, CLS_WANTS_WIDE = 4;
constexpr int WIDE_FROM = 11;                         // control tables this full go wide when they can (the other groups add values)
constexpr int HB_NONE = 0, HB_LIST = 1, HB_ALL = 2;   // hand-back modes (control block [2])
constexpr int GC_MU = 0, GC_NRNT = 1, GC_PROD12 = 2, GC_DENOM = 3, GC_INV_NT = 4, GC_N = 5;

size_t gtab_bytes(int b, int G) {
    const size_t bs = (size_t)((b + 63) & ~63), Gs = (size_t)((G + 63) & ~63);
    return bs * ((size_t)DCAP * 20 + 4 + 8 + 8 + 1 + 8 + 2 + (size_t)DW * 2) + Gs * 8 * GC_N + 1024;
}
Gtab gtab_carve(void* ws, int b, int G) {
    const size_t bs = (size_t)((b + 63) & ~63), Gs = (size_t)((G + 63) & ~63);
    char* p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    Gtab c;
    c.Gs = (int)Gs;
    c.gc = reinterpret_cast<double*>(p); p += Gs * 8 * GC_N;
    c.fval = reinterpret_cast<double*>(p); p += bs * 8 * DCAP;
    c.tie = reinterpret_cast<unsigned long long*>(p); p += bs * 8;
    c.sum = reinterpret_cast<double*>(p); p += bs * 8;
    c.key = reinterpret_cast<float*>(p); p += bs * 4 * DCAP;
    c.mult = reinterpret_cast<uint32_t*>(p); p += bs * 4 * DCAP;
    c.wgt = reinterpret_cast<uint32_t*>(p); p += bs * 4 * DCAP;
    c.nnz = reinterpret_cast<uint32_t*>(p); p += bs * 4;
    c.n_bad = reinterpret_cast<int*>(p); p += 64;
    c.list = reinterpret_cast<int*>(p); p += bs * 4;
    c.cmap = reinterpret_cast<int*>(p); p += bs * 4;
    c.wm = reinterpret_cast<uint32_t*>(p); p += bs * 2 * DW;
    c.bad = reinterpret_cast<unsigned char*>(p); p += bs;
    c.cls = reinterpret_cast<unsigned char*>(p); p += bs;
    c.mode = reinterpret_cast<unsigned char*>(p);
    return c;
}

// ---- 1. per-gene tables from the staged segments [seg_lo, seg_hi) -------------------------------------------------
// One warp per gene; lane t holds table slot t in registers.  Equal values of a 32-value load are merged with
// match.any, their leaders are inserted one after the other.
// Two tables are tried at once.  NARROW: at most DCAP distinct values of any kind (keys + multiplicities, slots in
// ascending value order).  WIDE (wide_on, one-versus-reference only): every value is an integer count in 1 .. DW, the
// table is indexed by the value itself (wm[v - 1] = multiplicity) and holds no keys.  What the gene qualifies for goes to
// gt.cls; fused_mode_kernel turns that into the gene's mode.
constexpr float ROUND_MAGIC = 12582912.0f;            // 1.5 * 2^23: v + MAGIC has the integer nearest to v in its low mantissa bits
constexpr uint32_t ROUND_MAGIC_BITS = 0x4B400000u;
// bin (value - 1) of an integer count in 1 .. DW; anything else (zero, negative, fractional, huge, NaN) gives ok = false
__device__ __forceinline__ uint32_t count_bin(float v, bool& ok) {
    const float tt = __fadd_rn(v, ROUND_MAGIC);
    const uint32_t q1 = __float_as_uint(tt) - (ROUND_MAGIC_BITS + 1u);
    ok = (__fsub_rn(tt, ROUND_MAGIC) == v) && (q1 < (uint32_t)DW);
    return q1;
}

__global__ void __launch_bounds__(256) fused_ctab_kernel(const float* __restrict__ ir_vals, const uint32_t* __restrict__ ir_cnt,
                                                         int b, const illico_plan_t pl, int seg_lo, int seg_hi, int is_log1p,
                                                         Gtab gt, int bs, int wide_on) {
    __shared__ uint32_t wh[8][DW];
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int S = pl.n_segments;
    for (int j = warp; j < b; j += nwarps) {
        float mykey = 0.0f;
        uint32_t mycnt = 0;
        int D = 0;
        bool nbad = false;                 // the narrow table does not hold the gene
        bool general = false;              // a negative value or a NaN: neither table
        for (int s = seg_lo; s < seg_hi && !nbad; ++s) {
            const int c = (int)ir_cnt[(long long)j * S + s];
            const float* src = ir_vals + (long long)j * pl.slot_cap + pl.seg_base[s];
            for (int i0 = 0; i0 < c && !nbad; i0 += 32) {
                const bool valid = i0 + lane < c;
                const float v = valid ? src[i0 + lane] : 0.0f;
                if (__any_sync(FULL, valid && !(v > 0.0f))) { nbad = general = true; break; }   // negative or NaN: general path
                const unsigned same = __match_any_sync(FULL, __float_as_uint(v));
                const bool leader = valid && (__ffs(same) - 1 == lane);
                const uint32_t n = (uint32_t)__popc(same);
                unsigned leaders = __ballot_sync(FULL, leader);
                while (leaders) {
                    const int l = __ffs(leaders) - 1;
                    leaders &= leaders - 1;
                    const float vv = __shfl_sync(FULL, v, l);
                    const uint32_t nn = __shfl_sync(FULL, n, l);
                    const unsigned hit = __ballot_sync(FULL, lane < D && mykey == vv);
                    if (hit) {
                        if (lane == __ffs(hit) - 1) mycnt += nn;
                    } else if (D < DCAP) {
                        if (lane == D) { mykey = vv; mycnt = nn; }
                        ++D;
                    } else {
                        nbad = true;
                        break;
                    }
                }
            }
        }
        // ---- wide table: the multiplicities by value.  A gene the narrow table holds gets it from that table; one it
        // does not hold has its control values read once more (they are in L2).
        bool ident = wide_on != 0 && !general;
        if (ident) {
            wh[wl][lane] = 0u;
            wh[wl][lane + 32] = 0u;
            __syncwarp();
            if (!nbad) {
                bool okv = true;
                const uint32_t q1 = count_bin(mykey, okv);
                if (__any_sync(FULL, lane < D && !okv)) ident = false;
                else if (lane < D) wh[wl][q1] = mycnt;
            } else {
                for (int s = seg_lo; s < seg_hi && ident; ++s) {
                    const int c = (int)ir_cnt[(long long)j * S + s];
                    const float* src = ir_vals + (long long)j * pl.slot_cap + pl.seg_base[s];
                    for (int i0 = 0; i0 < c; i0 += 32) {
                        const bool valid = i0 + lane < c;
                        const float v = valid ? src[i0 + lane] : 0.0f;
                        bool okv;
                        const uint32_t q1 = count_bin(v, okv);
                        if (__any_sync(FULL, valid && !okv)) { ident = false; break; }
                        const unsigned same = __match_any_sync(FULL, __float_as_uint(v));
                        if (valid && (__ffs(same) - 1 == lane)) wh[wl][q1] += (uint32_t)__popc(same);   // leaders: distinct bins
                        __syncwarp();
                    }
                }
            }
            __syncwarp();
        }
        int cls = nbad ? 0 : CLS_NARROW;
        if (ident) {
            const uint32_t c0 = wh[wl][lane], c1 = wh[wl][lane + 32];
            if (__any_sync(FULL, (c0 | c1) > 0xffffu)) {
                ident = false;                                        // (16-bit multiplicities in the pass's shared table)
            } else {
                // packed as the pass keeps it: word q = multiplicities of the values 2 q + 1 | 2 q + 2
                const uint32_t e0 = wh[wl][2 * lane], e1 = wh[wl][2 * lane + 1];
                gt.wm[(long long)lane * bs + j] = e0 | (e1 << 16);
                cls |= CLS_IDENT;
                if (nbad || D >= WIDE_FROM) cls |= CLS_WANTS_WIDE;
            }
        }
        __syncwarp();
        if (lane == 0) gt.cls[j] = (unsigned char)cls;
        if (nbad) continue;
        // slots in ascending value order (position = number of smaller values); the rest are free
        int pos = 0;
        for (int t = 0; t < D; ++t) pos += (__shfl_sync(FULL, mykey, t) < mykey) ? 1 : 0;
        const bool mine = lane < D;
        if (mine) { gt.key[(long long)pos * bs + j] = mykey; gt.mult[(long long)pos * bs + j] = mycnt; }
        if (lane >= D && lane < DCAP) { gt.key[(long long)lane * bs + j] = 0.0f; gt.mult[(long long)lane * bs + j] = 0u; }
        const uint32_t nnz = warp_sum<uint32_t>(mine ? mycnt : 0u);
        const unsigned long long tie = warp_sum_u64(mine ? (unsigned long long)cube_minus((long long)mycnt) : 0ull);
        const double sum = warp_sum_f64(mine ? (double)mycnt * fc_value(mykey, is_log1p) : 0.0);
        if (lane == 0) { gt.nnz[j] = nnz; gt.tie[j] = tie; gt.sum[j] = sum; }
    }
}

// Mode of every gene, per tile of FUSED_LANES genes (= one CTA column of the passes): a tile goes wide when one of its
// genes needs the wide table (too many distinct values for the narrow one, or nearly so); every gene of such a tile that
// qualifies then rides along, the others keep the narrow pass (both passes then stream the tile; raw-count matrices
// never mix the two).  Genes that fit neither table are flagged for the general path and counted.
__global__ void __launch_bounds__(256) fused_mode_kernel(int b, Gtab gt) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = (j < b) ? gt.cls[j] : 0;
    const bool tile_wide = __syncthreads_or((c & CLS_WANTS_WIDE) != 0) != 0;
    const int mode = (tile_wide && (c & CLS_IDENT)) ? 1 : 0;
    const bool bad = j < b && mode == 0 && !(c & CLS_NARROW);
    if (j < b) { gt.mode[j] = (unsigned char)mode; gt.bad[j] = bad ? 1 : 0; }
    const int nb = __syncthreads_count(bad);
    if (threadIdx.x == 0 && nb) atomicAdd(gt.n_bad, nb);
}

// ---- 2. the pass over the matrix ------------------------------------------------------------------------------------
template <int ROWS, int STAGES, int BUF>
struct FusedLayout {
    static constexpr int ROW_BYTES = FUSED_LANES * 4;
    static constexpr int STAGE_BYTES = ROWS * ROW_BYTES;
    static constexpr int RING_OFF = 0;
    static constexpr int NZ_OFF = STAGES * STAGE_BYTES;            // float [BUF][256]   compacted non-zeros of the group
    static constexpr int KEY_OFF = NZ_OFF + BUF * ROW_BYTES;       // float [DCAP][256]  the lane's copy of the gene's table
    static constexpr int HIST_OFF = KEY_OFF + DCAP * ROW_BYTES;    // u16   [DCAP][256]  multiplicity in the current group
    static constexpr int BAR_OFF = HIST_OFF + DCAP * FUSED_LANES * 2;
    static constexpr int BYTES = BAR_OFF + 2 * STAGES * 8;
};

// OVO = true: the control group's rows are skipped (its table is what the others are ranked against).
// OVO = false: every row is streamed and the CTA's share of each gene's whole histogram is added to gt.mult.
template <int ROWS, int STAGES, int BUF, int MINB, bool OVO>
__global__ void __launch_bounds__(FUSED_THREADS, MINB) fused_pass_kernel(const float* __restrict__ X, long long ld, int gene_lb,
                                                                         int b, const illico_plan_t pl, int groups_per_cta,
                                                                         Gtab gt, int bs, unsigned long long* __restrict__ rec,
                                                                         long long gstride, int share_1024) {
    using L = FusedLayout<ROWS, STAGES, BUF>;
    static_assert(32 % ROWS == 0 && BUF > ROWS, "layout");
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t smem_a = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = smem_a + L::BAR_OFF;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int G = pl.n_groups, ref = OVO ? pl.ref_group : -1;
    const int gy0 = blockIdx.y * groups_per_cta, gy1 = min(G, gy0 + groups_per_cta);
    const int p_begin = pl.seg_pos[pl.group_seg[gy0]], p_end = pl.seg_pos[pl.group_seg[gy1]];
    const bool ref_in = ref >= gy0 && ref < gy1;
    const int ref_p0 = ref_in ? pl.seg_pos[pl.group_seg[ref]] : 0;
    const int ref_len = ref_in ? pl.seg_pos[pl.group_seg[ref + 1]] - ref_p0 : 0;
    const int nv = p_end - p_begin - ref_len;                   // rows this CTA streams (the control's are skipped)
    const int g0 = blockIdx.x * FUSED_LANES;
    const uint32_t row_bytes = (uint32_t)min(FUSED_LANES, (b - g0 + 3) & ~3) * 4u;
    if (nv <= 0) return;
    // every gene of this CTA was already handed back by the table step (continuous data: all of them): nothing to stream.
    // The decision is the CTA's own, taken on the device: the host enqueues the pass without knowing.
    // Likewise when the table step flagged more genes than are handed back one by one: the whole batch will be redone by
    // the general path (fused_list_kernel takes the same decision from the same count), so the pass has nothing to add.
    if ((long long)gt.n_bad[0] * 1024 > (long long)b * share_1024) return;
    if (__syncthreads_and(t >= FUSED_LANES || g0 + t >= b || gt.bad[g0 + t] != 0 || gt.mode[g0 + t] != 0)) return;

    if (t == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(bars + 8 * i, 1);
            mbar_init(bars + 8 * (STAGES + i), FUSED_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (w == FUSED_WARPS) {
        // ---------------- producer warp (as in stage_dense_tma.cu); virtual row i -> position in perm, control skipped
        // (reading the permutation two groups ahead, or the group boundaries one group ahead, measured 5-10 % slower)
        uint64_t policy;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
        const char* base = reinterpret_cast<const char*>(X + gene_lb + g0);
        const unsigned long long ldb = (unsigned long long)ld * 4ull;
        auto row_of = [&](int i) {
            int p = p_begin + i;
            if (ref_in && p >= ref_p0) p += ref_len;
            return pl.perm[p];
        };
        int myrow = (lane < nv) ? row_of(lane) : 0;
        int k = 0;
        for (int i0 = 0; i0 < nv; i0 += 32) {
            const int nxt = (i0 + 32 + lane < nv) ? row_of(i0 + 32 + lane) : 0;
            const int nrows = min(32, nv - i0);
#pragma unroll
            for (int q = 0; q < 32 / ROWS; ++q, ++k) {
                if (q * ROWS >= nrows) break;
                const int slot = k % STAGES;
                const uint32_t full = bars + 8 * slot, empty = bars + 8 * (STAGES + slot);
                mbar_wait(empty, ((k / STAGES) & 1) ^ 1);
                const int rows_here = min(ROWS, nrows - q * ROWS);
                if (lane == 0) mbar_expect_tx(full, (uint32_t)rows_here * row_bytes);
                __syncwarp();
                const int u = lane - q * ROWS;
                if (u >= 0 && u < rows_here)
                    bulk_g2s(smem_a + L::RING_OFF + slot * L::STAGE_BYTES + u * L::ROW_BYTES,
                             base + (unsigned long long)(uint32_t)myrow * ldb, row_bytes, full, policy);
            }
            myrow = nxt;
        }
        return;
    }

    // ---------------- consumer warps: lane = gene.  All shared-memory traffic below uses explicit 32-bit shared
    // addresses (entry q of the lane's column of an array lives at array + q * 1024 + 4 * t).
    const int j = g0 + t;
    const bool in_batch = j < b;
    const uint32_t keys_a = smem_a + L::KEY_OFF + t * 4;
    const uint32_t hist_a = smem_a + L::HIST_OFF + t * 2;
    const uint32_t nz_a = smem_a + L::NZ_OFF + t * 4;
    auto lds_f = [](uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; };
    auto sts_f = [](uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); };
    auto lds_h = [](uint32_t a) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a)); return (uint32_t)v; };
    auto sts_h = [](uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory"); };
    const bool mine = in_batch && gt.bad[j] == 0 && gt.mode[j] == 0;   // (wide-table genes belong to fused_wide_pass_kernel)
    bool bad = !mine;
    float* gkey = gt.key + (in_batch ? j : 0);
    // The gene's table is global: slots are filled in order, the sample's values first; every slot already taken is
    // cached in the lane's shared column, later ones are found (or claimed) on a miss.
    int D = 0;
#pragma unroll
    for (int q = 0; q < DCAP; ++q) {
        const float kq = bad ? 0.0f : __ldcg(gkey + (long long)q * bs);
        if (kq != 0.0f) D = q + 1;
        sts_f(keys_a + q * L::ROW_BYTES, kq);
        sts_h(hist_a + q * (FUSED_LANES * 2), 0u);
    }
    uint32_t Hacc[OVO ? 1 : DCAP];                            // OVR: this CTA's share of the gene's whole histogram
#pragma unroll
    for (int q = 0; q < (OVO ? 1 : DCAP); ++q) Hacc[q] = 0u;
    uint32_t wr = nz_a;                                       // shared address of the lane's next free nz entry

    // looks the buffered non-zeros up in the lane's table and bumps the group's histogram
    auto drain = [&]() {
        const uint32_t mywr = bad ? nz_a : wr;
        const uint32_t maxwr = __reduce_max_sync(FULL, mywr - nz_a);
        for (uint32_t o = 0; o < maxwr; o += L::ROW_BYTES) {
            if (nz_a + o < mywr) {
                const float v = lds_f(nz_a + o);
                // counts: value c usually sits in slot c - 1; otherwise scan for equality
                int q = (int)v - 1;
                if (!(q >= 0 && q < D && lds_f(keys_a + q * L::ROW_BYTES) == v)) {
                    q = 0;
                    while (q < D && lds_f(keys_a + q * L::ROW_BYTES) != v) ++q;
                    if (q == D) {
                        // not cached: find or claim the value's slot in the gene's global table
                        int slot = -1;
                        if (v > 0.0f) {
                            for (int r = D; r < DCAP && slot < 0; ++r) {
                                const unsigned old = atomicCAS(reinterpret_cast<unsigned*>(gkey + (long long)r * bs), 0u,
                                                               __float_as_uint(v));
                                const float kv = old ? __uint_as_float(old) : v;
                                sts_f(keys_a + r * L::ROW_BYTES, kv);
                                D = r + 1;
                                if (kv == v) slot = r;
                            }
                        }
                        if (slot < 0) { bad = true; q = 0; }   // a 13th distinct value, a negative one or a NaN: general path
                        else q = slot;
                    }
                }
                const uint32_t ha = hist_a + q * (FUSED_LANES * 2);
                sts_h(ha, lds_h(ha) + 1u);
            }
        }
        wr = nz_a;
    };
    // record of group g = its histogram over the gene's table, 12 x u16 = 24 bytes, written where the result goes
    auto close_group = [&](int g) {
        drain();
        unsigned long long wds[3] = {0ull, 0ull, 0ull};
#pragma unroll
        for (int q = 0; q < DCAP; ++q) {
            const uint32_t bq = lds_h(hist_a + q * (FUSED_LANES * 2));
            wds[q >> 2] |= (unsigned long long)bq << (16 * (q & 3));
            if (!OVO) Hacc[OVO ? 0 : q] += bq;
            sts_h(hist_a + q * (FUSED_LANES * 2), 0u);
        }
        if (!bad) {
            unsigned long long* o = rec + (long long)g * gstride + (long long)j * 3;
            o[0] = wds[0]; o[1] = wds[1]; o[2] = wds[2];
        }
    };
    auto group_end_v = [&](int gg) { return pl.seg_pos[pl.group_seg[gg + 1]] - p_begin - ((ref_in && gg > ref) ? ref_len : 0); };
    int g = (gy0 == ref) ? gy0 + 1 : gy0;
    int gend = group_end_v(g);

    auto append = [&](float v) {
        asm volatile("{ .reg .pred p; setp.neu.f32 p, %1, 0f00000000; @p st.shared.f32 [%0], %1; @p add.u32 %0, %0, %2; }"
                     : "+r"(wr)
                     : "f"(v), "n"(L::ROW_BYTES)
                     : "memory");
    };
    const uint32_t ring_a = smem_a + L::RING_OFF + t * 4;
    const uint32_t wr_limit = nz_a + (uint32_t)(BUF - ROWS) * L::ROW_BYTES;
    int slot = 0;
    uint32_t parity = 0;
    for (int i = 0; i < nv; i += ROWS) {
        mbar_wait(bars + 8 * slot, parity);
        const uint32_t src = ring_a + slot * L::STAGE_BYTES;
        if (i + ROWS <= gend) {
            // the whole stage lies inside the current group (the usual case): independent shared loads first
            float v[ROWS];
#pragma unroll
            for (int u = 0; u < ROWS; ++u) v[u] = lds_f(src + u * L::ROW_BYTES);
#pragma unroll
            for (int u = 0; u < ROWS; ++u) append(v[u]);
        } else {
            const int nr = min(ROWS, nv - i);
#pragma unroll 1
            for (int u = 0; u < nr; ++u) {
                if (i + u == gend) {                                     // CTA-uniform: the next group starts here
                    close_group(g);
                    ++g;
                    if (g == ref) ++g;
                    gend = group_end_v(g);
                }
                append(lds_f(src + u * L::ROW_BYTES));
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (STAGES + slot));
        if (++slot == STAGES) { slot = 0; parity ^= 1u; }
        if (__any_sync(FULL, wr > wr_limit)) drain();                     // keep room for one more stage
    }
    close_group(g);
    if (mine) {
        if (bad) {
            gt.bad[j] = 1;
        } else if (!OVO) {
#pragma unroll
            for (int q = 0; q < (OVO ? 1 : DCAP); ++q)
                if (Hacc[q]) atomicAdd(gt.mult + (long long)q * bs + j, Hacc[q]);
        }
    }
}

// ---- 2b. the pass over the matrix with the wide table (integer counts 1 .. DW; one-versus-reference) --------------------
// Same TMA ring and lane = gene layout as fused_pass_kernel.  The table is indexed by the value itself, so an element costs
// no look-up: the lane's own 16-bit counter of that value is bumped in shared memory (plain LDS / STS, laid out so that a
// warp never meets a bank conflict).  A 24-byte record cannot hold DW counters, so the histogram is folded
// at the end of each group against the control's multiplicities, which the CTA keeps in shared memory in the same packed
// layout: with a_t the control's multiplicity of value t + 1 and b_t the group's,
//      2U_nz = sum_t b_t (2 #{control > t + 1} + a_t),   T_nz = sum_t [(a_t + b_t)^3 - (a_t + b_t) - (a_t^3 - a_t)],
// and the record is (2U_nz | non-zeros << 40, T_nz, sum of the values) -- all exact integers.  Values the control does not
// have need no special case (a_t = 0).  A value that is not an integer count in 1 .. DW flags the gene for the general path.
// The grid is persistent (CTA = one tile of 256 genes, walking every GY-th chunk of groups): the launch is enqueued
// without knowing whether any gene is wide, a no costs 296 CTA starts, and the control's table is loaded once per CTA.
template <int ROWS, int STAGES>
struct WideLayout {
    static constexpr int ROW_BYTES = FUSED_LANES * 4;
    static constexpr int STAGE_BYTES = ROWS * ROW_BYTES;
    static constexpr int RING_OFF = 0;
    static constexpr int HIST_OFF = STAGES * STAGE_BYTES;          // u16 [DW][256]      the group's count of each value
    static constexpr int ATAB_OFF = HIST_OFF + (DW / 2) * ROW_BYTES;   // u32 [DW / 2][256]  the control's counts of values 2 q + 1 | 2 q + 2
    static constexpr int BAR_OFF = ATAB_OFF + (DW / 2) * ROW_BYTES;
    static constexpr int BYTES = BAR_OFF + 2 * STAGES * 8;
};
constexpr int WIDE_M_SHIFT = 40;                                   // 2U_nz < 2^37 (pairs of at most PAIR_MAX cells)
static_assert(DW % 2 == 0 && DW <= 64, "packed layout: two 16-bit bins per word; the table step keeps two bins per lane");

template <int ROWS, int STAGES, int MINB>
__global__ void __launch_bounds__(FUSED_THREADS, MINB) fused_wide_pass_kernel(const float* __restrict__ X, long long ld, int gene_lb,
                                                                              int b, const illico_plan_t pl, int groups_per_cta,
                                                                              Gtab gt, int bs, unsigned long long* __restrict__ rec,
                                                                              long long gstride, int share_1024) {
    using L = WideLayout<ROWS, STAGES>;
    static_assert(32 % ROWS == 0, "layout");
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t smem_a = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = smem_a + L::BAR_OFF;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int G = pl.n_groups, ref = pl.ref_group;
    const int g0 = blockIdx.x * FUSED_LANES;
    const uint32_t row_bytes = (uint32_t)min(FUSED_LANES, (b - g0 + 3) & ~3) * 4u;
    if ((long long)gt.n_bad[0] * 1024 > (long long)b * share_1024) return;   // the general path redoes the batch
    if (__syncthreads_and(t >= FUSED_LANES || g0 + t >= b || gt.bad[g0 + t] != 0 || gt.mode[g0 + t] != 1)) return;

    if (t == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(bars + 8 * i, 1);
            mbar_init(bars + 8 * (STAGES + i), FUSED_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int n_chunks = (G + groups_per_cta - 1) / groups_per_cta;
    // rows of chunk c: the positions of its groups, the control's skipped
    struct Chunk { int gy0, p_begin, ref_p0, ref_len, nv; bool ref_in; };
    auto chunk_of = [&](int c) {
        Chunk k;
        k.gy0 = c * groups_per_cta;
        const int gy1 = min(G, k.gy0 + groups_per_cta);
        k.p_begin = pl.seg_pos[pl.group_seg[k.gy0]];
        const int p_end = pl.seg_pos[pl.group_seg[gy1]];
        k.ref_in = ref >= k.gy0 && ref < gy1;
        k.ref_p0 = k.ref_in ? pl.seg_pos[pl.group_seg[ref]] : 0;
        k.ref_len = k.ref_in ? pl.seg_pos[pl.group_seg[ref + 1]] - k.ref_p0 : 0;
        k.nv = p_end - k.p_begin - k.ref_len;
        return k;
    };

    if (w == FUSED_WARPS) {
        // ---------------- producer warp (as in fused_pass_kernel); the ring's stage counter runs on across chunks
        uint64_t policy;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
        const char* base = reinterpret_cast<const char*>(X + gene_lb + g0);
        const unsigned long long ldb = (unsigned long long)ld * 4ull;
        int k = 0;
        for (int c = blockIdx.y; c < n_chunks; c += gridDim.y) {
            const Chunk ch = chunk_of(c);
            auto row_of = [&](int i) {
                int p = ch.p_begin + i;
                if (ch.ref_in && p >= ch.ref_p0) p += ch.ref_len;
                return pl.perm[p];
            };
            int myrow = (lane < ch.nv) ? row_of(lane) : 0;
            for (int i0 = 0; i0 < ch.nv; i0 += 32) {
                const int nxt = (i0 + 32 + lane < ch.nv) ? row_of(i0 + 32 + lane) : 0;
                const int nrows = min(32, ch.nv - i0);
#pragma unroll
                for (int q = 0; q < 32 / ROWS; ++q, ++k) {
                    if (q * ROWS >= nrows) break;
                    const int slot = k % STAGES;
                    const uint32_t full = bars + 8 * slot, empty = bars + 8 * (STAGES + slot);
                    mbar_wait_backoff(empty, ((k / STAGES) & 1) ^ 1);
                    const int rows_here = min(ROWS, nrows - q * ROWS);
                    if (lane == 0) mbar_expect_tx(full, (uint32_t)rows_here * row_bytes);
                    __syncwarp();
                    const int u = lane - q * ROWS;
                    if (u >= 0 && u < rows_here)
                        bulk_g2s(smem_a + L::RING_OFF + slot * L::STAGE_BYTES + u * L::ROW_BYTES,
                                 base + (unsigned long long)(uint32_t)myrow * ldb, row_bytes, full, policy);
                }
                myrow = nxt;
            }
        }
        return;
    }

    // ---------------- consumer warps: lane = gene
    const int j = g0 + t;
    const bool in_batch = j < b;
    const bool mine = in_batch && gt.bad[j] == 0 && gt.mode[j] == 1;
    // counters: u16 [DW][256], bin stride 512 bytes.  Inside a bin row the 32 lanes of a warp sit in 32 different words
    // (warps 2 i and 2 i + 1 share the words of quarter i, one half each), so a warp's read-modify-write never meets a
    // bank conflict whatever the values are, and the address of bin q is one multiply-add away
    const uint32_t hist_a = smem_a + L::HIST_OFF + (uint32_t)(w >> 1) * 128u + (uint32_t)lane * 4u + (uint32_t)(w & 1) * 2u;
    const uint32_t atab_a = smem_a + L::ATAB_OFF + t * 4;     // u32 [DW / 2][256]: the control's multiplicities, two per word
    constexpr uint32_t BIN_BYTES = FUSED_LANES * 2;
    auto lds_f = [](uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; };
    auto lds_u = [](uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; };
    auto sts_u = [](uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); };
    auto lds_h = [](uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; };
    auto sts_h = [](uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); };
    // (lanes that are not `mine` count along -- their columns are private and their records are not written)
    {
        const uint32_t* wm_j = gt.wm + (in_batch ? j : 0);
#pragma unroll 8
        for (int q = 0; q < DW / 2; ++q) {
            sts_h(hist_a + (2 * q) * BIN_BYTES, 0u);
            sts_h(hist_a + (2 * q + 1) * BIN_BYTES, 0u);
            sts_u(atab_a + q * L::ROW_BYTES, mine ? __ldg(wm_j + (long long)q * bs) : 0u);
        }
    }
    bool bad = false;

    // one element: bump the 16-bit counter of its value (bin q1 = value - 1); one predicated read-modify-write, no branch
    auto take = [&](float v) {
        bool ok;
        const uint32_t q1 = count_bin(v, ok);
        const uint32_t a = hist_a + q1 * BIN_BYTES;
        asm volatile(
            "{ .reg .pred p; .reg .u32 h;\n"
            "setp.ne.u32 p, %1, 0;\n"
            "@p ld.shared.u16 h, [%0];\n"
            "@p add.u32 h, h, 1;\n"
            "@p st.shared.u16 [%0], h; }"
            ::"r"(a), "r"((uint32_t)ok) : "memory");
        bad |= !ok && v != 0.0f;                                  // not an integer count in 1 .. DW: general path
    };
    // end of group g: fold the histogram against the control's multiplicities (values descending, so that the number of
    // control values above the current one is a running sum), write the record, clear the counters
    auto close_group = [&](int g) {
        uint32_t m = 0, s1 = 0, above = 0;
        unsigned long long u2 = 0, tie = 0;
        // a, b < 2^16 (checked by the table step / the group-size limit): every product below is formed from 32-bit
        // factors, so each term is one widening multiply-add
        auto bin = [&](uint32_t ha, uint32_t a, int q) {
            const uint32_t bq = lds_h(ha);
            if (bq) {
                sts_h(ha, 0u);
                u2 += (unsigned long long)bq * (2u * above + a);
                // (a+b)^3 - (a+b) - (a^3 - a) = 3 a b (a + b) + b^3 - b
                tie += (unsigned long long)(a * bq) * (3u * (a + bq));
                tie += (unsigned long long)(bq * bq) * bq;
                s1 += bq * (uint32_t)(q + 1);
                m += bq;
            }
            above += a;
        };
#pragma unroll 4
        for (int q = DW / 2 - 1; q >= 0; --q) {                     // word q of the control's table: values 2 q + 2 | 2 q + 1
            const uint32_t ab = lds_u(atab_a + q * L::ROW_BYTES);
            bin(hist_a + (2 * q + 1) * BIN_BYTES, ab >> 16, 2 * q + 1);
            bin(hist_a + (2 * q) * BIN_BYTES, ab & 0xffffu, 2 * q);
        }
        if (mine && !bad) {
            unsigned long long* o = rec + (long long)g * gstride + (long long)j * 3;
            o[0] = u2 | ((unsigned long long)m << WIDE_M_SHIFT);
            o[1] = tie - m;
            o[2] = (unsigned long long)s1;
        }
    };

    const uint32_t ring_a = smem_a + L::RING_OFF + t * 4;
    int slot = 0;
    uint32_t parity = 0;
    for (int c = blockIdx.y; c < n_chunks; c += gridDim.y) {
        const Chunk ch = chunk_of(c);
        if (ch.nv <= 0) continue;
        auto group_end_v = [&](int gg) {
            return pl.seg_pos[pl.group_seg[gg + 1]] - ch.p_begin - ((ch.ref_in && gg > ref) ? ch.ref_len : 0);
        };
        int g = (ch.gy0 == ref) ? ch.gy0 + 1 : ch.gy0;
        int gend = group_end_v(g);
        for (int i = 0; i < ch.nv; i += ROWS) {
            mbar_wait(bars + 8 * slot, parity);
            const uint32_t src = ring_a + slot * L::STAGE_BYTES;
            if (i + ROWS <= gend) {
                float v[ROWS];
#pragma unroll
                for (int u = 0; u < ROWS; ++u) v[u] = lds_f(src + u * L::ROW_BYTES);
#pragma unroll
                for (int u = 0; u < ROWS; ++u) take(v[u]);
            } else {
                const int nr = min(ROWS, ch.nv - i);
#pragma unroll 1
                for (int u = 0; u < nr; ++u) {
                    if (i + u == gend) {                                     // CTA-uniform: the next group starts here
                        close_group(g);
                        ++g;
                        if (g == ref) ++g;
                        gend = group_end_v(g);
                    }
                    take(lds_f(src + u * L::ROW_BYTES));
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 8 * (STAGES + slot));
            if (++slot == STAGES) { slot = 0; parity ^= 1u; }
        }
        close_group(g);
    }
    if (mine && bad) gt.bad[j] = 1;
}

// ---- 3a. per-gene weights ---------------------------------------------------------------------------------------------
// Thread per gene.  Visits the gene's claimed slots in ascending value order.
// OVO: weight of slot t = 2 #{control > v_t} + a_t (rank_ovo.cu's dw); the control's sums are already in gt.
// OVR: gt.mult holds the whole gene's histogram; weight = doubled mid-rank r2 = 2 lo + c + 1 with the zero block below
//      every (positive) value, as in ovr_table_kernel (rank_ovr.cu); tie sum in the dense kernels' order
//      (illico/utils/ranking.py:31-47): zero block, then the runs ascending, sequential f64 once the exact total
//      reaches 2^53 (SURVEY.md appendix A.4).
template <bool OVO>
__global__ void __launch_bounds__(128) fused_gene_kernel(int b, const illico_plan_t pl, illico_flags_t fl, Gtab gt, int bs,
                                                         double* dbg_tie, long long* dbg_tie_exact) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b || gt.bad[j]) return;
    if (OVO && gt.mode[j] == 1) {
        // wide table: the control's own sums from its multiplicities by value (value of bin q = q + 1)
        unsigned long long nnz = 0, tie = 0, sum = 0;
        for (int q = 0; q < DW; ++q) {
            const unsigned long long c = (gt.wm[(long long)(q >> 1) * bs + j] >> (16 * (q & 1))) & 0xffffu;
            nnz += c;
            tie += (unsigned long long)cube_minus((long long)c);
            sum += c * (unsigned long long)(q + 1);
        }
        gt.nnz[j] = (uint32_t)nnz;
        gt.tie[j] = tie;
        gt.sum[j] = (double)sum;
        return;
    }
    float key[DCAP];
    int order[DCAP];
    int D = 0;
    for (int q = 0; q < DCAP; ++q) {
        const float kq = gt.key[(long long)q * bs + j];
        if (kq == 0.0f) break;
        int a = D - 1;
        while (a >= 0 && key[order[a]] > kq) { order[a + 1] = order[a]; --a; }
        key[q] = kq;
        order[a + 1] = q;
        ++D;
    }
    for (int q = D; q < DCAP; ++q) { gt.wgt[(long long)q * bs + j] = 0u; gt.fval[(long long)q * bs + j] = 0.0; }
    if (OVO) {
        unsigned long long above = 0, nnz = 0, tie = 0;                          // control values greater than the slot's
        for (int a = D - 1; a >= 0; --a) {
            const int q = order[a];
            const unsigned long long c = gt.mult[(long long)q * bs + j];
            gt.wgt[(long long)q * bs + j] = (uint32_t)(2ull * above + c);
            gt.fval[(long long)q * bs + j] = fc_value(key[q], fl.is_log1p);
            above += c;
        }
        double sum = 0.0;
        for (int a = 0; a < D; ++a) {                                            // the control's own sums, ascending
            const int q = order[a];
            const unsigned long long c = gt.mult[(long long)q * bs + j];
            nnz += c;
            tie += (unsigned long long)cube_minus((long long)c);
            sum += (double)c * gt.fval[(long long)q * bs + j];
        }
        gt.nnz[j] = (uint32_t)nnz;
        gt.tie[j] = tie;
        gt.sum[j] = sum;
        return;
    }
    const long long n = pl.n_cells;
    const bool sparse_order = fl.tie_order == ILLICO_TIES_SPARSE;                // ovr/sparse_ovr.py:83: zero block added last
    unsigned long long nnz = 0;
    for (int q = 0; q < D; ++q) nnz += gt.mult[(long long)q * bs + j];
    const long long n0 = n - (long long)nnz;
    unsigned long long lo = (unsigned long long)n0, t_exact = 0;
    double total = 0.0;
    const unsigned long long zterm = (unsigned long long)cube_minus(n0);
    double walk = sparse_order ? 0.0 : (double)(long long)zterm;                 // sequential accumulation of the runs
    for (int a = 0; a < D; ++a) {
        const int q = order[a];
        const unsigned long long c = gt.mult[(long long)q * bs + j];
        gt.wgt[(long long)q * bs + j] = (uint32_t)(2ull * lo + c + 1ull);
        const double f = fc_value(key[q], fl.is_log1p);
        gt.fval[(long long)q * bs + j] = f;
        total += (double)c * f;
        const unsigned long long t3 = (unsigned long long)cube_minus((long long)c);
        t_exact += t3;
        walk += (double)(long long)t3;
        lo += c;
    }
    double tie;
    if (sparse_order) {
        const double x = (double)n0;                                             // n0^3 - n0 in f64, as the reference forms it
        tie = __dadd_rn(((double)t_exact >= TWO53) ? walk : (double)t_exact, __dsub_rn(__dmul_rn(__dmul_rn(x, x), x), x));
    } else {
        tie = ((double)t_exact + (double)zterm >= TWO53) ? walk : (double)(t_exact + zterm);
    }
    gt.nnz[j] = (uint32_t)(n0 + 1);                                              // doubled mid-rank of the zero block
    gt.sum[j] = total;
    // the gene's tie correction, as compute_pval forms it (illico/utils/math.py:95): one division per gene, not per test
    const double tie_corr = __dsub_rn(1.0, __ddiv_rn(fl.tie_correct ? tie : 0.0, (double)(n * (n - 1) * (n + 1))));
    gt.tie[j] = (unsigned long long)__double_as_longlong(tie_corr);
    if (dbg_tie) dbg_tie[j] = tie;
    if (dbg_tie_exact) dbg_tie_exact[j] = (long long)(t_exact + zterm);
}

// ---- 3b. per-group constants of the p-value ------------------------------------------------------------------------
// Everything in compute_pval (illico/utils/math.py:95-103) that depends on the group sizes only: evaluated once per group
// with the reference's operations (int64 products, then float) instead of once per (group, gene).
template <bool OVO>
__global__ void __launch_bounds__(256) fused_group_kernel(const illico_plan_t pl, Gtab gt) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pl.n_groups) return;
    const long long n = pl.n_cells, n_t = pl.group_size[g];
    const long long n_r = OVO ? (long long)pl.group_size[pl.ref_group] : n - n_t;
    const long long nn = n_r + n_t;
    gt.gc[GC_MU * gt.Gs + g] = (double)(n_r * n_t) / 2.0;
    gt.gc[GC_NRNT * gt.Gs + g] = (double)(n_r * n_t);
    gt.gc[GC_PROD12 * gt.Gs + g] = __ddiv_rn((double)(n_r * n_t * (n_r + n_t + 1)), 12.0);
    gt.gc[GC_DENOM * gt.Gs + g] = (double)(nn * (nn - 1) * (nn + 1));
    gt.gc[GC_INV_NT * gt.Gs + g] = 1.0 / (double)n_t;
}

// ---- 3c. epilogue: 24-byte record -> (p, U, fold change), in place ----------------------------------------------------
// Thread = gene, looping over a slice of the groups; records of adjacent genes are adjacent, so every warp access is a
// contiguous 768-byte run, and the next group's record is loaded before the current one is folded.  The gene's slot
// constants (weight, control multiplicity, f(value)) sit in a private column of shared memory: in registers they would
// be spilled to the stack.  A CTA none of whose genes has the launch's record kind leaves before any other load.
// Narrow fold: slots past the warp's highest non-zero counter are skipped (a uniform trip count); every sum is an exact
// integer below 2^53 and reordered as such, while the f64 `sum` keeps its order (ascending slot, zero counts add
// nothing).  The fold change is a ratio of means compared at 1e-10: its divisions by the group sizes are multiplications
// by precomputed reciprocals; everything that feeds the p-value keeps the reference's IEEE operations.
constexpr int EPI_GROUPS = 16;   // groups per thread
constexpr int EPI_THREADS = 256;
struct __align__(16) EpiSlot {
    uint32_t wgt;   // OVO: 2 #{control > v} + a; OVR: doubled mid-rank
    uint32_t a;     // OVO: multiplicity in the control
    double fval;    // f(value) for the fold change
};
constexpr int EPI_SMEM = DCAP * EPI_THREADS * (int)sizeof(EpiSlot);   // 48 KB: 4 CTAs per SM
// SCORE: also writes the score plane (illico_flags_t::scores); a separate instantiation, so that the default call's
// epilogue is the same code as without the plane.
template <bool OVO, bool WIDE, bool SCORE>
__global__ void __launch_bounds__(EPI_THREADS, 4) fused_epilogue_kernel(int b, const illico_plan_t pl, const illico_flags_t fl, Gtab gt,
                                                                     int bs, double* __restrict__ results, long long gstride,
                                                                     int share_1024) {
    extern __shared__ __align__(128) unsigned char smem[];
    EpiSlot* const cst = reinterpret_cast<EpiSlot*>(smem) + threadIdx.x;   // slot q of this thread's gene: cst[q * EPI_THREADS]
    __shared__ double gcs[GC_N][EPI_GROUPS];
    __shared__ int nts[EPI_GROUPS];
    // the batch is being handed back as a whole (the table step flagged too many genes): nothing here will be kept
    if ((long long)gt.n_bad[0] * 1024 > (long long)b * share_1024) return;
    // WIDE: the genes of the wide table, whose record is (2U_nz | non-zeros << 40, T_nz, sum) and not a histogram.
    // The other genes stay in the loop without loads or stores: the narrow fold's trip count is a warp vote.
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = j < b && !gt.bad[j] && (gt.mode[j] == 1) == WIDE;
    if (!__syncthreads_or(live)) return;
    const int G = pl.n_groups, ref = pl.ref_group;
    const int ga = blockIdx.y * EPI_GROUPS, gb = min(G, ga + EPI_GROUPS);
    if (threadIdx.x < GC_N * EPI_GROUPS) {
        const int c = threadIdx.x / EPI_GROUPS, k = threadIdx.x % EPI_GROUPS;
        if (ga + k < gb) gcs[c][k] = gt.gc[c * gt.Gs + ga + k];
    } else if (threadIdx.x < GC_N * EPI_GROUPS + EPI_GROUPS) {
        const int k = threadIdx.x - GC_N * EPI_GROUPS;
        if (ga + k < gb) nts[k] = pl.group_size[ga + k];
    }
    __syncthreads();
    if (live && !WIDE) {
#pragma unroll 4
        for (int q = 0; q < DCAP; ++q)
            cst[q * EPI_THREADS] = {gt.wgt[(long long)q * bs + j], OVO ? gt.mult[(long long)q * bs + j] : 0u, gt.fval[(long long)q * bs + j]};
    }
    const long long n = pl.n_cells;
    const double cc = fl.use_continuity ? 0.5 : 0.0;
    const long long g_nnz = live ? gt.nnz[j] : 0;            // OVO: control non-zeros; OVR: doubled mid-rank of the zero block
    const unsigned long long g_tie = live ? gt.tie[j] : 0;   // OVO: control tie term; OVR: f64 bits of the gene's tie correction
    const double g_sum = live ? gt.sum[j] : 0.0;             // OVO: control sum; OVR: whole-gene sum
    const long long n_ref = OVO ? (long long)pl.group_size[ref] : 0;
    const double ovr_tie_corr = __longlong_as_double((long long)g_tie);
    // OVO: the control's mean is a per-gene constant
    const double ovo_rsum = (OVO && live) ? (fl.group_sums ? fl.group_sums[(long long)ref * b + j] : g_sum) : 0.0;
    const double ovo_mean_r = OVO ? ovo_rsum / (double)n_ref : 0.0;
    const double ovo_inv_mean_r = 1.0 / ovo_mean_r;
    const unsigned long long* rec = reinterpret_cast<const unsigned long long*>(results) + (long long)j * 3;
    unsigned long long nx0 = 0, nx1 = 0, nx2 = 0;           // the next group's record
    if (live) { nx0 = rec[(long long)ga * gstride]; nx1 = rec[(long long)ga * gstride + 1]; nx2 = rec[(long long)ga * gstride + 2]; }
    for (int g = ga; g < gb; ++g) {
        const unsigned long long w0 = nx0, w1 = nx1, w2 = nx2;
        if (live && g + 1 < gb) {
            const unsigned long long* r = rec + (long long)(g + 1) * gstride;
            nx0 = r[0]; nx1 = r[1]; nx2 = r[2];
        }
        const int k = g - ga;
        const long long n_t = nts[k];
        const long long n_r = OVO ? n_ref : n - n_t;         // the sample U is reported for
        double* o = results + (long long)g * gstride + (long long)j * 3;
        if (OVO && g == ref) {
            // control row: (1, -1, fold change of the control against itself), as ovo_kernel writes it
            if (live) {
                o[0] = 1.0; o[1] = -1.0; o[2] = (ovo_mean_r == 0.0) ? INFINITY : ovo_mean_r / ovo_mean_r;
                if (SCORE) fl.scores[(long long)g * fl.score_group_stride + j] = 0.0;
            }
            continue;
        }
        unsigned long long acc = 0, tie_nz = 0;              // acc: OVO 2U without the zero block, OVR 2R without it
        uint32_t m = 0;
        double sum = 0.0;
        if (WIDE) {
            acc = w0 & ((1ull << WIDE_M_SHIFT) - 1ull);
            m = (uint32_t)(w0 >> WIDE_M_SHIFT);
            tie_nz = w1;
            sum = (double)w2;
        } else {
            int top = 0;                                     // slots to visit: up to the warp's highest non-zero counter
            if (w0) top = 4 - (__clzll((long long)w0) >> 4);
            if (w1) top = 8 - (__clzll((long long)w1) >> 4);
            if (w2) top = 12 - (__clzll((long long)w2) >> 4);
            top = __reduce_max_sync(FULL, top);
            const unsigned long long wds[3] = {w0, w1, w2};
            unsigned long long tq = 0;                       // OVO: sum of bq (3a^2 + bq (3a + bq))
#pragma unroll
            for (int q = 0; q < DCAP; ++q) {
                if (q == top) break;
                const uint32_t bq = (uint32_t)(wds[q >> 2] >> (16 * (q & 3))) & 0xffffu;
                const EpiSlot c = cst[q * EPI_THREADS];
                acc += (unsigned long long)bq * c.wgt;
                const double t = (double)bq * c.fval;
                sum = bq ? sum + t : sum;                    // (a select: f(value) can be inf, and 0 * inf is NaN)
                m += bq;
                if (OVO) {
                    // (a+b)^3 - (a+b) - (a^3 - a) = b (3a^2 + b (3a + b)) - b; the - b of every slot is - m below.
                    // 3a < 2^20 and b < 2^16, so every product is a 32 x 32 -> 64-bit multiply-add but the last.
                    const uint32_t a3 = 3u * c.a;
                    const unsigned long long x = (unsigned long long)a3 * c.a + (unsigned long long)bq * (a3 + bq);
                    tq += bq * x;
                }
            }
            if (OVO) tie_nz = tq - m;
        }
        if (!live) continue;
        const long long z_t = n_t - (long long)m;
        double p, U, fc;
        if (OVO) {
            const long long zeros_r = n_r - g_nnz;           // every control value is positive
            if (fl.group_sums) sum = fl.group_sums[(long long)g * b + j];
            const long long Z = zeros_r + z_t;
            const unsigned long long u2 = acc + (unsigned long long)(z_t * (2ll * g_nnz + zeros_r));
            const unsigned long long tie_exact = g_tie + tie_nz + (unsigned long long)cube_minus(Z);
            const double tie = (double)tie_exact;            // < 2^53: pairs of at most 208 063 cells
            U = (double)u2 * 0.5;
            const double tie_corr = __dsub_rn(1.0, __ddiv_rn(fl.tie_correct ? tie : 0.0, gcs[GC_DENOM][k]));
            p = pval_core(gcs[GC_NRNT][k], gcs[GC_MU][k], gcs[GC_PROD12][k], tie_corr, U, cc, fl.alternative);
            if (SCORE) fl.scores[(long long)g * fl.score_group_stride + j] = score_core(gcs[GC_MU][k], gcs[GC_PROD12][k], tie_corr, U);
            fc = (ovo_mean_r == 0.0) ? INFINITY : (sum * gcs[GC_INV_NT][k]) * ovo_inv_mean_r;
        } else {
            const unsigned long long R2 = acc + (unsigned long long)z_t * (unsigned long long)g_nnz;
            const long long u2 = 2 * n_r * n_t + n_t * (n_t + 1) - (long long)R2;
            U = (double)u2 * 0.5;
            p = pval_core(gcs[GC_NRNT][k], gcs[GC_MU][k], gcs[GC_PROD12][k], ovr_tie_corr, U, cc, fl.alternative);
            if (SCORE)
                fl.scores[(long long)g * fl.score_group_stride + j] = score_core(gcs[GC_MU][k], gcs[GC_PROD12][k], ovr_tie_corr, U);
            // rest-of-cells mean: exactly zero when this group holds every non-zero of the gene (the reference's total is
            // the sum of the per-group sums, so its `total - sum` is an exact 0 there; a total accumulated in another
            // order could leave an ulp and turn the +inf fold change into 1e16)
            const bool all_here = (long long)m == n - (g_nnz - 1);
            const double mu_t = sum * gcs[GC_INV_NT][k], mu_r = all_here ? 0.0 : (g_sum - sum) / (double)(n - n_t);
            fc = (mu_r == 0.0) ? INFINITY : mu_t / mu_r;
        }
        o[0] = p; o[1] = U; o[2] = fc;
    }
}

// the epilogue of the narrow records (WIDE = false) or of the wide ones, for the dense and the CSR path
template <bool OVO, bool WIDE>
int launch_fused_epilogue(int b, const illico_plan_t* plan, const illico_flags_t* flags, Gtab gt, int bs, double* results,
                          long long gstride, int share_1024, cudaStream_t stream) {
    auto epi = flags->scores ? fused_epilogue_kernel<OVO, WIDE, true> : fused_epilogue_kernel<OVO, WIDE, false>;
    const int smem = WIDE ? 0 : EPI_SMEM;
    ILLICO_CUDA_OK(cudaFuncSetAttribute(epi, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const dim3 grid((unsigned)((b + EPI_THREADS - 1) / EPI_THREADS), (unsigned)((plan->n_groups + EPI_GROUPS - 1) / EPI_GROUPS));
    ILLICO_LAUNCH(WIDE ? "fused_wide_epilogue_kernel" : "fused_epilogue_kernel", stream,
                  epi<<<grid, EPI_THREADS, smem, stream>>>(b, *plan, *flags, gt, bs, results, gstride, share_1024));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

// ===================== CSR input: the same histograms, built in shared memory ==========================================
// Replaces, for count-like data, stage_csr_kernel + rank kernel (illico/ovr/sparse_ovr.py:23-208,
// illico/ovo/sparse_ovo.py:22-260, illico/utils/sparse/csr.py:103-257).  One CTA per plan segment (<= 512 cells of one
// group) and gene tile: it walks the segment's CSR rows once (warp per row, coalesced index/value loads) and counts
// every stored value in a shared-memory histogram [gene][slot] (12 x u16 per gene = the 24-byte record), then writes
// the records.  No staged lists, no sort: 8 bytes read per stored value, 24 bytes written per (gene, group).
constexpr int CSRF_THREADS = 1024;
constexpr int CSRF_TILE = 8192;                    // genes per CTA: 8192 x 24 B = 192 KB of shared memory

// slot of value v in gene j's global table (claims a free slot if the value is new); -1 = the gene is handed back
__device__ __forceinline__ int gtab_slot(float* gkey, int bs, float v) {
    int q = (int)v - 1;                                                          // counts: value c sits in slot c - 1
    if (q >= 0 && q < DCAP && __ldcg(gkey + (long long)q * bs) == v) return q;
    if (!(v > 0.0f)) return -1;                                                  // negative or NaN
    for (q = 0; q < DCAP; ++q) {
        float k = __ldcg(gkey + (long long)q * bs);
        if (k == 0.0f) {
            const unsigned old = atomicCAS(reinterpret_cast<unsigned*>(gkey + (long long)q * bs), 0u, __float_as_uint(v));
            k = old ? __uint_as_float(old) : v;
        }
        if (k == v) return q;
    }
    return -1;                                                                   // a 13th distinct value
}

__global__ void fused_seed_kernel(Gtab gt, int bs, int identity) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= bs) return;
#pragma unroll
    for (int q = 0; q < DCAP; ++q) {
        gt.key[(long long)q * bs + i] = identity ? (float)(q + 1) : 0.0f;       // raw counts: slots 1 .. 12 up front
        gt.mult[(long long)q * bs + i] = 0u;
    }
    gt.bad[i] = 0;
    gt.mode[i] = 0;
    if (i == 0) *gt.n_bad = 0;
}

// records of groups cut into several segments are accumulated with atomics: they start from zero
__global__ void fused_zero_multi_kernel(int b, const illico_plan_t pl, unsigned long long* __restrict__ rec, long long gstride) {
    const int g = blockIdx.y;
    if (pl.group_seg[g + 1] - pl.group_seg[g] < 2) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * b; i += gridDim.x * blockDim.x) rec[(long long)g * gstride + i] = 0ull;
}

template <bool OVO>
__global__ void __launch_bounds__(CSRF_THREADS, 1) fused_csr_pass_kernel(const float* __restrict__ data, const int32_t* __restrict__ indices,
                                                                        const long long* __restrict__ indptr, int gene_lb, int b,
                                                                        const illico_plan_t pl, Gtab gt, int bs,
                                                                        unsigned long long* __restrict__ rec, long long gstride) {
    extern __shared__ __align__(16) uint32_t hist[];             // [genes of the tile][6]: 12 u16 counters per gene
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int s = blockIdx.y, g = pl.seg_group[s];
    const int j_lo = blockIdx.x * CSRF_TILE, ng = min(CSRF_TILE, b - j_lo);
    __shared__ int stop;
    if (t == 0) stop = 8 * *reinterpret_cast<volatile int*>(gt.n_bad) > b;   // many genes handed back: the general path redoes the batch
    for (int i = t; i < ng * 6; i += CSRF_THREADS) hist[i] = 0u;
    __syncthreads();
    if (stop) return;
    const int c_lo = gene_lb + j_lo, c_hi = c_lo + ng;
    const int p0 = pl.seg_pos[s], p1 = pl.seg_pos[s + 1];
    constexpr int NW = CSRF_THREADS / 32;
    // the warp's rows are p0 + w, p0 + w + 32, ...: their extents are fetched up front (lane k holds row k's), so the
    // perm -> indptr -> indices dependency is paid once per warp and not once per row
    long long my_e0 = 0, my_e1 = 0;
    {
        const int p = p0 + w + lane * NW;
        if (p < p1) {
            const long long r = pl.perm[p];
            my_e0 = indptr[r];
            my_e1 = indptr[r + 1];
        }
    }
    for (int p = p0 + w, k = 0; p < p1; p += NW, ++k) {
        // continuous data: every gene overflows its 12 slots within a few rows -- stop before the (slow) miss path
        // has been walked for a whole segment; the host then runs the general path
        if (8 * *reinterpret_cast<volatile int*>(gt.n_bad) > b) break;
        if (k == 32) {                                            // (segments are at most 512 cells: one round; kept general)
            const int pp = p + lane * NW;
            my_e0 = my_e1 = 0;
            if (pp < p1) { const long long r = pl.perm[pp]; my_e0 = indptr[r]; my_e1 = indptr[r + 1]; }
            k = 0;
        }
        long long e0 = __shfl_sync(FULL, my_e0, k);
        const long long e1 = __shfl_sync(FULL, my_e1, k);
        if (c_lo > 0) {                                           // first stored element of the row inside the gene window
            long long lo = e0, hi = e1;
            while (lo < hi) { const long long mid = (lo + hi) >> 1; if (indices[mid] < c_lo) lo = mid + 1; else hi = mid; }
            e0 = lo;
        }
        // four 32-element chunks per step: the index / value loads, then the table probes, are issued together
        for (long long e = e0 + lane; ; e += 128) {
            int c[4];
            float v[4], kq[4];
            // indices and values are requested together (one DRAM latency per step, not two)
#pragma unroll
            for (int u = 0; u < 4; ++u) c[u] = (e + 32 * u < e1) ? __ldcs(indices + e + 32 * u) : 0x7fffffff;
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = (e + 32 * u < e1) ? __ldcs(data + e + 32 * u) : 0.0f;
            if (__all_sync(FULL, c[0] >= c_hi)) break;            // column indices ascend inside a row
#pragma unroll
            for (int u = 0; u < 4; ++u) if (c[u] >= c_hi) v[u] = 0.0f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {                         // probe of the usual slot (counts: value c in slot c - 1)
                const int q = min(max((int)v[u] - 1, 0), DCAP - 1);
                kq[u] = (v[u] != 0.0f) ? __ldcg(gt.key + (long long)q * bs + j_lo + (c[u] - c_lo)) : 0.0f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (v[u] != 0.0f) {                               // explicitly stored zeros are zeros
                    const int jj = c[u] - c_lo;
                    int q = min(max((int)v[u] - 1, 0), DCAP - 1);
                    if (kq[u] != v[u]) q = gt.bad[j_lo + jj] ? -1 : gtab_slot(gt.key + j_lo + jj, bs, v[u]);
                    if (q >= 0) {
                        atomicAdd(&hist[jj * 6 + (q >> 1)], 1u << (16 * (q & 1)));
                    } else {                                      // hand the gene back, counted once
                        const int j = j_lo + jj;
                        const unsigned bit = 1u << (8 * (j & 3));
                        const unsigned old = atomicOr(reinterpret_cast<unsigned*>(gt.bad + (j & ~3)), bit);
                        if (!(old & bit)) atomicAdd(gt.n_bad, 1);
                    }
                }
            }
        }
    }
    __syncthreads();
    const bool multi = pl.group_seg[g + 1] - pl.group_seg[g] > 1;
    for (int jj = t; jj < ng; jj += CSRF_THREADS) {
        const int j = j_lo + jj;
        uint32_t wd[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) wd[k] = hist[jj * 6 + k];
        if (OVO && g == pl.ref_group) {
            // the control's histogram is the table's multiplicity column
#pragma unroll
            for (int q = 0; q < DCAP; ++q) {
                const uint32_t cq = (wd[q >> 1] >> (16 * (q & 1))) & 0xffffu;
                if (cq) atomicAdd(gt.mult + (long long)q * bs + j, cq);
            }
        } else if (!multi) {
            unsigned long long* o = rec + (long long)g * gstride + (long long)j * 3;
#pragma unroll
            for (int k = 0; k < 3; ++k) o[k] = (unsigned long long)wd[2 * k] | ((unsigned long long)wd[2 * k + 1] << 32);
        } else {
            uint32_t* o = reinterpret_cast<uint32_t*>(rec + (long long)g * gstride + (long long)j * 3);
#pragma unroll
            for (int k = 0; k < 6; ++k) if (wd[k]) atomicAdd(o + k, wd[k]);   // u16 pairs: no carry, a group has < 65536 cells
        }
    }
}

// one-versus-rest: the whole gene's histogram = the sum of its groups' records
__global__ void __launch_bounds__(256) fused_hist_sum_kernel(int b, int G, int groups_per_block, Gtab gt, int bs,
                                                             const unsigned long long* __restrict__ rec, long long gstride) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b || gt.bad[j]) return;
    const int ga = blockIdx.y * groups_per_block, gb = min(G, ga + groups_per_block);
    uint32_t acc[DCAP];
#pragma unroll
    for (int q = 0; q < DCAP; ++q) acc[q] = 0u;
    for (int g = ga; g < gb; ++g) {
        const unsigned long long* r = rec + (long long)g * gstride + (long long)j * 3;
        const unsigned long long wds[3] = {r[0], r[1], r[2]};
#pragma unroll
        for (int q = 0; q < DCAP; ++q) acc[q] += (uint32_t)((wds[q >> 2] >> (16 * (q & 3))) & 0xffffull);
    }
#pragma unroll
    for (int q = 0; q < DCAP; ++q)
        if (acc[q]) atomicAdd(gt.mult + (long long)q * bs + j, acc[q]);
}

// ---- hand-back, decided on the device -----------------------------------------------------------------------------------
// After the epilogue: the genes flagged during the table step or the pass, in ascending order, become `list` (and, for the
// CSR staging, cmap[gene] = position in the list).  Few of them (<= b * num / den): HB_LIST, only those are staged and ranked
// by the general path; more: HB_ALL, the list is the whole batch (the fused results are simply overwritten); none: HB_NONE,
// the kernels enqueued behind this one find an empty list and leave.  One CTA: the flags are a few kilobytes.
__global__ void __launch_bounds__(1024) fused_list_kernel(int b, Gtab gt, int num, int den, int force_all) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) base_s = 0;
    __syncthreads();
    for (int j0 = 0; j0 < b; j0 += 1024) {
        const int j = j0 + t;
        const bool flag = j < b && gt.bad[j] != 0;
        const unsigned bal = __ballot_sync(FULL, flag);
        if (lane == 0) wsum[w] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int ww = 0; ww < 32; ++ww) { const int c = wsum[ww]; if (ww < w) before += c; total += c; }
        const int base = base_s;
        if (j < b) {
            const int k = base + before + __popc(bal & ((1u << lane) - 1u));
            if (flag) gt.list[k] = j;
            gt.cmap[j] = flag ? k : -1;
        }
        __syncthreads();
        if (t == 0) base_s = base + total;
        __syncthreads();
    }
    const int n = base_s;
    const bool all = force_all || (long long)n * den > (long long)b * num;
    if (all && n > 0) {
        for (int j = t; j < b; j += 1024) { gt.list[j] = j; gt.cmap[j] = j; }
    }
    if (t == 0) {
        gt.n_bad[1] = (n == 0) ? 0 : (all ? b : n);
        gt.n_bad[2] = (n == 0) ? HB_NONE : (all ? HB_ALL : HB_LIST);
    }
}

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}
// largest share of a batch (in 1/1024) that is handed back gene by gene; above it the general path redoes the batch
int list_share_1024() {
    const char* v = getenv("ILLICO_FUSED_LIST_SHARE");
    const double f = v ? atof(v) : 0.125;
    return (int)(f * 1024.0 + 0.5);
}

thread_local float g_last_fused_ms = -1.0f;   // >= 0: the last dispatcher call of this thread enqueued a fused pass

constexpr int PASS_ROWS = 1536;          // rows a CTA of the passes streams: groups per CTA = PASS_ROWS / average group size
constexpr int OVR_SAMPLE_CELLS = 16384;  // one-versus-rest: cells staged to seed the tables

// The whole fused path for one gene batch, enqueued without a single host read-back.
// 0 = enqueued, 1 = error, -1 = not applicable (the caller runs the general path).
template <bool OVO>
int run_fused(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, const illico_flags_t* flags,
              const illico_batch_buffers_t* buf, double* results, long long gstride, const illico_debug_t* dbg,
              cudaStream_t stream) {
    g_last_fused_ms = -1.0f;
    if (env_int(OVO ? "ILLICO_OVO_FUSED" : "ILLICO_OVR_FUSED", 1) == 0 || b <= 0) return -1;
    if (!stage_dense_tma_ok(X, ld, gene_lb, b, plan)) return -1;
    // u16 counters hold the groups that are ranked (the control's rows are skipped; its histogram is the u32 table)
    if (plan->max_target_group_size >= 65536 || plan->n_groups < 2 || plan->n_groups > 65535) return -1;   // + grid.y
    if (OVO && (long long)plan->ref_group_size + plan->max_target_group_size > PAIR_MAX) return -1;  // tie sums below 2^53
    if (!OVO && flags->group_sums) return -1;
    if (dbg) return -1;   // the exact integers / tie sums of every gene come from the general path's kernels
    if (buf->workspace_bytes < gtab_bytes(b, plan->n_groups)) return -1;
    const int bs = (b + 63) & ~63;
    Gtab gt = gtab_carve(buf->workspace, b, plan->n_groups);

    // wide table (integer counts up to DW, folded against the control at the end of each group): one-versus-reference on
    // raw counts only -- the ranks of one-versus-rest are not known before the whole gene has been seen
    const bool wide_on = OVO && !flags->is_log1p && env_int("ILLICO_FUSED_WIDE", 1) != 0;
    // 1. table segments: the control group (OVO) or a sample of about 16k cells (OVR: the first segments)
    int seg_lo = plan->ref_seg_begin, seg_hi = plan->ref_seg_end;
    if (!OVO) {
        long long avg = plan->n_cells / plan->n_segments;
        if (avg < 1) avg = 1;
        seg_lo = 0;
        seg_hi = (int)((OVR_SAMPLE_CELLS + avg - 1) / avg);
        if (seg_hi < 1) seg_hi = 1;
        if (seg_hi > plan->n_segments) seg_hi = plan->n_segments;
    }
    ILLICO_CUDA_OK(cudaMemsetAsync(gt.n_bad, 0, 16 * sizeof(int), stream));
    {
        const int rc = launch_stage_dense_tma(X, ld, gene_lb, b, plan, buf->ir_vals, buf->ir_cnt, seg_lo, seg_hi, stream, 1);
        if (rc != 0) return rc;
        int blocks = (b + 7) / 8;
        if (blocks > 148 * 8) blocks = 148 * 8;
        ILLICO_LAUNCH("fused_ctab_kernel", stream, fused_ctab_kernel<<<blocks, 256, 0, stream>>>(buf->ir_vals, buf->ir_cnt, b, *plan, seg_lo, seg_hi, flags->is_log1p, gt, bs, wide_on ? 1 : 0));
        ILLICO_LAUNCH("fused_mode_kernel", stream, fused_mode_kernel<<<(b + FUSED_LANES - 1) / FUSED_LANES, FUSED_LANES, 0, stream>>>(b, gt));
        ILLICO_CUDA_OK(cudaGetLastError());
    }
    if (!OVO)   // the sample only seeds the slots; gt.mult restarts as the whole gene's histogram
        ILLICO_CUDA_OK(cudaMemsetAsync(gt.mult, 0, (size_t)bs * DCAP * sizeof(uint32_t), stream));

    // 2. the pass over the matrix (CTAs whose genes were all handed back by the table step leave at once)
    long long avg_g = plan->n_cells / plan->n_groups;
    if (avg_g < 1) avg_g = 1;
    int gpc = (int)(PASS_ROWS / avg_g);
    if (gpc < 1) gpc = 1;
    {
        // ring / buffer shapes measured at the K562 shape (profiles/README.md): stages of 8 rows, a 16-entry group buffer,
        // 3 CTAs per SM; the 5-stage ring (74 KB of shared memory per CTA) is 6-7 % faster than the 4-stage one
        using L = FusedLayout<8, 5, 16>;
        auto kern = fused_pass_kernel<8, 5, 16, 3, OVO>;
        ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::BYTES));
        const dim3 grid((unsigned)((b + FUSED_LANES - 1) / FUSED_LANES), (unsigned)((plan->n_groups + gpc - 1) / gpc));
        ILLICO_LAUNCH("fused_pass_kernel", stream, kern<<<grid, FUSED_THREADS, L::BYTES, stream>>>(X, ld, gene_lb, b, *plan, gpc, gt, bs,
                                                        reinterpret_cast<unsigned long long*>(results), gstride, list_share_1024()));
        ILLICO_CUDA_OK(cudaGetLastError());
    }
    if (wide_on) {
        // (a 6-stage ring -- 112 KB per CTA, the most two CTAs per SM leave room for -- makes the pass 3 % faster and the
        // whole step 9 % slower: measured, and removed after commit 216d8fd)
        auto kern = fused_wide_pass_kernel<8, 5, 2>;
        const int wide_smem = WideLayout<8, 5>::BYTES;
        ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, wide_smem));
        // persistent: two CTAs per SM, each a tile of 256 genes walking every gy-th chunk of groups
        const int tiles = (b + FUSED_LANES - 1) / FUSED_LANES, chunks = (plan->n_groups + gpc - 1) / gpc;
        int gy = (2 * 148) / tiles;
        if (gy < 1) gy = 1;
        if (gy > chunks) gy = chunks;
        const dim3 grid((unsigned)tiles, (unsigned)gy);
        ILLICO_LAUNCH("fused_wide_pass_kernel", stream, kern<<<grid, FUSED_THREADS, wide_smem, stream>>>(
                X, ld, gene_lb, b, *plan, gpc, gt, bs, reinterpret_cast<unsigned long long*>(results), gstride, list_share_1024()));
        ILLICO_CUDA_OK(cudaGetLastError());
    }
    g_last_fused_ms = 0.0f;

    // 3. per-group constants, per-gene weights, then the epilogue
    ILLICO_LAUNCH("fused_group_kernel", stream, fused_group_kernel<OVO><<<(plan->n_groups + 255) / 256, 256, 0, stream>>>(*plan, gt));
    ILLICO_LAUNCH("fused_gene_kernel", stream, fused_gene_kernel<OVO><<<(b + 127) / 128, 128, 0, stream>>>(b, *plan, *flags, gt, bs, nullptr, nullptr));
    ILLICO_CUDA_OK(cudaGetLastError());
    if (launch_fused_epilogue<OVO, false>(b, plan, flags, gt, bs, results, gstride, list_share_1024(), stream)) return 1;
    if (wide_on && launch_fused_epilogue<OVO, true>(b, plan, flags, gt, bs, results, gstride, list_share_1024(), stream)) return 1;

    // 4. genes handed back: listed on the device, staged from the matrix by a persistent kernel, ranked by the general
    // path with the device-side count (an empty list costs three nearly empty launches)
    ILLICO_LAUNCH("fused_list_kernel", stream, fused_list_kernel<<<1, 1024, 0, stream>>>(b, gt, list_share_1024(), 1024, 0));
    ILLICO_CUDA_OK(cudaGetLastError());
    if (launch_stage_dense_list(X, ld, gene_lb, gt.list, gt.n_bad + 1, gt.n_bad + 2, HB_LIST, plan, buf->ir_vals, buf->ir_cnt, stream))
        return 1;
    if (launch_stage_dense_tma_if(X, ld, gene_lb, b, plan, buf->ir_vals, buf->ir_cnt, 0, plan->n_segments, stream, 0, gt.n_bad + 2,
                                  HB_ALL))
        return 1;
    // the rank kernels' scratch lies behind the tables (they are read until the list has been ranked)
    const size_t tab = (gtab_bytes(b, plan->n_groups) + 255) & ~(size_t)255;
    if (buf->workspace_bytes <= tab) return 1;
    char* ws = reinterpret_cast<char*>(buf->workspace) + tab;
    const size_t ws_bytes = buf->workspace_bytes - tab;
    return OVO ? launch_ovo_mapped(buf->ir_vals, buf->ir_cnt, b, gt.n_bad + 1, gt.list, b, plan, flags, results, gstride, ws, ws_bytes,
                                   nullptr, stream)
               : launch_ovr_mapped(buf->ir_vals, buf->ir_cnt, b, gt.n_bad + 1, gt.list, b, plan, flags, results, gstride, ws, ws_bytes,
                                   nullptr, stream);
}

}  // namespace

float ovo_fused_last_ms() { return g_last_fused_ms; }

size_t ovo_fused_workspace_bytes(int b, int n_groups) { return gtab_bytes(b, n_groups); }

int launch_ovo_dense_fused(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan,
                           const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results, long long gstride,
                           const illico_debug_t* dbg, cudaStream_t stream) {
    return run_fused<true>(X, ld, gene_lb, b, plan, flags, buf, results, gstride, dbg, stream);
}

int launch_ovr_dense_fused(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan,
                           const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results, long long gstride,
                           const illico_debug_t* dbg, cudaStream_t stream) {
    return run_fused<false>(X, ld, gene_lb, b, plan, flags, buf, results, gstride, dbg, stream);
}


namespace {

// The fused path for one gene batch of a CSR matrix, enqueued without a host read-back.  0 = enqueued, 1 = error,
// -1 = not applicable.
template <bool OVO>
int run_fused_csr(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                  const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results,
                  long long gstride, const illico_debug_t* dbg, cudaStream_t stream) {
    g_last_fused_ms = -1.0f;
    if (env_int(OVO ? "ILLICO_OVO_FUSED" : "ILLICO_OVR_FUSED", 1) == 0 || env_int("ILLICO_CSR_FUSED", 1) == 0 || b <= 0) return -1;
    if (plan->max_target_group_size >= 65536 || plan->n_groups < 2 || plan->n_groups > 65535 || plan->n_segments > 65535) return -1;
    if (OVO && (long long)plan->ref_group_size + plan->max_target_group_size > PAIR_MAX) return -1;
    if (!OVO && flags->group_sums) return -1;
    if (dbg) return -1;
    if (buf->workspace_bytes < gtab_bytes(b, plan->n_groups)) return -1;
    const int bs = (b + 63) & ~63;
    Gtab gt = gtab_carve(buf->workspace, b, plan->n_groups);
    unsigned long long* rec = reinterpret_cast<unsigned long long*>(results);
    const int G = plan->n_groups;

    // tables: raw counts get slots 1 .. 12 up front (log1p data claims its slots while streaming)
    ILLICO_CUDA_OK(cudaMemsetAsync(gt.n_bad, 0, 16 * sizeof(int), stream));
    ILLICO_LAUNCH("fused_seed_kernel", stream, fused_seed_kernel<<<(bs + 255) / 256, 256, 0, stream>>>(gt, bs, flags->is_log1p ? 0 : 1));
    ILLICO_LAUNCH("fused_zero_multi_kernel", stream, fused_zero_multi_kernel<<<dim3(8, (unsigned)G), 256, 0, stream>>>(b, *plan, rec, gstride));
    ILLICO_CUDA_OK(cudaGetLastError());
    {
        // (An atomics-free variant -- the whole CTA applies one row at a time, plain LDS/STS -- measured 1.5-2.7 x
        // slower: 150 CTA-wide barriers per segment cost more than the shared atomics they avoid.  Counting part of the
        // updates in a per-SM global histogram with L2 reductions instead of shared atomics measured 1.4-1.9 x slower.
        // A warp per gene range without atomics measured 1.57 ms against 1.15 ms at the K562 shape: finding the range's
        // start in every row costs more than the atomics it saves; it was removed after commit 216d8fd.)
        auto kern = fused_csr_pass_kernel<OVO>;
        const int tile = b < CSRF_TILE ? b : CSRF_TILE;
        const size_t smem = (size_t)tile * 24;
        ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const dim3 grid((unsigned)((b + CSRF_TILE - 1) / CSRF_TILE), (unsigned)plan->n_segments);
        ILLICO_LAUNCH("fused_csr_pass_kernel", stream, kern<<<grid, CSRF_THREADS, smem, stream>>>(data, indices, indptr, gene_lb, b, *plan, gt, bs, rec, gstride));
        ILLICO_CUDA_OK(cudaGetLastError());
    }
    g_last_fused_ms = 0.0f;
    // (when the pass stopped early -- an eighth of the genes flagged: continuous data -- the kernels below work on
    // incomplete records; the list kernel then hands the WHOLE batch to the general path, which overwrites everything)
    if (!OVO) {
        const int gpb = 64;
        ILLICO_LAUNCH("fused_hist_sum_kernel", stream, fused_hist_sum_kernel<<<dim3((unsigned)((b + 255) / 256), (unsigned)((G + gpb - 1) / gpb)), 256, 0, stream>>>(b, G, gpb, gt, bs, rec,
                                                                                                                 gstride));
    }
    ILLICO_LAUNCH("fused_group_kernel", stream, fused_group_kernel<OVO><<<(plan->n_groups + 255) / 256, 256, 0, stream>>>(*plan, gt));
    ILLICO_LAUNCH("fused_gene_kernel", stream, fused_gene_kernel<OVO><<<(b + 127) / 128, 128, 0, stream>>>(b, *plan, *flags, gt, bs, nullptr, nullptr));
    if (launch_fused_epilogue<OVO, false>(b, plan, flags, gt, bs, results, gstride, 128, stream)) return 1;   // (the CSR pass stops at an eighth)

    // hand-back, decided on the device: a few scattered genes -> one filtered pass over the stored values (HB_LIST);
    // many (or a pass that stopped early: 8 n_bad > b) -> the general CSR staging of the whole batch (HB_ALL)
    int share = list_share_1024();
    if (share > 128) share = 128;                       // the pass itself stops at an eighth
    ILLICO_LAUNCH("fused_list_kernel", stream, fused_list_kernel<<<1, 1024, 0, stream>>>(b, gt, share, 1024, 0));
    ILLICO_CUDA_OK(cudaGetLastError());
    const size_t tab = (gtab_bytes(b, plan->n_groups) + 255) & ~(size_t)255;
    if (buf->workspace_bytes <= tab) return 1;
    char* ws = reinterpret_cast<char*>(buf->workspace) + tab;
    const size_t ws_bytes = buf->workspace_bytes - tab;
    const int max_list = (int)(((long long)b * share) / 1024) + 1;
    if (launch_stage_csr_list(data, indices, indptr, gene_lb, b, gt.cmap, gt.n_bad + 2, HB_LIST, max_list < b ? max_list : b, plan,
                              buf->ir_vals, buf->ir_cnt, stream)) return 1;
    if (launch_stage_csr_if(data, indices, indptr, gene_lb, b, plan, buf->ir_vals, buf->ir_cnt, ws, ws_bytes, gt.n_bad + 2, HB_ALL, stream))
        return 1;
    return OVO ? launch_ovo_mapped(buf->ir_vals, buf->ir_cnt, b, gt.n_bad + 1, gt.list, b, plan, flags, results, gstride, ws, ws_bytes,
                                   nullptr, stream)
               : launch_ovr_mapped(buf->ir_vals, buf->ir_cnt, b, gt.n_bad + 1, gt.list, b, plan, flags, results, gstride, ws, ws_bytes,
                                   nullptr, stream);
}

}  // namespace

int launch_ovo_csr_fused(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                         const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results,
                         long long gstride, const illico_debug_t* dbg, cudaStream_t stream) {
    return run_fused_csr<true>(data, indices, indptr, gene_lb, b, plan, flags, buf, results, gstride, dbg, stream);
}
int launch_ovr_csr_fused(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                         const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results,
                         long long gstride, const illico_debug_t* dbg, cudaStream_t stream) {
    return run_fused_csr<false>(data, indices, indptr, gene_lb, b, plan, flags, buf, results, gstride, dbg, stream);
}

}  // namespace illico
