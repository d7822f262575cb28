// stage_dense_tma.cu -- dense staging with the rows brought in by the TMA engine (sm_100a).
//
// Same contract as stage_dense_kernel (stage.cu; replaces chunk_and_fortranize, illico/utils/math.py:247-278, and
// the per-group row gathers of illico/ovo/dense_ovo.py:111-123): every element of the batch is read exactly once,
// the non-zero values of each (gene, segment) are compacted at the start of the segment's slot, counts go to ir_cnt.
//
// What is different: the loads are not issued by the threads that compact.  One producer warp walks the CTA's
// permuted cell rows and issues one bulk copy per row piece (`cp.async.bulk.shared.global`, SASS UBLKCP: 4 * GENES
// bytes, global -> shared, completion counted on an mbarrier); the eight consumer warps read the rows from shared
// memory.  The bytes in flight per SM are then a property of the ring (STAGES * ROWS * row piece per CTA), not of
// the consumers' registers or issue slots, and a consumer spends one LDS per element instead of an address
// computation, a shuffle and a global load.  The compaction is lane-private as before, but the lane's buffer holds
// 8 + ROWS entries and is inspected once per ring stage instead of once per element, which removes the divergent
// flush branch from the per-element path (it was a third of the old kernel's instructions).
#include "common.cuh"
#include "tma.cuh"

#include <stdlib.h>

namespace illico {

namespace {

constexpr int TMA_CONSUMER_WARPS = 8;
constexpr int TMA_CONSUMERS = TMA_CONSUMER_WARPS * 32;
constexpr int TMA_THREADS = TMA_CONSUMERS + 32;   // + one producer warp
constexpr int TMA_MAX_SEGS = 16;

// Lane-private compaction buffer: ENTRIES floats per (thread, gene stream), contiguous per lane.
__device__ __forceinline__ void append_nz(uint32_t& off, float v, uint32_t buf) {
    asm volatile("{ .reg .pred p; setp.neu.f32 p, %2, 0f00000000; @p st.shared.f32 [%1], %2; @p add.u32 %0, %0, 4; }"
                 : "+r"(off)
                 : "r"(buf + off), "f"(v)
                 : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 q;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(q.x), "=f"(q.y), "=f"(q.z), "=f"(q.w) : "r"(a));
    return q;
}
__device__ __forceinline__ void sts128(uint32_t a, float4 q) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(q.x), "f"(q.y), "f"(q.z), "f"(q.w) : "memory");
}
// writes entries [0, 8) of the lane's buffer as one aligned 32-byte sector: a single 256-bit streaming store
// (sm_100 STG.256), so L2 receives the sector whole
__device__ __forceinline__ void flush_sector(float* dst, uint32_t buf) {
    const float4 a = lds128(buf), b = lds128(buf + 16);
    asm volatile("st.global.cs.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "f"(a.x), "f"(a.y), "f"(a.z),
                 "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w)
                 : "memory");
}

template <int ROWS, int STAGES>
struct TmaLayout {
    static constexpr int GENES = TMA_CONSUMERS;               // genes per CTA: one per consumer lane
    static constexpr int ROW_BYTES = GENES * 4;               // bytes of one row piece
    static constexpr int STAGE_BYTES = ROWS * ROW_BYTES;
    static constexpr int ENTRIES = 8 + ROWS;                  // lane buffer: < 8 left over + one stage's appends
    static constexpr int WBUF_BYTES = TMA_CONSUMERS * ENTRIES * 4;
    static constexpr int RING_OFF = 0;
    static constexpr int WBUF_OFF = STAGES * STAGE_BYTES;
    static constexpr int BAR_OFF = WBUF_OFF + WBUF_BYTES;     // 2 * STAGES mbarriers
    static constexpr int CNT_OFF = BAR_OFF + 2 * STAGES * 8;  // uint16 [segs_per_cta][GENES]
    static size_t bytes(int segs_per_cta) { return (size_t)CNT_OFF + (size_t)segs_per_cta * GENES * 2; }
};

template <int ROWS, int STAGES, int MINB>
__global__ void __launch_bounds__(TMA_THREADS, MINB) stage_dense_tma_kernel(const float* __restrict__ X, long long ld, int gene_lb,
                                                                      int b, const illico_plan_t pl,
                                                                      float* __restrict__ ir_vals,
                                                                      uint32_t* __restrict__ ir_cnt, int segs_per_cta, int seg_lo,
                                                                      int seg_hi, int tiles_x, int tiles_y,
                                                                      const int* __restrict__ mode_dev, int want_mode) {
    // A decision taken on the device (hand-back of the fused paths): the host enqueued this launch without knowing
    // whether it is needed.  Such launches are persistent (a fixed 1-D grid walking the tiles), so a no costs microseconds.
    if (mode_dev && *mode_dev != want_mode) return;
    using L = TmaLayout<ROWS, STAGES>;
    static_assert(32 % ROWS == 0, "a 32-row group of the permutation holds whole stages");
    extern __shared__ __align__(128) unsigned char smem[];
    const uint32_t smem_a = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = smem_a + L::BAR_OFF;                 // full[i] = bars + 8 i, empty[i] = bars + 8 (STAGES + i)
    uint16_t* cnt_tile = reinterpret_cast<uint16_t*>(smem + L::CNT_OFF);
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int S = pl.n_segments;
    // tiles: (256 genes) x (segs_per_cta segments).  A 2-D grid gives every CTA its own tile; a 1-D (persistent)
    // grid walks them.  The ring's stage counters run on across tiles, so the producer fills the ring with the next
    // tile's rows while the consumers finish the current one.
    const int n_tiles = tiles_x * tiles_y;
    const bool own_tile = gridDim.y > 1 || gridDim.x == (unsigned)n_tiles;
    const int tile0 = own_tile ? (int)(blockIdx.y * gridDim.x + blockIdx.x) : (int)blockIdx.x;
    const int tile_step = own_tile ? n_tiles : (int)gridDim.x;

    if (t == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(bars + 8 * i, 1);                                  // producer's arrive.expect_tx
            mbar_init(bars + 8 * (STAGES + i), TMA_CONSUMER_WARPS);      // one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (w == TMA_CONSUMER_WARPS) {
        // ---------------- producer warp: one bulk copy per (row, CTA gene range)
        uint64_t policy;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
        const unsigned long long ldb = (unsigned long long)ld * 4ull;
        int k = 0;                                                       // stage counter (runs on across tiles)
        for (int tile = tile0; tile < n_tiles; tile += tile_step) {
        const int bx = tile % tiles_x, by = tile / tiles_x;
        const int s_begin = seg_lo + by * segs_per_cta, s_end = min(seg_hi, s_begin + segs_per_cta);
        const int p_begin = pl.seg_pos[s_begin], p_end = pl.seg_pos[s_end];
        const int g0 = bx * L::GENES;                              // first gene of the tile inside the batch
        // bytes of the row piece this tile reads: whole 16-byte units (the host checked that the round-up stays in the row)
        const uint32_t row_bytes = (uint32_t)min(L::GENES, (b - g0 + 3) & ~3) * 4u;
        const char* base = reinterpret_cast<const char*>(X + gene_lb + g0);
        int myrow = (p_begin + lane < p_end) ? pl.perm[p_begin + lane] : 0;
        for (int p = p_begin; p < p_end; p += 32) {
            const int nxt = (p + 32 + lane < p_end) ? pl.perm[p + 32 + lane] : 0;   // next group's rows, ahead of use
            const int nrows = min(32, p_end - p);
#pragma unroll
            for (int q = 0; q < 32 / ROWS; ++q, ++k) {
                if (q * ROWS >= nrows) break;
                const int slot = k % STAGES;
                const uint32_t full = bars + 8 * slot, empty = bars + 8 * (STAGES + slot);
                mbar_wait(empty, ((k / STAGES) & 1) ^ 1);                // passes at once the first time round
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
    int k = 0;                                                           // stage counter (runs on across tiles)
    for (int tile = tile0; tile < n_tiles; tile += tile_step) {
    const int bx = tile % tiles_x, by = tile / tiles_x;
    const int s_begin = seg_lo + by * segs_per_cta, s_end = min(seg_hi, s_begin + segs_per_cta);
    const int p_begin = pl.seg_pos[s_begin], p_end = pl.seg_pos[s_end];
    const int g0 = bx * L::GENES;
    const int j = g0 + t;
    const bool act = j < b;
    float* const gene_base = ir_vals + (long long)(act ? j : 0) * pl.slot_cap;
    uint32_t done = 0, off = 0;
    const uint32_t buf = smem_a + L::WBUF_OFF + t * L::ENTRIES * 4;
    int s = s_begin;
    int seg_end = pl.seg_pos[s + 1];
    int seg_off = pl.seg_base[s];
    // closes segment s: the lane's leftovers leave as one or two padded sectors, the count goes to the tile
    auto finalize = [&]() {
        if (act) {
            float* dst = gene_base + seg_off + done;
            for (uint32_t o = 0; o < off; o += 32u) flush_sector(dst + (o >> 2), buf + o);
        }
        cnt_tile[(s - s_begin) * L::GENES + t] = (uint16_t)(done + (off >> 2));
        done = 0;
        off = 0;
    };
    const unsigned char* my_ring = smem + L::RING_OFF + t * 4;
    for (int p = p_begin; p < p_end; p += ROWS, ++k) {
        const int slot = k % STAGES;
        mbar_wait(bars + 8 * slot, (k / STAGES) & 1);
        const int nr = min(ROWS, p_end - p);
        const unsigned char* src = my_ring + slot * L::STAGE_BYTES;
        auto load_row = [&](int u) { return *reinterpret_cast<const float*>(src + u * L::ROW_BYTES); };
        if (p + ROWS <= seg_end) {
            // the whole stage lies inside the current segment (the usual case): the stage's rows first
            // (independent shared loads), then the dependent appends
            float v[ROWS];
#pragma unroll
            for (int u = 0; u < ROWS; ++u) v[u] = load_row(u);
#pragma unroll
            for (int u = 0; u < ROWS; ++u) append_nz(off, v[u], buf);
        } else {
            // a segment ends inside this stage (or the CTA's rows do): row by row
#pragma unroll 1
            for (int u = 0; u < nr; ++u) {
                while (p + u == seg_end) {                               // CTA-uniform: the next segment starts here
                    finalize();
                    ++s;
                    seg_end = pl.seg_pos[s + 1];
                    seg_off = pl.seg_base[s];
                }
                append_nz(off, load_row(u), buf);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (STAGES + slot));          // this warp is done with the stage
        // once per stage: full sectors leave, the (< 8) leftovers move to the front of the lane's buffer
        if (off >= 32u) {
            const uint32_t full_bytes = off & ~31u;
            if (act) {
                float* dst = gene_base + seg_off + done;
                for (uint32_t o = 0; o < full_bytes; o += 32u) flush_sector(dst + (o >> 2), buf + o);
            }
            sts128(buf, lds128(buf + full_bytes));
            if (ROWS >= 8) sts128(buf + 16, lds128(buf + full_bytes + 16));
            done += full_bytes >> 2;
            off -= full_bytes;
        }
    }
    for (;;) {                                                           // closes the last segment (and empty ones after it)
        finalize();
        if (++s >= s_end) break;
        seg_off = pl.seg_base[s];
    }
    // counts: thread t writes the consecutive segments of gene t (contiguous runs per gene)
    asm volatile("bar.sync 1, %0;" ::"r"(TMA_CONSUMERS) : "memory");
    const int nseg = s_end - s_begin;
    if (act) {
        uint32_t* dst = ir_cnt + (long long)j * S + s_begin;
        for (int ls = 0; ls < nseg; ++ls) dst[ls] = cnt_tile[ls * L::GENES + t];
    }
    asm volatile("bar.sync 1, %0;" ::"r"(TMA_CONSUMERS) : "memory");   // the count tile is free for the next tile
    }
}

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}

constexpr int STAGE_ROWS = 512;   // rows a CTA stages: segments per CTA = STAGE_ROWS / average segment size

template <int ROWS, int STAGES, int MINB>
int launch_t(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt,
             int segs_per_cta, int seg_lo, int seg_hi, cudaStream_t stream, const int* mode_dev, int want_mode) {
    using L = TmaLayout<ROWS, STAGES>;
    const unsigned gx = (unsigned)((b + L::GENES - 1) / L::GENES);
    const unsigned gy = (unsigned)((seg_hi - seg_lo + segs_per_cta - 1) / segs_per_cta);
    const size_t smem = L::bytes(segs_per_cta);
    auto kern = stage_dense_tma_kernel<ROWS, STAGES, MINB>;
    ILLICO_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(gx, gy);
    if (mode_dev) {   // decided on the device: persistent 1-D grid
        int occ = 0;
        ILLICO_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TMA_THREADS, smem));
        long long ctas = 148ll * (occ > 0 ? occ : 1);
        if (ctas > (long long)gx * gy) ctas = (long long)gx * gy;
        if (ctas == (long long)gx * gy && gy > 1) ctas -= 1;   // (a 1-D grid of exactly n_tiles CTAs would read as 2-D)
        grid = dim3((unsigned)ctas, 1);
    }
    ILLICO_LAUNCH("stage_dense_tma_kernel", stream,
                  kern<<<grid, TMA_THREADS, smem, stream>>>(X, ld, gene_lb, b, *plan, ir_vals, ir_cnt, segs_per_cta, seg_lo, seg_hi,
                                                            (int)gx, (int)gy, mode_dev, want_mode));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace

// The bulk copies need 16-byte aligned row pieces, and every segment must fit the 16-bit count tile.
bool stage_dense_tma_ok(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan) {
    if (env_int("ILLICO_STAGE_TMA", 1) == 0) return false;
    if ((reinterpret_cast<uintptr_t>(X) & 15) || (ld & 3) || (gene_lb & 3)) return false;
    if (gene_lb + ((b + 3) & ~3) > ld) return false;            // the last piece would leave the row
    // (a partial check only, for plans whose groups were not cut at all: every plan must keep its segments under
    // 65536 cells -- HostPlan refuses longer ones, see seg_pos in illico_b200.h)
    if (plan->max_group_size >= 65536 && plan->n_segments == plan->n_groups) return false;
    return true;
}

// Stages segments [seg_lo, seg_hi) of the plan (the whole plan: 0, n_segments; the control group alone for the fused
// one-versus-reference path).
int launch_stage_dense_tma_if(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                              uint32_t* ir_cnt, int seg_lo, int seg_hi, cudaStream_t stream, int segs_per_cta_req,
                              const int* mode_dev, int want_mode) {
    const int S = plan->n_segments;
    if (seg_lo < 0 || seg_hi > S || seg_lo >= seg_hi) { set_error("segment range [%d, %d) out of bounds", seg_lo, seg_hi); return 1; }
    long long avg = plan->n_cells / S;
    if (avg < 1) avg = 1;
    int segs_per_cta = segs_per_cta_req > 0 ? segs_per_cta_req : (int)(STAGE_ROWS / avg);
    if (segs_per_cta < 1) segs_per_cta = 1;
    if (segs_per_cta > TMA_MAX_SEGS) segs_per_cta = TMA_MAX_SEGS;
    if (!mode_dev && (S + segs_per_cta - 1) / segs_per_cta > 65535) return -1;      // caller falls back to the plain kernel
    // Ring configurations measured at the K562 shape (profiles/README.md): one gene per lane (1 KB row pieces) is the
    // fastest and has the smallest footprint.  Measured on the continuous K562 shape: 72 registers / 3 CTAs per SM
    // 2.01 ms as a 2-D grid and 2.14 ms persistent; 96 registers / 2 CTAs per SM with a 6-stage ring 2.05 / 2.09 ms;
    // 56 registers / 4 CTAs per SM spills in the per-element loop and takes 3.4 ms.  A launch decided on the device
    // has to be persistent, and takes the 6-stage ring.
    if (mode_dev)
        return launch_t<8, 6, 2>(X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta, seg_lo, seg_hi, stream, mode_dev, want_mode);
    return launch_t<8, 4, 3>(X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta, seg_lo, seg_hi, stream, mode_dev, want_mode);
}

int launch_stage_dense_tma(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                           uint32_t* ir_cnt, int seg_lo, int seg_hi, cudaStream_t stream, int segs_per_cta_req) {
    return launch_stage_dense_tma_if(X, ld, gene_lb, b, plan, ir_vals, ir_cnt, seg_lo, seg_hi, stream, segs_per_cta_req, nullptr, 0);
}

}  // namespace illico
