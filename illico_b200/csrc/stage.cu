// stage.cu -- input formats -> group-segmented, gene-major lists of non-zero values (sm_100a).
//
// Replaces the reference's batch re-layout steps: chunk_and_fortranize (illico/utils/math.py:247-278),
// the CSR/CSC slicers (illico/utils/sparse/csr.py:103-257, csc.py:99-183).  The output ("IR") is the same
// for every input format, so one pair of rank kernels serves all six reference dispatchers:
//
//   ir_vals[gene, seg_base[s] + k]  k-th non-zero value of the cells of segment s (a slice of one group)
//   ir_cnt [gene, s]                how many there are
//
// Zeros are dropped here -- for dense input too -- because the rank kernels treat them as one analytic
// tie block (SURVEY.md appendix A.3).  This is HBM-bound byte shuffling: the dense kernel reads every
// element exactly once with warp-coalesced row segments and writes only the ~10 % that are non-zero.
#include "common.cuh"

namespace illico {

constexpr int STAGE_WARPS = 8;
constexpr int STAGE_MAX_SEGS = 16;
constexpr int STAGE_INFLIGHT = 8;   // cell rows per load batch (two batches in flight per warp)

// Appends v to the lane's slot when it is non-zero.  Non-zeros are collected eight at a time in a lane-private
// 32-byte shared-memory row and leave as ONE full, aligned 32-byte sector (slots are 32-byte aligned and padded),
// so L2 never sees a partial-sector write that it would have to merge with a DRAM fill.  The row is contiguous
// per lane: only the ~3 lanes of a warp that hold a non-zero store at a time, so bank conflicts are rare, and
// the flush is two 128-bit shared loads + two 128-bit global stores.
__device__ __forceinline__ void flush8(float* out0, uint32_t first, uint32_t row_addr) {
    float4 a, b;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(row_addr));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(row_addr + 16));
    float4* dst = reinterpret_cast<float4*>(out0 + first);
    __stcs(dst, a);
    __stcs(dst + 1, b);
}
// `off` = byte offset of the next free entry in the lane's 32-byte row; `done` = values already written to the
// slot.  Six instructions per element, no divergent branch except the flush every eighth non-zero.
__device__ __forceinline__ void append_nonzero(float* out0, uint32_t& done, uint32_t& off, float v, uint32_t row_addr) {
    asm volatile("{ .reg .pred p; setp.neu.f32 p, %2, 0f00000000; @p st.shared.f32 [%1], %2; @p add.u32 %0, %0, 4; }"
                 : "+r"(off) : "r"(row_addr + off), "f"(v) : "memory");
    if (off == 32u) {
        flush8(out0, done, row_addr);
        done += 8u;
        off = 0u;
    }
}
// row * ld in one wide multiply-add (row < 2^31, ld * 4 < 2^32: checked by the host)
__device__ __forceinline__ const float* row_ptr(const float* col, int row, uint32_t ld_bytes) {
    return reinterpret_cast<const float*>(reinterpret_cast<const char*>(col) +
                                          (unsigned long long)(uint32_t)row * (unsigned long long)ld_bytes);
}

// One warp = 32 * VEC adjacent genes: lane = VEC adjacent genes, so every cell row is one coalesced 128 * VEC
// byte request per warp and the CTA's 8 warps cover 1 KB * VEC of the row.  Each lane owns VEC (gene, segment)
// slots at a time and appends the non-zeros of the segment's cells in plan order: deterministic layout, no
// atomics, no shared-memory transposition.  The per-(gene, segment) counts go through a shared tile so that
// each gene's counts leave as one contiguous run.
template <bool TILE_COUNTS, int VEC>
__global__ void __launch_bounds__(STAGE_WARPS * 32) stage_dense_kernel(const float* __restrict__ X, long long ld,
                                                                       int gene_lb, int b, const illico_plan_t pl,
                                                                       float* __restrict__ ir_vals,
                                                                       uint32_t* __restrict__ ir_cnt,
                                                                       int segs_per_cta) {
    constexpr int NT = STAGE_WARPS * 32;
    __shared__ uint16_t cnt_tile[TILE_COUNTS ? STAGE_MAX_SEGS : 1][TILE_COUNTS ? NT * VEC : 1];
    __shared__ __align__(16) float wbuf[VEC][NT][8];
    const int lane = threadIdx.x & 31;
    const int t = threadIdx.x;
    const int jb = (blockIdx.x * NT + t) * VEC;          // first of this lane's VEC genes inside the batch
    const bool active = jb < b;                          // b is a multiple of VEC (host)
    const int jj = active ? jb : 0;                      // inactive lanes shadow gene 0 and never store
    const float* col = X + gene_lb + jj;
    const uint32_t ldb = (uint32_t)(ld * 4);
    const uint32_t wbuf_t = (uint32_t)__cvta_generic_to_shared(&wbuf[0][t][0]);
    const int S = pl.n_segments;
    const int s_begin = blockIdx.y * segs_per_cta, s_end = min(S, s_begin + segs_per_cta);
    for (int s = s_begin; s < s_end; ++s) {
        const int p0 = pl.seg_pos[s], p1 = pl.seg_pos[s + 1];
        float* out0[VEC];
        uint32_t done[VEC], off[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            out0[e] = ir_vals + (long long)(jj + e) * pl.slot_cap + pl.seg_base[s];
            done[e] = 0;
            off[e] = 0;
        }
        for (int p = p0; p < p1; p += 32) {
            const int nrows = min(32, p1 - p);
            const int myrow = pl.perm[p + min(lane, nrows - 1)];   // tail lanes repeat the last cell (never stored)
            const bool full = nrows == 32;
            // software pipeline over the chunk's rows in batches of STAGE_INFLIGHT: the next batch's loads are
            // issued before the current batch is compacted (two register buffers, manually alternated)
            auto load_batch = [&](float (&v)[STAGE_INFLIGHT][VEC], int k0) {
#pragma unroll
                for (int u = 0; u < STAGE_INFLIGHT; ++u) {
                    const float* src = row_ptr(col, __shfl_sync(FULL, myrow, (k0 + u) & 31), ldb);
                    if (VEC == 2) {
                        const float2 q = __ldcs(reinterpret_cast<const float2*>(src));
                        v[u][0] = q.x; v[u][VEC - 1] = q.y;
                    } else {
                        v[u][0] = __ldcs(src);
                    }
                }
            };
            auto compact_batch = [&](const float (&v)[STAGE_INFLIGHT][VEC], int k0) {
                if (!active) return;
#pragma unroll
                for (int u = 0; u < STAGE_INFLIGHT; ++u) {
                    if (full || k0 + u < nrows) {
#pragma unroll
                        for (int e = 0; e < VEC; ++e)
                            append_nonzero(out0[e], done[e], off[e], v[u][e], wbuf_t + e * NT * 32);
                    }
                }
            };
            float va[STAGE_INFLIGHT][VEC], vb[STAGE_INFLIGHT][VEC];
            load_batch(va, 0);
#pragma unroll
            for (int k0 = 0; k0 < 32; k0 += 2 * STAGE_INFLIGHT) {
                if (k0 >= nrows) break;
                if (k0 + STAGE_INFLIGHT < nrows) load_batch(vb, k0 + STAGE_INFLIGHT);
                compact_batch(va, k0);
                if (k0 + STAGE_INFLIGHT >= nrows) break;
                if (k0 + 2 * STAGE_INFLIGHT < nrows) load_batch(va, k0 + 2 * STAGE_INFLIGHT);
                compact_batch(vb, k0 + STAGE_INFLIGHT);
            }
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            if (active && off[e]) flush8(out0[e], done[e], wbuf_t + e * NT * 32);  // tail: one padded full sector
            const uint32_t cnt = done[e] + (off[e] >> 2);
            if (TILE_COUNTS) cnt_tile[s - s_begin][t * VEC + e] = (uint16_t)cnt;
            else if (active) ir_cnt[(long long)(jb + e) * S + s] = cnt;
        }
    }
    if (TILE_COUNTS) {
        __syncthreads();
        // thread t writes the consecutive segments of genes t, t + NT, ... of the CTA's NT * VEC genes
        const int nseg = s_end - s_begin;
        for (int g = t; g < NT * VEC; g += NT) {
            const int j = blockIdx.x * NT * VEC + g;
            if (j < b) {
                uint32_t* dst = ir_cnt + (long long)j * S + s_begin;
                for (int ls = 0; ls < nseg; ++ls) dst[ls] = cnt_tile[ls][g];
            }
        }
    }
}

// Hand-back of the fused paths: the genes to stage are named by a list that was built ON THE DEVICE (n = *n_list_dev of
// them; gene k of the list is column gene_lb + list[k] of X and goes to slot space k of ir_vals / ir_cnt).  Nothing about
// the list is known on the host when this kernel is enqueued, so the grid is persistent (a fixed number of CTAs walking
// the (256-gene tile, segment chunk) work items) and an empty list costs a few microseconds.  Same compaction as
// stage_dense_kernel<true, 1>; a scattered list reads one 32-byte sector per 4-byte element.
__global__ void __launch_bounds__(STAGE_WARPS * 32) stage_dense_list_kernel(const float* __restrict__ X, long long ld, int gene_lb,
                                                                            const int* __restrict__ list,
                                                                            const int* __restrict__ n_list_dev,
                                                                            const int* __restrict__ mode_dev, int want_mode,
                                                                            const illico_plan_t pl, float* __restrict__ ir_vals,
                                                                            uint32_t* __restrict__ ir_cnt, int segs_per_cta) {
    constexpr int NT = STAGE_WARPS * 32;
    __shared__ __align__(16) float wbuf[NT][8];
    const int lane = threadIdx.x & 31, t = threadIdx.x;
    if (mode_dev && *mode_dev != want_mode) return;
    const int n = *n_list_dev;
    if (n <= 0) return;
    const int S = pl.n_segments;
    const int tiles_x = (n + NT - 1) / NT, tiles_y = (S + segs_per_cta - 1) / segs_per_cta;
    const uint32_t ldb = (uint32_t)(ld * 4);
    const uint32_t wbuf_t = (uint32_t)__cvta_generic_to_shared(&wbuf[t][0]);
    for (long long tile = blockIdx.x; tile < (long long)tiles_x * tiles_y; tile += gridDim.x) {
        const int bx = (int)(tile % tiles_x), by = (int)(tile / tiles_x);
        const int jb = bx * NT + t;                        // position in the list = gene index of the staged lists
        const bool active = jb < n;
        const float* col = X + gene_lb + (active ? list[jb] : list[0]);
        const int s_begin = by * segs_per_cta, s_end = min(S, s_begin + segs_per_cta);
        for (int s = s_begin; s < s_end; ++s) {
            const int p0 = pl.seg_pos[s], p1 = pl.seg_pos[s + 1];
            float* out0 = ir_vals + (long long)(active ? jb : 0) * pl.slot_cap + pl.seg_base[s];
            uint32_t done = 0, off = 0;
            for (int p = p0; p < p1; p += 32) {
                const int nrows = min(32, p1 - p);
                const int myrow = pl.perm[p + min(lane, nrows - 1)];
                for (int k0 = 0; k0 < nrows; k0 += STAGE_INFLIGHT) {
                    float v[STAGE_INFLIGHT];
#pragma unroll
                    for (int u = 0; u < STAGE_INFLIGHT; ++u)
                        v[u] = __ldcs(row_ptr(col, __shfl_sync(FULL, myrow, (k0 + u) & 31), ldb));
                    if (active) {
#pragma unroll
                        for (int u = 0; u < STAGE_INFLIGHT; ++u)
                            if (k0 + u < nrows) append_nonzero(out0, done, off, v[u], wbuf_t);
                    }
                }
            }
            if (active) {
                if (off) flush8(out0, done, wbuf_t);
                ir_cnt[(long long)jb * S + s] = done + (off >> 2);   // (a thread's segments are consecutive: one short run)
            }
        }
    }
}

__device__ __forceinline__ long long lower_bound_i32(const int32_t* a, long long n, int key) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// ---- CSR ----------------------------------------------------------------------------------------------
// Pass 1 (csr_split_kernel): for every cell row, the position of each gene-range boundary of the batch inside the
// row's sorted indices (binary search, as illico/utils/sparse/csr.py:171,226 does for the batch bounds).
// Pass 2 (stage_csr_kernel): a CTA owns (a few segments) x (one range of CSR_GC genes).  It counting-sorts the
// tile's stored values by gene in shared memory and writes every (gene, segment) run with aligned, padded
// 32-byte sectors -- no global atomics and no partial-sector writes (which cost one DRAM fill each).  The order
// inside a slot is arbitrary (shared-memory cursor atomics); ranks, U and tie sums do not depend on it.
constexpr int CSR_GC = 512;        // genes per range
constexpr int CSR_CAP = 8192;      // values per shared tile pass
constexpr int CSR_THREADS = 256;
constexpr int CSR_MAX_SEGS = 16;

__global__ void __launch_bounds__(256) csr_split_kernel(const int32_t* __restrict__ indices, const long long* __restrict__ indptr,
                                                        int n_rows, int gene_lb, int b, int K, int32_t* __restrict__ split,
                                                        const int* __restrict__ mode_dev, int want_mode) {
    if (mode_dev && *mode_dev != want_mode) return;   // (hand-back decided on the device: see launch_stage_csr_if)
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < n_rows; r += nwarps) {
        const long long start = indptr[r], len = indptr[r + 1] - start;
        for (int k = lane; k <= K; k += 32) {
            const int bound = gene_lb + min(k * CSR_GC, b);
            split[r * (K + 1) + k] = (int32_t)lower_bound_i32(indices + start, len, bound);
        }
    }
}

constexpr int CSR_MAX_ROWS = 1024;  // cells per segment this kernel accepts (the plan cuts groups at 512)

__global__ void __launch_bounds__(CSR_THREADS) stage_csr_kernel(const float* __restrict__ data, const int32_t* __restrict__ indices,
                                                                const long long* __restrict__ indptr, int gene_lb, int b, int K,
                                                                const int32_t* __restrict__ split, const illico_plan_t pl,
                                                                float* __restrict__ ir_vals, uint32_t* __restrict__ ir_cnt,
                                                                int segs_per_cta, const int* __restrict__ mode_dev, int want_mode) {
    if (mode_dev && *mode_dev != want_mode) return;
    extern __shared__ __align__(16) unsigned char csr_smem[];
    long long* row_a = reinterpret_cast<long long*>(csr_smem);             // [CSR_MAX_ROWS] first stored element of each row in the range
    float* vals = reinterpret_cast<float*>(row_a + CSR_MAX_ROWS);          // [CSR_CAP]
    uint32_t* hist = reinterpret_cast<uint32_t*>(vals + CSR_CAP);          // [CSR_GC] per-gene count, then scatter cursor
    uint32_t* offs = hist + CSR_GC;                                        // [CSR_GC + 1] exclusive prefix of the counts
    int* row_n = reinterpret_cast<int*>(offs + CSR_GC + 1);                // [CSR_MAX_ROWS] stored elements per row in the range
    uint32_t* wsum = reinterpret_cast<uint32_t*>(row_n + CSR_MAX_ROWS);    // [8]
    int* chunk_end_p = reinterpret_cast<int*>(wsum + 8);                   // [1]
    uint16_t (*done)[CSR_GC] = reinterpret_cast<uint16_t (*)[CSR_GC]>(chunk_end_p + 1);  // [CSR_MAX_SEGS][CSR_GC] values written
    int& chunk_end = *chunk_end_p;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    constexpr int NW = CSR_THREADS / 32;
    const int k = blockIdx.x;                          // gene range
    const int g0 = k * CSR_GC;                         // first gene of the range inside the batch
    const int ng = min(CSR_GC, b - g0);
    const int S = pl.n_segments;
    const int s_begin = blockIdx.y * segs_per_cta, s_end = min(S, s_begin + segs_per_cta);
    for (int s = s_begin; s < s_end; ++s) {
        const int ls = s - s_begin;
        __syncthreads();
        for (int g = t; g < CSR_GC; g += CSR_THREADS) done[ls][g] = 0;
      // segments longer than the row table are walked in blocks of CSR_MAX_ROWS cells (the plan cuts at 512)
      for (int pb = pl.seg_pos[s]; pb < pl.seg_pos[s + 1]; pb += CSR_MAX_ROWS) {
        const int p0 = pb, nrows = min(CSR_MAX_ROWS, pl.seg_pos[s + 1] - pb);
        __syncthreads();
        uint32_t mine = 0;
        for (int i = t; i < nrows; i += CSR_THREADS) {
            const long long r = pl.perm[p0 + i];
            const int a = split[r * (K + 1) + k], z = split[r * (K + 1) + k + 1];
            row_a[i] = indptr[r] + a;
            row_n[i] = z - a;
            mine += (uint32_t)(z - a);
        }
        // total stored values of the tile: the whole segment goes in one pass when it fits (the usual case)
        mine = warp_sum<uint32_t>(mine);
        if (lane == 0) wsum[w] = mine;
        __syncthreads();
        uint32_t tile_total = 0;
        for (int ww = 0; ww < NW; ++ww) tile_total += wsum[ww];
        int rc = 0;                                    // first row of the current pass
        while (rc < nrows) {
            __syncthreads();
            if (t == 0) {
                int e = nrows;
                if (tile_total > CSR_CAP) {
                    int tot = 0;
                    e = rc;
                    while (e < nrows && (tot + row_n[e] <= CSR_CAP || e == rc)) { tot += row_n[e]; ++e; }
                }
                chunk_end = e;
            }
            for (int g = t; g < CSR_GC; g += CSR_THREADS) hist[g] = 0;
            __syncthreads();
            const int re = chunk_end;
            // ---- count per gene
            // eight lanes per row, four elements per lane in flight: the loads of 32 rows x 4 elements overlap
            for (int i = rc + (t >> 3); i < re; i += CSR_THREADS / 8) {
                const long long a = row_a[i];
                const int nrow = row_n[i];
                for (int e0 = (t & 7); e0 < nrow; e0 += 32) {
                    float d[4];
                    int c[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int ee = e0 + 8 * u;
                        d[u] = (ee < nrow) ? data[a + ee] : 0.0f;
                        c[u] = (ee < nrow) ? indices[a + ee] : 0;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (d[u] != 0.0f) atomicAdd(&hist[c[u] - gene_lb - g0], 1u);
                }
            }
            __syncthreads();
            // ---- exclusive scan of hist[0..CSR_GC) (2 entries per thread)
            {
                const uint32_t c0 = hist[2 * t], c1 = hist[2 * t + 1];
                const uint32_t incl = warp_incl_scan(c0 + c1, lane);
                if (lane == 31) wsum[w] = incl;
                __syncthreads();
                uint32_t basev = incl - (c0 + c1);
                for (int ww = 0; ww < w; ++ww) basev += wsum[ww];
                offs[2 * t] = basev;
                offs[2 * t + 1] = basev + c0;
                if (t == CSR_THREADS - 1) offs[CSR_GC] = basev + c0 + c1;
                hist[2 * t] = basev;                   // cursors start at the offsets
                hist[2 * t + 1] = basev + c0;
            }
            __syncthreads();
            if (offs[CSR_GC] <= CSR_CAP) {
                // ---- scatter the values by gene into the shared tile
                for (int i = rc + (t >> 3); i < re; i += CSR_THREADS / 8) {
                    const long long a = row_a[i];
                    const int nrow = row_n[i];
                    for (int e0 = (t & 7); e0 < nrow; e0 += 32) {
                        float d[4];
                        int c[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int ee = e0 + 8 * u;
                            d[u] = (ee < nrow) ? data[a + ee] : 0.0f;
                            c[u] = (ee < nrow) ? indices[a + ee] : 0;
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (d[u] != 0.0f) vals[atomicAdd(&hist[c[u] - gene_lb - g0], 1u)] = d[u];
                    }
                }
                __syncthreads();
                // ---- write every gene's run: aligned padded sectors while the slot start is sector aligned
                for (int g = t; g < ng; g += CSR_THREADS) {
                    const uint32_t o = offs[g], c = offs[g + 1] - o;
                    if (c == 0) continue;
                    const uint32_t prior = done[ls][g];
                    float* dst = ir_vals + (long long)(g0 + g) * pl.slot_cap + pl.seg_base[s] + prior;
                    if ((prior & 7u) == 0u) {
                        for (uint32_t i = 0; i < c; i += 8) {
                            float q[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u) q[u] = vals[min(o + i + u, (uint32_t)CSR_CAP - 1)];
                            __stcs(reinterpret_cast<float4*>(dst + i), make_float4(q[0], q[1], q[2], q[3]));
                            __stcs(reinterpret_cast<float4*>(dst + i) + 1, make_float4(q[4], q[5], q[6], q[7]));
                        }
                    } else {
                        for (uint32_t i = 0; i < c; ++i) dst[i] = vals[o + i];
                    }
                    done[ls][g] = (uint16_t)(prior + c);
                }
            } else {
                // one row holds more values in this range than the tile (cannot happen with CSR_GC <= CSR_CAP and
                // unique column indices; kept as a safe path): write it directly, one warp per row
                for (int i = rc + w; i < re; i += NW) {
                    const long long a = row_a[i], z = a + row_n[i];
                    for (long long e = a + lane; e < z; e += 32) {
                        const float v = data[e];
                        if (v == 0.0f) continue;
                        const int g = indices[e] - gene_lb - g0;
                        const uint32_t slot = atomicAdd(&hist[g], 1u) - offs[g] + done[ls][g];
                        ir_vals[(long long)(g0 + g) * pl.slot_cap + pl.seg_base[s] + slot] = v;
                    }
                }
                __syncthreads();
                for (int g = t; g < ng; g += CSR_THREADS) done[ls][g] += (uint16_t)(offs[g + 1] - offs[g]);
            }
            rc = re;
        }
      }
    }
    __syncthreads();
    const int nseg = s_end - s_begin;
    for (int g = t; g < ng; g += CSR_THREADS) {
        uint32_t* dst = ir_cnt + (long long)(g0 + g) * S + s_begin;
        for (int ls = 0; ls < nseg; ++ls) dst[ls] = done[ls][g];
    }
}

// CSR hand-back of a few scattered genes (device-side list): one pass over the stored values of the batch's gene window;
// a value whose gene is on the list (cmap[gene] = its position k, else -1) is appended to slot space k with one atomic
// (the counts of the listed genes were zeroed).  Only runs when *mode_dev == want_mode.
__global__ void __launch_bounds__(256) stage_csr_list_kernel(const float* __restrict__ data, const int32_t* __restrict__ indices,
                                                             const long long* __restrict__ indptr, int n_rows, int gene_lb, int b,
                                                             const int* __restrict__ cmap, const int* __restrict__ mode_dev,
                                                             int want_mode, const illico_plan_t pl, float* __restrict__ ir_vals,
                                                             uint32_t* __restrict__ ir_cnt) {
    if (*mode_dev != want_mode) return;
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int S = pl.n_segments, c_hi = gene_lb + b;
    for (long long r = warp; r < n_rows; r += nwarps) {
        long long e0 = indptr[r];
        const long long e1 = indptr[r + 1];
        if (gene_lb > 0) e0 += lower_bound_i32(indices + e0, e1 - e0, gene_lb);
        const int seg = pl.cell_seg[r];
        const int base = pl.seg_base[seg], cap = pl.seg_base[seg + 1] - base;
        for (long long e = e0 + lane; ; e += 32) {
            const int c = (e < e1) ? __ldcs(indices + e) : 0x7fffffff;
            if (__all_sync(FULL, c >= c_hi)) break;
            if (c < c_hi) {
                const int k = cmap[c - gene_lb];
                const float v = __ldcs(data + e);
                if (k >= 0 && v != 0.0f) {
                    const uint32_t slot = atomicAdd(&ir_cnt[(long long)k * S + seg], 1u);
                    if (slot < (uint32_t)cap) ir_vals[(long long)k * pl.slot_cap + base + slot] = v;
                }
            }
        }
    }
}

// CSC: one CTA per gene column of the batch.
__global__ void __launch_bounds__(256) stage_csc_kernel(const float* __restrict__ data, const int32_t* __restrict__ indices,
                                                        const long long* __restrict__ indptr, int gene_lb, int b,
                                                        const illico_plan_t pl, float* __restrict__ ir_vals,
                                                        uint32_t* __restrict__ ir_cnt) {
    const int S = pl.n_segments;
    for (int j = blockIdx.x; j < b; j += gridDim.x) {
        const long long start = indptr[gene_lb + j], end = indptr[gene_lb + j + 1];
        for (long long k = start + threadIdx.x; k < end; k += blockDim.x) {
            const float v = __ldcs(data + k);
            if (v == 0.0f) continue;
            const int s = pl.cell_seg[indices[k]];
            const int base = pl.seg_base[s], cap = pl.seg_base[s + 1] - base;
            const uint32_t slot = atomicAdd(&ir_cnt[(long long)j * S + s], 1u);
            if (slot < (uint32_t)cap) ir_vals[(long long)j * pl.slot_cap + base + slot] = v;
        }
    }
}

// illico/utils/ranking.py:245-273: every row's indices must ascend
__global__ void check_csr_sorted_kernel(const int32_t* __restrict__ indices, const long long* __restrict__ indptr,
                                        long long n_rows, int* flag) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < n_rows; r += nwarps) {
        const long long start = indptr[r], end = indptr[r + 1];
        for (long long k = start + 1 + lane; k < end; k += 32)
            if (indices[k] < indices[k - 1]) *flag = 0;
    }
}

// ------------------------------------------------------------------------------------------------------
template <bool TILE, int VEC>
static void launch_stage_dense_t(dim3 grid, cudaStream_t stream, const float* X, long long ld, int gene_lb, int b,
                                 const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, int segs_per_cta) {
    ILLICO_LAUNCH("stage_dense_kernel", stream,
                  stage_dense_kernel<TILE, VEC><<<grid, STAGE_WARPS * 32, 0, stream>>>(X, ld, gene_lb, b, *plan, ir_vals, ir_cnt, segs_per_cta));
}

// stage_dense_tma.cu
bool stage_dense_tma_ok(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan);
int launch_stage_dense_tma(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                           uint32_t* ir_cnt, int seg_lo, int seg_hi, cudaStream_t stream, int segs_per_cta = 0);

int launch_stage_dense(const float* X, long long ld, int gene_lb, int b, const illico_plan_t* plan, float* ir_vals,
                       uint32_t* ir_cnt, cudaStream_t stream) {
    if (b <= 0 || plan->n_segments <= 0) return 0;
    if (ld <= 0 || ld >= (1ll << 30)) { set_error("leading dimension %lld out of range", ld); return 1; }
    // 16-byte aligned batches: rows come in through the TMA engine; anything else takes the plain-load kernel below
    if (stage_dense_tma_ok(X, ld, gene_lb, b, plan)) {
        const int rc = launch_stage_dense_tma(X, ld, gene_lb, b, plan, ir_vals, ir_cnt, 0, plan->n_segments, stream);
        if (rc >= 0) return rc;
    }
    const int S = plan->n_segments;
    long long avg = plan->n_cells / S;
    if (avg < 1) avg = 1;
    // ~512 cells per CTA: enough CTAs (tens of waves) that the last partial wave costs a few percent
    int segs_per_cta = (int)(512 / avg);
    if (segs_per_cta < 1) segs_per_cta = 1;
    if (segs_per_cta > STAGE_MAX_SEGS) segs_per_cta = STAGE_MAX_SEGS;
    long long gy = (S + segs_per_cta - 1) / segs_per_cta;
    // two genes per lane (64-bit loads) when the batch is 8-byte aligned
    const bool vec2 = ((reinterpret_cast<uintptr_t>(X) & 7) == 0) && (ld % 2 == 0) &&
                      (gene_lb % 2 == 0) && (b % 2 == 0);
    const int gpc = STAGE_WARPS * 32 * (vec2 ? 2 : 1);
    const unsigned gx = (unsigned)((b + gpc - 1) / gpc);
    const bool tile = gy <= 65535 && plan->max_group_size < 65536;
    if (!tile) {  // more than a million segments: any number of segments per CTA, counts written directly
        while (gy > 65535) { segs_per_cta *= 2; gy = (S + segs_per_cta - 1) / segs_per_cta; }
    }
    const dim3 grid(gx, (unsigned)gy);
    if (tile && vec2) launch_stage_dense_t<true, 2>(grid, stream, X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta);
    else if (tile) launch_stage_dense_t<true, 1>(grid, stream, X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta);
    else if (vec2) launch_stage_dense_t<false, 2>(grid, stream, X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta);
    else launch_stage_dense_t<false, 1>(grid, stream, X, ld, gene_lb, b, plan, ir_vals, ir_cnt, segs_per_cta);
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

size_t stage_csr_workspace_bytes(const illico_plan_t* plan, int b) {
    const int K = (b + CSR_GC - 1) / CSR_GC;
    return (size_t)plan->n_cells * (size_t)(K + 1) * sizeof(int32_t) + 256;
}

// mode_dev != NULL: the kernels only run when *mode_dev == want_mode (a decision taken on the device)
int launch_stage_csr_if(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                        const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, void* workspace, size_t workspace_bytes,
                        const int* mode_dev, int want_mode, cudaStream_t stream) {
    if (b <= 0 || plan->n_cells <= 0) return 0;
    const int K = (b + CSR_GC - 1) / CSR_GC;
    if (!workspace || workspace_bytes < stage_csr_workspace_bytes(plan, b)) {
        set_error("illico_stage_csr_f32: workspace too small (%zu < %zu bytes)", workspace_bytes, stage_csr_workspace_bytes(plan, b));
        return 1;
    }
    int32_t* split = reinterpret_cast<int32_t*>(workspace);
    long long blocks = ((long long)plan->n_cells + 7) / 8;
    if (blocks > 148 * 32) blocks = 148 * 32;
    ILLICO_LAUNCH("csr_split_kernel", stream, csr_split_kernel<<<(unsigned)blocks, 256, 0, stream>>>(indices, indptr, plan->n_cells, gene_lb, b, K, split, mode_dev, want_mode));
    ILLICO_CUDA_OK(cudaGetLastError());
    const int S = plan->n_segments;
    long long avg = plan->n_cells / S;
    if (avg < 1) avg = 1;
    int segs_per_cta = (int)(1024 / avg);
    if (segs_per_cta < 1) segs_per_cta = 1;
    if (segs_per_cta > CSR_MAX_SEGS) segs_per_cta = CSR_MAX_SEGS;
    const long long gy = (S + segs_per_cta - 1) / segs_per_cta;
    if (gy > 65535) { set_error("too many segments (%d) for one CSR staging launch", S); return 1; }
    // (a partial check only: it catches plans whose groups were not cut at all.  The guarantee that every segment has
    // fewer than 65536 cells is the plan's own -- HostPlan refuses longer segments, see seg_pos in illico_b200.h)
    if (plan->max_group_size >= 65536 && plan->n_segments == plan->n_groups) {
        set_error("segments of 65536 or more cells are not supported by the CSR staging kernel");
        return 1;
    }
    const size_t smem = CSR_MAX_ROWS * 8 + CSR_CAP * 4 + (2 * CSR_GC + 1) * 4 + CSR_MAX_ROWS * 4 + 9 * 4 +
                        CSR_MAX_SEGS * CSR_GC * 2 + 16;
    ILLICO_CUDA_OK(cudaFuncSetAttribute(stage_csr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ILLICO_LAUNCH("stage_csr_kernel", stream, stage_csr_kernel<<<dim3((unsigned)K, (unsigned)gy), CSR_THREADS, smem, stream>>>(data, indices, indptr, gene_lb, b, K, split,
                                                                                     *plan, ir_vals, ir_cnt, segs_per_cta, mode_dev, want_mode));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_stage_csr(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                     const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, void* workspace, size_t workspace_bytes,
                     cudaStream_t stream) {
    return launch_stage_csr_if(data, indices, indptr, gene_lb, b, plan, ir_vals, ir_cnt, workspace, workspace_bytes, nullptr, 0, stream);
}

// stages the genes of a device-side list (see stage_csr_list_kernel); the counts of up to `max_list` genes are zeroed first
int launch_stage_csr_list(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b, const int* cmap,
                          const int* mode_dev, int want_mode, int max_list, const illico_plan_t* plan, float* ir_vals,
                          uint32_t* ir_cnt, cudaStream_t stream) {
    if (b <= 0 || plan->n_cells <= 0 || max_list <= 0) return 0;
    ILLICO_CUDA_OK(cudaMemsetAsync(ir_cnt, 0, (size_t)max_list * (size_t)plan->n_segments * sizeof(uint32_t), stream));
    long long blocks = ((long long)plan->n_cells + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ILLICO_LAUNCH("stage_csr_list_kernel", stream,
                  stage_csr_list_kernel<<<(unsigned)blocks, 256, 0, stream>>>(data, indices, indptr, plan->n_cells, gene_lb, b, cmap, mode_dev,
                                                                              want_mode, *plan, ir_vals, ir_cnt));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

// stages the genes of a device-side list from a dense matrix (see stage_dense_list_kernel)
int launch_stage_dense_list(const float* X, long long ld, int gene_lb, const int* list, const int* n_list_dev,
                            const int* mode_dev, int want_mode, const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt,
                            cudaStream_t stream) {
    const int S = plan->n_segments;
    if (S <= 0) return 0;
    if (ld <= 0 || ld >= (1ll << 30)) { set_error("leading dimension %lld out of range", ld); return 1; }
    long long avg = plan->n_cells / S;
    if (avg < 1) avg = 1;
    int segs_per_cta = (int)(512 / avg);
    if (segs_per_cta < 1) segs_per_cta = 1;
    if (segs_per_cta > STAGE_MAX_SEGS) segs_per_cta = STAGE_MAX_SEGS;
    ILLICO_LAUNCH("stage_dense_list_kernel", stream,
                  stage_dense_list_kernel<<<148 * 8, STAGE_WARPS * 32, 0, stream>>>(X, ld, gene_lb, list, n_list_dev, mode_dev, want_mode,
                                                                                     *plan, ir_vals, ir_cnt, segs_per_cta));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_stage_csc(const float* data, const int32_t* indices, const long long* indptr, int gene_lb, int b,
                     const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, cudaStream_t stream) {
    if (b <= 0) return 0;
    int blocks = b < 148 * 32 ? b : 148 * 32;
    ILLICO_LAUNCH("stage_csc_kernel", stream, stage_csc_kernel<<<blocks, 256, 0, stream>>>(data, indices, indptr, gene_lb, b, *plan, ir_vals, ir_cnt));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int launch_check_csr_sorted(const int32_t* indices, const long long* indptr, long long n_rows, int* d_flag,
                            int* h_sorted, cudaStream_t stream) {
    int one = 1;
    ILLICO_CUDA_OK(cudaMemcpyAsync(d_flag, &one, sizeof(int), cudaMemcpyHostToDevice, stream));
    if (n_rows > 0) {
        long long blocks = (n_rows + 7) / 8;
        if (blocks > 148 * 32) blocks = 148 * 32;
        ILLICO_LAUNCH("check_csr_sorted_kernel", stream, check_csr_sorted_kernel<<<(unsigned)blocks, 256, 0, stream>>>(indices, indptr, n_rows, d_flag));
        ILLICO_CUDA_OK(cudaGetLastError());
    }
    int h = -1;
    ILLICO_CUDA_OK(cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, stream));
    ILLICO_CUDA_OK(cudaStreamSynchronize(stream));
    *h_sorted = h;
    return 0;
}

}  // namespace illico
