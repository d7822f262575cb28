// sort.cuh -- block / warp sorting primitives on 32-bit keys (sm_100a).
//
// Ranking never moves payloads: the rank kernels sort KEYS ONLY (the order-preserving image of the
// non-zero values) and look ranks up by binary search, so group labels stay where they were staged.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace illico {

// Shared scratch of the block radix sort: one digit histogram per warp + digit totals.
//   hist : [NW * 256] uint32 (NW = blockDim.x / 32, blockDim.x >= 256)
//   aux  : [40] uint32
constexpr int RADIX_AUX_WORDS = 40;

// Stable LSD radix sort of `n` keys, 8-bit digits, ping-pong between `a` (input) and `b`, optionally carrying one
// payload per key (ValT, ping-pong between `va` and `vb`: it moves with its key).  Pointers may be shared or global
// (generic addressing).  Passes in which every key has the same digit are skipped (integer-valued floats have two constant
// low bytes).  Returns the buffer that holds the sorted keys; the payloads are in `va` if that is `a`, else in `vb`.
// Must be called by all threads of the block.
struct NoPayload {};
template <typename KeyT, typename ValT>
static __device__ __forceinline__ KeyT* block_radix_sort_impl(KeyT* a, KeyT* b, ValT* va, ValT* vb, int n, uint32_t* hist,
                                                              uint32_t* aux) {
    constexpr bool PAY = !std::is_same<ValT, NoPayload>::value;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, NW = blockDim.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    if (n <= 1) return a;
    const int chunk = (((n + NW - 1) / NW) + 31) & ~31;
    const int beg = min(w * chunk, n), end = min(beg + chunk, n);
    uint32_t* myhist = hist + w * 256;

    for (int shift = 0; shift < (int)sizeof(KeyT) * 8; shift += 8) {
        for (int i = tid; i < NW * 256; i += blockDim.x) hist[i] = 0;
        if (tid == 0) aux[32] = 0;
        __syncthreads();
        // ---- per-warp digit counts (warp-private counters: match_any aggregates equal digits)
        // (the next 32 keys are requested before the current ones are counted: the loop is one dependent load per round)
        KeyT nxt = (beg + lane < end) ? a[beg + lane] : KeyT(0);
        for (int i0 = beg; i0 < end; i0 += 32) {
            int i = i0 + lane;
            bool valid = i < end;
            const KeyT cur = nxt;
            if (i + 32 < end) nxt = a[i + 32];
            uint32_t d = valid ? ((uint32_t)(cur >> shift) & 255u) : (256u + lane);
            unsigned peers = __match_any_sync(FULL, d);
            if (valid && lane == __ffs(peers) - 1) myhist[d] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        // ---- digit totals, exclusive scan over (digit major, warp minor)
        uint32_t total = 0;
        if (tid < 256) {
            for (int ww = 0; ww < NW; ++ww) {
                uint32_t c = hist[ww * 256 + tid];
                hist[ww * 256 + tid] = total;
                total += c;
            }
            if (total == (uint32_t)n) aux[32] = 1;  // every key shares this digit: nothing to do
        }
        uint32_t incl = warp_incl_scan(total, lane);
        if (tid < 256 && lane == 31) aux[w] = incl;
        __syncthreads();
        const bool skip = aux[32] != 0;  // block-uniform
        __syncthreads();                 // everyone has read the flag before the next pass clears it
        if (skip) continue;
        if (tid < 256) {
            uint32_t base = incl - total;
            for (int ww = 0; ww < w; ++ww) base += aux[ww];
            for (int ww = 0; ww < NW; ++ww) hist[ww * 256 + tid] += base;
        }
        __syncthreads();
        // ---- stable scatter: each warp walks its chunk in order
        nxt = (beg + lane < end) ? a[beg + lane] : KeyT(0);
        for (int i0 = beg; i0 < end; i0 += 32) {
            int i = i0 + lane;
            bool valid = i < end;
            const KeyT key = nxt;
            if (i + 32 < end) nxt = a[i + 32];
            uint32_t d = valid ? ((uint32_t)(key >> shift) & 255u) : (256u + lane);
            unsigned peers = __match_any_sync(FULL, d);
            uint32_t pos = valid ? myhist[d] + __popc(peers & lt) : 0u;
            if (valid) b[pos] = key;
            if constexpr (PAY) {
                if (valid) vb[pos] = va[i];
            }
            __syncwarp();
            if (valid && lane == __ffs(peers) - 1) myhist[d] += __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        KeyT* t = a; a = b; b = t;
        if constexpr (PAY) {
            ValT* tv = va; va = vb; vb = tv;
        }
    }
    return a;
}
template <typename KeyT>
static __device__ __noinline__ KeyT* block_radix_sort_t(KeyT* a, KeyT* b, int n, uint32_t* hist, uint32_t* aux) {
    return block_radix_sort_impl<KeyT, NoPayload>(a, b, nullptr, nullptr, n, hist, aux);
}
template <typename KeyT, typename ValT>
static __device__ __noinline__ KeyT* block_radix_sort_t(KeyT* a, KeyT* b, int n, uint32_t* hist, uint32_t* aux, ValT* va,
                                                        ValT* vb) {
    return block_radix_sort_impl<KeyT, ValT>(a, b, va, vb, n, hist, aux);
}
static __device__ __forceinline__ uint32_t* block_radix_sort(uint32_t* a, uint32_t* b, int n, uint32_t* hist, uint32_t* aux) {
    return block_radix_sort_t<uint32_t>(a, b, n, hist, aux);
}

// Bitonic sort of P (power of two) keys in shared memory by ONE warp.
__device__ __forceinline__ void warp_bitonic_sort(uint32_t* buf, int P, int lane) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (P >> 1); t += 32) {
                int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                int ixj = i | j;
                bool up = (i & k) == 0;
                uint32_t x = buf[i], y = buf[ixj];
                if ((x > y) == up) { buf[i] = y; buf[ixj] = x; }
            }
            __syncwarp();
        }
    }
}

// Bitonic sort of P (power of two) (key, value) pairs in shared memory by the whole block.
__device__ __forceinline__ void block_bitonic_sort_pairs(uint32_t* keys, uint32_t* vals, int P) {
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
                int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                int ixj = i | j;
                bool up = (i & k) == 0;
                uint32_t x = keys[i], y = keys[ixj];
                if ((x > y) == up) {
                    keys[i] = y; keys[ixj] = x;
                    uint32_t vx = vals[i]; vals[i] = vals[ixj]; vals[ixj] = vx;
                }
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace illico
