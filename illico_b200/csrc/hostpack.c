/* hostpack.c -- host side of the packed upload (plain C, compiled by gcc and linked into libillico_b200.so).
 *
 * A dense float32 expression matrix is ~90 % zeros, and its upload is what the end-to-end time consists of (9.6 GB over
 * PCIe at the K562 shape: 0.17 of 0.18 s).  The reference has no such boundary (zero-copy InRAMDataHandler.fetch,
 * illico/utils/registry.py:97-100).  Here the host threads that used to copy row chunks into pinned staging buffers
 * squeeze them instead: per row, one bit per element (non-zero or not) and the non-zero values in order, i.e. 1/8 + 4 d
 * bytes per element at density d -- 0.13 of the raw bytes at d = 0.1.  The packed chunk goes over PCIe and
 * illico_unpack_rows_f32 (csrc/extras.cu) rebuilds the dense rows in HBM at memory speed; everything downstream sees the
 * same dense matrix.  The scan runs at the host's memory bandwidth (AVX-512 compress-store, AVX2 permute table or scalar
 * code, chosen at run time).  -0.0 packs as a zero, NaN as a value (x != 0), like every kernel treats them.
 */
#include <immintrin.h>
#include <stdint.h>
#include <stddef.h>
#include <string.h>

#define PREFETCH_AHEAD 4096

static void scalar_words(const float* row, const int32_t* cols, long c0, long c1, uint32_t* mask, float** out) {
    /* columns [c0, c1) of one row (element k is row[cols[k]] with a column list), c0 a multiple of 32 */
    float* o = *out;
    for (long c = c0; c < c1; c += 32) {
        uint32_t m = 0;
        const long e = c + 32 < c1 ? c + 32 : c1;
        for (long k = c; k < e; ++k) {
            const float v = cols ? row[cols[k]] : row[k];
            if (v != 0.0f) { m |= 1u << (k - c); *o++ = v; }
        }
        mask[c >> 5] = m;
    }
    *out = o;
}

__attribute__((target("avx512f"))) static void row_avx512(const float* row, long n_cols, uint32_t* mask, float** out) {
    float* o = *out;
    const __m512 zero = _mm512_setzero_ps();
    const long full = n_cols & ~31L;
    for (long c = 0; c < full; c += 32) {
        /* the scan is bound by how many cache lines a core keeps in flight: ask for the lines 4 KB ahead (they may belong
         * to the next row -- rows of a chunk are adjacent or a fixed stride apart -- or lie past the end: harmless) */
        _mm_prefetch((const char*)(row + c) + PREFETCH_AHEAD, _MM_HINT_T0);
        _mm_prefetch((const char*)(row + c) + PREFETCH_AHEAD + 64, _MM_HINT_T0);
        const __m512 a = _mm512_loadu_ps(row + c), b = _mm512_loadu_ps(row + c + 16);
        const __mmask16 ma = _mm512_cmp_ps_mask(a, zero, _CMP_NEQ_UQ), mb = _mm512_cmp_ps_mask(b, zero, _CMP_NEQ_UQ);
        /* compress in a register, store all 16 lanes, advance by the count: the memory form of vcompressps is microcoded
         * (very slow) on some CPUs; the caller leaves 16 floats of slack */
        _mm512_storeu_ps(o, _mm512_maskz_compress_ps(ma, a));
        o += __builtin_popcount((unsigned)ma);
        _mm512_storeu_ps(o, _mm512_maskz_compress_ps(mb, b));
        o += __builtin_popcount((unsigned)mb);
        mask[c >> 5] = (uint32_t)ma | ((uint32_t)mb << 16);
    }
    *out = o;
    if (full < n_cols) scalar_words(row, NULL, full, n_cols, mask, out);
}

/* row_avx512 over the elements row[cols[k]]: the hardware gather loads them (cols ascend, so a gather's 16 lanes touch few
 * cache lines), the squeeze is the same */
__attribute__((target("avx512f"))) static void gather_avx512(const float* row, const int32_t* cols, long n_cols, uint32_t* mask,
                                                            float** out) {
    float* o = *out;
    const __m512 zero = _mm512_setzero_ps();
    const long full = n_cols & ~31L;
    for (long c = 0; c < full; c += 32) {
        const __m512 a = _mm512_i32gather_ps(_mm512_loadu_si512((const void*)(cols + c)), row, 4);
        const __m512 b = _mm512_i32gather_ps(_mm512_loadu_si512((const void*)(cols + c + 16)), row, 4);
        const __mmask16 ma = _mm512_cmp_ps_mask(a, zero, _CMP_NEQ_UQ), mb = _mm512_cmp_ps_mask(b, zero, _CMP_NEQ_UQ);
        _mm512_storeu_ps(o, _mm512_maskz_compress_ps(ma, a));
        o += __builtin_popcount((unsigned)ma);
        _mm512_storeu_ps(o, _mm512_maskz_compress_ps(mb, b));
        o += __builtin_popcount((unsigned)mb);
        mask[c >> 5] = (uint32_t)ma | ((uint32_t)mb << 16);
    }
    *out = o;
    if (full < n_cols) scalar_words(row, cols, full, n_cols, mask, out);
}

static int32_t g_perm[256][8];
static int g_perm_ready = 0;
static void build_perm(void) {
    for (int m = 0; m < 256; ++m) {
        int k = 0;
        for (int b = 0; b < 8; ++b) if (m & (1 << b)) g_perm[m][k++] = b;
        for (; k < 8; ++k) g_perm[m][k] = 0;
    }
    g_perm_ready = 1;
}

__attribute__((target("avx2"))) static void row_avx2(const float* row, long n_cols, uint32_t* mask, float** out) {
    /* stores 8 floats per step and advances by the number of non-zeros: the caller leaves 8 floats of slack */
    float* o = *out;
    const __m256 zero = _mm256_setzero_ps();
    const long full = n_cols & ~31L;
    for (long c = 0; c < full; c += 32) {
        uint32_t m = 0;
        _mm_prefetch((const char*)(row + c) + PREFETCH_AHEAD, _MM_HINT_T0);
        _mm_prefetch((const char*)(row + c) + PREFETCH_AHEAD + 64, _MM_HINT_T0);
        for (int q = 0; q < 4; ++q) {
            const __m256 v = _mm256_loadu_ps(row + c + 8 * q);
            const int mm = _mm256_movemask_ps(_mm256_cmp_ps(v, zero, _CMP_NEQ_UQ));
            const __m256i idx = _mm256_loadu_si256((const __m256i*)g_perm[mm]);
            _mm256_storeu_ps(o, _mm256_permutevar8x32_ps(v, idx));
            o += __builtin_popcount((unsigned)mm);
            m |= (uint32_t)mm << (8 * q);
        }
        mask[c >> 5] = m;
    }
    *out = o;
    if (full < n_cols) scalar_words(row, NULL, full, n_cols, mask, out);
}

__attribute__((target("avx2"))) static void gather_avx2(const float* row, const int32_t* cols, long n_cols, uint32_t* mask, float** out) {
    float* o = *out;
    const __m256 zero = _mm256_setzero_ps();
    const long full = n_cols & ~31L;
    for (long c = 0; c < full; c += 32) {
        uint32_t m = 0;
        for (int q = 0; q < 4; ++q) {
            const __m256 v = _mm256_i32gather_ps(row, _mm256_loadu_si256((const __m256i*)(cols + c + 8 * q)), 4);
            const int mm = _mm256_movemask_ps(_mm256_cmp_ps(v, zero, _CMP_NEQ_UQ));
            const __m256i idx = _mm256_loadu_si256((const __m256i*)g_perm[mm]);
            _mm256_storeu_ps(o, _mm256_permutevar8x32_ps(v, idx));
            o += __builtin_popcount((unsigned)mm);
            m |= (uint32_t)mm << (8 * q);
        }
        mask[c >> 5] = m;
    }
    *out = o;
    if (full < n_cols) scalar_words(row, cols, full, n_cols, mask, out);
}

/* which code path this CPU takes: 2 = AVX-512, 1 = AVX2, 0 = scalar */
int illico_host_pack_isa(void) {
    __builtin_cpu_init();
    if (__builtin_cpu_supports("avx512f")) return 2;
    if (__builtin_cpu_supports("avx2")) return 1;
    return 0;
}

static long pack_rows(const float* src, long row_stride, const int64_t* rows, long n_rows, const int32_t* cols, long n_cols,
                      uint32_t* mask, uint32_t* row_off, float* vals, long vals_cap) {
    const int isa = illico_host_pack_isa();
    if (isa == 1 && !g_perm_ready) build_perm();
    const long W = (n_cols + 31) / 32;
    float* o = vals;
    for (long r = 0; r < n_rows; ++r) {
        if ((o - vals) + n_cols + 16 > vals_cap) return -1;
        row_off[r] = (uint32_t)(o - vals);
        const float* row = src + (rows ? rows[r] : r) * row_stride;
        if (cols) {
            if (isa == 2) gather_avx512(row, cols, n_cols, mask + r * W, &o);
            else if (isa == 1) gather_avx2(row, cols, n_cols, mask + r * W, &o);
            else scalar_words(row, cols, 0, n_cols, mask + r * W, &o);
        } else if (isa == 2) row_avx512(row, n_cols, mask + r * W, &o);
        else if (isa == 1) row_avx2(row, n_cols, mask + r * W, &o);
        else scalar_words(row, NULL, 0, n_cols, mask + r * W, &o);
    }
    row_off[n_rows] = (uint32_t)(o - vals);
    return (long)(o - vals);
}

/* Packs rows [0, n_rows) of a row-major float32 matrix (row stride in elements, n_cols columns read per row):
 *   mask    [n_rows][W] uint32, W = (n_cols + 31) / 32: bit k of word w = element 32 w + k is non-zero
 *   row_off [n_rows + 1] uint32: position of each row's first value in vals
 *   vals    the non-zero values, row by row, in column order; capacity vals_cap floats (16 floats of slack included)
 * Returns the number of values, or -1 when they do not fit (the caller then sends the chunk as it is). */
long illico_host_pack_rows_f32(const float* src, long row_stride, long n_rows, long n_cols, uint32_t* mask, uint32_t* row_off,
                               float* vals, long vals_cap) {
    return pack_rows(src, row_stride, NULL, n_rows, NULL, n_cols, mask, row_off, vals, vals_cap);
}

/* The same for the rows rows[0 .. n_rows) of the matrix (any order; packed row r is source row rows[r]): the upload of the
 * cells of the groups a call tests gathers them while it squeezes them. */
long illico_host_pack_row_list_f32(const float* src, long row_stride, const int64_t* rows, long n_rows, long n_cols, uint32_t* mask,
                                   uint32_t* row_off, float* vals, long vals_cap) {
    return pack_rows(src, row_stride, rows, n_rows, NULL, n_cols, mask, row_off, vals, vals_cap);
}

/* The same for the columns cols[0 .. n_cols) of rows rows[0 .. n_rows) (rows [0, n_rows) when rows is NULL): packed row r
 * holds src[rows[r], cols[k]] as its element k.  The upload of the genes a call tests (mask_var=) gathers them while it
 * squeezes them, so that only their bytes cross PCIe. */
long illico_host_pack_cols_f32(const float* src, long row_stride, const int64_t* rows, long n_rows, const int32_t* cols, long n_cols,
                               uint32_t* mask, uint32_t* row_off, float* vals, long vals_cap) {
    return pack_rows(src, row_stride, rows, n_rows, cols, n_cols, mask, row_off, vals, vals_cap);
}
