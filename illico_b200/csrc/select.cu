// select.cu -- the cells of the groups a call tests (scanpy's rank_genes_groups(groups=...)), one-versus-reference, and the
// genes it tests (mask_var=) (sm_100a).
//
// A one-versus-reference test of a few groups needs only their cells and the reference's.  These kernels cut those rows
// out of a device-resident matrix, keeping their ascending order, so that the group plan built from the same rows gives
// every selected group the segments and summation order of the full call and the six dispatchers run unchanged on the
// result.  A call that tests a subset of the genes needs only their columns: the dense gather takes a column list (and an
// optional row list, in the same pass), and a CSR row is compacted through a new_col table by the CSC kernels with the
// roles of rows and columns swapped.  Values are moved as bit patterns: float32 or float64 (a float64 matrix stays float64
// and keeps going through the recode path).  Every call only enqueues work on `stream`.
#include "common.cuh"

namespace illico {

namespace {

constexpr int SEL_THREADS = 256;
constexpr int SEL_SCAN_THREADS = 1024;

// One CTA per (output row, tile of 4 * 256 columns): the four loads of a thread are issued before its stores.  Columns
// [n_cols, out_ld) of the output row are written as zeros (the padding that keeps rows 16-byte aligned).  ROWS: output row r
// is source row rows[r] (else r).  COLS: output column c is source column cols[c] (else c); lane t of a warp reads the
// t-th of 32 consecutive entries of the ascending list, so a warp's loads fall into as few sectors as the list allows.
template <typename T, bool ROWS, bool COLS>
__global__ void __launch_bounds__(SEL_THREADS) select_dense_kernel(const T* __restrict__ X, long long ld, long long n_cols,
                                                                   const int32_t* __restrict__ rows, const int32_t* __restrict__ cols,
                                                                   T* __restrict__ out, long long out_ld) {
    const long long r = blockIdx.x;
    const T* src = X + (ROWS ? (long long)rows[r] : r) * ld;
    T* dst = out + r * out_ld;
    const long long c0 = (long long)blockIdx.y * (4 * SEL_THREADS) + threadIdx.x;
    T v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long c = c0 + k * SEL_THREADS;
        v[k] = c < n_cols ? src[COLS ? (long long)__ldg(cols + c) : c] : T(0);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long c = c0 + k * SEL_THREADS;
        if (c < out_ld) dst[c] = v[k];
    }
}

// out_indptr[i + 1] = stored entries of row rows[i]
__global__ void __launch_bounds__(SEL_THREADS) csr_row_lengths_kernel(const long long* __restrict__ indptr, const int32_t* __restrict__ rows,
                                                                      long long n_rows, long long* __restrict__ out_indptr) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (long long)gridDim.x * blockDim.x) {
        const int32_t r = rows[i];
        out_indptr[i + 1] = indptr[r + 1] - indptr[r];
    }
}

// One CTA per column: out_indptr[c + 1] = entries of column c whose row is kept (new_row[row] >= 0)
__global__ void __launch_bounds__(SEL_THREADS) csc_kept_count_kernel(const int32_t* __restrict__ indices, const long long* __restrict__ indptr,
                                                                     const int32_t* __restrict__ new_row, long long* __restrict__ out_indptr) {
    __shared__ unsigned long long red[32];
    const int c = blockIdx.x;
    const long long e0 = indptr[c], e1 = indptr[c + 1];
    unsigned long long n = 0;
    for (long long e = e0 + threadIdx.x; e < e1; e += SEL_THREADS) n += new_row[indices[e]] >= 0;
    n = block_sum(n, red);
    if (threadIdx.x == 0) out_indptr[c + 1] = (long long)n;
}

// In place, one CTA: a[1..n] holds lengths on entry, a[0..n] their exclusive scan on exit (a[0] = 0, a[n] = the total).
// Thread t owns a contiguous run of the lengths: it sums its run, the CTA scans the 1024 sums, and each thread rewrites its
// run from its offset.  (At most a few million lengths -- the rows of a matrix or the columns of a batch -- so one CTA
// reads them in well under a millisecond.)
__global__ void __launch_bounds__(SEL_SCAN_THREADS) scan_lengths_kernel(long long* __restrict__ a, long long n) {
    __shared__ long long part[SEL_SCAN_THREADS];
    const long long per = (n + SEL_SCAN_THREADS - 1) / SEL_SCAN_THREADS;
    const long long b0 = 1 + threadIdx.x * per;
    const long long b1 = b0 + per < n + 1 ? b0 + per : n + 1;
    long long s = 0;
    for (long long i = b0; i < b1; ++i) s += a[i];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < SEL_SCAN_THREADS; o <<= 1) {       // Hillis-Steele inclusive scan of the 1024 sums
        const long long t = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += t;
        __syncthreads();
    }
    long long run = part[threadIdx.x] - s;
    for (long long i = b0; i < b1; ++i) {
        run += a[i];
        a[i] = run;
    }
    if (threadIdx.x == 0) a[0] = 0;
}

// Warp per output row: the row's stored values and column indices, copied as they are (they stay sorted)
template <typename T>
__global__ void __launch_bounds__(SEL_THREADS) csr_copy_rows_kernel(const T* __restrict__ data, const int32_t* __restrict__ indices,
                                                                    const long long* __restrict__ indptr, const int32_t* __restrict__ rows,
                                                                    long long n_rows, const long long* __restrict__ out_indptr,
                                                                    T* __restrict__ out_data, int32_t* __restrict__ out_indices) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp; i < n_rows; i += nwarps) {
        const long long s = indptr[rows[i]], o = out_indptr[i], len = out_indptr[i + 1] - o;
        for (long long k = lane; k < len; k += 32) {
            out_data[o + k] = data[s + k];
            out_indices[o + k] = indices[s + k];
        }
    }
}

// One CTA per column, tiles of 256 entries in order: a warp ballots which of its 32 entries are kept, the eight warp counts
// are scanned in shared memory, and each kept entry lands at the column's output offset + the kept entries before it --
// a stable compaction, so the renumbered rows of a column still ascend.
template <typename T>
__global__ void __launch_bounds__(SEL_THREADS) csc_compact_kernel(const T* __restrict__ data, const int32_t* __restrict__ indices,
                                                                  const long long* __restrict__ indptr, const int32_t* __restrict__ new_row,
                                                                  const long long* __restrict__ out_indptr, T* __restrict__ out_data,
                                                                  int32_t* __restrict__ out_indices) {
    constexpr int NW = SEL_THREADS / 32;
    __shared__ int wcnt[NW];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c = blockIdx.x;
    const long long e0 = indptr[c], e1 = indptr[c + 1];
    long long o = out_indptr[c];
    for (long long base = e0; base < e1; base += SEL_THREADS) {
        const long long e = base + threadIdx.x;
        int nr = -1;
        T v = T(0);
        if (e < e1) {
            nr = new_row[indices[e]];
            v = data[e];
        }
        const unsigned m = __ballot_sync(FULL, nr >= 0);
        if (lane == 0) wcnt[w] = __popc(m);
        __syncthreads();
        int before = 0, tile = 0;
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            before += k < w ? wcnt[k] : 0;
            tile += wcnt[k];
        }
        if (nr >= 0) {
            const long long pos = o + before + __popc(m & ((1u << lane) - 1u));
            out_data[pos] = v;
            out_indices[pos] = nr;
        }
        o += tile;
        __syncthreads();     // wcnt is rewritten by the next tile
    }
}

unsigned grid_for(long long work, long long per_block) {
    long long blocks = (work + per_block - 1) / per_block;
    if (blocks > 148 * 16) blocks = 148 * 16;
    return (unsigned)(blocks > 0 ? blocks : 1);
}

int value_bytes(int32_t dtype, const char* who) {
    if (dtype == ILLICO_DTYPE_F32) return 4;
    if (dtype == ILLICO_DTYPE_F64) return 8;
    set_error("%s: dtype must be ILLICO_DTYPE_F32 or ILLICO_DTYPE_F64, got %d", who, (int)dtype);
    return 0;
}

int scan_lengths(long long* out_indptr, long long n, cudaStream_t st) {
    ILLICO_LAUNCH("scan_lengths_kernel", st, scan_lengths_kernel<<<1, SEL_SCAN_THREADS, 0, st>>>(out_indptr, n));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename T, bool ROWS, bool COLS>
int launch_select_dense(const void* X, long long ld, long long n_cols, const int32_t* rows, const int32_t* cols, dim3 grid, void* out,
                        long long out_ld, cudaStream_t st) {
    ILLICO_LAUNCH("select_dense_kernel", st,
                  (select_dense_kernel<T, ROWS, COLS><<<grid, SEL_THREADS, 0, st>>>((const T*)X, ld, n_cols, rows, cols, (T*)out, out_ld)));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

// out[i, c] = X[rows ? rows[i] : i, cols ? cols[c] : c] for c < n_cols, zeros up to out_ld
int select_dense(const void* X, int vb, long long ld, long long n_cols, const int32_t* rows, const int32_t* cols, long long n_rows,
                 void* out, long long out_ld, cudaStream_t st, const char* who) {
    const long long tiles = (out_ld + 4 * SEL_THREADS - 1) / (4 * SEL_THREADS);
    if (tiles > 65535) { set_error("%s: rows wider than %d elements", who, 65535 * 4 * SEL_THREADS); return 1; }
    const dim3 grid((unsigned)n_rows, (unsigned)tiles);
    if (vb == 4) {
        if (!cols) return launch_select_dense<float, true, false>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
        if (rows) return launch_select_dense<float, true, true>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
        return launch_select_dense<float, false, true>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
    }
    if (!cols) return launch_select_dense<double, true, false>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
    if (rows) return launch_select_dense<double, true, true>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
    return launch_select_dense<double, false, true>(X, ld, n_cols, rows, cols, grid, out, out_ld, st);
}

}  // namespace

}  // namespace illico

using namespace illico;

extern "C" int illico_select_rows_dense(const void* X, int32_t dtype, int64_t ld, int64_t n_cols, const int32_t* rows, int64_t n_rows,
                                        void* out, int64_t out_ld, void* stream) {
    const int vb = value_bytes(dtype, "illico_select_rows_dense");
    if (!vb) return 1;
    if (n_rows <= 0 || out_ld <= 0) return 0;
    if (!X || !rows || !out || n_cols < 0 || ld < n_cols || out_ld < n_cols) {
        set_error("illico_select_rows_dense: bad argument");
        return 1;
    }
    if (n_rows > 0x7fffffffLL) { set_error("illico_select_rows_dense: more than 2^31 - 1 rows"); return 1; }
    return select_dense(X, vb, ld, n_cols, rows, nullptr, n_rows, out, out_ld, (cudaStream_t)stream, "illico_select_rows_dense");
}

extern "C" int illico_select_cols_dense(const void* X, int32_t dtype, int64_t ld, const int32_t* rows, int64_t n_rows, const int32_t* cols,
                                        int64_t n_cols, void* out, int64_t out_ld, void* stream) {
    const int vb = value_bytes(dtype, "illico_select_cols_dense");
    if (!vb) return 1;
    if (n_rows <= 0 || out_ld <= 0) return 0;
    if (!X || !out || n_cols < 0 || out_ld < n_cols || ld <= 0 || (n_cols > 0 && !cols)) {
        set_error("illico_select_cols_dense: bad argument");
        return 1;
    }
    if (n_rows > 0x7fffffffLL) { set_error("illico_select_cols_dense: more than 2^31 - 1 rows"); return 1; }
    return select_dense(X, vb, ld, n_cols, rows, cols, n_rows, out, out_ld, (cudaStream_t)stream, "illico_select_cols_dense");
}

extern "C" int illico_select_rows_csr_indptr(const int64_t* indptr, const int32_t* rows, int64_t n_rows, int64_t* out_indptr,
                                             void* stream) {
    if (!indptr || !out_indptr || (n_rows > 0 && !rows) || n_rows < 0) { set_error("illico_select_rows_csr_indptr: bad argument"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows > 0)
        ILLICO_LAUNCH("csr_row_lengths_kernel", st,
                      csr_row_lengths_kernel<<<grid_for(n_rows, SEL_THREADS), SEL_THREADS, 0, st>>>((const long long*)indptr, rows, n_rows,
                                                                                                 (long long*)out_indptr));
    ILLICO_CUDA_OK(cudaGetLastError());
    return scan_lengths((long long*)out_indptr, n_rows, st);
}

extern "C" int illico_select_rows_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, const int32_t* rows,
                                      int64_t n_rows, const int64_t* out_indptr, void* out_data, int32_t* out_indices, void* stream) {
    const int vb = value_bytes(dtype, "illico_select_rows_csr");
    if (!vb) return 1;
    if (n_rows <= 0) return 0;
    if (!data || !indices || !indptr || !rows || !out_indptr || !out_data || !out_indices) {
        set_error("illico_select_rows_csr: NULL argument");
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = grid_for(n_rows, SEL_THREADS / 32);
    if (vb == 4)
        ILLICO_LAUNCH("csr_copy_rows_kernel", st,
                      csr_copy_rows_kernel<float><<<grid, SEL_THREADS, 0, st>>>((const float*)data, indices, (const long long*)indptr, rows, n_rows,
                                                                               (const long long*)out_indptr, (float*)out_data, out_indices));
    else
        ILLICO_LAUNCH("csr_copy_rows_kernel", st,
                      csr_copy_rows_kernel<double><<<grid, SEL_THREADS, 0, st>>>((const double*)data, indices, (const long long*)indptr, rows,
                                                                                n_rows, (const long long*)out_indptr, (double*)out_data,
                                                                                out_indices));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int illico_select_rows_csc_indptr(const int32_t* indices, const int64_t* indptr, int32_t n_cols, const int32_t* new_row,
                                             int64_t* out_indptr, void* stream) {
    if (!indptr || !out_indptr || n_cols < 0 || (n_cols > 0 && (!indices || !new_row))) {
        set_error("illico_select_rows_csc_indptr: bad argument");
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (n_cols > 0)
        ILLICO_LAUNCH("csc_kept_count_kernel", st,
                      csc_kept_count_kernel<<<(unsigned)n_cols, SEL_THREADS, 0, st>>>(indices, (const long long*)indptr, new_row,
                                                                                      (long long*)out_indptr));
    ILLICO_CUDA_OK(cudaGetLastError());
    return scan_lengths((long long*)out_indptr, n_cols, st);
}

extern "C" int illico_select_rows_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t n_cols,
                                      const int32_t* new_row, const int64_t* out_indptr, void* out_data, int32_t* out_indices, void* stream) {
    const int vb = value_bytes(dtype, "illico_select_rows_csc");
    if (!vb) return 1;
    if (n_cols <= 0) return 0;
    if (!data || !indices || !indptr || !new_row || !out_indptr || !out_data || !out_indices) {
        set_error("illico_select_rows_csc: NULL argument");
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (vb == 4)
        ILLICO_LAUNCH("csc_compact_kernel", st,
                      csc_compact_kernel<float><<<(unsigned)n_cols, SEL_THREADS, 0, st>>>((const float*)data, indices, (const long long*)indptr,
                                                                                        new_row, (const long long*)out_indptr, (float*)out_data,
                                                                                        out_indices));
    else
        ILLICO_LAUNCH("csc_compact_kernel", st,
                      csc_compact_kernel<double><<<(unsigned)n_cols, SEL_THREADS, 0, st>>>((const double*)data, indices,
                                                                                         (const long long*)indptr, new_row,
                                                                                         (const long long*)out_indptr, (double*)out_data,
                                                                                         out_indices));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}
