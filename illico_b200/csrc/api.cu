// api.cu -- extern "C" entry points of libillico_b200.so (see include/illico_b200.h).
#include <stdarg.h>
#include <stdio.h>

#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace illico {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-kernel profiling (ILLICO_PROFILE=1) ----------------------------------------------------------------
struct ProfRec { const char* name; cudaEvent_t e0, e1; };
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
static thread_local cudaEvent_t g_prof_open = nullptr;
static thread_local const char* g_prof_name = nullptr;

bool profiling_on() {
    const char* v = getenv("ILLICO_PROFILE");
    return v && v[0] != '0' && v[0] != 0;
}
void prof_begin(const char* name, cudaStream_t stream) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, stream);
    g_prof_open = e;
    g_prof_name = name;
}
void prof_end(cudaStream_t stream) {
    if (!g_prof_open) return;
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, stream);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(ProfRec{g_prof_name, g_prof_open, e});
    g_prof_open = nullptr;
}

// kernels' host launchers (stage.cu, rank_ovr.cu, rank_ovo.cu)
int launch_stage_dense(const float*, long long, int, int, const illico_plan_t*, float*, uint32_t*, cudaStream_t);
int launch_stage_csr(const float*, const int32_t*, const long long*, int, int, const illico_plan_t*, float*, uint32_t*,
                     void*, size_t, cudaStream_t);
size_t stage_csr_workspace_bytes(const illico_plan_t*, int);
int launch_stage_csc(const float*, const int32_t*, const long long*, int, int, const illico_plan_t*, float*, uint32_t*,
                     cudaStream_t);
int launch_check_csr_sorted(const int32_t*, const long long*, long long, int*, int*, cudaStream_t);
int launch_ovr(const float*, const uint32_t*, int, const illico_plan_t*, const illico_flags_t*, double*, long long, void*,
               size_t, const illico_debug_t*, cudaStream_t);
int launch_ovo(const float*, const uint32_t*, int, const illico_plan_t*, const illico_flags_t*, double*, long long, void*,
               size_t, const illico_debug_t*, cudaStream_t);
size_t ovr_slab_qwords(const illico_plan_t*);
// fused.cu: dense one-versus-reference in one pass (0 = done, 1 = error, -1 = not applicable)
int launch_ovo_dense_fused(const float*, long long, int, int, const illico_plan_t*, const illico_flags_t*,
                           const illico_batch_buffers_t*, double*, long long, const illico_debug_t*, cudaStream_t);
int launch_ovr_dense_fused(const float*, long long, int, int, const illico_plan_t*, const illico_flags_t*,
                           const illico_batch_buffers_t*, double*, long long, const illico_debug_t*, cudaStream_t);
int launch_ovo_csr_fused(const float*, const int32_t*, const long long*, int, int, const illico_plan_t*, const illico_flags_t*,
                         const illico_batch_buffers_t*, double*, long long, const illico_debug_t*, cudaStream_t);
int launch_ovr_csr_fused(const float*, const int32_t*, const long long*, int, int, const illico_plan_t*, const illico_flags_t*,
                         const illico_batch_buffers_t*, double*, long long, const illico_debug_t*, cudaStream_t);
size_t ovo_fused_workspace_bytes(int, int);
float ovo_fused_last_ms();
size_t ovr_table_rec_bytes(const illico_plan_t*);
// recode.cu
size_t recode_workspace_bytes(long long, int);
int launch_convert_values(const void*, int, long long, float*, double*, int*, cudaStream_t);
int launch_recode_dense(const double*, long long, int, int, long long, const int32_t*, int, int, float*, double*, void*, size_t, cudaStream_t);
int launch_recode_csc(const double*, const int32_t*, const long long*, int, int, const int32_t*, int, long long, int, float*, double*, void*,
                      size_t, cudaStream_t);
int launch_recode_csr(const double*, const int32_t*, const long long*, long long, int, int, const int32_t*, int, int, float*, double*, void*,
                      size_t, cudaStream_t);
// repart.cu
int launch_csr_shard_count(const int32_t*, const long long*, long long, const int32_t*, int, int32_t*, unsigned long long*, cudaStream_t);
int launch_csr_shard_scatter(const float*, const int32_t*, const long long*, long long, long long, const int32_t*, int, const int32_t*,
                             const long long*, float* const*, int32_t* const*, int32_t* const*, cudaStream_t);

static int check_plan(const illico_plan_t* p) {
    if (!p) { set_error("plan is NULL"); return 1; }
    if (p->n_cells <= 0 || p->n_groups <= 0 || p->n_segments < p->n_groups) { set_error("plan has invalid sizes"); return 1; }
    if (!p->perm || !p->cell_seg || !p->seg_pos || !p->seg_base || !p->seg_group || !p->group_seg || !p->group_size) {
        set_error("plan has NULL tables");
        return 1;
    }
    if (p->ref_group >= p->n_groups) { set_error("plan.ref_group out of range"); return 1; }
    if (p->max_target_group_size < 0 || p->max_target_group_size > p->max_group_size) { set_error("plan.max_target_group_size out of range"); return 1; }
    if (p->ref_group >= 0 && (p->ref_seg_begin < 0 || p->ref_seg_end > p->n_segments || p->ref_seg_begin >= p->ref_seg_end)) {
        set_error("plan.ref_seg_* out of range");
        return 1;
    }
    return 0;
}

static int max_resident_ctas() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms * 4;
}

}  // namespace illico

using namespace illico;

extern "C" {

int illico_abi_version(void) { return ILLICO_ABI_VERSION; }
const char* illico_last_error(void) { return g_err; }
int64_t illico_launch_count(void) { return (int64_t)g_launches.load(); }
double illico_last_fused_ms(void) { return (double)ovo_fused_last_ms(); }

int64_t illico_profile_report(char* out, int64_t cap) {
    std::vector<ProfRec> recs;
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        recs.swap(g_prof);
    }
    std::map<std::string, std::pair<double, long long>> acc;
    std::vector<std::string> order;
    for (auto& r : recs) {
        float ms = 0.0f;
        if (cudaEventSynchronize(r.e1) == cudaSuccess && cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) {
            auto it = acc.find(r.name);
            if (it == acc.end()) { order.push_back(r.name); acc[r.name] = {0.0, 0}; it = acc.find(r.name); }
            it->second.first += ms;
            it->second.second += 1;
        }
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    std::string txt;
    char line[256];
    for (auto& nm : order) {
        snprintf(line, sizeof(line), "%s\t%.6f\t%lld\n", nm.c_str(), acc[nm].first, acc[nm].second);
        txt += line;
    }
    if (out && cap > 0) {
        const size_t n = txt.size() < (size_t)(cap - 1) ? txt.size() : (size_t)(cap - 1);
        memcpy(out, txt.data(), n);
        out[n] = 0;
    }
    return (int64_t)txt.size();
}

int illico_memcpy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                          int kind, void* stream) {
    if (!dst || !src) { set_error("illico_memcpy2d_async: NULL pointer"); return 1; }
    if (kind < 1 || kind > 3) {
        set_error("illico_memcpy2d_async: kind must be 1 (host to device), 2 (device to host) or 3 (device to device)");
        return 1;
    }
    if (width_bytes == 0 || height == 0) return 0;
    // device to device: cudaMemcpyDefault lets the driver route a copy between two GPUs (peer or staged)
    const cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDefault;
    ILLICO_CUDA_OK(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, height, k, (cudaStream_t)stream));
    return 0;
}

static int check_recode(const void* values, int32_t dtype, const void* cell_group, const void* codes, const void* sums, const void* ws) {
    if (dtype != ILLICO_DTYPE_F64) { set_error("illico_recode_*: dtype %d (float32-exact dtypes are converted on upload; pass float64)", dtype); return 1; }
    if (!values || !cell_group || !codes || !sums || !ws) { set_error("illico_recode_*: NULL argument"); return 1; }
    return 0;
}
int illico_convert_values(const void* src, int32_t dtype, int64_t count, float* dst_f32, double* dst_f64, int32_t* inexact, void* stream) {
    if (count > 0 && (!src || (!dst_f32 && !dst_f64) || (dst_f32 && !inexact))) { set_error("illico_convert_values: NULL argument"); return 1; }
    return launch_convert_values(src, dtype, count, dst_f32, dst_f64, inexact, (cudaStream_t)stream);
}
size_t illico_recode_workspace_bytes(int64_t total_keys, int32_t n_genes_batch) {
    return recode_workspace_bytes(total_keys > 0 ? total_keys : 0, n_genes_batch > 0 ? n_genes_batch : 1);
}
int illico_recode_dense(const void* X, int32_t dtype, int64_t ld, int32_t gene_lb, int32_t nb, int64_t n_cells, const int32_t* cell_group,
                        int32_t n_groups, int32_t is_log1p, float* codes, double* group_sums, void* workspace, size_t workspace_bytes,
                        void* stream) {
    if (check_recode(X, dtype, cell_group, codes, group_sums, workspace)) return 1;
    return launch_recode_dense((const double*)X, ld, gene_lb, nb, n_cells, cell_group, n_groups, is_log1p, codes, group_sums, workspace,
                               workspace_bytes, (cudaStream_t)stream);
}
int illico_recode_csc(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int32_t gene_lb, int32_t nb,
                      int64_t batch_nnz, const int32_t* cell_group, int32_t n_groups, int32_t is_log1p, float* codes, double* group_sums,
                      void* workspace, size_t workspace_bytes, void* stream) {
    if (batch_nnz > 0 && check_recode(data, dtype, cell_group, codes, group_sums, workspace)) return 1;
    if (!indptr || !group_sums || !workspace) { set_error("illico_recode_csc: NULL argument"); return 1; }
    return launch_recode_csc((const double*)data, indices, (const long long*)indptr, gene_lb, nb, cell_group, n_groups, batch_nnz, is_log1p,
                             codes, group_sums, workspace, workspace_bytes, (cudaStream_t)stream);
}
int illico_recode_csr(const void* data, int32_t dtype, const int32_t* indices, const int64_t* indptr, int64_t n_cells, int32_t gene_lb,
                      int32_t nb, const int32_t* cell_group, int32_t n_groups, int32_t is_log1p, float* codes, double* group_sums,
                      void* workspace, size_t workspace_bytes, void* stream) {
    if (!indptr || !group_sums || !workspace || !cell_group) { set_error("illico_recode_csr: NULL argument"); return 1; }
    if (dtype != ILLICO_DTYPE_F64) { set_error("illico_recode_csr: dtype %d (pass float64)", dtype); return 1; }
    return launch_recode_csr((const double*)data, indices, (const long long*)indptr, n_cells, gene_lb, nb, cell_group, n_groups, is_log1p,
                             codes, group_sums, workspace, workspace_bytes, (cudaStream_t)stream);
}

int illico_enable_peer_access(int32_t device, int32_t peer_device) {
    if (device == peer_device) return 0;
    int can = 0;
    ILLICO_CUDA_OK(cudaDeviceCanAccessPeer(&can, device, peer_device));
    if (!can) { set_error("GPU %d cannot access GPU %d's memory", device, peer_device); return 1; }
    int cur = 0;
    ILLICO_CUDA_OK(cudaGetDevice(&cur));
    ILLICO_CUDA_OK(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
    cudaSetDevice(cur);
    if (e != cudaSuccess) { set_error("cudaDeviceEnablePeerAccess(%d -> %d) failed: %s", device, peer_device, cudaGetErrorString(e)); return 1; }
    return 0;
}

int illico_csr_shard_count(const int32_t* indices, const int64_t* indptr, int64_t n_rows, const int32_t* bounds, int32_t n_shards,
                           int32_t* cnt, uint64_t* totals, void* stream) {
    if (!indptr || !bounds || !cnt || !totals) { set_error("illico_csr_shard_count: NULL argument"); return 1; }
    return launch_csr_shard_count(indices, (const long long*)indptr, n_rows, bounds, n_shards, cnt, (unsigned long long*)totals,
                                  (cudaStream_t)stream);
}

int illico_csr_shard_scatter(const float* data, const int32_t* indices, const int64_t* indptr, int64_t n_rows, int64_t row0,
                             const int32_t* bounds, int32_t n_shards, const int32_t* cnt, const int64_t* out_pos,
                             float* const* out_data, int32_t* const* out_indices, int32_t* const* out_row_cnt, void* stream) {
    if (!indptr || !bounds || !cnt || !out_pos || !out_data || !out_indices || !out_row_cnt) {
        set_error("illico_csr_shard_scatter: NULL argument");
        return 1;
    }
    return launch_csr_shard_scatter(data, indices, (const long long*)indptr, n_rows, row0, bounds, n_shards, cnt, (const long long*)out_pos,
                                    out_data, out_indices, out_row_cnt, (cudaStream_t)stream);
}

int illico_stage_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t n_genes_batch, const illico_plan_t* plan,
                           float* ir_vals, uint32_t* ir_cnt, void* stream) {
    if (check_plan(plan)) return 1;
    if (!X || !ir_vals || !ir_cnt) { set_error("illico_stage_dense_f32: NULL buffer"); return 1; }
    return launch_stage_dense(X, ld, gene_lb, n_genes_batch, plan, ir_vals, ir_cnt, (cudaStream_t)stream);
}

int illico_zero_counts(uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan, void* stream) {
    if (check_plan(plan)) return 1;
    ILLICO_CUDA_OK(cudaMemsetAsync(ir_cnt, 0, (size_t)n_genes_batch * plan->n_segments * sizeof(uint32_t),
                                   (cudaStream_t)stream));
    return 0;
}

size_t illico_stage_csr_workspace_bytes(const illico_plan_t* plan, int32_t n_genes_batch) {
    if (check_plan(plan)) return 0;
    return stage_csr_workspace_bytes(plan, n_genes_batch);
}

int illico_stage_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                         int32_t n_genes_batch, const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt,
                         void* workspace, size_t workspace_bytes, void* stream) {
    if (check_plan(plan)) return 1;
    if (!indptr || !ir_vals || !ir_cnt) { set_error("illico_stage_csr_f32: NULL buffer"); return 1; }
    return launch_stage_csr(data, indices, (const long long*)indptr, gene_lb, n_genes_batch, plan, ir_vals, ir_cnt,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

int illico_stage_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb,
                         int32_t n_genes_batch, const illico_plan_t* plan, float* ir_vals, uint32_t* ir_cnt, void* stream) {
    if (check_plan(plan)) return 1;
    if (!indptr || !ir_vals || !ir_cnt) { set_error("illico_stage_csc_f32: NULL buffer"); return 1; }
    return launch_stage_csc(data, indices, (const long long*)indptr, gene_lb, n_genes_batch, plan, ir_vals, ir_cnt,
                            (cudaStream_t)stream);
}

int illico_check_csr_sorted(const int32_t* indices, const int64_t* indptr, int64_t n_rows, int32_t* d_flag, void* stream) {
    int sorted = -1;
    if (launch_check_csr_sorted(indices, (const long long*)indptr, n_rows, d_flag, &sorted, (cudaStream_t)stream)) return -1;
    return sorted;
}

size_t illico_rank_workspace_bytes(const illico_plan_t* plan, int32_t n_genes_batch) {
    if (check_plan(plan)) return 0;
    size_t ctas = (size_t)max_resident_ctas();
    if ((size_t)n_genes_batch < ctas) ctas = (size_t)(n_genes_batch > 0 ? n_genes_batch : 1);
    size_t per_cta = plan->ref_group >= 0 ? 4 * (size_t)plan->max_group_size * sizeof(uint32_t)
                                          : ovr_slab_qwords(plan) * 8;
    size_t rank = ctas * per_cta + 256 + (((size_t)(n_genes_batch > 0 ? n_genes_batch : 1) + 64) * sizeof(int) + 255);
    if (plan->ref_group < 0) rank += 2 * ctas * ovr_table_rec_bytes(plan) + 256;  // table kernel: up to 8 CTAs per SM
    else rank += 1024 + ((size_t)plan->n_groups + 64) * 5 * sizeof(double);       // gene counter + per-group constants
    const size_t stage = stage_csr_workspace_bytes(plan, n_genes_batch);  // CSR staging reuses the rank kernels' scratch
    // the fused paths keep their per-gene tables in front of that scratch until the handed-back genes have been ranked
    const size_t fused = (ovo_fused_workspace_bytes(n_genes_batch > 0 ? n_genes_batch : 1, plan->n_groups) + 511) & ~(size_t)255;
    return fused + (rank > stage ? rank : stage);
}

int illico_rank_ovr(const float* ir_vals, const uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan,
                    const illico_flags_t* flags, double* results, int64_t result_group_stride, void* workspace,
                    size_t workspace_bytes, const illico_debug_t* dbg, void* stream) {
    if (check_plan(plan)) return 1;
    if (plan->ref_group >= 0) { set_error("illico_rank_ovr: plan has a reference group"); return 1; }
    if (!flags || !results || !workspace) { set_error("illico_rank_ovr: NULL argument"); return 1; }
    return launch_ovr(ir_vals, ir_cnt, n_genes_batch, plan, flags, results, result_group_stride, workspace,
                      workspace_bytes, dbg, (cudaStream_t)stream);
}

int illico_rank_ovo(const float* ir_vals, const uint32_t* ir_cnt, int32_t n_genes_batch, const illico_plan_t* plan,
                    const illico_flags_t* flags, double* results, int64_t result_group_stride, void* workspace,
                    size_t workspace_bytes, const illico_debug_t* dbg, void* stream) {
    if (check_plan(plan)) return 1;
    if (plan->ref_group < 0) { set_error("illico_rank_ovo: plan has no reference group"); return 1; }
    if (!flags || !results || !workspace) { set_error("illico_rank_ovo: NULL argument"); return 1; }
    return launch_ovo(ir_vals, ir_cnt, n_genes_batch, plan, flags, results, result_group_stride, workspace,
                      workspace_bytes, dbg, (cudaStream_t)stream);
}

// ---- the six dispatchers ------------------------------------------------------------------------------
#define ILLICO_CHECK_BUF(b)                                                            \
    if (!(b) || !(b)->ir_vals || !(b)->ir_cnt || !(b)->workspace) {                    \
        set_error("batch buffers missing");                                            \
        return 1;                                                                      \
    }

int illico_ovr_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t nb, const illico_plan_t* plan,
                         const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results,
                         int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (check_plan(plan)) return 1;
    if (plan->ref_group >= 0) { set_error("illico_ovr_dense_f32: plan has a reference group"); return 1; }
    if (!X || !flags || !results) { set_error("illico_ovr_dense_f32: NULL argument"); return 1; }
    // count-like data: one pass over the matrix, per-group histograms instead of staged lists (fused.cu)
    const int rc = launch_ovr_dense_fused(X, ld, gene_lb, nb, plan, flags, buf, results, gstride, dbg, (cudaStream_t)stream);
    if (rc >= 0) return rc;
    if (illico_stage_dense_f32(X, ld, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, stream)) return 1;
    return illico_rank_ovr(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}
int illico_ovo_dense_f32(const float* X, int64_t ld, int32_t gene_lb, int32_t nb, const illico_plan_t* plan,
                         const illico_flags_t* flags, const illico_batch_buffers_t* buf, double* results,
                         int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (check_plan(plan)) return 1;
    if (plan->ref_group < 0) { set_error("illico_ovo_dense_f32: plan has no reference group"); return 1; }
    if (!X || !flags || !results) { set_error("illico_ovo_dense_f32: NULL argument"); return 1; }
    // count-like data: one pass over the matrix, no staged lists (fused.cu); anything else: stage + rank
    const int rc = launch_ovo_dense_fused(X, ld, gene_lb, nb, plan, flags, buf, results, gstride, dbg, (cudaStream_t)stream);
    if (rc >= 0) return rc;
    if (illico_stage_dense_f32(X, ld, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, stream)) return 1;
    return illico_rank_ovo(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}
int illico_ovr_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb, int32_t nb,
                       const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                       double* results, int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (check_plan(plan)) return 1;
    if ((plan->ref_group >= 0) != false) { set_error("illico_ovr_csr_f32: plan / test mismatch"); return 1; }
    if (!indptr || !flags || !results) { set_error("illico_ovr_csr_f32: NULL argument"); return 1; }
    // count-like data: per-group histograms built in shared memory, no staged lists (fused.cu)
    const int rc = launch_ovr_csr_fused(data, indices, (const long long*)indptr, gene_lb, nb, plan, flags, buf, results, gstride, dbg,
                                        (cudaStream_t)stream);
    if (rc >= 0) return rc;
    if (illico_stage_csr_f32(data, indices, indptr, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, buf->workspace,
                             buf->workspace_bytes, stream)) return 1;
    return illico_rank_ovr(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}
int illico_ovo_csr_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb, int32_t nb,
                       const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                       double* results, int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (check_plan(plan)) return 1;
    if ((plan->ref_group >= 0) != true) { set_error("illico_ovo_csr_f32: plan / test mismatch"); return 1; }
    if (!indptr || !flags || !results) { set_error("illico_ovo_csr_f32: NULL argument"); return 1; }
    // count-like data: per-group histograms built in shared memory, no staged lists (fused.cu)
    const int rc = launch_ovo_csr_fused(data, indices, (const long long*)indptr, gene_lb, nb, plan, flags, buf, results, gstride, dbg,
                                        (cudaStream_t)stream);
    if (rc >= 0) return rc;
    if (illico_stage_csr_f32(data, indices, indptr, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, buf->workspace,
                             buf->workspace_bytes, stream)) return 1;
    return illico_rank_ovo(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}
int illico_ovr_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb, int32_t nb,
                       const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                       double* results, int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (illico_zero_counts(buf->ir_cnt, nb, plan, stream)) return 1;
    if (illico_stage_csc_f32(data, indices, indptr, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, stream)) return 1;
    return illico_rank_ovr(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}
int illico_ovo_csc_f32(const float* data, const int32_t* indices, const int64_t* indptr, int32_t gene_lb, int32_t nb,
                       const illico_plan_t* plan, const illico_flags_t* flags, const illico_batch_buffers_t* buf,
                       double* results, int64_t gstride, const illico_debug_t* dbg, void* stream) {
    ILLICO_CHECK_BUF(buf);
    if (illico_zero_counts(buf->ir_cnt, nb, plan, stream)) return 1;
    if (illico_stage_csc_f32(data, indices, indptr, gene_lb, nb, plan, buf->ir_vals, buf->ir_cnt, stream)) return 1;
    return illico_rank_ovo(buf->ir_vals, buf->ir_cnt, nb, plan, flags, results, gstride, buf->workspace,
                           buf->workspace_bytes, dbg, stream);
}

}  // extern "C"
