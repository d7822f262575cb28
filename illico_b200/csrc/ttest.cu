// ttest.cu -- Welch's t-test from per-(group, gene) moments: scanpy's rank_genes_groups(method="t-test" /
// "t-test_overestim_var"), restated operation by operation.
//
//   illico_welch_ttest      sums / sums of squares / fold-change sums of every (group, gene) (illico_group_moments_*)
//                           -> (p, t, fold_change) records and the score plane: welch_ttest_kernel (CTA = 32 genes x 16
//                           group lanes) for t, df and the fold change, welch_pvalue_kernel (a thread per test) for p.
//   illico_student_t_batch  the device Student t CDF on arrays of (df, t): the known-answer hook of the p-value.
//
// Per group and gene, with n cells, S1 = sum x, S2 = sum x*x (scanpy 1.10 _get_mean_var, dense branch, one pass):
//   mean = S1 / n;  var = S2 / n - mean * mean;  if n != 1: var *= n / (n - 1)
// The comparison sample is the reference group (one-versus-reference) or all other cells (one-versus-rest: sums = the
// gene's total over the groups, added in a fixed order, minus the group's).  Then scipy 1.18 ttest_ind_from_stats(mean_g,
// sqrt(var_g), n_g, mean_r, sqrt(var_r), n_r', equal_var=False, alternative) (scipy/stats/_stats_py.py,
// _unequal_var_ttest_denom / _ttest_ind_from_stats / _get_pvalue), n_r' = n_r for "t-test" and n_g for
// "t-test_overestim_var":
//   v = sqrt(var)**2;  vn = v / n;  df = (vn1 + vn2)**2 / (vn1**2 / (n1 - 1) + vn2**2 / (n2 - 1)), NaN -> 1
//   t = (mean1 - mean2) / sqrt(vn1 + vn2)
//   p = 2 stdtr(df, -|t|) (two-sided), stdtr(df, -t) (greater), stdtr(df, t) (less)
// and scanpy's replacement: score = t with NaN -> 0, p NaN -> 1.  The record keeps the raw t.  Every operation is an
// explicit __d*_rn (the library is built with -fmad=false besides).
#include <math.h>

#include "common.cuh"

namespace illico {

namespace {

constexpr int TT_COLS = 32;    // epilogue CTA: genes (one warp row) x group lanes
constexpr int TT_ROWS = 16;
constexpr double MACHEP = 1.11022302462515654042e-16;
constexpr double BIG = 4.503599627370496e15;
constexpr double BIGINV = 2.22044604925031308085e-16;

// Stirling series of ln Gamma(z) without its leading terms, z >= 16 (|error| < 1e-19 there)
__device__ __forceinline__ double stirling_tail(double z) {
    const double z2 = z * z;
    return (1.0 / 12.0 - (1.0 / 360.0 - (1.0 / 1260.0 - (1.0 / 1680.0 - 1.0 / (1188.0 * z2)) / z2) / z2) / z2) / z;
}

// ln Gamma(a + 1/2) - ln Gamma(a), to an absolute error of a few ulps at every a (the difference of two lgamma values
// would lose ~1e-8 at a = 5e6).  Large a: the Stirling terms in closed form, a ln(1 + 1/(2a)) - 1/2 + ln(a) / 2.
__device__ __forceinline__ double lgamma_half_ratio(double a) {
    if (a < 16.0) return lgamma(a + 0.5) - lgamma(a);
    return (a * log1p(0.5 / a) - 0.5) + 0.5 * log(a) + (stirling_tail(a + 0.5) - stirling_tail(a));
}

// Continued fraction #1 of the incomplete beta integral (Lentz; Numerical Recipes betacf), for I_y(1/2, a) at small y
__device__ __forceinline__ double betacf(double a, double b, double x) {
    const double tiny = 1e-300;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (fabs(d) < tiny) d = tiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m < 10000; ++m) {
        const double m2 = 2.0 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
        c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < MACHEP) break;
    }
    return h;
}

// Continued fraction #2 of the incomplete beta integral (Cephes incbd) in z = x / (1 - x), with b = 1/2: every partial
// numerator is positive, so the recurrence never cancels -- the tail I_x(a, 1/2) stays accurate where x is within 1e-7
// of 1 (df up to 1e7 and more), which continued fraction #1 in x cannot do.
__device__ __forceinline__ double betacf_z(double a, double b, double z) {
    double k1 = a, k2 = b - 1.0, k3 = a, k4 = a + 1.0, k5 = 1.0, k6 = a + b, k7 = a + 1.0, k8 = a + 2.0;
    double pkm2 = 0.0, qkm2 = 1.0, pkm1 = 1.0, qkm1 = 1.0, ans = 1.0;
    for (int n = 0; n < 10000; ++n) {
        double xk = -(z * k1 * k2) / (k3 * k4);
        double pk = pkm1 + pkm2 * xk, qk = qkm1 + qkm2 * xk;
        pkm2 = pkm1; pkm1 = pk; qkm2 = qkm1; qkm1 = qk;
        xk = (z * k5 * k6) / (k7 * k8);
        pk = pkm1 + pkm2 * xk; qk = qkm1 + qkm2 * xk;
        pkm2 = pkm1; pkm1 = pk; qkm2 = qkm1; qkm1 = qk;
        const double r = pk / qk;
        const double err = fabs((ans - r) / r);
        ans = r;
        if (err < MACHEP) break;
        k1 += 1.0; k2 -= 1.0; k3 += 2.0; k4 += 2.0; k5 += 1.0; k6 += 1.0; k7 += 2.0; k8 += 2.0;
        if (fabs(qk) + fabs(pk) > BIG) { pkm2 *= BIGINV; pkm1 *= BIGINV; qkm2 *= BIGINV; qkm1 *= BIGINV; }
        if (fabs(qk) < BIGINV || fabs(pk) < BIGINV) { pkm2 *= BIG; pkm1 *= BIG; qkm2 *= BIG; qkm1 *= BIG; }
    }
    return ans;
}

// Lower tail P(T <= -|t|) of Student's t with df degrees of freedom: (1/2) I_x(df/2, 1/2), x = df / (df + t^2).
// |t| >= 1: the tail itself, x^a y^(-1/2) / (a B(a, 1/2)) * betacf_z(a, 1/2, df / t^2), y = 1 - x = t^2 / (df + t^2).
// |t| < 1: 1/2 - (1/2) I_y(1/2, a) (the result is above 0.25, nothing cancels).  x and y are each formed directly, and
// ln x as log1p(-y) when y is small, so that a ln x keeps its absolute accuracy at large a.
__device__ __forceinline__ double student_t_tail(double df, double t) {
    t = fabs(t);
    if (t != t || !(df > 0.0)) return NAN;
    if (t == 0.0) return 0.5;
    if (isinf(t)) return 0.0;
    if (isinf(df)) return 0.5 * erfc(t / 1.4142135623730951);
    const double a = 0.5 * df;
    const double t2 = t * t;
    if (t2 == 0.0) return 0.5;
    double x, y, lx, ly, z;
    if (isinf(t2)) {                                    // |t| > 1.3e154: in terms of q = df / t^2
        const double q = (df / t) / t;
        x = q / (1.0 + q); y = 1.0 / (1.0 + q);
        lx = log(df) - 2.0 * log(t) - log1p(q); ly = -log1p(q); z = q;
    } else {
        x = df / (df + t2); y = t2 / (df + t2);
        lx = (y < 0.5) ? log1p(-y) : log(x);
        ly = log(y); z = df / t2;
    }
    const double lnB = 0.5 * 1.1447298858494002 - lgamma_half_ratio(a);   // ln B(a, 1/2) = ln sqrt(pi) - (ln G(a+1/2) - ln G(a))
    if (t2 >= 1.0) return 0.5 * (exp(a * lx - 0.5 * ly - lnB) * betacf_z(a, 0.5, z) / a);
    return 0.5 * (1.0 - exp(a * lx + 0.5 * ly - lnB) * betacf(0.5, a, y) / 0.5);
}

// scipy.special.stdtr(df, t)
__device__ __forceinline__ double stdtr(double df, double t) {
    const double q = student_t_tail(df, t);
    return (t > 0.0) ? 1.0 - q : q;
}

// p of the t statistic: two-sided 2 stdtr(df, -|t|), greater stdtr(df, -t), less stdtr(df, t)
__device__ __forceinline__ double t_pvalue(double df, double t, int alternative) {
    if (alternative == ILLICO_TWO_SIDED) return __dmul_rn(2.0, student_t_tail(df, t));
    return stdtr(df, alternative == ILLICO_GREATER ? -t : t);
}

// _get_mean_var, dense branch: mean = S1 / n, var = S2 / n - mean^2, times n / (n - 1) unless n == 1
__device__ __forceinline__ void mean_var(double s1, double s2, long long n, double& mean, double& var) {
    const double dn = (double)n;
    mean = __ddiv_rn(s1, dn);
    var = __dsub_rn(__ddiv_rn(s2, dn), __dmul_rn(mean, mean));
    if (n != 1) var = __dmul_rn(var, __ddiv_rn(dn, (double)(n - 1)));
}

// ttest_ind_from_stats(equal_var=False) from (mean, var, n) of both samples: t and df
__device__ __forceinline__ void welch(double m1, double var1, long long n1, double m2, double var2, long long n2, double& t,
                                      double& df) {
    const double sd1 = __dsqrt_rn(var1), sd2 = __dsqrt_rn(var2);
    const double vn1 = __ddiv_rn(__dmul_rn(sd1, sd1), (double)n1);
    const double vn2 = __ddiv_rn(__dmul_rn(sd2, sd2), (double)n2);
    const double s = __dadd_rn(vn1, vn2);
    df = __ddiv_rn(__dmul_rn(s, s), __dadd_rn(__ddiv_rn(__dmul_rn(vn1, vn1), (double)(n1 - 1)),
                                              __ddiv_rn(__dmul_rn(vn2, vn2), (double)(n2 - 1))));
    if (df != df) df = 1.0;
    t = __ddiv_rn(__dsub_rn(m1, m2), __dsqrt_rn(s));
}

// CTA = TT_COLS genes x TT_ROWS group lanes: thread (r, c) takes gene c of the CTA in groups r, r + TT_ROWS, ..
__global__ void __launch_bounds__(TT_COLS * TT_ROWS) welch_ttest_kernel(const double* __restrict__ S1, const double* __restrict__ S2,
                                                                        const double* __restrict__ SF, long long ms,
                                                                        const int32_t* __restrict__ group_size, int G, int N,
                                                                        int ref, long long n_cells, int overestim, int alternative,
                                                                        double* __restrict__ results, long long rstride,
                                                                        double* __restrict__ scores, long long sstride) {
    __shared__ double part[3][TT_ROWS][TT_COLS + 1];
    const int c = threadIdx.x % TT_COLS, r = threadIdx.x / TT_COLS;
    const int j = blockIdx.x * TT_COLS + c;
    const bool in = j < N;
    const double* F = SF ? SF : S1;      // fold-change sums: expm1(x) for log1p data, else x
    // comparison sample: the reference group, or the gene's totals for one-versus-rest (each lane's groups in order,
    // then the lanes in order: a fixed order)
    double r1 = 0.0, r2 = 0.0, rf = 0.0;
    long long nr = 0;
    if (ref >= 0) {
        if (in) { r1 = S1[(long long)ref * ms + j]; r2 = S2[(long long)ref * ms + j]; rf = F[(long long)ref * ms + j]; }
        nr = group_size[ref];
    } else {
        if (in)
            for (int g = r; g < G; g += TT_ROWS) {
                const long long o = (long long)g * ms + j;
                r1 = __dadd_rn(r1, S1[o]); r2 = __dadd_rn(r2, S2[o]); rf = __dadd_rn(rf, F[o]);
            }
        part[0][r][c] = r1; part[1][r][c] = r2; part[2][r][c] = rf;
        __syncthreads();
        r1 = r2 = rf = 0.0;
        for (int q = 0; q < TT_ROWS; ++q) {
            r1 = __dadd_rn(r1, part[0][q][c]); r2 = __dadd_rn(r2, part[1][q][c]); rf = __dadd_rn(rf, part[2][q][c]);
        }
    }
    if (!in) return;
    double ref_mean = 0.0, ref_var = 0.0, fc_mean_r = 0.0, fc_inv_r = 0.0;
    if (ref >= 0) {
        mean_var(r1, r2, nr, ref_mean, ref_var);
        fc_mean_r = rf / (double)nr;                    // rank_ovo.cu: R.mean = R.sum / n_ref, R.inv_mean = 1 / R.mean
        fc_inv_r = 1.0 / fc_mean_r;
    }
    for (int g = r; g < G; g += TT_ROWS) {
        const long long o = (long long)g * ms + j;
        double* rec = results + (long long)g * rstride + (long long)j * 3;
        const long long ng = group_size[g];
        const double s1 = S1[o], s2 = S2[o], sf = F[o];
        if (g == ref) {                                 // the reference row: (1, 0, fold change of the control with itself)
            rec[0] = 1.0; rec[1] = 0.0; rec[2] = (fc_mean_r == 0.0) ? INFINITY : fc_mean_r / fc_mean_r;
            if (scores) scores[(long long)g * sstride + j] = 0.0;
            continue;
        }
        double mg, vg, mr, vr, fc;
        long long nrest;
        mean_var(s1, s2, ng, mg, vg);
        if (ref >= 0) {
            mr = ref_mean; vr = ref_var; nrest = nr;
            fc = (fc_mean_r == 0.0) ? INFINITY : (sf * (1.0 / (double)ng)) * fc_inv_r;   // rank_ovo.cu finalize_group
        } else {
            nrest = n_cells - ng;
            mean_var(__dsub_rn(r1, s1), __dsub_rn(r2, s2), nrest, mr, vr);
            const double mu_t = sf * (1.0 / (double)ng);                                 // rank_ovr.cu phase D
            const double mu_r = (rf - sf) / (double)nrest;
            fc = (mu_r == 0.0) ? INFINITY : mu_t / mu_r;
        }
        double t, df;
        welch(mg, vg, ng, mr, vr, overestim ? ng : nrest, t, df);
        rec[0] = df; rec[1] = t; rec[2] = fc;           // (df: welch_pvalue_kernel replaces it by p)
        if (scores) scores[(long long)g * sstride + j] = (t != t) ? 0.0 : t;
    }
}

// The p-values, a thread per test: (df, t) -> p in the record's first slot, NaN -> 1.  A kernel of its own, so that little
// is live across the incomplete beta's library calls (nothing spills) and the tests' uneven iteration counts spread over
// the whole grid.
__global__ void __launch_bounds__(256) welch_pvalue_kernel(double* __restrict__ results, long long rstride, int G, int N, int ref,
                                                           int alternative) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= (long long)G * N) return;
    const int g = (int)(i / N), j = (int)(i - (long long)g * N);
    if (g == ref) return;
    double* rec = results + (long long)g * rstride + (long long)j * 3;
    const double p = t_pvalue(rec[0], rec[1], alternative);
    rec[0] = (p != p) ? 1.0 : p;
}

__global__ void student_t_batch_kernel(const double* df, const double* t, long long n, int alternative, double* out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = t_pvalue(df[i], t[i], alternative);
}

}  // namespace
}  // namespace illico

using namespace illico;

extern "C" {

int illico_welch_ttest(const double* sums, const double* sumsq, const double* fsums, int64_t group_stride, const int32_t* group_size,
                       int32_t n_groups, int32_t n_genes, int32_t ref_group, int64_t n_cells, int32_t overestim_var,
                       int32_t alternative, double* results, int64_t result_group_stride, double* scores, int64_t score_group_stride,
                       void* stream) {
    if (!sums || !sumsq || !group_size || !results) { set_error("illico_welch_ttest: NULL argument"); return 1; }
    if (n_groups <= 0 || n_genes <= 0) return 0;
    if (group_stride < n_genes || result_group_stride < 3ll * n_genes || ref_group >= n_groups ||
        (scores && score_group_stride < n_genes)) {
        set_error("illico_welch_ttest: a stride below the batch width or ref_group out of range");
        return 1;
    }
    if (alternative != ILLICO_TWO_SIDED && alternative != ILLICO_LESS && alternative != ILLICO_GREATER) {
        set_error("illico_welch_ttest: alternative %d", alternative);
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned ctas = (unsigned)(((long long)n_genes + TT_COLS - 1) / TT_COLS);
    ILLICO_LAUNCH("welch_ttest_kernel", st,
                  welch_ttest_kernel<<<ctas, TT_COLS * TT_ROWS, 0, st>>>(sums, sumsq, fsums, group_stride, group_size, n_groups, n_genes,
                                                                  ref_group < 0 ? -1 : ref_group, (long long)n_cells,
                                                                  overestim_var ? 1 : 0, alternative, results, result_group_stride,
                                                                  scores, score_group_stride));
    const long long tests = (long long)n_groups * n_genes;
    ILLICO_LAUNCH("welch_pvalue_kernel", st,
                  welch_pvalue_kernel<<<(unsigned)((tests + 255) / 256), 256, 0, st>>>(results, result_group_stride, n_groups, n_genes,
                                                                                     ref_group < 0 ? -1 : ref_group, alternative));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

int illico_student_t_batch(const double* df, const double* t, int64_t n, int32_t alternative, double* out, void* stream) {
    if (n <= 0) return 0;
    if (!df || !t || !out) { set_error("illico_student_t_batch: NULL argument"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    ILLICO_LAUNCH("student_t_batch_kernel", st,
                  student_t_batch_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(df, t, (long long)n, alternative, out));
    ILLICO_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
