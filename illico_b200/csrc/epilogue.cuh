// epilogue.cuh -- fused U -> z -> p-value epilogue, strict IEEE f64 in the reference's operation order.
//
// Restates illico/utils/math.py:64-118 (compute_pval).  The library is compiled with -fmad=false so
// no multiply-add is contracted; the explicit __d*_rn intrinsics below make that independent of
// compiler flags.  Integer products are formed in int64 first, exactly as numba does.
#pragma once
#include <math.h>

#include "common.cuh"

namespace illico {

// sigma = sqrt(n_ref * n_tgt * (n_ref + n_tgt + 1) / 12.0 * tie_corr)
__device__ __forceinline__ double pval_sigma(double prod12, double tie_corr) {
    return __dsqrt_rn(__dmul_rn(prod12, tie_corr));
}

// The part of compute_pval after the quantities that only depend on the group sizes: nrnt = float(n_ref * n_tgt),
// mu = nrnt / 2, prod12 = float(n_ref * n_tgt * (n_ref + n_tgt + 1)) / 12.0, tie_corr = 1 - tie_sum / float(n (n-1) (n+1)).
// The fused epilogue takes those from a per-group table (same operations, so the same bits, evaluated once per group
// instead of once per test).
__device__ __forceinline__ double pval_core(double nrnt, double mu, double prod12, double tie_corr, double U, double cc,
                                            int alternative) {
    if (!(tie_corr > 1.0e-9)) return 1.0;
    const double sigma = pval_sigma(prod12, tie_corr);
    const double sqrt2 = 1.4142135623730951;  // math.sqrt(2.0)
    if (alternative == ILLICO_TWO_SIDED) {
        const double other = __dsub_rn(nrnt, U);
        if (other < U) U = other;  // min(U, n_ref*n_tgt - U)
        const double delta = __dsub_rn(U, mu);
        const double sgn = (delta > 0.0) ? 1.0 : ((delta < 0.0) ? -1.0 : 0.0);
        const double z = __ddiv_rn(__dadd_rn(fabs(delta), __dmul_rn(sgn, cc)), sigma);
        return erfc(__ddiv_rn(z, sqrt2));
    } else if (alternative == ILLICO_GREATER) {
        const double delta = __dsub_rn(U, mu);
        const double z = __ddiv_rn(__dsub_rn(delta, cc), sigma);
        return __dmul_rn(0.5, erfc(__ddiv_rn(z, sqrt2)));
    } else {
        const double delta = __dsub_rn(U, mu);
        const double z = __ddiv_rn(__dadd_rn(delta, cc), sigma);
        return __dmul_rn(0.5, erfc(__ddiv_rn(-z, sqrt2)));
    }
}

// Signed effect score (illico_flags_t::scores): (mu - U) / sigma with the p-value's sigma, no continuity correction --
// the z of the normal approximation, positive when the group ranks above the reference / rest.  0 where the p-value is 1
// (tie correction <= 1e-9); NaN where sigma = 0 otherwise (a one-versus-rest run with a single group, where p is NaN).
__device__ __forceinline__ double score_core(double mu, double prod12, double tie_corr, double U) {
    if (!(tie_corr > 1.0e-9)) return 0.0;
    return __ddiv_rn(__dsub_rn(mu, U), pval_sigma(prod12, tie_corr));
}

// score_core from the group sizes and the tie sum, with compute_pval's operations
__device__ __forceinline__ double compute_score(long long n_ref, long long n_tgt, long long n, double tie_sum, double U,
                                                double mu) {
    const double denom = (double)(n * (n - 1) * (n + 1));
    const double tie_corr = __dsub_rn(1.0, __ddiv_rn(tie_sum, denom));
    const double prod12 = __ddiv_rn((double)(n_ref * n_tgt * (n_ref + n_tgt + 1)), 12.0);
    return score_core(mu, prod12, tie_corr, U);
}

__device__ __forceinline__ double compute_pval(long long n_ref, long long n_tgt, long long n, double tie_sum,
                                               double U, double mu, double cc, int alternative) {
    // tie_corr = 1.0 - tie_sum / (n * (n - 1) * (n + 1))
    const double denom = (double)(n * (n - 1) * (n + 1));
    const double tie_corr = __dsub_rn(1.0, __ddiv_rn(tie_sum, denom));
    const double prod12 = __ddiv_rn((double)(n_ref * n_tgt * (n_ref + n_tgt + 1)), 12.0);
    return pval_core((double)(n_ref * n_tgt), mu, prod12, tie_corr, U, cc, alternative);
}

// value fed to the fold-change sums: x, or expm1(x) when the data is log1p-transformed
// (illico/utils/math.py:212).  Evaluated in f64 on the f32 value (the reference evaluates expm1 in
// float32; see DESIGN.md, "fold change with is_log1p").
__device__ __forceinline__ double fc_value(float v, int is_log1p) {
    return is_log1p ? expm1((double)v) : (double)v;
}

}  // namespace illico
