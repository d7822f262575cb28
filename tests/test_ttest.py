"""Welch's t-test (``illico_b200.ttest``, ``rank_genes(method="t-test")``): the moments pass ``illico_group_moments_*``, the
epilogue ``illico_welch_ttest`` and the device Student t CDF ``illico_student_t_batch``.

The oracle is numpy float64: per-group sums of x and x*x, scanpy 1.10's ``_get_mean_var`` (dense branch) and scipy 1.18's
``ttest_ind_from_stats(equal_var=False)`` restated operation by operation, with ``scipy.special.stdtr`` for the p-value.
It is checked once against ``scipy.stats.ttest_ind(equal_var=False)`` on the raw arrays.  On integer counts every sum is
exact in any order, so t and the fold change are compared bit for bit and p at 1e-12 relative."""
import os
import shutil
import subprocess

import numpy as np
import pytest
from scipy import special, stats

from tests.golden import cases as C
from tests.test_rank_genes import bh_reference, rank_order
from tests.util import FakeAnnData

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_FUNCTIONS = ["illico_group_moments_dense", "illico_group_moments_csr", "illico_group_moments_csc", "illico_welch_ttest",
                 "illico_student_t_batch"]
METHODS = ["t-test", "t-test_overestim_var"]
ALTERNATIVES = ["two-sided", "less", "greater"]


# ---- numpy oracle ------------------------------------------------------------------------------------------------------

def dense_of(X):
    if hasattr(X, "toarray"):
        return X.toarray()
    if hasattr(X, "cpu"):
        return X.cpu().numpy()
    return np.asarray(X)


def group_sums(X, labels, is_log1p=False):
    """(groups, sizes int64, S1, S2, Sf) [G, N] float64; x widened to float64 before it is squared."""
    Xd = dense_of(X).astype(np.float64)
    groups, codes = np.unique(np.asarray(labels), return_inverse=True)
    G = groups.size
    sizes = np.bincount(codes, minlength=G).astype(np.int64)
    S1, S2, SF = (np.zeros((G, Xd.shape[1])) for _ in range(3))
    with np.errstate(invalid="ignore", over="ignore"):
        for g in range(G):
            rows = Xd[codes == g]
            S1[g], S2[g] = rows.sum(axis=0), (rows * rows).sum(axis=0)
            SF[g] = np.expm1(rows).sum(axis=0) if is_log1p else S1[g]
    return groups, sizes, S1, S2, SF


def mean_var(s1, s2, n):
    n = np.asarray(n, dtype=np.float64)
    mean = s1 / n
    var = s2 / n - mean * mean
    return mean, np.where(n != 1, var * (n / (n - 1)), var)


def welch(m1, v1, n1, m2, v2, n2):
    sd1, sd2 = np.sqrt(v1), np.sqrt(v2)
    vn1, vn2 = (sd1 * sd1) / n1, (sd2 * sd2) / n2
    s = vn1 + vn2
    df = (s * s) / ((vn1 * vn1) / (n1 - 1) + (vn2 * vn2) / (n2 - 1))
    df = np.where(np.isnan(df), 1.0, df)
    return (m1 - m2) / np.sqrt(s), df


def p_of(t, df, alternative):
    if alternative == "two-sided":
        return 2 * special.stdtr(df, -np.abs(t))
    return special.stdtr(df, -t if alternative == "greater" else t)


def oracle(X, labels, reference, method="t-test", alternative="two-sided", is_log1p=False):
    """(groups, results [G, N, 3] = (p, t, fold_change), score [G, N]) as the device computes them."""
    groups, sizes, S1, S2, SF = group_sums(X, labels, is_log1p)
    G, N = S1.shape
    out = np.empty((G, N, 3))
    score = np.empty((G, N))
    with np.errstate(all="ignore"):
        if reference is not None:
            r = int(np.flatnonzero(groups == reference)[0])
            n_r = np.full(G, sizes[r])
            m2, v2 = mean_var(S1[r], S2[r], sizes[r])
            m2, v2 = np.broadcast_to(m2, S1.shape), np.broadcast_to(v2, S1.shape)
            mean_r = SF[r] / np.float64(sizes[r])
            fc = np.where(mean_r == 0, np.inf, (SF * (1.0 / sizes.astype(np.float64))[:, None]) * (1.0 / mean_r))
        else:
            r = None
            n_r = sizes.sum() - sizes
            T1, T2, TF = (np.zeros(N) for _ in range(3))
            for g in range(G):                      # the gene's totals (the device adds them in another fixed order)
                T1, T2, TF = T1 + S1[g], T2 + S2[g], TF + SF[g]
            m2, v2 = mean_var(T1 - S1, T2 - S2, n_r[:, None])
            mu_t = SF * (1.0 / sizes.astype(np.float64))[:, None]
            mu_r = (TF - SF) / n_r.astype(np.float64)[:, None]
            fc = np.where(mu_r == 0, np.inf, mu_t / mu_r)
        m1, v1 = mean_var(S1, S2, sizes[:, None])
        n2 = sizes if method == "t-test_overestim_var" else n_r
        t, df = welch(m1, v1, sizes[:, None].astype(np.float64), m2, v2, n2[:, None].astype(np.float64))
        p = p_of(t, df, alternative)
        p = np.where(np.isnan(p), 1.0, p)
        out[:, :, 0], out[:, :, 1], out[:, :, 2] = p, t, fc
        score[:] = np.where(np.isnan(t), 0.0, t)
        if r is not None:
            out[r, :, 0], out[r, :, 1] = 1.0, 0.0
            out[r, :, 2] = np.where(mean_r == 0, np.inf, mean_r / mean_r)
            score[r] = 0.0
    return groups, out, score


def assert_close(got, want, rtol, what, floor=0.0):
    """Equal NaN / inf positions, |got - want| <= rtol |want| where |want| >= floor, both below floor elsewhere."""
    got, want = np.asarray(got), np.asarray(want)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=what)
    fin = np.isfinite(want)
    np.testing.assert_array_equal(got[~fin & ~np.isnan(want)], want[~fin & ~np.isnan(want)], err_msg=what)
    big = fin & (np.abs(want) >= floor)
    err = np.abs(got[big] - want[big]) / np.maximum(np.abs(want[big]), np.finfo(float).tiny)
    assert err.size == 0 or err.max() <= rtol, f"{what}: max relative error {err.max():.3g}"
    small = fin & ~big
    assert (np.abs(got[small]) < floor).all(), what
    return 0.0 if err.size == 0 else float(err.max())


# ---- test data ---------------------------------------------------------------------------------------------------------

def special_case(seed=5, n_cells=600, n_genes=24, integer=True, nan=True):
    """Counts with the genes and groups the t-test has to get right: an all-zero gene, a constant non-zero gene, a gene
    non-zero in one cell, negative values, a NaN (float only); groups of 1 and 2 cells, a large reference."""
    rng = np.random.RandomState(seed)
    X = (rng.poisson(2.0, size=(n_cells, n_genes)) * (rng.rand(n_cells, n_genes) < 0.4)).astype(np.float64)
    if not integer:
        X = X * rng.gamma(2.0, 0.37, size=X.shape)
    X[:, 0] = 0.0
    X[:, 1] = 3.0
    X[:, 2] = 0.0
    X[17, 2] = 5.0
    X[:, 3] = rng.randint(-4, 5, n_cells)
    if nan:
        X[11, 4] = np.nan
    labels = np.array(["ctrl"] * 200 + [f"g{i % 5}" for i in range(n_cells - 203)] + ["one", "two", "two"])
    return X, labels.tolist()


def to_dtype(X, dtype):
    return X.astype(dtype)


def run_ttest(X, labels, reference, **kw):
    from illico_b200 import ttest

    groups, var_names, out, extra = ttest(FakeAnnData(X, labels), "pert", reference, return_array=True, score=True, **kw)
    return groups, out, extra["score"]


def check_against_oracle(X, labels, reference, Xo=None, method="t-test", alternative="two-sided", exact=True, is_log1p=False,
                         what="", **kw):
    Xo = X if Xo is None else Xo
    groups, got, score = run_ttest(X, labels, reference, method=method, alternative=alternative, is_log1p=is_log1p, **kw)
    wg, want, wscore = oracle(Xo, labels, reference, method, alternative, is_log1p)
    assert list(groups) == list(wg)
    errs = {}
    if exact:
        np.testing.assert_array_equal(got[:, :, 1], want[:, :, 1], err_msg=f"{what} t")
        np.testing.assert_array_equal(got[:, :, 2], want[:, :, 2], err_msg=f"{what} fold change")
        np.testing.assert_array_equal(score, wscore, err_msg=f"{what} score")
        errs["p"] = assert_close(got[:, :, 0], want[:, :, 0], 1e-12, f"{what} p")
    else:
        errs["t"] = assert_close(got[:, :, 1], want[:, :, 1], 1e-10, f"{what} t")
        errs["fc"] = assert_close(got[:, :, 2], want[:, :, 2], 1e-10, f"{what} fold change")
        errs["p"] = assert_close(got[:, :, 0], want[:, :, 0], 1e-8, f"{what} p", floor=1e-280)
    return got, errs


# ---- CPU -----------------------------------------------------------------------------------------------------------------

def test_new_functions_are_bound_and_exported():
    from illico_b200 import _lib

    for name in NEW_FUNCTIONS:
        assert name in _lib.SIGNATURES
    if os.path.exists(_lib.LIB_PATH):
        out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True)
        if out.returncode == 0:
            for name in NEW_FUNCTIONS:
                assert f" {name}\n" in out.stdout + "\n", name


def test_header_declares_the_new_functions(tmp_path):
    src = tmp_path / "decl.c"
    src.write_text(
        '#include "illico_b200.h"\n'
        "int (*a)(const void*, int32_t, int64_t, int32_t, int32_t, const illico_plan_t*, int32_t, double*, double*, double*, int32_t*,"
        " int64_t, int64_t, void*) = illico_group_moments_dense;\n"
        "int (*b)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, int32_t, double*,"
        " double*, double*, int32_t*, int64_t, int64_t, void*) = illico_group_moments_csr;\n"
        "int (*c)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, int32_t, double*,"
        " double*, double*, int32_t*, int64_t, int64_t, void*) = illico_group_moments_csc;\n"
        "int (*d)(const double*, const double*, const double*, int64_t, const int32_t*, int32_t, int32_t, int32_t, int64_t, int32_t,"
        " int32_t, double*, int64_t, double*, int64_t, void*) = illico_welch_ttest;\n"
        "int (*e)(const double*, const double*, int64_t, int32_t, double*, void*) = illico_student_t_batch;\n"
        "int main(void) { return !(a && b && c && d && e); }\n")
    subprocess.check_call(["gcc", "-std=c11", "-Werror=incompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c",
                           str(src), "-o", str(tmp_path / "decl.o")])


@pytest.mark.parametrize("method", ["wilcox", "t_test", "logreg", None, 1])
def test_bad_method_raises_before_any_cuda_work(monkeypatch, method):
    from illico_b200 import engine, rank_genes, ttest

    def no_cuda(*a, **k):
        raise AssertionError("device work started")

    monkeypatch.setattr(engine, "require_cuda", no_cuda)
    X, labels = special_case(n_cells=300, n_genes=6)
    adata = FakeAnnData(X.astype(np.float32), labels)
    for call in (lambda: ttest(adata, "pert", None, method=method),
                 lambda: rank_genes(adata, is_log1p=False, group_keys="pert", method=method)):
        with pytest.raises(ValueError, match="'wilcoxon', 't-test', 't-test_overestim_var'"):
            call()


def test_oracle_matches_scipy_ttest_ind():
    """The oracle's t and p against scipy.stats.ttest_ind(equal_var=False) on the raw arrays (which computes the variance in
    two passes: agreement to rounding), for one-versus-reference and one-versus-rest and every alternative."""
    X, labels = special_case(integer=False, nan=False)
    labels = np.asarray(labels)
    Xd = X.astype(np.float64)
    for reference in ("ctrl", None):
        for alt in ALTERNATIVES:
            groups, out, _ = oracle(Xd, labels, reference, "t-test", alt)
            for g, name in enumerate(groups):
                if name == reference or (labels == name).sum() < 2:
                    continue
                a = Xd[labels == name]
                b = Xd[labels == reference] if reference is not None else Xd[labels != name]
                with np.errstate(all="ignore"):
                    res = stats.ttest_ind(a, b, equal_var=False, alternative=alt)
                ok = np.isfinite(res.statistic) & (np.abs(res.statistic) > 1e-6)
                np.testing.assert_allclose(out[g, ok, 1], res.statistic[ok], rtol=1e-9)
                np.testing.assert_allclose(out[g, ok, 0], res.pvalue[ok], rtol=1e-8)


def test_overestim_var_uses_the_group_size():
    X, labels = special_case(nan=False)
    _, a, _ = oracle(X, labels, "ctrl", "t-test")
    _, b, _ = oracle(X, labels, "ctrl", "t-test_overestim_var")
    assert not np.array_equal(a[:, :, 1], b[:, :, 1])
    np.testing.assert_array_equal(a[:, :, 2], b[:, :, 2])


def test_new_kernels_do_not_spill(tmp_path):
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from illico_b200.build import NVCC_FLAGS

    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    for src, kernels in (("counts.cu", ("count_dense_kernel", "count_csr_kernel", "count_csc_kernel")),
                         ("ttest.cu", ("welch_ttest_kernel", "welch_pvalue_kernel", "student_t_batch_kernel"))):
        res = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(ROOT, "illico_b200", "csrc", src), "-o",
                                               str(tmp_path / (src + ".o"))], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        seen, current = 0, None
        for line in res.stderr.splitlines():
            if "Function properties for" in line:
                current = line.split("for", 1)[1].strip()
            elif "spill" in line and current and any(k in current for k in kernels):
                seen += 1
                assert " 0 bytes spill stores, 0 bytes spill loads" in line, (current, line)
        assert seen >= len(kernels)


# ---- GPU: the device Student t -------------------------------------------------------------------------------------------

DF_GRID = [1, 1.5, 2, 3.7, 10, 29.5, 100, 1e3, 1e4, 1.5e5, 6e5, 1e7]
T_GRID = [0.0, 1e-300, -1e-300, 0.5, -0.5, 2, -2, 5, -5, 10, -10, 20, -20, 38, -38, 100, -100, np.inf, -np.inf, np.nan]


def device_p(df, t, alternative):
    import torch

    from illico_b200 import _lib

    lib = _lib.load()
    d = torch.tensor(np.asarray(df, dtype=np.float64), device="cuda")
    tt = torch.tensor(np.asarray(t, dtype=np.float64), device="cuda")
    out = torch.empty_like(d)
    _lib.check(lib.illico_student_t_batch(d.data_ptr(), tt.data_ptr(), d.numel(), _lib.ALTERNATIVES[alternative], out.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream), "illico_student_t_batch")
    return out.cpu().numpy()


def _grid():
    df, t = np.meshgrid(np.array(DF_GRID, dtype=np.float64), np.array(T_GRID, dtype=np.float64), indexing="ij")
    return df.ravel(), t.ravel()


@pytest.mark.gpu
@pytest.mark.parametrize("alternative", ALTERNATIVES)
def test_student_t_against_scipy_stdtr(alternative):
    df, t = _grid()
    got = device_p(df, t, alternative)
    want = p_of(t, df, alternative)
    err = assert_close(got, want, 1e-12, alternative, floor=1e-280)
    print(f"max relative error against scipy.special.stdtr ({alternative}): {err:.3g}")


@pytest.mark.gpu
def test_student_t_against_mpmath():
    """stdtr(df, t) = I_x(df/2, 1/2) / 2 for t < 0 from mpmath's betainc at 40 digits, df up to 6e5 (where mpmath's
    hypergeometric series converges; it gives up on tails far below 1e-280, which are left out)."""
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.dps = 40
    df, t = _grid()
    keep = np.isfinite(t) & (t != 0) & (df <= 6e5)
    df, t = df[keep], t[keep]
    want = np.full(df.size, np.nan)
    for i, (d, x) in enumerate(zip(df, t)):
        try:
            half = 0.5 * mpmath.betainc(d / 2, 0.5, 0, mpmath.mpf(d) / (d + mpmath.mpf(x) ** 2), regularized=True)
        except ValueError:
            continue
        want[i] = float(half if x < 0 else 1 - half)
    ok = ~np.isnan(want)
    assert ok.sum() > 0.9 * ok.size
    got = device_p(df[ok], t[ok], "less")
    assert_close(got, want[ok], 1e-12, "mpmath", floor=1e-280)


# ---- GPU: the full table against the oracle ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "int32", "float64"])
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_integer_counts_every_route_bit_identical(fmt, dtype):
    X, labels = special_case(nan=dtype != "int32")
    Xt = to_dtype(X, dtype)
    for reference in ("ctrl", None):
        for method in METHODS:
            for alt in ALTERNATIVES:
                check_against_oracle(C.to_format(Xt, fmt), labels, reference, X, method, alt, what=f"{fmt}:{reference}:{method}:{alt}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_non_integer_data(fmt, dtype):
    X, labels = special_case(integer=False)
    Xt = to_dtype(X, dtype)
    Xo = Xt.astype(np.float64)
    worst = {}
    for reference in ("ctrl", None):
        for method in METHODS:
            for alt in ALTERNATIVES:
                for log1p in (False, True):
                    _, errs = check_against_oracle(C.to_format(Xt, fmt), labels, reference, Xo, method, alt, exact=False,
                                                   is_log1p=log1p, what=f"{fmt}:{dtype}:{reference}:{method}:{alt}:{log1p}")
                    for k, v in errs.items():
                        worst[k] = max(worst.get(k, 0.0), v)
    print(f"non-integer {dtype} {fmt}: max relative errors {worst}")


@pytest.mark.gpu
def test_special_genes_and_groups():
    X, labels = special_case()
    for reference in ("ctrl", None):
        _, out, score = run_ttest(X.astype(np.float32), labels, reference)
        p, t = out[:, :, 0], out[:, :, 1]
        rows = np.arange(p.shape[0]) != (0 if reference == "ctrl" else -1)     # ("ctrl" is group 0)
        assert (p[:, 0] == 1).all() and (score[:, 0] == 0).all() and np.isnan(t[rows, 0]).all()   # all-zero gene: t = 0 / 0
        assert (p[:, 4] == 1).all() and (score[:, 4] == 0).all()        # NaN in the data
    groups, out, score = run_ttest(X.astype(np.float32), ["only"] * len(labels), None)   # one group: empty rest
    assert (out[:, :, 0] == 1).all() and (score == 0).all()
    check_against_oracle(X.astype(np.float32), ["only"] * len(labels), None, X, what="single group")


# ---- GPU: routes -----------------------------------------------------------------------------------------------------------

def _route_case():
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=83, n_cells=5000, n_genes=67, n_perts=9)
    X[:, 11] = np.random.RandomState(2).poisson(25.0, X.shape[0])
    return X, labels, synth.CONTROL


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_multi_segment_groups_and_batches(monkeypatch, fmt):
    X, labels, ctrl = _route_case()
    Xf = C.to_format(X, fmt)
    for reference in (ctrl, None):
        want, _ = check_against_oracle(Xf, labels, reference, X, what=f"{fmt}:{reference}")
        for kw in (dict(batch_size=7), dict(batch_size=30)):
            _, got, _ = run_ttest(Xf, labels, reference, **kw)
            np.testing.assert_array_equal(got, want)
        monkeypatch.setenv("ILLICO_B200_SEG_MAX", "37")
        _, got, _ = run_ttest(Xf, labels, reference, batch_size=16)
        monkeypatch.delenv("ILLICO_B200_SEG_MAX")
        np.testing.assert_array_equal(got, want)


@pytest.mark.gpu
def test_csc_many_groups_global_branch(monkeypatch):
    from illico_b200 import _lib

    X, labels, reference = C.CASES["c5_many_groups"][0]()
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    _lib.profile_report()
    for ref in (reference, None):
        check_against_oracle(C.to_format(X, "csc"), labels, ref, X, batch_size=5, what=f"csc:{ref}")
        check_against_oracle(C.to_format(X, "csr"), labels, ref, X, what=f"csr:{ref}")
    ran = _lib.profile_report()
    assert "moments_csc_global_kernel" in ran and "moments_csc_kernel" not in ran, ran


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["device_tensor", "backed_dense", "backed_csc", "devices_all", "layer"])
def test_input_routes(tmp_path, source):
    import torch
    from scipy import sparse

    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense

    X, labels, ctrl = _route_case()
    kw, layers, Xin = {}, None, X
    if source == "device_tensor":
        Xin = torch.from_numpy(X).cuda()
    elif source == "backed_dense":
        save_dense(str(tmp_path / "d.bin"), X)
        Xin, kw = MemmapDense(str(tmp_path / "d.bin")), dict(batch_size=16, n_threads=3)
    elif source == "backed_csc":
        Xc = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
        Xin, kw = MemmapCSC(str(tmp_path / "csc")), dict(batch_size=20, n_threads=2)
    elif source == "devices_all":
        kw = dict(devices="all")
    else:
        layers, Xin, kw = {"counts": X}, np.zeros_like(X), dict(layer="counts")
    from illico_b200 import ttest

    for reference in (ctrl, None):
        _, want, _ = run_ttest(X, labels, reference)
        _, _, got = ttest(FakeAnnData(Xin, labels, layers=layers), "pert", reference, return_array=True, **kw)
        np.testing.assert_array_equal(got, want, err_msg=source)
    if source == "devices_all":
        for devices in (["cuda:0"], torch.cuda.device_count()):
            _, _, got = ttest(FakeAnnData(X, labels), "pert", None, return_array=True, devices=devices)
            np.testing.assert_array_equal(got, run_ttest(X, labels, None)[1])


# ---- GPU: consistency with the Wilcoxon path -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_fold_change_and_counts_match_the_wilcoxon_call(fmt):
    from illico_b200 import asymptotic_wilcoxon, ttest

    X, labels, ctrl = _route_case()
    Xf = C.to_format(X, fmt)
    for reference in (ctrl, None):
        for method in METHODS:
            _, _, w, wx = asymptotic_wilcoxon(FakeAnnData(Xf, labels), is_log1p=False, group_keys="pert", reference=reference,
                                              return_array=True, pts=True)
            _, _, t, tx = ttest(FakeAnnData(Xf, labels), "pert", reference, method=method, return_array=True, pts=True)
            np.testing.assert_array_equal(t[:, :, 2], w[:, :, 2])
            for k in ("pct_nz_group", "pct_nz_reference"):
                np.testing.assert_array_equal(tx[k], wx[k])


@pytest.mark.gpu
def test_count_plane_of_a_ttest_run_equals_the_count_pass():
    from illico_b200 import rank_genes  # noqa: F401  (binds the package's public names first)
    from illico_b200.asymptotic_wilcoxon import _run_tests

    X, labels, ctrl = _route_case()
    for fmt in ("dense", "csr", "csc"):
        runs = [_run_tests(FakeAnnData(C.to_format(X, fmt), labels), False, "pert", ctrl, 1, "auto", "two-sided", True, True, None,
                           None, None, score=False, on_device=False, pts=True, method=m) for m in ("wilcoxon", "t-test")]
        np.testing.assert_array_equal(runs[0].nnz, runs[1].nnz)


@pytest.mark.gpu
def test_k562_shaped_slice():
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=91, n_cells=300_000, n_genes=256, n_perts=2000)
    for reference in (synth.CONTROL, None):
        check_against_oracle(X, labels, reference, what=f"k562:{reference}")


# ---- GPU: rank_genes(method=...) -------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("by_abs", [False, True])
@pytest.mark.parametrize("reference", ["ctrl", None])
def test_rank_genes_t_test_order_p_adj_and_filters(reference, by_abs):
    from illico_b200 import rank_genes

    X, labels = special_case(n_cells=900, n_genes=60)
    X = X.astype(np.float32)
    groups, out, score = oracle(X, labels, reference)
    padj = bh_reference(out[:, :, 0])
    for method in METHODS:
        groups, out, score = oracle(X, labels, reference, method)
        padj = bh_reference(out[:, :, 0])
        for kw in (dict(), dict(pts=True), dict(min_in_group_fraction=0.2, min_fold_change=1.0)):
            df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=reference, n_genes=None,
                            rankby_abs=by_abs, method=method, **kw)
            pert = df.index.get_level_values("pert").to_numpy()
            for g, name in enumerate(groups):
                rows = df[pert == name]
                if name == reference:
                    assert rows.shape[0] == 0
                    continue
                keep = np.ones(out.shape[1], dtype=bool)
                if "min_in_group_fraction" in kw:
                    Xg = X[np.asarray(labels) == name]
                    keep &= (Xg != 0).sum(axis=0) / Xg.shape[0] >= 0.2
                    fc = out[g, :, 2]
                    keep &= (fc >= 1.0) | ((fc <= 1.0) if by_abs else False)
                kept = np.flatnonzero(keep)
                sel = kept[rank_order(score[g, kept], by_abs)]
                assert list(rows["feature"].astype(str)) == [f"gene_{j}" for j in sel], name
                np.testing.assert_array_equal(rows["score"].to_numpy(), score[g, sel])
                np.testing.assert_array_equal(rows["statistic"].to_numpy(), out[g, sel, 1])
                np.testing.assert_array_equal(rows["fold_change"].to_numpy(), out[g, sel, 2])
                assert_close(rows["p_value"].to_numpy(), out[g, sel, 0], 1e-12, name)
                assert_close(rows["p_adj"].to_numpy(), padj[g, sel], 1e-12, name)
                if kw:
                    assert "pct_nz_group" in rows.columns
