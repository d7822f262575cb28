"""Cells expressing each gene (``pts``): the count pass ``illico_count_nonzero_*``, the fractions ``illico_nonzero_fractions``
and the filtered selection ``illico_top_genes_filtered`` behind ``asymptotic_wilcoxon(pts=True)`` and ``rank_genes``' marker
filter.

The oracle is numpy: ``(X != 0)`` summed per group in int64 (so -0.0 and stored zeros do not count, NaN does), and the
fractions restated with one float64 division each.  Every comparison is bit for bit."""
import os
import subprocess

import numpy as np
import pytest

from tests.golden import cases as C
from tests.test_rank_genes import bh_reference, rank_order
from tests.util import FakeAnnData

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_FUNCTIONS = ["illico_count_nonzero_dense", "illico_count_nonzero_csr", "illico_count_nonzero_csc", "illico_nonzero_fractions",
                 "illico_top_genes_filtered"]


# ---- numpy oracle ------------------------------------------------------------------------------------------------------

def dense_of(X):
    if hasattr(X, "toarray"):
        return X.toarray()
    if hasattr(X, "cpu"):
        return X.cpu().numpy()
    return np.asarray(X)


def want_counts(X, labels):
    """(groups in np.unique order, group sizes, int64 counts [G, N]) of x != 0."""
    groups, codes = np.unique(np.asarray(labels), return_inverse=True)
    nz = dense_of(X) != 0
    order = np.argsort(codes, kind="stable")
    sizes = np.bincount(codes, minlength=groups.size)
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    counts = np.add.reduceat(nz[order].astype(np.int64), starts, axis=0)
    return groups, sizes.astype(np.int64), counts


def want_fractions(counts, sizes, ref_row):
    n_g = sizes.astype(np.float64)[:, None]
    with np.errstate(divide="ignore", invalid="ignore"):
        pg = counts.astype(np.float64) / n_g
        if ref_row is not None:
            pr = np.broadcast_to(counts[ref_row].astype(np.float64) / np.float64(sizes[ref_row]), counts.shape).copy()
        else:
            total = counts.sum(axis=0, dtype=np.int64)
            pr = (total[None, :] - counts).astype(np.float64) / (sizes.sum() - sizes).astype(np.float64)[:, None]
    return pg, pr


def _aw():
    """``asymptotic_wilcoxon``, once ``illico_b200.__getattr__`` has bound the package's public names: importing the
    submodule before that would leave the module under the package attribute of the same name for the tests that follow."""
    from illico_b200 import rank_genes  # noqa: F401
    from illico_b200.asymptotic_wilcoxon import asymptotic_wilcoxon

    return asymptotic_wilcoxon


def _run(X, labels, reference, **kw):
    """(groups, count plane, pct_group, pct_ref) as asymptotic_wilcoxon(pts=True) computes them."""
    _aw()
    from illico_b200.asymptotic_wilcoxon import _host_fractions, _run_tests

    kw.setdefault("batch_size", "auto")
    run = _run_tests(FakeAnnData(X, labels), kw.pop("is_log1p", False), "pert", reference, kw.pop("n_threads", 1),
                     kw.pop("batch_size"), "two-sided", True, True, None, None, kw.pop("devices", None), score=False,
                     on_device=False, pts=True)
    assert not kw
    pg, pr = _host_fractions(run)
    return run.groups, run.nnz.copy(), pg, pr


def check_pts(X, labels, reference, Xo=None, what="", **kw):
    """The count plane and both fractions of X equal the oracle on Xo (default X)."""
    groups, counts, pg, pr = _run(X, labels, reference, **kw)
    wg, sizes, wc = want_counts(X if Xo is None else Xo, labels)
    assert list(groups) == list(wg), what
    assert counts.dtype == np.int32
    np.testing.assert_array_equal(counts.astype(np.int64), wc, err_msg=what)
    ref_row = int(np.searchsorted(wg, reference)) if reference is not None else None
    wpg, wpr = want_fractions(wc, sizes, ref_row)
    np.testing.assert_array_equal(pg, wpg, err_msg=what)
    np.testing.assert_array_equal(pr, wpr, err_msg=what)
    return counts


def _profile(monkeypatch):
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_PROFILE", "1")
    _lib.profile_report()
    return _lib.profile_report


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_header_declares_the_new_functions(tmp_path):
    """The header declares the count, fraction and filtered-selection entry points with the argument lists the bindings
    use: a C program taking their addresses through typed pointers compiles."""
    from illico_b200 import _lib

    src = tmp_path / "decl.c"
    src.write_text(
        '#include "illico_b200.h"\n'
        "int (*a)(const void*, int32_t, int64_t, int32_t, int32_t, const illico_plan_t*, int32_t*, int64_t, void*) = "
        "illico_count_nonzero_dense;\n"
        "int (*b)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, int32_t*, int64_t,"
        " void*) = illico_count_nonzero_csr;\n"
        "int (*c)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, int32_t*, int64_t,"
        " void*) = illico_count_nonzero_csc;\n"
        "int (*d)(const int32_t*, int64_t, const int32_t*, int32_t, int32_t, int32_t, int64_t, double*, double*, void*) = "
        "illico_nonzero_fractions;\n"
        "int (*e)(const double*, int64_t, const double*, int64_t, const double*, const double*, const double*, int32_t, int32_t,"
        " int32_t, int32_t, double, double, double, double, int32_t*, double*, int32_t*, void*, size_t, void*) = "
        "illico_top_genes_filtered;\n"
        "int main(void) { return !(a && b && c && d && e) || ILLICO_ABI_VERSION != 3; }\n")
    obj = tmp_path / "decl.o"
    subprocess.check_call(["gcc", "-std=c11", "-Werror=incompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c",
                           str(src), "-o", str(obj)])
    for name in NEW_FUNCTIONS:
        assert name in _lib.SIGNATURES


def _tiny():
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=3, n_cells=200, n_genes=8, n_perts=3)
    return FakeAnnData(X, labels)


BAD_FRACTIONS = [-0.1, 1.5, float("nan"), True, "0.25", np.inf]


@pytest.mark.parametrize("name", ["min_in_group_fraction", "max_out_group_fraction"])
@pytest.mark.parametrize("value", BAD_FRACTIONS)
def test_rank_genes_rejects_bad_fractions(name, value):
    from illico_b200 import rank_genes

    with pytest.raises(ValueError, match=name):
        rank_genes(_tiny(), is_log1p=False, group_keys="pert", **{name: value})


@pytest.mark.parametrize("value", [-1.0, float("nan"), False, "1"])
def test_rank_genes_rejects_bad_fold_change(value):
    from illico_b200 import rank_genes

    with pytest.raises(ValueError, match="min_fold_change"):
        rank_genes(_tiny(), is_log1p=False, group_keys="pert", min_fold_change=value)


@pytest.mark.parametrize("value", [1, 0, None, "yes", 1.0])
def test_pts_must_be_a_bool(value):
    from illico_b200 import rank_genes

    asymptotic_wilcoxon = _aw()

    for f in (rank_genes, asymptotic_wilcoxon):
        with pytest.raises(ValueError, match="pts"):
            f(_tiny(), is_log1p=False, group_keys="pert", pts=value)


def test_pts_without_gpu_raises(monkeypatch):
    import torch

    from illico_b200 import _lib, rank_genes

    asymptotic_wilcoxon = _aw()

    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(_lib.IllicoCudaError):
        asymptotic_wilcoxon(_tiny(), is_log1p=False, group_keys="pert", pts=True)
    with pytest.raises(_lib.IllicoCudaError):
        rank_genes(_tiny(), is_log1p=False, group_keys="pert", min_in_group_fraction=0.25, max_out_group_fraction=0.5,
                   min_fold_change=1)


# ---- GPU: the count plane and the fractions ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", list(C.CASES))
def test_counts_and_fractions_on_golden_cases(name):
    builder, grid, batch_size = C.CASES[name]
    X, labels, reference = builder()
    for fmt in sorted({g[0] for g in grid}):
        for ref in (reference, None):
            check_pts(C.to_format(X, fmt), labels, ref, X, what=f"{name}:{fmt}:{ref}", batch_size=batch_size)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_stored_zeros_negative_zero_and_nan(fmt):
    """-0.0 and explicitly stored zeros are not counted, NaN is."""
    from scipy import sparse

    rng = np.random.RandomState(41)
    n, N = 3000, 37
    X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) > 0.5)).astype(np.float32)
    labels = [f"g{v}" for v in rng.randint(0, 5, n)]
    if fmt == "dense":
        X[rng.rand(n, N) < 0.05] = -0.0
        X[rng.rand(n, N) < 0.01] = np.nan
        Xin = X
    else:
        S = sparse.coo_matrix(X)
        extra_r, extra_c = rng.randint(0, n, 4000), rng.randint(0, N, 4000)
        free = X[extra_r, extra_c] == 0
        r = np.concatenate([S.row, extra_r[free]])
        c = np.concatenate([S.col, extra_c[free]])
        v = np.concatenate([S.data, np.where(rng.rand(free.sum()) < 0.5, 0.0, -0.0).astype(np.float32)])
        v[rng.rand(v.size) < 0.01] = np.nan
        M = sparse.coo_matrix((v, (r, c)), shape=(n, N))
        Xin = M.tocsr() if fmt == "csr" else M.tocsc()
        Xin.sum_duplicates()
        assert (Xin.data == 0).sum() > 1000                                # stored zeros survive the conversion
        X = Xin.toarray()
    assert np.isnan(X).any()
    for ref in ("g2", None):
        check_pts(Xin, labels, ref, X, what=f"{fmt}:{ref}", batch_size=16)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_recoded_float64_counted_once_on_the_original_values(monkeypatch, fmt):
    """A float64 matrix float32 cannot hold is recoded per batch; the count pass runs once per batch on the float64 values,
    before the batch is cut into sub-batches."""
    rng = np.random.RandomState(43)
    n, N = 70_000, 1000 if fmt == "dense" else 300
    X = rng.poisson(0.5, (n, N)).astype(np.float64) * (1.0 + 1e-12)
    X[rng.rand(n, N) < 0.01] = 1e-300                                     # float32 would make these zeros
    X[:, 5] = -0.0
    labels = [f"g{v}" for v in rng.randint(0, 9, n)]
    report = _profile(monkeypatch)
    check_pts(C.to_format(X, fmt), labels, "g4", X, what=fmt)
    ran = report()
    assert any(k.startswith("wide_recode") for k in ran), ran
    assert ran[f"count_{fmt}_kernel"][1] == 1, ran
    if fmt == "dense":
        assert ran["wide_recode_dense_kernel"][1] >= 2                   # two sub-batches, one count


DTYPES = ["float16", "int8", "uint16", "int64_above_2_24", "bool"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", DTYPES)
def test_dtype_sample(name):
    rng = np.random.RandomState(47)
    n, N = 4000, 13
    k = rng.poisson(1.0, (n, N)) * (rng.rand(n, N) > 0.6)
    X = {"float16": lambda: (k * 0.5).astype(np.float16),
         "int8": lambda: (k - 2 * (rng.rand(n, N) < 0.1)).astype(np.int8),
         "uint16": lambda: (k * 300).astype(np.uint16),
         "int64_above_2_24": lambda: (k * ((1 << 24) + 1)).astype(np.int64),
         "bool": lambda: k > 0}[name]()
    labels = [f"g{v}" for v in rng.randint(0, 6, n)]
    formats = ["dense"] if name in ("float16", "int8", "bool") else ["dense", "csr", "csc"]
    for fmt in formats:
        for ref in ("g1", None):
            check_pts(C.to_format(X, fmt), labels, ref, X, what=f"{name}:{fmt}:{ref}")


@pytest.mark.gpu
@pytest.mark.parametrize("batch_size", [7, 30, 66])
def test_batch_widths_not_multiples_of_4(batch_size):
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=53, n_cells=5000, n_genes=131, n_perts=9)
    for fmt in ("dense", "csr", "csc"):
        for ref in (synth.CONTROL, None):
            check_pts(C.to_format(X, fmt), labels, ref, X, what=f"{fmt}:{ref}", batch_size=batch_size)


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["device_tensor", "backed_dense", "backed_csc", "devices_all"])
def test_input_routes(tmp_path, source):
    import torch
    from scipy import sparse

    from illico_b200 import synth
    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense

    X, labels = synth.k562_like(seed=59, n_cells=5000, n_genes=67, n_perts=9)
    kw = {}
    if source == "device_tensor":
        Xin = torch.from_numpy(X).cuda()
    elif source == "backed_dense":
        save_dense(str(tmp_path / "d.bin"), X)
        Xin, kw = MemmapDense(str(tmp_path / "d.bin")), dict(batch_size=16, n_threads=3)
    elif source == "backed_csc":
        Xc = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
        Xin, kw = MemmapCSC(str(tmp_path / "csc")), dict(batch_size=20, n_threads=2)
    else:
        Xin, kw = X, dict(devices="all")
    for ref in (synth.CONTROL, None):
        check_pts(Xin, labels, ref, X, what=source, **kw)


@pytest.mark.gpu
def test_many_groups_csc_fallback(monkeypatch):
    """10 001 groups: more than the CSC kernel's shared histogram holds, so each CTA counts into its global column."""
    X, labels, reference = C.CASES["c5_many_groups"][0]()
    report = _profile(monkeypatch)
    for ref in (reference, None):
        check_pts(C.to_format(X, "csc"), labels, ref, X, what=f"csc:{ref}", batch_size=5)
    ran = report()
    assert "count_csc_global_kernel" in ran and "count_csc_kernel" not in ran, ran


@pytest.mark.gpu
def test_long_column_and_group_above_16_bits():
    """One gene over 300 000 cells, and a group of 200 000 cells whose counts pass 65 535."""
    rng = np.random.RandomState(61)
    n = 300_000
    X = np.zeros((n, 3), dtype=np.float32)
    X[:, 0] = rng.poisson(2.0, n)
    X[:, 1] = 1.0
    X[:, 2] = rng.rand(n) < 0.3
    labels = np.where(np.arange(n) % 3 == 0, "b", "a")
    labels[rng.rand(n) < 0.01] = "c"
    for fmt in ("dense", "csr", "csc"):
        for ref in ("b", None):
            counts = check_pts(C.to_format(X, fmt), labels.tolist(), ref, X, what=f"{fmt}:{ref}")
            assert counts.max() > 65_535
        check_pts(C.to_format(X[:, :1], fmt), labels.tolist(), None, X[:, :1], what=f"{fmt}:one gene")


# ---- GPU: nothing else changes -------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_pts_leaves_the_tests_unchanged(fmt):
    from illico_b200 import synth

    asymptotic_wilcoxon = _aw()

    X, labels = synth.k562_like(seed=67, n_cells=6000, n_genes=90, n_perts=7)
    Xf = C.to_format(X, fmt)
    for ref in (synth.CONTROL, None):
        kw = dict(group_keys="pert", reference=ref, is_log1p=False, batch_size=32, return_array=True)
        g0, v0, base = asymptotic_wilcoxon(FakeAnnData(Xf, labels), **kw)
        g1, v1, out, extra = asymptotic_wilcoxon(FakeAnnData(Xf, labels), pts=True, **kw)
        assert list(extra) == ["pct_nz_group", "pct_nz_reference"]
        np.testing.assert_array_equal(out, base)                           # integer counts: the fold change too
        wg, sizes, wc = want_counts(X, labels)
        wpg, wpr = want_fractions(wc, sizes, int(np.searchsorted(wg, ref)) if ref else None)
        np.testing.assert_array_equal(extra["pct_nz_group"], wpg)
        np.testing.assert_array_equal(extra["pct_nz_reference"], wpr)
        df = asymptotic_wilcoxon(FakeAnnData(Xf, labels), pts=True, p_adjust=True, **{**kw, "return_array": False})
        assert list(df.columns) == ["p_value", "statistic", "fold_change", "p_adj", "pct_nz_group", "pct_nz_reference"]
        np.testing.assert_array_equal(df["pct_nz_reference"].to_numpy(), wpr.reshape(-1))


@pytest.mark.gpu
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_rank_genes_pts_adds_two_columns(test):
    import pandas as pd

    from illico_b200 import rank_genes, synth

    X, labels = synth.k562_like(seed=71, n_cells=4000, n_genes=300, n_perts=6)
    ref = synth.CONTROL if test == "ovo" else None
    kw = dict(is_log1p=False, group_keys="pert", reference=ref, n_genes=40)
    base = rank_genes(FakeAnnData(X, labels), **kw)
    df = rank_genes(FakeAnnData(X, labels), pts=True, **kw)
    assert list(df.columns) == list(base.columns) + ["pct_nz_group", "pct_nz_reference"]
    pd.testing.assert_frame_equal(df[list(base.columns)], base, check_exact=True)
    wg, sizes, wc = want_counts(X, labels)
    wpg, wpr = want_fractions(wc, sizes, int(np.searchsorted(wg, ref)) if ref else None)
    gene = df["feature"].cat.codes.to_numpy()
    grow = np.searchsorted(wg, df.index.get_level_values("pert").to_numpy())
    np.testing.assert_array_equal(df["pct_nz_group"].to_numpy(), wpg[grow, gene])
    np.testing.assert_array_equal(df["pct_nz_reference"].to_numpy(), wpr[grow, gene])


# ---- GPU: the marker filter ----------------------------------------------------------------------------------------------

def _filter_case(single_group=False):
    """Counts with planted fold changes of +inf (absent from the reference / rest), 0 (absent from a group) and NaN (a NaN
    value in a group's cells), and a group that expresses nothing, so that no gene passes a fraction filter."""
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=73, n_cells=4000, n_genes=150, n_perts=7)
    labels = np.asarray(labels)
    if single_group:
        return X, ["only"] * len(labels)
    X[:, :30] *= ((labels == "p0001") * 4 + 1)[:, None]
    X[labels != "p0001", 40] = 0.0
    X[labels == "p0001", 40] = 2.0
    X[labels == "p0002", 41] = 0.0
    X[np.flatnonzero(labels == "p0004")[:3], 42] = np.nan
    X[labels == "p0003"] = 0.0
    return X, labels.tolist()


FILTERS = [dict(min_in_group_fraction=0.25, max_out_group_fraction=0.5, min_fold_change=1),   # scanpy's defaults
           dict(min_in_group_fraction=0.1), dict(max_out_group_fraction=0.3), dict(min_fold_change=1.5),
           dict(min_in_group_fraction=0.05, max_out_group_fraction=0.9), dict(min_in_group_fraction=0.0, min_fold_change=0),
           dict(max_out_group_fraction=1.0, min_fold_change=np.inf), dict()]


def check_filtered(df, X, labels, reference, n_genes, by_abs, flt):
    """rank_genes' filtered frame against np.lexsort over the kept genes of the full pts=True frame."""
    asymptotic_wilcoxon = _aw()

    groups, _, out, extra = asymptotic_wilcoxon(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=reference,
                                                score=True, p_adjust=True, pts=True, return_array=True)
    np.testing.assert_array_equal(extra["p_adj"], bh_reference(out[:, :, 0]))   # (one group and no rest: p, p_adj NaN)
    fc = out[:, :, 2]
    ok = np.ones(fc.shape, dtype=bool)
    if flt.get("min_in_group_fraction") is not None:
        ok &= extra["pct_nz_group"] >= flt["min_in_group_fraction"]
    if flt.get("max_out_group_fraction") is not None:
        ok &= extra["pct_nz_reference"] <= flt["max_out_group_fraction"]
    m = flt.get("min_fold_change")
    if m is not None:
        with np.errstate(divide="ignore"):
            ok &= (fc >= m) | ((fc <= np.float64(1.0) / np.float64(m)) if by_abs else False)
    assert list(df.columns)[-2:] == ["pct_nz_group", "pct_nz_reference"]
    got = df.to_numpy()
    pert = df.index.get_level_values("pert").to_numpy()
    rank = df.index.get_level_values("rank").to_numpy()
    N = X.shape[1]
    k = N if n_genes is None else min(n_genes, N)
    empty = 0
    for g, name in enumerate(groups):
        rows = got[pert == name]
        if name == reference:
            assert rows.shape[0] == 0
            continue
        kept = np.flatnonzero(ok[g])
        sel = kept[rank_order(extra["score"][g, kept], by_abs)][:k]
        assert rows.shape[0] == sel.size, f"group {name}"
        empty += sel.size == 0
        assert list(rank[pert == name]) == list(range(sel.size))
        assert list(rows[:, 0]) == [f"gene_{j}" for j in sel], f"group {name}"
        for col, plane in ((1, extra["score"]), (2, out[:, :, 0]), (3, extra["p_adj"]), (4, out[:, :, 1]), (5, fc),
                           (7, extra["pct_nz_group"]), (8, extra["pct_nz_reference"])):
            np.testing.assert_array_equal(rows[:, col].astype(float), plane[g, sel], err_msg=f"group {name} column {col}")
    return empty


@pytest.mark.gpu
@pytest.mark.parametrize("by_abs", [False, True])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_rank_genes_filters_against_full_frame(test, by_abs):
    from illico_b200 import rank_genes, synth

    asymptotic_wilcoxon = _aw()

    X, labels = _filter_case()
    ref = synth.CONTROL if test == "ovo" else None
    empties = 0
    for flt in FILTERS:
        for n_genes in (10, None):
            df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=ref, n_genes=n_genes,
                            rankby_abs=by_abs, pts=True, **flt)
            empties += check_filtered(df, X, labels, ref, n_genes, by_abs, flt)
    assert empties > 0                                                     # "p0003" expresses nothing
    _, _, out = asymptotic_wilcoxon(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=ref, return_array=True)
    fc = out[:, :, 2]
    assert np.isposinf(fc).any() and (fc == 0).any() and np.isnan(fc).any()


@pytest.mark.gpu
def test_rank_genes_single_group_one_versus_rest():
    """One group: the rest is empty, pct_nz_reference is NaN, and a max_out filter keeps nothing."""
    from illico_b200 import rank_genes

    X, labels = _filter_case(single_group=True)
    df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", n_genes=20, pts=True)
    assert len(df) == 20 and np.isnan(df["pct_nz_reference"].to_numpy()).all()
    for flt in (dict(max_out_group_fraction=1.0), dict(min_in_group_fraction=0.2)):
        df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", n_genes=20, **flt)
        check_filtered(df, X, labels, None, 20, False, flt)
    assert len(rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", max_out_group_fraction=1.0)) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("by_abs", [False, True])
def test_top_genes_filtered_entry_point_on_planted_planes(by_abs):
    """illico_top_genes_filtered directly: dropped genes after kept NaN scores, kept[g], gene -1 / NaN padding when k >
    kept[g], NULL planes give NaN fields, and no filter reproduces illico_top_genes."""
    import torch

    from illico_b200 import _lib

    rng = np.random.RandomState(79)
    G, N = 5, 2000
    s = np.round(rng.randn(G, N) * 3, 1)
    s[:, rng.choice(N, 150, replace=False)] = np.nan
    res = rng.rand(G, N, 3) * 2
    res[:, rng.choice(N, 50, replace=False), 2] = np.nan
    res[:, rng.choice(N, 50, replace=False), 2] = np.inf
    res[:, rng.choice(N, 50, replace=False), 2] = 0.0
    pg, pr = rng.rand(G, N), rng.rand(G, N)
    pg[:, rng.choice(N, 40, replace=False)] = np.nan
    pr[:, rng.choice(N, 40, replace=False)] = np.nan
    pg[3] = 0.0                                                            # group 3 keeps nothing under min_in
    padj = rng.rand(G, N)
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in dict(s=s, res=res, pg=pg, pr=pr, padj=padj).items()}
    ws = torch.empty(int(lib.illico_top_genes_workspace_bytes(G, N)), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    nan = float("nan")

    def call(k, min_in, max_out, fc_lo, fc_hi, planes=True):
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 7), dtype=torch.float64, device=dev)
        kept = torch.empty(G, dtype=torch.int32, device=dev)
        rc = lib.illico_top_genes_filtered(d["s"].data_ptr(), N, d["res"].data_ptr(), 3 * N, d["padj"].data_ptr(),
                                           d["pg"].data_ptr() if planes else None, d["pr"].data_ptr() if planes else None, G, N, k,
                                           int(by_abs), min_in, max_out, fc_lo, fc_hi, gene.data_ptr(), rec.data_ptr(),
                                           kept.data_ptr(), ws.data_ptr(), ws.numel(), st)
        _lib.check(rc, "illico_top_genes_filtered")
        return gene.cpu().numpy(), rec.cpu().numpy(), kept.cpu().numpy()

    fc = res[:, :, 2]
    for min_in, max_out, fc_lo, fc_hi in ((0.3, 0.7, 0.8, nan), (0.3, nan, nan, nan), (nan, 0.5, 1.2, 1 / 1.2),
                                          (nan, nan, 0.0, np.inf), (nan, nan, nan, nan)):
        ok = np.ones((G, N), dtype=bool)
        if min_in == min_in:
            ok &= pg >= min_in
        if max_out == max_out:
            ok &= pr <= max_out
        if fc_lo == fc_lo or fc_hi == fc_hi:
            ok &= (fc >= fc_lo) | (fc <= fc_hi)
        for k in (1, 600, N):
            gene, rec, kept = call(k, min_in, max_out, fc_lo, fc_hi)
            np.testing.assert_array_equal(kept, ok.sum(axis=1))
            for g in range(G):
                idx = np.flatnonzero(ok[g])
                sel = idx[rank_order(s[g, idx], by_abs)][:k]
                m = sel.size
                assert m == min(k, kept[g])
                np.testing.assert_array_equal(gene[g, :m], sel, err_msg=f"{g} {k} {min_in} {max_out} {fc_lo}")
                np.testing.assert_array_equal(rec[g, :m, 0], s[g, sel])
                np.testing.assert_array_equal(rec[g, :m, 1:4], res[g, sel])
                np.testing.assert_array_equal(rec[g, :m, 4], padj[g, sel])
                np.testing.assert_array_equal(rec[g, :m, 5], pg[g, sel])
                np.testing.assert_array_equal(rec[g, :m, 6], pr[g, sel])
                assert (gene[g, m:] == -1).all() and np.isnan(rec[g, m:]).all()
        if min_in == min_in:
            assert kept[3] == 0
    # no filter and no planes: the records of illico_top_genes, NaN fractions
    gene, rec, kept = call(N, nan, nan, nan, nan, planes=False)
    assert (kept == N).all() and np.isnan(rec[:, :, 5:]).all()
    g5 = torch.empty((G, N), dtype=torch.int32, device=dev)
    r5 = torch.empty((G, N, 5), dtype=torch.float64, device=dev)
    _lib.check(lib.illico_top_genes(d["s"].data_ptr(), N, d["res"].data_ptr(), 3 * N, d["padj"].data_ptr(), G, N, N, int(by_abs),
                                    g5.data_ptr(), r5.data_ptr(), ws.data_ptr(), ws.numel(), st), "illico_top_genes")
    np.testing.assert_array_equal(gene, g5.cpu().numpy())
    np.testing.assert_array_equal(rec[:, :, :5], r5.cpu().numpy())
    # a fraction bound without its plane is refused
    assert lib.illico_top_genes_filtered(d["s"].data_ptr(), N, d["res"].data_ptr(), 3 * N, None, None, None, G, N, 1, 0, 0.25,
                                         nan, nan, nan, g5.data_ptr(), r5.data_ptr(), None, ws.data_ptr(), ws.numel(), st) != 0
