"""``mask_var=`` (scanpy's ``rank_genes_groups(mask_var=...)``) for ``asymptotic_wilcoxon``, ``ttest`` and ``rank_genes``.

The defining property: every selected gene's values equal its values in the same call without ``mask_var``, and ``p_adj`` is
Benjamini-Hochberg over the selected genes of each group.  Shards and batches span the selected genes; the matrix a batch runs
on holds only their columns -- gathered by the staging threads and ``illico_host_pack_cols_f32`` (dense host input), scipy's
CSC column index and the backed readers (CSC), ``illico_select_cols_dense`` (CUDA tensors), or compacted on the device through
a ``new_col`` table by the CSC selection kernels with rows and columns swapped (host CSR).  The kernels are checked against
numpy / scipy slicing."""
import numpy as np
import pandas as pd
import pytest
from scipy import sparse

from tests.test_groups import CONTROL, METHODS, ROUTES, _route_input, assert_rows_of_full_call, labelled_counts
from tests.test_rank_genes import bh_reference
from tests.util import FakeAnnData


class VarAnnData(FakeAnnData):
    """``FakeAnnData`` with a ``var`` frame (indexed by ``var_names``) holding boolean columns such as ``highly_variable``."""

    def __init__(self, X, labels, var=None, **kw):
        super().__init__(X, labels, **kw)
        self.var = pd.DataFrame(var or {}, index=self.var_names)


def scattered_mask(n_genes, share=0.25, seed=0):
    """About ``share`` of the genes, scattered, gene 0 and gene n_genes - 1 among them."""
    rng = np.random.RandomState(seed)
    mask = rng.rand(n_genes) < share
    mask[0] = mask[-1] = True
    return mask


# ---- CPU: validation, shards and batches, backed fetch, host pack --------------------------------------------------------

def test_resolve_mask_var_validation():
    from illico_b200.select import resolve_mask_var

    n = 10
    m = np.zeros(n, bool)
    m[[0, 3, 9]] = True
    ad = VarAnnData(np.zeros((4, n), np.float32), ["a"] * 4,
                    var={"highly_variable": m, "score": np.arange(n, dtype=float), "nullable": pd.array(m, dtype="boolean")})
    assert resolve_mask_var(ad, None, n) is None
    for given in (m, list(m), pd.Series(m), "highly_variable", "nullable", pd.Series(m, dtype="boolean")):
        got = resolve_mask_var(ad, given, n)
        assert got.dtype == np.int64
        np.testing.assert_array_equal(got, [0, 3, 9])
    assert resolve_mask_var(ad, np.ones(n, bool), n) is None               # every gene: the call without mask_var
    with pytest.raises(ValueError, match="positions"):
        resolve_mask_var(ad, np.array([0, 3, 9]), n)                       # integer indices are refused
    with pytest.raises(ValueError, match="positions"):
        resolve_mask_var(ad, m.astype(np.int8), n)
    with pytest.raises(ValueError, match="positions"):
        resolve_mask_var(ad, "score", n)                                   # a column that is not boolean
    with pytest.raises(ValueError, match="not a column"):
        resolve_mask_var(ad, "missing", n)
    with pytest.raises(ValueError, match="not a column"):
        resolve_mask_var(FakeAnnData(np.zeros((4, n)), ["a"] * 4), "highly_variable", n)   # no var frame at all
    with pytest.raises(ValueError, match="shape"):
        resolve_mask_var(ad, m[:-1], n)
    with pytest.raises(ValueError, match="shape"):
        resolve_mask_var(ad, m.reshape(2, 5), n)
    with pytest.raises(ValueError, match="no gene"):
        resolve_mask_var(ad, np.zeros(n, bool), n)
    with pytest.raises(ValueError, match="positions"):
        resolve_mask_var(ad, pd.Series(pd.array([True, None] * 5, dtype="boolean")), n)   # a missing value


def test_bad_mask_fails_before_device_work():
    """The mask is refused before a device is looked for (so this runs without a GPU too)."""
    from illico_b200 import asymptotic_wilcoxon, rank_genes, ttest

    X, labels = labelled_counts(0, 200, 8, 4)
    ad = VarAnnData(X, labels, var={"hv": np.arange(8) % 2 == 0})
    for call in (lambda m: asymptotic_wilcoxon(ad, False, "pert", CONTROL, mask_var=m),
                 lambda m: ttest(ad, "pert", None, mask_var=m), lambda m: rank_genes(ad, False, "pert", None, mask_var=m)):
        with pytest.raises(ValueError, match="positions"):
            call(np.array([0, 2]))
        with pytest.raises(ValueError, match="no gene"):
            call(np.zeros(8, bool))
        with pytest.raises(ValueError, match="not a column"):
            call("nope")
        with pytest.raises(ValueError, match="shape"):
            call(np.ones(7, bool))


class _BatchSizer:
    def __init__(self, step):
        self.step = step

    def max_batch_genes(self, n_genes, method):
        return self.step


def test_shards_and_batches_cover_the_selected_genes():
    from illico_b200.asymptotic_wilcoxon import _batches
    from illico_b200.parallel import gene_shard
    from illico_b200.select import ColumnSelection

    n_genes = 1000
    names = np.array([f"g{i}" for i in range(n_genes)])
    for mask in (scattered_mask(n_genes), np.arange(n_genes) == 517, np.arange(n_genes) < 999):
        sel = ColumnSelection(np.flatnonzero(mask), n_genes)
        for world in (1, 3, 8):
            seen = []
            for r in range(world):
                lb, ub = gene_shard(sel.size, r, world)
                for step in (1, 7, 64):
                    got = [g for blb, bub in _batches(lb, ub, step, _BatchSizer(step), True) for g in range(blb, bub)]
                    assert got == list(range(lb, ub))
                seen += list(range(lb, ub))
            assert seen == list(range(sel.size))                      # each selected gene exactly once, in order
            np.testing.assert_array_equal(names[sel.cols[seen]], names[mask])
        for lb, ub in ((0, sel.size), (1, max(1, sel.size - 1)), (sel.size // 2, sel.size)):
            runs = sel.runs(lb, ub)
            assert sum(c1 - c0 for c0, c1 in runs) == ub - lb
            np.testing.assert_array_equal(np.concatenate([np.arange(c0, c1) for c0, c1 in runs] or [[]]), sel.cols[lb:ub])
            assert all(a[1] < b[0] for a, b in zip(runs, runs[1:]))   # maximal runs: a gap between two


def test_backed_readers_fetch_the_selected_columns(tmp_path):
    """ColumnSelection.fetch reads each run of consecutive columns as one slice of a backed matrix and joins them."""
    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense
    from illico_b200.registry import data_handler_registry
    from illico_b200.select import ColumnSelection

    X, _ = labelled_counts(1, 300, 97, 3)
    save_dense(str(tmp_path / "d.bin"), X)
    Xc = sparse.csc_matrix(X)
    save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
    mask = scattered_mask(97, seed=2)
    mask[40:50] = True                                                  # one long run
    sel = ColumnSelection(np.flatnonzero(mask), 97)
    for backed in (MemmapDense(str(tmp_path / "d.bin")), MemmapCSC(str(tmp_path / "csc"))):
        handler = data_handler_registry.get(backed)
        for lb, ub in ((0, sel.size), (3, 4), (5, sel.size - 2)):
            data, bounds = sel.fetch(handler, lb, ub)
            assert bounds == (0, ub - lb)
            got = data.toarray() if sparse.issparse(data) else np.asarray(data)
            np.testing.assert_array_equal(got, X[:, sel.cols[lb:ub]])
            if sparse.issparse(data):
                assert data.format == "csc" and data.has_sorted_indices


def _pack(lib, fn, *args, nr, b):
    W = (b + 31) // 32
    mask = np.zeros((nr, W), np.uint32)
    off = np.zeros(nr + 1, np.uint32)
    vals = np.zeros(nr * b + 16, np.float32)
    cnt = fn(*args, mask.ctypes.data, off.ctypes.data, vals.ctypes.data, vals.size)
    return cnt, mask, off, vals[:max(cnt, 0)]


@pytest.mark.parametrize("which", ["scattered", "unaligned", "one", "all", "ends"])
@pytest.mark.parametrize("with_rows", [False, True])
def test_host_column_list_pack_matches_contiguous_pack(which, with_rows):
    """illico_host_pack_cols_f32 over (rows, cols) packs byte for byte what illico_host_pack_rows_f32 makes of the contiguous
    array src[rows][:, cols] (this CPU's code path: AVX-512, AVX2 or scalar)."""
    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(4)
    n, N = 300, 173
    X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) < 0.2)).astype(np.float32)
    X[4, 5], X[9, 6], X[11, 0], X[12, N - 1] = -0.0, np.nan, 3.0, 2.0
    cols = {"scattered": np.sort(rng.choice(N, 97, replace=False)), "unaligned": np.sort(rng.choice(N, 33, replace=False)),
            "one": np.array([6]), "all": np.arange(N), "ends": np.array([0, 1, N - 2, N - 1])}[which]
    cols32 = np.ascontiguousarray(cols, dtype=np.int32)
    rows = np.ascontiguousarray(np.sort(rng.choice(n, 77, replace=False)), dtype=np.int64) if with_rows else None
    nr, b = (rows.size if with_rows else n), cols.size
    got = _pack(lib, lib.illico_host_pack_cols_f32, X.ctypes.data, N, rows.ctypes.data if with_rows else None, nr,
                cols32.ctypes.data, b, nr=nr, b=b)
    contiguous = np.ascontiguousarray((X[rows] if with_rows else X)[:, cols])
    want = _pack(lib, lib.illico_host_pack_rows_f32, contiguous.ctypes.data, b, nr, b, nr=nr, b=b)
    assert got[0] == want[0] > 0
    for g, w in zip(got[1:], want[1:]):
        np.testing.assert_array_equal(g.view(np.uint32), w.view(np.uint32))
    mask, off, vals = np.zeros((nr, (b + 31) // 32), np.uint32), np.zeros(nr + 1, np.uint32), np.zeros(b, np.float32)
    assert lib.illico_host_pack_cols_f32(X.ctypes.data, N, rows.ctypes.data if with_rows else None, nr, cols32.ctypes.data, b,
                                         mask.ctypes.data, off.ctypes.data, vals.ctypes.data, b) == -1     # does not fit


# ---- GPU: the kernels ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("which", ["scattered", "one", "all", "wide"])
@pytest.mark.parametrize("with_rows", [False, True])
def test_dense_gather_kernel_matches_numpy(dtype, which, with_rows):
    import torch

    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(5)
    n, N, ld = 700, 3001, 3005                                 # a source whose rows are longer than its columns (ld padding)
    X = np.zeros((n, ld), dtype)
    X[:, :N] = (rng.rand(n, N) < 0.3) * rng.standard_normal((n, N))
    X[:, N:] = 99.0                                            # never read
    cols = {"scattered": np.sort(rng.choice(N, 757, replace=False)), "one": np.array([N - 1]), "all": np.arange(N),
            "wide": np.sort(rng.choice(N, 2100, replace=False))}[which]
    rows = np.sort(rng.choice(n, 333, replace=False)) if with_rows else None
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    src = torch.from_numpy(X).to(dev)
    d_cols = torch.from_numpy(cols.astype(np.int32)).to(dev)
    d_rows = torch.from_numpy(rows.astype(np.int32)).to(dev) if with_rows else None
    n_out, b = (rows.size if with_rows else n), cols.size
    out_ld = (b + 3) & ~3
    out = torch.full((n_out, out_ld), 7.0, dtype=src.dtype, device=dev)
    code = _lib.DTYPE_F32 if dtype == np.float32 else _lib.DTYPE_F64
    _lib.check(lib.illico_select_cols_dense(src.data_ptr(), code, ld, d_rows.data_ptr() if with_rows else None, n_out,
                                            d_cols.data_ptr(), b, out.data_ptr(), out_ld, st), "illico_select_cols_dense")
    got = out.cpu().numpy()
    want = (X[rows] if with_rows else X)[:, cols]
    np.testing.assert_array_equal(got[:, :b].view(np.uint8), np.ascontiguousarray(want).view(np.uint8))
    assert not got[:, b:].any()                               # the padding is zeroed


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_csr_column_compaction_matches_scipy(dtype):
    """A CSR matrix compacted through new_col by illico_select_rows_csc[_indptr] (rows and columns swapped) is scipy's
    X[:, cols]: same row pointer, column indices renumbered and still sorted, same values."""
    import torch

    from illico_b200 import _lib
    from illico_b200.select import ColumnSelection, compact

    rng = np.random.RandomState(6)
    n, N = 2500, 1300
    X = (rng.rand(n, N) < 0.05) * rng.standard_normal((n, N))
    X[rng.rand(n) < 0.2] = 0.0                                 # empty rows
    X[:, rng.rand(N) < 0.3] = 0.0                              # columns with no entries
    X = sparse.csr_matrix(X.astype(dtype))
    dev = torch.device("cuda", 0)
    code = _lib.DTYPE_F32 if dtype == np.float32 else _lib.DTYPE_F64
    data = torch.from_numpy(X.data).to(dev)
    idx = torch.from_numpy(X.indices.astype(np.int32)).to(dev)
    ptr = torch.from_numpy(X.indptr.astype(np.int64)).to(dev)
    for cols in (np.sort(rng.choice(N, 321, replace=False)), np.array([0]), np.flatnonzero(np.diff(sparse.csc_matrix(X).indptr) == 0)):
        sel = ColumnSelection(cols, N)
        new_col = torch.from_numpy(sel.new_col()).to(dev)
        indptr, d, i = compact(data, code, idx, ptr.data_ptr(), n, new_col)
        want = X[:, cols]
        want.sort_indices()
        np.testing.assert_array_equal(indptr.cpu().numpy(), want.indptr)
        np.testing.assert_array_equal(i.cpu().numpy(), want.indices)
        np.testing.assert_array_equal(d.cpu().numpy(), want.data)
        got = i.cpu().numpy()
        p = want.indptr
        assert all(np.all(np.diff(got[p[r]:p[r + 1]]) > 0) for r in range(n))


@pytest.mark.gpu
def test_csr_repartition_over_the_selected_genes():
    """repartition_csr with a column selection: every row block is compacted before it is cut, so shard j holds the
    selected genes [edges[j], edges[j + 1]) -- scipy's X[:, cols][:, edges[j]:edges[j + 1]].  (Several shards on one GPU:
    the same code path as one shard per GPU, peer stores included.)"""
    import torch

    from illico_b200 import repartition
    from illico_b200.select import ColumnSelection

    rng = np.random.RandomState(14)
    n, N = 3000, 700
    X = (rng.rand(n, N) < 0.08) * rng.poisson(3.0, (n, N)).astype(np.float32)
    X[rng.rand(n) < 0.1] = 0.0
    X = sparse.csr_matrix(X.astype(np.float32))
    cols = np.flatnonzero(scattered_mask(N, seed=15))
    dev = torch.device("cuda", 0)
    edges = [0, 1, cols.size // 3, cols.size]                          # a one-gene shard among them
    shards = repartition.repartition_csr(X, [dev] * (len(edges) - 1), edges, cols=ColumnSelection(cols, N))
    torch.cuda.synchronize()
    sub = X[:, cols]
    sub.sort_indices()
    for j, M in enumerate(shards):
        want = sub[:, edges[j]:edges[j + 1]]
        assert M.shape == want.shape
        np.testing.assert_array_equal(M.indptr.cpu().numpy(), want.indptr)
        np.testing.assert_array_equal(M.indices.cpu().numpy(), want.indices)
        np.testing.assert_array_equal(M.data.cpu().numpy(), want.data)


# ---- GPU: the equivalence property ---------------------------------------------------------------------------------------

def _call(method, Xin, labels, reference, mask, groups, pts, kw):
    from illico_b200 import asymptotic_wilcoxon, ttest

    ad = VarAnnData(Xin, labels, var={"hv": mask if mask is not None else np.ones(Xin.shape[1], bool)})
    common = dict(return_array=True, score=True, pts=pts, p_adjust=True, groups=groups,
                  mask_var="hv" if mask is not None else None, **kw)
    if method == "wilcoxon":
        return asymptotic_wilcoxon(ad, False, "pert", reference, **common)
    return ttest(ad, "pert", reference, method=method, **common)


def assert_columns_of_full_call(sub, full, mask, method, integer, what):
    """sub: (groups, var, results, extra) of a call with mask_var (and perhaps groups); full: the same call without either.
    Every selected gene's values are its values in the full call; p_adj is Benjamini-Hochberg over the selected genes."""
    g_sub, var_sub, res_sub, ex_sub = sub
    g_full, var_full, res_full, ex_full = full
    cols = np.flatnonzero(mask)
    np.testing.assert_array_equal(var_sub, var_full[cols], err_msg=what)
    assert res_sub.shape[1] == cols.size
    # p_adj over the selected genes: bit for bit against statsmodels' restatement, on the call's own p-values and -- where
    # they are the full call's bit for bit -- on those
    np.testing.assert_array_equal(ex_sub["p_adj"], bh_reference(res_sub[:, :, 0]), err_msg=f"{what}: p_adj")
    restricted = {k: v[:, cols] for k, v in ex_full.items()}
    restricted["p_adj"] = bh_reference(res_full[:, cols, 0])
    assert_rows_of_full_call(sub, (g_full, var_full[cols], np.ascontiguousarray(res_full[:, cols]), restricted), method, integer,
                             what)


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("test", ["ovo", "ovr"])
@pytest.mark.parametrize("route", ROUTES)
def test_selected_genes_equal_the_full_call(route, test, method, monkeypatch, tmp_path):
    X, labels = labelled_counts(7, 5000, 320, 12, control_share=0.6)
    Xin, kw, integer = _route_input(route, X, monkeypatch, tmp_path)
    reference = CONTROL if test == "ovo" else None
    N = X.shape[1]
    names = sorted(set(labels) - {CONTROL})
    masks = [("one", np.arange(N) == 1, None), ("scattered", scattered_mask(N), None), ("all", np.ones(N, bool), None),
             ("with groups", scattered_mask(N, seed=3), [names[1], names[6]])]
    for pts in (False, True):
        full = _call(method, Xin, labels, reference, None, None, pts, kw)
        for name, mask, groups in masks:
            sub = _call(method, Xin, labels, reference, mask, groups, pts, kw)
            if groups is not None:
                assert list(sub[0]) == sorted(set(groups) | ({CONTROL} if reference else set()))
            else:
                assert list(sub[0]) == list(full[0])
            assert_columns_of_full_call(sub, full, mask, method, integer, f"{route} {test} {method} pts={pts} mask={name}")


@pytest.mark.gpu
def test_packed_upload_moves_only_the_selected_columns(monkeypatch):
    """A mostly-zero dense host matrix with a 25 % mask: the packed upload squeezes only the selected columns
    (illico_host_pack_cols_f32), so its bytes over PCIe stay below 0.35 of the selected columns' raw bytes."""
    from illico_b200 import hostio

    monkeypatch.setenv("ILLICO_PACK_UPLOAD", "1")
    X, labels = labelled_counts(12, 31000, 2240, 12, control_share=0.5, density=0.1)
    mask = np.zeros(X.shape[1], bool)
    mask[np.sort(np.random.RandomState(13).choice(X.shape[1], 560, replace=False))] = True
    mask[0] = mask[-1] = True
    n_sel = int(mask.sum())
    assert X.shape[0] * n_sel * 4 >= 64 << 20                 # large enough to be squeezed
    full = _call("wilcoxon", X, labels, CONTROL, None, None, True, {})
    hostio.LAST_UPLOAD.clear()
    sub = _call("wilcoxon", X, labels, CONTROL, mask, None, True, {})
    st = hostio.LAST_UPLOAD
    assert st.get("packed", 0) > 0 and st["raw"] == 0
    assert st["bytes"] < 0.35 * X.shape[0] * n_sel * 4
    assert_columns_of_full_call(sub, full, mask, "wilcoxon", True, "packed 25 %")


def _host_ranking(full, mask, k, reference_row, filt):
    """rank_genes by hand from a full call's arrays: per group, the selected genes (passing the filters) by score descending,
    ties by gene index, NaN last; p_adj over the selected genes."""
    g, var, res, ex = full
    cols = np.flatnonzero(mask)
    p, score = res[:, cols, 0], ex["score"][:, cols]
    padj = bh_reference(p)
    out = {}
    for gi in range(len(g)):
        if gi == reference_row:
            continue
        keep = np.ones(cols.size, bool)
        with np.errstate(invalid="ignore"):
            if "min_in_group_fraction" in filt:
                keep &= ex["pct_nz_group"][gi, cols] >= filt["min_in_group_fraction"]
            if "max_out_group_fraction" in filt:
                keep &= ex["pct_nz_reference"][gi, cols] <= filt["max_out_group_fraction"]
            if "min_fold_change" in filt:
                keep &= res[gi, cols, 2] >= filt["min_fold_change"]
        cand = np.flatnonzero(keep)
        s = score[gi, cand]
        order = cand[np.lexsort((cand, np.where(np.isnan(s), np.inf, -s)))][:k]
        rec = {"feature": var[cols[order]], "score": score[gi, order], "p_value": p[gi, order], "p_adj": padj[gi, order],
               "statistic": res[gi, cols[order], 1], "fold_change": res[gi, cols[order], 2]}
        if filt:                                               # (a filter implies pts)
            rec["pct_nz_group"], rec["pct_nz_reference"] = ex["pct_nz_group"][gi, cols[order]], ex["pct_nz_reference"][gi, cols[order]]
        out[g[gi]] = rec
    return out


@pytest.mark.gpu
def test_rank_genes_with_mask_var_equals_a_host_ranking(monkeypatch, tmp_path):
    from illico_b200 import rank_genes

    X, labels = labelled_counts(8, 4000, 200, 8, control_share=0.5)
    mask = scattered_mask(X.shape[1], seed=9)
    for route in ("dense_pageable", "csr", "cuda_tensor"):
        Xin, kw, _ = _route_input(route, X, monkeypatch, tmp_path)
        ad = VarAnnData(Xin, labels, var={"highly_variable": mask})
        for reference in (CONTROL, None):
            for method in ("wilcoxon", "t-test"):
                full = _call(method, Xin, labels, reference, None, None, True, kw)
                ref_row = list(full[0]).index(CONTROL) if reference else None
                for filt in ({}, dict(min_in_group_fraction=0.1, max_out_group_fraction=0.5, min_fold_change=1.0)):
                    for n_genes in (15, 10_000):
                        sub = rank_genes(ad, False, "pert", reference, n_genes=n_genes, method=method, mask_var="highly_variable",
                                         **filt, **kw)
                        want = _host_ranking(full, mask, n_genes, ref_row, filt)
                        what = f"{route} ref={reference} {method} {filt} n_genes={n_genes}"
                        assert list(sub.index.get_level_values("pert").unique()) == [g for g in want if want[g]["score"].size], what
                        assert set(sub["feature"].cat.categories) == set(np.asarray(ad.var_names)[mask]), what
                        for g, rec in want.items():
                            part = sub.xs(g, level="pert") if rec["score"].size else sub.iloc[:0]
                            assert len(part) == rec["score"].size <= int(mask.sum()), what
                            np.testing.assert_array_equal(np.asarray(part["feature"]), rec["feature"], err_msg=what)
                            for col, v in rec.items():
                                if col != "feature":
                                    np.testing.assert_array_equal(part[col].to_numpy(), v, err_msg=f"{what} {g} {col}")


@pytest.mark.gpu
def test_mask_var_on_every_gpu():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    X, labels = labelled_counts(10, 5000, 333, 12, control_share=0.6)
    mask = scattered_mask(X.shape[1], seed=11)
    names = sorted(set(labels) - {CONTROL})
    for Xin in (X, sparse.csr_matrix(X), sparse.csc_matrix(X), torch.from_numpy(X).to("cuda:0")):
        for reference in (CONTROL, None):
            for method in ("wilcoxon", "t-test"):
                full = _call(method, Xin, labels, reference, None, None, True, dict(devices="all"))
                for groups in (None, [names[2], names[5]]):
                    sub = _call(method, Xin, labels, reference, mask, groups, True, dict(devices="all"))
                    assert_columns_of_full_call(sub, full, mask, method, True,
                                                f"devices=all {type(Xin)} {reference} {method} groups={groups}")
