"""``rank_genes_groups``: scanpy's call and result layout (``adata.uns``), and the kernels under it -- the group sums pass
``illico_group_sums_*``, ``illico_log_fold_changes``, ``illico_bonferroni_adjust`` and ``illico_top_genes_columns``.

The oracle is a numpy / scipy restatement of scanpy 1.10's ``_RankGenes``: group means and variances from float64 sums,
Wilcoxon ranks from ``scipy.stats.rankdata`` (over group and reference, or over all cells) with scanpy's ``_tiecorrect``,
the t-test through ``ttest_ind_from_stats`` with scanpy's NaN replacements, Benjamini-Hochberg as statsmodels' ``fdr_bh``,
Bonferroni as ``np.minimum(p * n_genes, 1)`` and the log fold change from the group means."""
import ctypes
import os
import subprocess

import numpy as np
import pandas as pd
import pytest
from scipy import sparse, stats

from tests.test_rank_genes import bh_reference
from tests.util import FakeAnnData

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_FUNCTIONS = ["illico_group_sums_dense", "illico_group_sums_csr", "illico_group_sums_csc", "illico_log_fold_changes",
                 "illico_bonferroni_adjust", "illico_top_genes_columns"]
FIELDS_DTYPE = {"names": "O", "scores": "float32", "logfoldchanges": "float32", "pvals": "float64", "pvals_adj": "float64"}


class AnnData(FakeAnnData):
    """FakeAnnData with what scanpy's call reads and writes besides: ``uns``, ``var``, ``raw`` and ``copy()``."""

    def __init__(self, X, labels, var_names=None, key="pert", layers=None, uns=None, var=None, raw=None, categories=None):
        super().__init__(X, labels, var_names, key, layers)
        if categories is not None:
            self.obs[key] = pd.Categorical(list(labels), categories=categories)
        self.uns = uns if uns is not None else {}
        self.var = var if var is not None else pd.DataFrame(index=self.var_names)
        self.raw = raw

    def copy(self):
        out = AnnData.__new__(AnnData)
        out.__dict__.update({k: (v.copy() if hasattr(v, "copy") and k != "raw" else v) for k, v in self.__dict__.items()})
        out.uns = {k: v for k, v in self.uns.items()}
        return out


class Raw:
    def __init__(self, X, var_names, var=None):
        self.X, self.var_names = X, pd.Index(var_names)
        self.var = var if var is not None else pd.DataFrame(index=self.var_names)


def data(seed=3, n_cells=900, n_genes=40, n_perts=6, dtype=np.float32):
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=seed, n_cells=n_cells, n_genes=n_genes, n_perts=n_perts, lam=1.5, masked=0.6, dtype=dtype)
    X[:, 0] = 0                      # an all-zero gene (every test tied: score 0, p 1, lfc 0)
    X[:, 1] = 2                      # a constant gene
    return X, np.asarray(labels)


# ---- the oracle: scanpy 1.10 _RankGenes ---------------------------------------------------------------------------------

def _tiecorrect(ranks):
    size = ranks.shape[0]
    if size < 2:
        return np.ones(ranks.shape[1])
    arr = np.sort(ranks, axis=0)
    out = np.empty(ranks.shape[1])
    for j in range(ranks.shape[1]):
        a = arr[:, j]
        idx = np.nonzero(np.r_[True, a[1:] != a[:-1], True])[0]
        cnt = np.diff(idx).astype(np.float64)
        out[j] = 1.0 - (cnt ** 3 - cnt).sum() / float(size ** 3 - size)
    return out


def _mean_var(X):
    mean = X.mean(axis=0)
    var = (X * X).mean(axis=0) - mean ** 2
    return mean, var * (X.shape[0] / (X.shape[0] - 1))


def scanpy_oracle(X, labels, order, reference="rest", method="t-test", corr_method="benjamini-hochberg", tie_correct=False,
                  log_scale=1.0):
    """{group: (scores, pvals, pvals_adj, lfc)} over every gene of ``X`` (dense float64), and (pts, pts_rest) [G, N]."""
    X = np.asarray(X, dtype=np.float64)
    n_cells, N = X.shape
    masks = [labels == g for g in order]
    iref = None if reference == "rest" else order.index(reference)
    ns = np.array([m.sum() for m in masks])
    means, vars_ = zip(*[_mean_var(X[m]) for m in masks])
    out = {}
    with np.errstate(all="ignore"):
        pts = np.array([(X[m] != 0).sum(0) / m.sum() for m in masks])
        pts_rest = np.array([(X[~m] != 0).sum(0) / (~m).sum() for m in masks]) if iref is None else None
        for i, g in enumerate(order):
            if i == iref:
                continue
            m = masks[i]
            if iref is None:
                mean_r, var_r = _mean_var(X[~m])
                n_r = n_cells - ns[i]
            else:
                mean_r, var_r, n_r = means[iref], vars_[iref], ns[iref]
            if method in ("t-test", "t-test_overestim_var"):
                nobs2 = ns[i] if method == "t-test_overestim_var" else n_r
                s, p = stats.ttest_ind_from_stats(means[i], np.sqrt(vars_[i]), ns[i], mean_r, np.sqrt(var_r), nobs2, equal_var=False)
                s, p = np.where(np.isnan(s), 0.0, s), np.where(np.isnan(p), 1.0, p)
            else:
                if iref is None:
                    ranks = stats.rankdata(X, axis=0)
                    T = _tiecorrect(ranks) if tie_correct else 1.0
                    sd = np.sqrt(T * ns[i] * (n_cells - ns[i]) * (n_cells + 1) / 12.0)
                    s = (ranks[m].sum(0) - ns[i] * (n_cells + 1) / 2.0) / sd
                else:
                    both = np.vstack([X[m], X[masks[iref]]])
                    ranks = stats.rankdata(both, axis=0)
                    T = _tiecorrect(ranks) if tie_correct else 1.0
                    n1, n2 = ns[i], ns[iref]
                    sd = np.sqrt(T * n1 * n2 * (n1 + n2 + 1) / 12.0)
                    s = (ranks[:n1].sum(0) - n1 * (n1 + n2 + 1) / 2.0) / sd
                s = np.where(np.isnan(s), 0.0, s)
                p = 2 * stats.norm.sf(np.abs(s))
            if corr_method == "benjamini-hochberg":
                padj = bh_reference(np.where(np.isnan(p), 1.0, p)[None, :])[0]
            else:
                padj = np.minimum(p * N, 1.0)
            f = lambda x: np.expm1(x * log_scale)  # noqa: E731
            lfc = np.log2((f(means[i]) + 1e-9) / (f(mean_r) + 1e-9))
            out[str(g)] = (s, p, padj, lfc)
    return out, pts, pts_rest


def f32_match(got32, want64, rel=1e-13):
    """got (float32) is want rounded to float32, or its neighbour where want is within ``rel`` of the rounding boundary."""
    got32, want64 = np.asarray(got32, np.float32), np.asarray(want64, np.float64)
    w = want64.astype(np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        lo, hi = (want64 * (1 - rel)).astype(np.float32), (want64 * (1 + rel)).astype(np.float32)
    same = (got32 == w) | (np.isnan(got32) & np.isnan(w)) | (got32 == lo) | (got32 == hi)
    return same


def p_match(got, want, rel=1e-12):
    got, want = np.asarray(got), np.asarray(want)
    both0 = (got == 0) & (want == 0)
    return both0 | (np.abs(got - want) <= rel * np.abs(want)) | (np.isnan(got) & np.isnan(want))


def check_uns(res, want, var_names, k, rankby_abs=False, what=""):
    """The record arrays of ``res`` against the oracle ``want`` ({group: (scores, p, padj, lfc)})."""
    fields = list(want)
    for key, dt in FIELDS_DTYPE.items():
        rec = res[key]
        assert isinstance(rec, np.recarray) and rec.shape == (k,), (what, key, rec.shape)
        assert list(rec.dtype.names) == fields, (what, key)
        assert all(rec.dtype[f] == np.dtype(dt) for f in fields), (what, key, rec.dtype)
    pos = {n: i for i, n in enumerate(var_names)}
    for g, (s, p, padj, lfc) in want.items():
        gene = np.array([pos[n] for n in res["names"][g]])
        assert len(set(gene)) == k, what
        key = np.abs(s) if rankby_abs else s
        order = np.lexsort((np.arange(s.size), -key))
        # names: the oracle's order wherever the scores are distinct; a near-tie (1e-12 relative) may swap
        exp = order[:k]
        bad = gene != exp
        if bad.any():
            a, b = key[gene[bad]], key[exp[bad]]
            assert np.all(np.abs(a - b) <= 1e-12 * np.maximum(np.abs(a), np.abs(b)) + 1e-300), (what, g, gene[bad], exp[bad])
        assert f32_match(res["scores"][g], s[gene]).all(), (what, g, "scores")
        assert f32_match(res["logfoldchanges"][g], lfc[gene]).all(), (what, g, "lfc", res["logfoldchanges"][g], lfc[gene])
        assert p_match(res["pvals"][g], p[gene]).all(), (what, g, "pvals")
        assert p_match(res["pvals_adj"][g], padj[gene]).all(), (what, g, "pvals_adj")


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_new_functions_are_bound_and_declared(tmp_path):
    from illico_b200 import _lib

    for name in NEW_FUNCTIONS:
        assert name in _lib.SIGNATURES
    src = tmp_path / "decl.c"
    src.write_text(
        '#include "illico_b200.h"\n'
        "int (*a)(const void*, int32_t, int64_t, int32_t, int32_t, const illico_plan_t*, double*, int32_t*, int64_t, int64_t, void*)"
        " = illico_group_sums_dense;\n"
        "int (*b)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, double*, int32_t*,"
        " int64_t, int64_t, void*) = illico_group_sums_csr;\n"
        "int (*c)(const void*, int32_t, const int32_t*, const int64_t*, int32_t, int32_t, const illico_plan_t*, double*, int32_t*,"
        " int64_t, int64_t, void*) = illico_group_sums_csc;\n"
        "int (*d)(const double*, int64_t, const int32_t*, int32_t, int32_t, int32_t, int64_t, double, double*, int64_t, void*)"
        " = illico_log_fold_changes;\n"
        "int (*e)(const double*, int64_t, int64_t, int32_t, int32_t, double*, void*) = illico_bonferroni_adjust;\n"
        "int (*f)(const double*, int64_t, const double*, int64_t, const double*, const double*, int64_t, int32_t, int32_t,"
        " const int32_t*, int32_t, int32_t, int32_t, int32_t*, float*, float*, double*, double*, void*, size_t, void*)"
        " = illico_top_genes_columns;\n"
        "int main(void) { return !(a && b && c && d && e && f) || ILLICO_ABI_VERSION != 3; }\n")
    subprocess.check_call(["gcc", "-std=c11", "-Werror=incompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c",
                           str(src), "-o", str(tmp_path / "decl.o")])


def test_new_kernels_do_not_spill(tmp_path):
    import shutil

    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from illico_b200.build import NVCC_FLAGS

    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    for src, kernels in (("counts.cu", ("count_dense_kernelIfLi1", "count_dense_kernelIdLi1", "count_csr_kernelIfLi1",
                                        "count_csr_kernelIdLi1", "count_csc_kernelIfLb1ELi1", "count_csc_kernelIfLb0ELi1",
                                        "count_csc_kernelIdLb1ELi1", "count_csc_kernelIdLb0ELi1")),
                         ("ttest.cu", ("log_fold_change_kernel",)),
                         ("extras.cu", ("bonferroni_kernel", "top_genes_kernelILb1"))):
        res = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(ROOT, "illico_b200", "csrc", src), "-o",
                                               str(tmp_path / (src + ".o"))], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        seen, current = set(), None
        for line in res.stderr.splitlines():
            if "Function properties for" in line:
                current = line.split("for", 1)[1].strip()
            elif "spill" in line and current:
                for k in kernels:
                    if k in current:
                        seen.add(k)
                        assert " 0 bytes spill stores, 0 bytes spill loads" in line, (current, line)
        assert seen == set(kernels), (src, set(kernels) - seen)


def _no_cuda(monkeypatch):
    from illico_b200 import engine

    def no_cuda(*a, **k):
        raise AssertionError("device work started")

    monkeypatch.setattr(engine, "require_cuda", no_cuda)


@pytest.mark.parametrize("kw", [dict(groups="p0000"), dict(reference="nope"), dict(method="logreg"), dict(method="wilcox"),
                                dict(corr_method="holm"), dict(use_raw=True), dict(use_raw=True, layer="L", raw=True),
                                dict(groups=["p0000", "single"]), dict(single_in_all=True), dict(empty_category=True),
                                dict(groups=["p0000", "nope"]), dict(n_genes=0), dict(mask_var="missing")])
def test_errors_are_raised_before_any_device_work(monkeypatch, kw):
    from illico_b200 import rank_genes_groups

    kw = dict(kw)
    X, labels = data(n_cells=300, n_genes=8)
    categories = None
    if kw.pop("single_in_all", False) or "single" in str(kw.get("groups", "")):
        labels = labels.copy()
        labels[0] = "single"
    if kw.pop("empty_category", False):
        categories = sorted(set(labels)) + ["zzz_empty"]
    raw = Raw(X, [f"gene_{i}" for i in range(X.shape[1])]) if kw.pop("raw", False) else None
    ad = AnnData(X, labels, layers={"L": X}, raw=raw, categories=categories)
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError):
        rank_genes_groups(ad, "pert", **kw)
    assert "rank_genes_groups" not in ad.uns


def test_group_order():
    from illico_b200.scanpy_compat import group_order

    labels = pd.Series(["b", "a", "c", "a", "b", "c", "d", "d"])
    assert group_order(labels, "all", "rest") == ["a", "b", "c", "d"]
    cat = pd.Series(pd.Categorical(labels, categories=["c", "a", "d", "b"]))
    assert group_order(cat, "all", "rest") == ["c", "a", "d", "b"]
    assert group_order(cat, "all", "b") == ["c", "a", "d", "b"]
    assert group_order(labels, ["d", "b"], "rest") == ["d", "b"]
    assert group_order(labels, ["d", "b"], "a") == ["d", "b", "a"]
    assert group_order(labels, ["d", "a", "b"], "a") == ["d", "a", "b"]
    assert group_order(pd.Series([1, 1, 0, 0, 2, 2]).astype(str), [2, 0], "rest") == ["2", "0"]


def test_records_match_pandas_to_records():
    from illico_b200.scanpy_compat import name_records, records

    rng = np.random.RandomState(0)
    k, fields = 7, ["g1", "ctrl", "10"]
    var_names = pd.Index([f"v{i}" for i in range(20)])
    gene = rng.randint(0, 20, size=(k, 3)).astype(np.int32)
    planes = {"scores": rng.randn(k, 3).astype(np.float32), "pvals": rng.rand(k, 3), "pvals_adj": rng.rand(k, 3),
              "logfoldchanges": rng.randn(k, 3).astype(np.float32)}
    for key, plane in planes.items():
        want = pd.DataFrame(plane.astype(np.float64), columns=fields).to_records(index=False, column_dtypes=FIELDS_DTYPE[key])
        got = records(plane, fields)
        assert got.dtype == want.dtype and isinstance(got, np.recarray)
        assert got.base is not None and np.shares_memory(got, plane)          # a view, not a copy
        for f in fields:
            np.testing.assert_array_equal(got[f], want[f])
    want = pd.DataFrame({f: var_names[gene[:, c]] for c, f in enumerate(fields)}).to_records(index=False, column_dtypes="O")
    got = name_records(gene, var_names, fields)
    assert got.dtype == want.dtype
    for f in fields:
        assert list(got[f]) == list(want[f])


def test_use_raw_resolution():
    from illico_b200.scanpy_compat import resolve_use_raw

    X, labels = data(n_cells=50, n_genes=4)
    plain = AnnData(X, labels)
    with_raw = AnnData(X, labels, raw=Raw(X, ["a", "b", "c", "d"]))
    assert resolve_use_raw(plain, None, None) is False
    assert resolve_use_raw(with_raw, None, None) is True
    assert resolve_use_raw(with_raw, None, "L") is False
    assert resolve_use_raw(with_raw, False, None) is False
    with pytest.raises(ValueError):
        resolve_use_raw(plain, True, None)
    with pytest.raises(ValueError):
        resolve_use_raw(with_raw, True, "L")


def test_public_name_whatever_the_import_order():
    import sys

    code = ("from illico_b200 import rank_genes_groups; import illico_b200 as m; from illico_b200 import asymptotic_wilcoxon; "
            "assert callable(rank_genes_groups) and callable(m.asymptotic_wilcoxon) and callable(asymptotic_wilcoxon)")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


# ---- GPU: uns against the oracle -----------------------------------------------------------------------------------------

def run_and_check(X, labels, *, Xo=None, var_names=None, ad_kw=None, oracle_labels=None, **kw):
    """rank_genes_groups on ``X`` against the oracle on ``Xo`` (dense float64, default ``X``)."""
    from illico_b200 import rank_genes_groups
    from illico_b200.scanpy_compat import group_order

    ad = AnnData(X, labels, var_names=var_names, **(ad_kw or {}))
    Xo = np.asarray(X.toarray() if hasattr(X, "toarray") else (X.cpu().numpy() if hasattr(X, "cpu") else X), np.float64) \
        if Xo is None else Xo
    order = group_order(ad.obs["pert"], kw.get("groups", "all"), kw.get("reference", "rest"))
    base = ad.uns.get("log1p", {}).get("base")
    want, pts, pts_rest = scanpy_oracle(Xo, np.asarray(labels), order, kw.get("reference", "rest"), kw.get("method") or "t-test",
                                        kw.get("corr_method", "benjamini-hochberg"), kw.get("tie_correct", False),
                                        np.log(base) if base is not None else 1.0)
    out = rank_genes_groups(ad, "pert", **kw)
    key = kw.get("key_added") or "rank_genes_groups"
    if kw.get("copy"):
        assert key not in ad.uns
        ad = out
    else:
        assert out is None
    res = ad.uns[key]
    names = list(ad.var_names) if var_names is None else list(var_names)
    k = Xo.shape[1] if kw.get("n_genes") is None else min(kw["n_genes"], Xo.shape[1])
    check_uns(res, want, names, k, kw.get("rankby_abs", False), what=str(kw))
    assert res["params"] == dict(groupby="pert", reference=kw.get("reference", "rest"), method=kw.get("method") or "t-test",
                                 use_raw=False, layer=kw.get("layer"), corr_method=kw.get("corr_method", "benjamini-hochberg"))
    if kw.get("pts"):
        cols = [str(g) for g in order]
        assert list(res["pts"].columns) == cols and list(res["pts"].index) == names
        np.testing.assert_array_equal(res["pts"].to_numpy(), pts.T)
        if kw.get("reference", "rest") == "rest":
            np.testing.assert_array_equal(res["pts_rest"].to_numpy(), pts_rest.T)
        else:
            assert "pts_rest" not in res
    return res


CASES = [
    dict(method="wilcoxon"),
    dict(method="wilcoxon", tie_correct=True),
    dict(method="wilcoxon", reference="non-targeting", tie_correct=True, pts=True),
    dict(),
    dict(method="t-test", reference="non-targeting", corr_method="bonferroni"),
    dict(method="t-test_overestim_var", pts=True),
    dict(method="wilcoxon", rankby_abs=True, n_genes=7),
    dict(method="t-test", rankby_abs=True, n_genes=1, corr_method="bonferroni"),
    dict(method="wilcoxon", n_genes=1000, corr_method="bonferroni", key_added="mine"),
    dict(method="wilcoxon", groups=["p0003", "p0000"], pts=True),
    dict(method="wilcoxon", groups=["p0003", "p0000"], reference="non-targeting"),
    dict(method="t-test", groups=["p0004", "non-targeting", "p0001"], reference="non-targeting", copy=True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("kw", CASES, ids=[str(i) for i in range(len(CASES))])
def test_against_the_oracle(kw):
    X, labels = data()
    run_and_check(X, labels, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["dense", "csr", "csc", "float64", "cuda", "backed_csc", "all_gpus"])
@pytest.mark.parametrize("method", ["wilcoxon", "t-test"])
def test_input_routes(route, method, tmp_path):
    import torch

    X, labels = data(n_cells=1100, n_genes=37)
    Xo = X.astype(np.float64)
    kw = dict(method=method, pts=True)
    if route == "csr":
        Xr = sparse.csr_matrix(X)
    elif route == "csc":
        Xr = sparse.csc_matrix(X)
    elif route == "float64":
        Xo = Xo.copy()
        Xo[5, 9] = 16777217.0                  # float32 cannot hold it: the recode path, exact float64 sums
        Xr = Xo
    elif route == "cuda":
        Xr = torch.from_numpy(X).cuda()
    elif route == "backed_csc":
        from illico_b200.backed import MemmapCSC, save_csc

        C = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), C.data, C.indices, C.indptr, C.shape)
        Xr = MemmapCSC(str(tmp_path / "csc"))
        kw["batch_size"] = 8
    elif route == "all_gpus":
        Xr, kw["devices"] = X, "all"
    else:
        Xr = X
    for ref in ("rest", "non-targeting"):
        run_and_check(Xr, labels, Xo=Xo, reference=ref, **kw)


@pytest.mark.gpu
def test_mask_var_layer_use_raw_and_log1p_base():
    X, labels = data(n_cells=800, n_genes=30)
    names = [f"g{i}" for i in range(30)]
    mask = np.zeros(30, bool)
    mask[[1, 2, 5, 6, 7, 20, 29]] = True
    var = pd.DataFrame({"hv": mask}, index=names)
    # mask_var: only those genes, Bonferroni over their number
    from illico_b200 import rank_genes_groups

    for method in ("wilcoxon", "t-test"):
        ad = AnnData(X, labels, var_names=names, var=var)
        rank_genes_groups(ad, "pert", method=method, mask_var="hv", corr_method="bonferroni", pts=True)
        res = ad.uns["rank_genes_groups"]
        want, pts, pts_rest = scanpy_oracle(X[:, mask].astype(np.float64), labels, sorted(set(labels)), method=method,
                                            corr_method="bonferroni")
        check_uns(res, want, list(np.asarray(names)[mask]), int(mask.sum()), what=f"mask_var {method}")
        np.testing.assert_array_equal(res["pts"].to_numpy(), pts.T)
        assert list(res["pts"].index) == list(np.asarray(names)[mask])
    # layer: the layer's values, not X
    L = (X * 2).astype(np.float32)
    ad = AnnData(np.zeros_like(X), labels, layers={"L": L})
    rank_genes_groups(ad, "pert", method="wilcoxon", layer="L")
    want, _, _ = scanpy_oracle(L.astype(np.float64), labels, sorted(set(labels)), method="wilcoxon")
    check_uns(ad.uns["rank_genes_groups"], want, list(ad.var_names), 30, what="layer")
    assert ad.uns["rank_genes_groups"]["params"]["layer"] == "L"
    # use_raw (default with a raw): raw.X, raw.var_names, mask_var looked up in raw.var
    raw_names = [f"r{i}" for i in range(30)]
    ad = AnnData(np.zeros((X.shape[0], 3), np.float32), labels,
                 raw=Raw(X, raw_names, pd.DataFrame({"hv": mask}, index=raw_names)))
    rank_genes_groups(ad, "pert", method="t-test", mask_var="hv")
    want, _, _ = scanpy_oracle(X[:, mask].astype(np.float64), labels, sorted(set(labels)))
    check_uns(ad.uns["rank_genes_groups"], want, list(np.asarray(raw_names)[mask]), int(mask.sum()), what="use_raw")
    assert ad.uns["rank_genes_groups"]["params"]["use_raw"] is True
    # log1p in base 2: expm1(x ln 2)
    Xl = np.log2(1 + X).astype(np.float32)
    run_and_check(Xl, labels, Xo=Xl.astype(np.float64), ad_kw=dict(uns={"log1p": {"base": 2}}), method="wilcoxon")
    run_and_check(Xl, labels, Xo=Xl.astype(np.float64), ad_kw=dict(uns={"log1p": {"base": None}}), method="t-test")


@pytest.mark.gpu
def test_categorical_order():
    X, labels = data(n_cells=700, n_genes=12)
    cats = ["p0002", "non-targeting", "p0005", "p0000", "p0001", "p0003", "p0004"]
    res = run_and_check(X, labels, ad_kw=dict(categories=cats), method="wilcoxon", pts=True)
    assert list(res["scores"].dtype.names) == cats and list(res["pts"].columns) == cats
    res = run_and_check(X, labels, ad_kw=dict(categories=cats), reference="p0000", method="t-test", pts=True)
    assert list(res["scores"].dtype.names) == [c for c in cats if c != "p0000"] and list(res["pts"].columns) == cats


@pytest.mark.gpu
def test_other_calls_are_unchanged():
    """A rank_genes_groups call leaves asymptotic_wilcoxon and rank_genes bit-identical (no state survives it)."""
    from illico_b200 import asymptotic_wilcoxon, rank_genes, rank_genes_groups

    X, labels = data(n_cells=900, n_genes=33)
    ad = AnnData(X, labels)
    before = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference="non-targeting", p_adjust=True, score=True,
                                 pts=True)
    rg_before = rank_genes(ad, is_log1p=False, group_keys="pert", n_genes=10, pts=True)
    rank_genes_groups(ad, "pert", method="wilcoxon", pts=True)
    rank_genes_groups(ad, "pert", method="t-test", reference="non-targeting")
    after = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference="non-targeting", p_adjust=True, score=True,
                                pts=True)
    rg_after = rank_genes(ad, is_log1p=False, group_keys="pert", n_genes=10, pts=True)
    pd.testing.assert_frame_equal(before, after, check_exact=True)
    pd.testing.assert_frame_equal(rg_before, rg_after, check_exact=True)


# ---- GPU: the kernels ------------------------------------------------------------------------------------------------

def _engine(labels, reference=None, seg_max=None):
    from illico_b200.engine import Engine
    from illico_b200.groups import build_plan, encode_and_count_groups

    _, grpc = encode_and_count_groups(np.asarray(labels), reference)
    return Engine(grpc, "cuda:0", host_plan=build_plan(grpc, seg_max)), grpc


def _device_matrix(X, fmt, dtype):
    import torch

    from illico_b200.engine import DeviceMatrix

    t = torch.float64 if dtype == np.float64 else torch.float32
    if fmt == "dense":
        return DeviceMatrix("dense", X.shape, torch.from_numpy(X.astype(dtype)).cuda())
    S = sparse.csr_matrix(X) if fmt == "csr" else sparse.csc_matrix(X)
    return DeviceMatrix(fmt, X.shape, torch.from_numpy(S.data.astype(dtype)).to("cuda", t),
                        torch.from_numpy(S.indices.astype(np.int32)).cuda(), torch.from_numpy(S.indptr.astype(np.int64)).cuda())


def _call_pass(eng, M, kind, lb, b, counts=True):
    """(sums [G, b], counts [G, b]) of ``illico_group_sums_*`` (kind "sums") or (S1, counts) of ``illico_group_moments_*``
    (kind "moments"), or the counts of ``illico_count_nonzero_*`` (kind "count")."""
    import torch

    from illico_b200 import _lib

    lib, G = _lib.load(), eng.n_groups
    st = torch.cuda.current_stream().cuda_stream
    dt = _lib.DTYPE_F64 if M.data.dtype == torch.float64 else _lib.DTYPE_F32
    sums = torch.full((3, G, b), np.nan, dtype=torch.float64, device="cuda")
    cnt = torch.full((G, b), -7, dtype=torch.int32, device="cuda")
    plan = ctypes.byref(eng.plan)
    head = [M.data.data_ptr(), dt] + ([M.data.stride(0)] if M.fmt == "dense" else [M.indices.data_ptr(), M.indptr.data_ptr()]) + \
        [lb, b, plan]
    cp = cnt.data_ptr() if counts else None
    if kind == "sums":
        rc = getattr(lib, f"illico_group_sums_{M.fmt}")(*head, sums[0].data_ptr(), cp, b, b, st)
    elif kind == "moments":
        rc = getattr(lib, f"illico_group_moments_{M.fmt}")(*head, 0, sums[0].data_ptr(), sums[1].data_ptr(), None, cp, b, b, st)
    else:
        rc = getattr(lib, f"illico_count_nonzero_{M.fmt}")(*head, cnt.data_ptr(), b, st)
    _lib.check(rc, kind)
    torch.cuda.synchronize()
    return sums[0].cpu().numpy(), cnt.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_group_sums_pass(fmt, dtype):
    """Bit-identical to the moments pass's S1, to numpy (integer data) and, for its count plane, to illico_count_nonzero_*;
    groups of several plan segments (seg_max 64), a batch inside the matrix, and wide batches (CSR tiles)."""
    X, labels = data(n_cells=2000, n_genes=4500 if fmt == "csr" else 300)
    X[3, 7] = -2.0
    eng, grpc = _engine(labels, seg_max=64)
    M = _device_matrix(X, fmt, dtype)
    codes = grpc.encoded_groups
    for lb, ub in ((0, X.shape[1]), (5, X.shape[1] - 3)):
        b = ub - lb
        s, c = _call_pass(eng, M, "sums", lb, b)
        m, cm = _call_pass(eng, M, "moments", lb, b)
        _, cn = _call_pass(eng, M, "count", lb, b)
        want = np.stack([X[codes == g, lb:ub].astype(np.float64).sum(0) for g in range(eng.n_groups)])
        np.testing.assert_array_equal(s, want)
        np.testing.assert_array_equal(s, m)
        np.testing.assert_array_equal(c, cn)
        np.testing.assert_array_equal(cm, cn)
        s2, _ = _call_pass(eng, M, "sums", lb, b, counts=False)
        np.testing.assert_array_equal(s2, want)


@pytest.mark.gpu
def test_group_sums_csc_global_branch(monkeypatch):
    """More groups than the shared histogram holds (4096): the CTA adds into its global columns."""
    from illico_b200 import _lib

    rng = np.random.RandomState(2)
    G = 4200
    labels = np.repeat([f"c{i:05d}" for i in range(G)], 2)
    X = (rng.poisson(1.0, size=(labels.size, 6)) * (rng.rand(labels.size, 6) < 0.5)).astype(np.float32)
    eng, grpc = _engine(labels)
    M = _device_matrix(X, "csc", np.float32)
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    _lib.profile_report()
    s, c = _call_pass(eng, M, "sums", 0, 6)
    ran = _lib.profile_report()
    assert "sums_csc_global_kernel" in ran and "sums_csc_kernel" not in ran, ran
    codes = grpc.encoded_groups
    want = np.zeros((G, 6))
    np.add.at(want, codes, X.astype(np.float64))
    np.testing.assert_array_equal(s, want)
    _, cn = _call_pass(eng, M, "count", 0, 6)
    np.testing.assert_array_equal(c, cn)


@pytest.mark.gpu
@pytest.mark.parametrize("ref", [None, 2])
def test_log_fold_changes_kernel(ref):
    import torch

    from illico_b200 import _lib

    rng = np.random.RandomState(4)
    G, N = 37, 70
    sizes = rng.randint(2, 50, size=G).astype(np.int32)
    S = rng.randint(0, 200, size=(G, N)).astype(np.float64)
    S[:, 0] = 0.0                                              # mean 0 everywhere
    S[3, 1] = 0.0                                              # mean 0 in one group
    n_cells = int(sizes.sum())
    for log_scale in (1.0, float(np.log(2.0))):
        out = torch.full((G, N + 5), np.nan, dtype=torch.float64, device="cuda")
        d = torch.from_numpy(S).cuda()
        gs = torch.from_numpy(sizes).cuda()
        _lib.check(_lib.load().illico_log_fold_changes(d.data_ptr(), N, gs.data_ptr(), G, N, -1 if ref is None else ref, n_cells,
                                                       log_scale, out.data_ptr(), N + 5, torch.cuda.current_stream().cuda_stream),
                   "illico_log_fold_changes")
        got = out[:, :N].cpu().numpy()
        mg = S / sizes[:, None]
        mr = np.broadcast_to(S[ref] / sizes[ref], S.shape) if ref is not None else (S.sum(0) - S) / (n_cells - sizes)[:, None]
        want = np.log2((np.expm1(mg * log_scale) + 1e-9) / (np.expm1(mr * log_scale) + 1e-9))
        np.testing.assert_allclose(got, want, rtol=1e-14, atol=1e-13)
        assert (got[:, 0] == 0).all()


@pytest.mark.gpu
def test_bonferroni_kernel():
    import torch

    from illico_b200 import _lib

    rng = np.random.RandomState(5)
    G, N = 9, 333
    res = rng.rand(G, N, 3) ** 4
    res[0, 3, 0] = np.nan
    res[1, :, 0] = 0.0
    res[2, 5, 0] = 1.0 / N
    d = torch.from_numpy(res).cuda()
    out = torch.empty((G, N), dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().illico_bonferroni_adjust(d.data_ptr(), 3 * N, 3, G, N, out.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "illico_bonferroni_adjust")
    got = out.cpu().numpy()
    np.testing.assert_array_equal(got, np.minimum(res[:, :, 0] * N, 1.0))
    assert np.isnan(got[0, 3])


@pytest.mark.gpu
@pytest.mark.parametrize("by_abs", [0, 1])
def test_top_genes_columns_agrees_with_top_genes(by_abs):
    import torch

    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(6)
    G, N = 11, 600
    scores = np.round(rng.randn(G, N), 1)                       # many ties
    scores[0, :5] = np.nan
    scores[1, 7] = -0.0
    res = rng.rand(G, N, 3)
    lfc = rng.randn(G, N)
    padj = rng.rand(G, N)
    rows = np.array([4, 0, 9, 1], dtype=np.int32)
    st = torch.cuda.current_stream().cuda_stream
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in
         dict(scores=scores, res=res, lfc=lfc, padj=padj, rows=rows).items()}
    for k in (1, 17, N):
        ws = torch.empty(int(lib.illico_top_genes_workspace_bytes(G, N)), dtype=torch.uint8, device="cuda")
        gene = torch.empty((G, k), dtype=torch.int32, device="cuda")
        rec = torch.empty((G, k, 5), dtype=torch.float64, device="cuda")
        _lib.check(lib.illico_top_genes(d["scores"].data_ptr(), N, d["res"].data_ptr(), 3 * N, d["padj"].data_ptr(), G, N, k, by_abs,
                                        gene.data_ptr(), rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "illico_top_genes")
        C = rows.size
        cg = torch.empty((k, C), dtype=torch.int32, device="cuda")
        cs, cl = (torch.empty((k, C), dtype=torch.float32, device="cuda") for _ in range(2))
        cp, cq = (torch.empty((k, C), dtype=torch.float64, device="cuda") for _ in range(2))
        _lib.check(lib.illico_top_genes_columns(d["scores"].data_ptr(), N, d["res"].data_ptr(), 3 * N, d["padj"].data_ptr(),
                                                d["lfc"].data_ptr(), N, G, N, d["rows"].data_ptr(), C, k, by_abs, cg.data_ptr(),
                                                cs.data_ptr(), cl.data_ptr(), cp.data_ptr(), cq.data_ptr(), ws.data_ptr(), ws.numel(),
                                                st), "illico_top_genes_columns")
        gene, rec = gene.cpu().numpy(), rec.cpu().numpy()
        cg, cs, cl, cp, cq = (t.cpu().numpy() for t in (cg, cs, cl, cp, cq))
        for c, g in enumerate(rows):
            np.testing.assert_array_equal(cg[:, c], gene[g])
            np.testing.assert_array_equal(cs[:, c], rec[g, :, 0].astype(np.float32))
            np.testing.assert_array_equal(cp[:, c], rec[g, :, 1])
            np.testing.assert_array_equal(cq[:, c], rec[g, :, 4])
            np.testing.assert_array_equal(cl[:, c], lfc[g, gene[g]].astype(np.float32))
