"""``filter_rank_genes_groups``: scanpy's marker filter over a stored ``rank_genes_groups`` result, the run mode without tests
that gives it fractions and fold changes (``_run_tests(stats_only=True)``), and its kernel ``illico_filter_marker_pairs``.

The oracle is a numpy / pandas restatement of scanpy 1.10's ``filter_rank_genes_groups``: fractions and fold changes from
``uns`` when the result is one-versus-rest on the same ``groupby`` and ``use_raw``, otherwise from ``X`` with each group's
out-group taken as its own cells (every other cell), the fold change in float64; strict comparisons, NaN failing each."""
import os
import subprocess

import numpy as np
import pandas as pd
import pytest
from scipy import sparse

from tests.test_rank_genes_groups import ROOT, AnnData, Raw, _no_cuda, data

KEY, FILTERED = "rank_genes_groups", "rank_genes_groups_filtered"


# ---- the oracle: scanpy 1.10 filter_rank_genes_groups ----------------------------------------------------------------------

def dense64(X):
    if hasattr(X, "toarray"):
        X = X.toarray()
    elif hasattr(X, "cpu"):
        X = X.cpu().numpy()
    return np.asarray(X, dtype=np.float64)


def oracle_quantities(ad, key=None, groupby=None, use_raw=None, X=None):
    """(names DataFrame, in, out, fc) with in / out / fc ``[k, C]``: float64, or the stored float32 ``logfoldchanges``.
    ``X``: the matrix to read in place of ``adata.X`` / ``adata.raw.X`` (the same values held in RAM, for backed input)."""
    st = ad.uns[key or KEY]
    params = st["params"]
    groupby = params["groupby"] if groupby is None else groupby
    use_raw = params["use_raw"] if use_raw is None else use_raw
    same = params["groupby"] == groupby and params["reference"] == "rest" and params["use_raw"] == use_raw
    use_lfc, use_frac = same and "logfoldchanges" in st, same and "pts_rest" in st
    names = pd.DataFrame(st["names"])
    k, C = names.shape
    fin, fout, fc = (np.full((k, C), np.nan) for _ in range(3))
    if use_lfc:
        fc = np.column_stack([np.asarray(st["logfoldchanges"][f]) for f in names.columns]).astype(np.float32)
    if not (use_lfc and use_frac):
        src = ad.raw if use_raw else ad
        X = src.X if X is None else X
        pos = {g: i for i, g in enumerate(src.var_names)}
        labels = np.asarray([str(x) for x in ad.obs[groupby]])
        base = ad.uns.get("log1p", {}).get("base")
        f = (lambda x: np.expm1(x * np.log(base))) if base is not None else np.expm1
    for c, cluster in enumerate(names.columns):
        genes = names[cluster]
        ok = genes.notna().to_numpy()
        if use_frac:
            fin[ok, c] = st["pts"][cluster].loc[genes[ok]].to_numpy()
            fout[ok, c] = st["pts_rest"][cluster].loc[genes[ok]].to_numpy()
        if use_lfc and use_frac:
            continue
        Xg = dense64(X[:, [pos[g] for g in genes[ok]]])
        inside = labels == cluster
        X_in, X_out = Xg[inside], Xg[~inside]
        with np.errstate(all="ignore"):
            if not use_frac:
                fin[ok, c] = (X_in != 0).sum(0) / X_in.shape[0]
                fout[ok, c] = (X_out != 0).sum(0) / X_out.shape[0]
            if not use_lfc:
                fc[ok, c] = np.log2((f(X_in.mean(0)) + 1e-9) / (f(X_out.mean(0)) + 1e-9))
    return names, fin, fout, fc


def oracle_keep(ad, key=None, groupby=None, use_raw=None, min_in_group_fraction=0.25, min_fold_change=1,
                max_out_group_fraction=0.5, compare_abs=False, X=None):
    names, fin, fout, fc = oracle_quantities(ad, key, groupby, use_raw, X)
    if compare_abs:
        fc = np.abs(fc)
    with np.errstate(invalid="ignore"):
        keep = (fin > min_in_group_fraction) & (fout < max_out_group_fraction) & (fc > min_fold_change)
    return keep & names.notna().to_numpy()


def names_where(names, keep):
    return pd.DataFrame(names).where(keep).to_records(index=False)


def assert_names_equal(got, want):
    assert isinstance(got, np.recarray)
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    for f in want.dtype.names:
        a, b = list(got[f]), list(want[f])
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert (x == y) or (pd.isna(x) and pd.isna(y) and isinstance(x, float)), (f, x, y)


def run_filter(ad, Xo=None, **kw):
    """``filter_rank_genes_groups`` against the oracle's keep mask (the oracle reading ``Xo`` when given); returns the mask."""
    from illico_b200 import filter_rank_genes_groups

    key, key_added = kw.get("key") or KEY, kw.get("key_added", FILTERED)
    fkw = {k: v for k, v in kw.items() if k not in ("device", "devices", "n_threads", "batch_size")}
    keep = oracle_keep(ad, **{k: v for k, v in fkw.items() if k != "key_added"}, X=Xo)
    stored = ad.uns[key]
    assert filter_rank_genes_groups(ad, **kw) is None
    out = ad.uns[key_added]
    want = names_where(stored["names"], keep)
    assert_names_equal(out["names"], want)
    assert set(out) == set(stored) and all(out[k] is stored[k] for k in stored if k != "names")
    return keep


# ---- CPU -------------------------------------------------------------------------------------------------------------------

def test_new_function_is_bound_and_declared(tmp_path):
    from illico_b200 import _lib

    assert "illico_filter_marker_pairs" in _lib.SIGNATURES
    src = tmp_path / "decl.c"
    src.write_text(
        '#include "illico_b200.h"\n'
        "int (*a)(const int32_t*, const int32_t*, int32_t, int32_t, int64_t, const void*, int32_t, const void*, int32_t,"
        " const void*, int32_t, double, double, double, int32_t, uint8_t*, void*) = illico_filter_marker_pairs;\n"
        "int main(void) { return !a || ILLICO_ABI_VERSION != 3 || ILLICO_PAIRS_PLANE != 0 || ILLICO_PAIRS_F64 != 1"
        " || ILLICO_PAIRS_F32 != 2; }\n")
    subprocess.check_call(["gcc", "-std=c11", "-Werror=incompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c",
                           str(src), "-o", str(tmp_path / "decl.o")])
    assert (_lib.PAIRS_PLANE, _lib.PAIRS_F64, _lib.PAIRS_F32) == (0, 1, 2)


def test_new_kernel_does_not_spill(tmp_path):
    import shutil

    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from illico_b200.build import NVCC_FLAGS

    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    res = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(ROOT, "illico_b200", "csrc", "extras.cu"), "-o",
                                           str(tmp_path / "extras.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    seen, current = False, None
    for line in res.stderr.splitlines():
        if "Function properties for" in line:
            current = line.split("for", 1)[1].strip()
        elif "spill" in line and current and "filter_marker_pairs_kernel" in current:
            seen = True
            assert " 0 bytes spill stores, 0 bytes spill loads" in line, (current, line)
    assert seen


def ranked(n_cells=300, n_genes=12, k=4, labels=None, reference="rest", pts=True, categories=None, raw=None, obs_extra=None):
    """An AnnData with a small stored result of scanpy's layout, written by hand (no device)."""
    X, lab = data(n_cells=n_cells, n_genes=n_genes)
    lab = lab if labels is None else labels
    ad = AnnData(X, lab, categories=categories, raw=raw)
    for col, vals in (obs_extra or {}).items():
        ad.obs[col] = vals
    groups = [g for g in (categories or sorted(set(map(str, lab)))) if g != reference]
    rng = np.random.RandomState(1)
    var = list(ad.var_names if raw is None else raw.var_names)
    names = pd.DataFrame({g: rng.choice(var, size=k, replace=False) for g in groups}).to_records(index=False)
    lfc = pd.DataFrame({g: rng.randn(k) for g in groups}).to_records(index=False, column_dtypes="float32")
    st = {"params": dict(groupby="pert", reference=reference, method="wilcoxon", use_raw=raw is not None, layer=None,
                         corr_method="benjamini-hochberg"), "names": names, "logfoldchanges": lfc}
    if pts:
        st["pts"] = pd.DataFrame(rng.rand(len(var), len(groups)), index=var, columns=groups)
        if reference == "rest":
            st["pts_rest"] = pd.DataFrame(rng.rand(len(var), len(groups)), index=var, columns=groups)
    ad.uns[KEY] = st
    return ad


def _bad(case):
    if case == "key":
        return ranked(), dict(key="nope"), KeyError
    if case == "groupby":
        return ranked(), dict(groupby="nope"), KeyError
    if case.startswith("bound"):
        v = {"bound_bool": True, "bound_str": "0.3", "bound_none": None}[case]
        return ranked(), dict(min_fold_change=v), ValueError
    if case == "compare_abs":
        return ranked(), dict(compare_abs=1), ValueError
    if case == "use_raw":
        return ranked(), dict(use_raw=True), ValueError
    if case == "dup_names":
        ad = ranked()
        ad.var_names = pd.Index(["a"] * 2 + list(ad.var_names[2:]))
        ad.uns[KEY]["names"] = pd.DataFrame({f: ["a"] * 4 for f in ad.uns[KEY]["names"].dtype.names}).to_records(index=False)
        return ad, {}, ValueError
    if case == "dup_raw_names":
        X, _ = data(n_cells=300, n_genes=12)
        ad = ranked(raw=Raw(X, ["r"] * 12))
        return ad, {}, ValueError
    if case == "unknown_field":
        ad = ranked(pts=False)
        ad.uns[KEY]["names"] = pd.DataFrame({"zzz": list(ad.var_names[:4])}).to_records(index=False)
        del ad.uns[KEY]["logfoldchanges"]          # (both quantities then come from X: the field must name a group)
        return ad, {}, ValueError
    if case == "same_str":
        ad = ranked(pts=False)
        n = len(ad.obs)
        ad.obs["mixed"] = [1 if i % 2 else "1" for i in range(n)]
        ad.uns[KEY]["names"] = pd.DataFrame({"1": list(ad.var_names[:4])}).to_records(index=False)
        return ad, dict(groupby="mixed"), ValueError
    if case == "unknown_gene":
        ad = ranked()
        names = ad.uns[KEY]["names"]
        names[names.dtype.names[0]][2] = "not_a_gene"
        return ad, {}, KeyError
    if case == "missing_label":
        ad = ranked(pts=False)
        ad.obs["pert"] = ad.obs["pert"].astype(object)
        ad.obs.loc[3, "pert"] = None
        return ad, {}, ValueError
    raise AssertionError(case)


BAD = ["key", "groupby", "bound_bool", "bound_str", "bound_none", "compare_abs", "use_raw", "dup_names", "dup_raw_names",
       "unknown_field", "same_str", "unknown_gene", "missing_label"]


@pytest.mark.parametrize("case", BAD)
def test_errors_are_raised_before_any_device_work(monkeypatch, case):
    from illico_b200 import filter_rank_genes_groups

    ad, kw, err = _bad(case)
    _no_cuda(monkeypatch)
    with pytest.raises(err) as info:
        filter_rank_genes_groups(ad, **kw)
    if case == "unknown_gene":
        assert "not_a_gene" in str(info.value)
    assert FILTERED not in ad.uns


class _Captured:
    """Stands in for the device: records what the filter hands to the run and to the kernel, and evaluates the criteria on
    the host (a restatement of illico_filter_marker_pairs) so the names assembly can be checked without a GPU."""

    def __init__(self, monkeypatch, planes=None):
        import torch

        from illico_b200 import scanpy_compat

        self.planes = planes or {}
        self.calls = {}

        def run_tests(target, *a, **kw):
            self.calls["run"] = dict(mask_var=kw["mask_var"], pts=kw["pts"], lfc=kw["lfc"], stats_only=kw["stats_only"],
                                     X=target.X)

            class R:
                device = torch.device("cpu")
                nnz, grpc = None, None
                lfc = self.planes.get("fc")
            return R()

        def fractions(nnz, grpc):
            return self.planes["in"], self.planes["out"]

        def filter_pairs(col, rows, sources, planes, stride, min_in, max_out, min_fc, compare_abs, dev):
            self.calls["pairs"] = dict(col=col, rows=rows, sources=sources, planes=planes, stride=stride)
            k, C = col.shape
            vals = {}
            for q in ("in", "out", "fc"):
                if q in planes:
                    p = planes[q].numpy()
                    vals[q] = np.where(col >= 0, p[rows[None, :].repeat(k, 0), np.maximum(col, 0)], np.nan)
                else:
                    vals[q] = sources[q]
            fc = np.abs(vals["fc"]) if compare_abs else vals["fc"]
            with np.errstate(invalid="ignore"):
                b = np.float32(min_fc) if fc.dtype == np.float32 else min_fc
                keep = (vals["in"] > min_in) & (vals["out"] < max_out) & (fc > b) & (col >= 0)
            return keep.astype(np.uint8)

        monkeypatch.setattr(scanpy_compat, "_run_tests", run_tests)
        monkeypatch.setattr(scanpy_compat, "nonzero_fractions", fractions)
        monkeypatch.setattr(scanpy_compat, "_filter_pairs", filter_pairs)
        monkeypatch.setattr(scanpy_compat, "_device_list", lambda device, devices: [torch.device("cpu")])


@pytest.mark.parametrize("column", ["str", "int", "categorical"])
def test_names_union_and_group_rows(monkeypatch, column):
    """Names become gene indices (nan: -1), the union goes to the run as an ascending boolean mask, each field maps to its
    row of the run's np.unique order, and ``names`` is ``DataFrame.where(keep).to_records``."""
    import torch

    from illico_b200 import filter_rank_genes_groups

    n = 60
    codes = np.arange(n) % 3
    if column == "str":
        labels, fields = np.array(["b", "c", "a"])[codes], ["c", "a"]
        rows_want = [2, 0]
    elif column == "int":
        labels, fields = np.array([10, 2, 7])[codes], ["10", "2"]
        rows_want = [2, 0]
    else:
        labels, fields = pd.Categorical(np.array(["b", "c", "a"])[codes], categories=["c", "b", "a"]), ["a", "c"]
        rows_want = [0, 2]
    X = np.zeros((n, 9), np.float32)
    ad = AnnData(X, list(labels))
    if column == "categorical":
        ad.obs["pert"] = labels
    v = list(ad.var_names)
    names = pd.DataFrame({fields[0]: [v[7], v[2], np.nan], fields[1]: [v[2], v[5], v[0]]}).to_records(index=False)
    ad.uns[KEY] = {"params": dict(groupby="pert", reference="p", use_raw=False), "names": names}
    rng = np.random.RandomState(0)
    G = 3
    planes = {q: torch.from_numpy(rng.rand(G, 4)) for q in ("in", "out")}
    planes["fc"] = torch.from_numpy(rng.randn(G, 4) * 2)
    cap = _Captured(monkeypatch, planes)
    filter_rank_genes_groups(ad, min_in_group_fraction=0.2, max_out_group_fraction=0.9, min_fold_change=-0.5)
    run, pairs = cap.calls["run"], cap.calls["pairs"]
    mask = np.zeros(9, bool)
    mask[[0, 2, 5, 7]] = True
    np.testing.assert_array_equal(run["mask_var"], mask)
    assert run["stats_only"] and run["pts"] and run["lfc"] and run["X"] is X
    np.testing.assert_array_equal(pairs["col"], [[3, 1], [1, 2], [-1, 0]])
    np.testing.assert_array_equal(pairs["rows"], rows_want)
    assert pairs["stride"] == 4 and not pairs["sources"]
    keep = filter_pairs_host(pairs["col"], pairs["rows"], planes, 0.2, 0.9, -0.5)
    assert_names_equal(ad.uns[FILTERED]["names"], names_where(names, keep))
    assert ad.uns[KEY]["names"] is names and pd.isna(names[fields[0]][2])


def filter_pairs_host(col, rows, planes, min_in, max_out, min_fc):
    k, C = col.shape
    v = {q: np.where(col >= 0, p.numpy()[np.broadcast_to(rows, (k, C)), np.maximum(col, 0)], np.nan) for q, p in planes.items()}
    with np.errstate(invalid="ignore"):
        return (v["in"] > min_in) & (v["out"] < max_out) & (v["fc"] > min_fc) & (col >= 0)


def test_no_read_branch_takes_every_quantity_from_uns(monkeypatch):
    """rest with pts on the same groupby: no run at all, the pairs come from uns (pts / pts_rest float64 by name, the stored
    float32 logfoldchanges by field), and the names equal the oracle's where()."""
    from illico_b200 import filter_rank_genes_groups

    ad = ranked()
    cap = _Captured(monkeypatch)
    ad.X = None
    filter_rank_genes_groups(ad, min_in_group_fraction=0.3, max_out_group_fraction=0.6, min_fold_change=0.1, compare_abs=True)
    assert "run" not in cap.calls
    src = cap.calls["pairs"]["sources"]
    assert src["fc"].dtype == np.float32 and src["in"].dtype == np.float64 and src["out"].dtype == np.float64
    names, fin, fout, fc = oracle_quantities(ad)
    np.testing.assert_array_equal(src["in"], fin)
    np.testing.assert_array_equal(src["out"], fout)
    np.testing.assert_array_equal(src["fc"], fc)
    keep = oracle_keep(ad, min_in_group_fraction=0.3, max_out_group_fraction=0.6, min_fold_change=0.1, compare_abs=True)
    assert_names_equal(ad.uns[FILTERED]["names"], names_where(ad.uns[KEY]["names"], keep))


def test_public_name_whatever_the_import_order():
    import sys

    code = ("from illico_b200 import filter_rank_genes_groups; import illico_b200 as m; from illico_b200 import rank_genes_groups; "
            "assert callable(filter_rank_genes_groups) and callable(m.rank_genes_groups) and callable(m.asymptotic_wilcoxon)")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


# ---- GPU: against the oracle --------------------------------------------------------------------------------------------

class Untouchable:
    """A matrix that must not be read."""

    shape = property(lambda self: (_ for _ in ()).throw(AssertionError("X was read")))

    def __getattr__(self, name):
        raise AssertionError(f"X was read ({name})")


def ranked_gpu(X=None, labels=None, ad_kw=None, **kw):
    from illico_b200 import rank_genes_groups

    if X is None:
        X, labels = data()
    ad = AnnData(X, labels, **(ad_kw or {}))
    rank_genes_groups(ad, "pert", **{"method": "wilcoxon", "n_genes": 7, **kw})
    return ad


BOUNDS = [dict(), dict(min_in_group_fraction=0.1, max_out_group_fraction=0.9, min_fold_change=0.2),
          dict(min_fold_change=0.5, compare_abs=True), dict(min_in_group_fraction=0, max_out_group_fraction=1, min_fold_change=0),
          dict(min_in_group_fraction=1, max_out_group_fraction=0, min_fold_change=-1e9)]


@pytest.mark.gpu
@pytest.mark.parametrize("branch", ["rest_pts", "rest", "reference", "other_groupby"])
def test_branches(branch):
    X, labels = data()
    kw = dict(rest_pts=dict(pts=True), rest=dict(), reference=dict(reference="non-targeting", pts=True), other_groupby=dict())[branch]
    ad = ranked_gpu(X, labels, n_genes=None if branch == "rest" else 7, **kw)
    fkw = {}
    if branch == "other_groupby":
        ad.obs["coarse"] = [lab if lab in ("p0000", "p0001") else "other" for lab in labels]
        ad.uns[KEY]["names"] = pd.DataFrame({f: ad.uns[KEY]["names"][f] for f in ("p0000", "p0001")}).to_records(index=False)
        fkw["groupby"] = "coarse"
    if branch == "rest_pts":
        ad.X = Untouchable()
    kept = 0
    for b in BOUNDS:
        kept += run_filter(ad, **fkw, **b).sum()
    assert kept > 0


@pytest.mark.gpu
def test_strictness_at_the_bounds():
    """A bound equal to a listed fraction drops that pair (strict), and a bound one float32 ulp either side of a stored float32
    fold change decides it as numpy's float32 comparison does."""
    from illico_b200 import filter_rank_genes_groups

    ad = ranked_gpu(pts=True)
    st = ad.uns[KEY]
    f = st["names"].dtype.names[0]
    gene = st["names"][f][0]
    frac = float(st["pts"][f].loc[gene])
    run_filter(ad, min_in_group_fraction=frac, max_out_group_fraction=2, min_fold_change=-1e9)
    assert pd.isna(ad.uns[FILTERED]["names"][f][0])
    run_filter(ad, min_in_group_fraction=float(np.nextafter(frac, -1)), max_out_group_fraction=2, min_fold_change=-1e9)
    assert ad.uns[FILTERED]["names"][f][0] == gene
    fc32 = st["logfoldchanges"][f][0]
    for bound, kept in ((float(np.nextafter(fc32, np.float32(-np.inf))), True), (float(fc32), False),
                        (float(np.nextafter(fc32, np.float32(np.inf))), False),
                        # halfway-ish below: rounds up to fc32 in float32, so the pair is dropped although bound < fc32
                        (float(fc32) - abs(float(np.spacing(fc32))) / 4, False)):
        filter_rank_genes_groups(ad, min_in_group_fraction=-1, max_out_group_fraction=2, min_fold_change=bound)
        assert (ad.uns[FILTERED]["names"][f][0] == gene) is kept, (bound, fc32)
        run_filter(ad, min_in_group_fraction=-1, max_out_group_fraction=2, min_fold_change=bound)


@pytest.mark.gpu
def test_stored_results():
    """n_genes None / 1 / 7; results ranked with groups=, mask_var=, layer= (the filter reads X); use_raw; a log1p base of 2;
    filtering twice; key and key_added; a result written by the oracle."""
    X, labels = data(n_cells=800, n_genes=30)
    b = BOUNDS[1]
    for n_genes in (None, 1, 7):
        run_filter(ranked_gpu(X, labels, n_genes=n_genes), **b)
        run_filter(ranked_gpu(X, labels, n_genes=n_genes, reference="p0002"), **b)
    run_filter(ranked_gpu(X, labels, groups=["p0003", "p0000"]), **b)
    run_filter(ranked_gpu(X, labels, groups=["p0003", "p0000"], reference="non-targeting"), **b)
    mask = np.zeros(30, bool)
    mask[[1, 2, 5, 6, 7, 20, 29]] = True
    ad = ranked_gpu(X, labels, ad_kw=dict(var=pd.DataFrame({"hv": mask}, index=[f"gene_{i}" for i in range(30)])), mask_var="hv")
    run_filter(ad, **b)
    # layer=: the ranking read the layer, the filter reads X (here different)
    L = (X * 3).astype(np.float32)
    ad = ranked_gpu(X, labels, ad_kw=dict(layers={"L": L}), layer="L", pts=True)
    run_filter(ad, **b)
    # use_raw
    raw_names = [f"r{i}" for i in range(30)]
    ad = ranked_gpu(np.zeros((X.shape[0], 3), np.float32), labels, ad_kw=dict(raw=Raw(X, raw_names)), reference="p0001")
    assert ad.uns[KEY]["params"]["use_raw"] is True
    run_filter(ad, **b)
    # log1p in base 2
    Xl = np.log2(1 + X).astype(np.float32)
    run_filter(ranked_gpu(Xl, labels, ad_kw=dict(uns={"log1p": {"base": 2}}), reference="non-targeting"), **b)
    # twice, with key and key_added
    ad = ranked_gpu(X, labels, key_added="mine", reference="non-targeting")
    run_filter(ad, key="mine", key_added="once", **BOUNDS[2])
    run_filter(ad, key="once", key_added="twice", **b)
    assert "rank_genes_groups" not in ad.uns and FILTERED not in ad.uns
    # a result written by the oracle (scanpy's layout), not by rank_genes_groups
    ad = AnnData(X, labels)
    rng = np.random.RandomState(9)
    groups = sorted(set(labels))
    ad.uns[KEY] = {"params": dict(groupby="pert", reference="non-targeting", method="t-test", use_raw=False, layer=None,
                                  corr_method="benjamini-hochberg"),
                   "names": pd.DataFrame({g: rng.choice(list(ad.var_names), 9, replace=False) for g in groups}).to_records(index=False),
                   "logfoldchanges": pd.DataFrame({g: rng.randn(9) for g in groups}).to_records(index=False, column_dtypes="float32")}
    run_filter(ad, **b)


@pytest.mark.gpu
def test_planes_against_the_oracle():
    """The stats-only run's fractions are the oracle's exactly; its fold changes match to 1e-14 relative (the same float64
    means on integer counts; expm1 / log2 of the device library)."""
    from illico_b200 import scanpy_compat
    from illico_b200.asymptotic_wilcoxon import _run_tests, nonzero_fractions

    X, labels = data(n_cells=1000, n_genes=40)
    ad = AnnData(X, labels)
    mask = np.zeros(40, bool)
    mask[[0, 1, 3, 9, 17, 18, 39]] = True
    for Xin in (X, sparse.csr_matrix(X), sparse.csc_matrix(X)):
        ad.X = Xin
        run = _run_tests(ad, False, "pert", None, 1, "auto", "two-sided", False, False, None, None, None, score=False, on_device=True,
                         pts=True, mask_var=mask, lfc=True, log_scale=scanpy_compat.log1p_scale(ad), stats_only=True)
        assert run.results is None and run.scores is None
        pin, pout = (p.cpu().numpy() for p in nonzero_fractions(run.nnz, run.grpc))
        lfc = run.lfc.cpu().numpy()
        Xs = X[:, mask].astype(np.float64)
        for g, name in enumerate(run.groups):
            inside = labels == name
            np.testing.assert_array_equal(pin[g], (Xs[inside] != 0).sum(0) / inside.sum())
            np.testing.assert_array_equal(pout[g], (Xs[~inside] != 0).sum(0) / (~inside).sum())
            want = np.log2((np.expm1(Xs[inside].mean(0)) + 1e-9) / (np.expm1(Xs[~inside].mean(0)) + 1e-9))
            np.testing.assert_allclose(lfc[g], want, rtol=1e-14, atol=1e-14)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["dense", "csr", "csc", "float64", "cuda", "backed_csc", "all_gpus"])
def test_input_routes(route, tmp_path, monkeypatch):
    import torch

    from illico_b200 import _lib

    X, labels = data(n_cells=1100, n_genes=37)
    ad = ranked_gpu(X, labels, reference="non-targeting")
    kw = {}
    if route == "csr":
        ad.X = sparse.csr_matrix(X)
    elif route == "csc":
        ad.X = sparse.csc_matrix(X)
    elif route == "float64":
        Xo = X.astype(np.float64)
        Xo[5, 9] = 16777217.0                  # float32 cannot hold it: summed as float64, never recoded
        ad.X = Xo
        monkeypatch.setenv("ILLICO_PROFILE", "1")
        _lib.profile_report()
    elif route == "cuda":
        ad.X = torch.from_numpy(X).cuda()
    elif route == "backed_csc":
        from illico_b200.backed import MemmapCSC, save_csc

        C = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), C.data, C.indices, C.indptr, C.shape)
        ad.X = MemmapCSC(str(tmp_path / "csc"))
        kw["batch_size"] = 4
    elif route == "all_gpus":
        kw["devices"] = "all"
    for b in BOUNDS[:3]:
        run_filter(ad, Xo=X if route == "backed_csc" else None, **kw, **b)
    if route == "float64":
        ran = _lib.profile_report()
        assert ran and not any("recode" in name for name in ran), ran


@pytest.mark.gpu
def test_dense_route_moves_only_the_listed_columns(monkeypatch):
    from illico_b200 import hostio

    X, labels = data(n_cells=1200, n_genes=300)
    ad = ranked_gpu(X, labels, reference="non-targeting", n_genes=5)
    listed = {g for f in ad.uns[KEY]["names"].dtype.names for g in ad.uns[KEY]["names"][f]}
    moved = []
    real = hostio.h2d_2d

    def counting(d, view, **kw):
        moved.append(d.numel() * d.element_size())
        return real(d, view, **kw)

    monkeypatch.setattr(hostio, "h2d_2d", counting)
    run_filter(ad, **BOUNDS[1])
    assert len(listed) < 300 and sum(moved) == X.shape[0] * len(listed) * 4, (sum(moved), len(listed))


@pytest.mark.gpu
def test_originals_unchanged():
    """After a filter call, uns[key] and its arrays are as they were, and rank_genes_groups gives the same bits again."""
    import copy

    from illico_b200 import filter_rank_genes_groups, rank_genes_groups

    X, labels = data(n_cells=900, n_genes=33)
    ad = ranked_gpu(X, labels, reference="non-targeting", pts=True)
    before = copy.deepcopy(ad.uns[KEY])
    filter_rank_genes_groups(ad, **BOUNDS[1])
    after = ad.uns[KEY]
    assert set(after) == set(before)
    for k, v in before.items():
        if isinstance(v, pd.DataFrame):
            pd.testing.assert_frame_equal(after[k], v, check_exact=True)
        elif isinstance(v, np.ndarray):
            assert after[k].dtype == v.dtype and all(list(after[k][f]) == list(v[f]) for f in v.dtype.names)
        else:
            assert after[k] == v
    ad2 = AnnData(X, labels)
    rank_genes_groups(ad2, "pert", method="wilcoxon", n_genes=7, reference="non-targeting", pts=True)
    for k in ("scores", "pvals", "pvals_adj", "logfoldchanges"):
        assert ad2.uns[KEY][k].tobytes() == before[k].tobytes()


# ---- GPU: the kernel directly --------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("compare_abs", [0, 1])
def test_filter_marker_pairs_kernel(compare_abs):
    import torch

    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(11)
    G, S, k, C = 13, 50, 17, 9
    special = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 0.25, 0.5, 1.0])

    def salt(a):
        a = a.copy()
        flat = a.reshape(-1)
        hit = rng.rand(flat.size) < 0.15
        flat[hit] = rng.choice(special, hit.sum())
        return a

    plane = {q: salt(rng.rand(G, S) * (4 if q == "fc" else 1) - (2 if q == "fc" else 0)) for q in ("in", "out", "fc")}
    pair = {q: salt(rng.rand(k, C) * (4 if q == "fc" else 1) - (2 if q == "fc" else 0)) for q in ("in", "out", "fc")}
    gene = rng.randint(0, S, size=(k, C)).astype(np.int32)
    gene[rng.rand(k, C) < 0.1] = -1
    rows = rng.randint(0, G, size=C).astype(np.int32)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    d_gene, d_rows = d(gene), d(rows)
    bounds = (0.25, 0.5, 1.0)
    kinds = [(a, b, c) for a in range(3) for b in range(3) for c in range(3)]
    for kind in kinds:
        vals, args, hold = {}, [], []
        for q, kd in zip(("in", "out", "fc"), kind):
            if kd == _lib.PAIRS_PLANE:
                v = np.where(gene >= 0, plane[q][np.broadcast_to(rows, (k, C)), np.maximum(gene, 0)], np.nan)
                t = d(plane[q])
            elif kd == _lib.PAIRS_F64:
                v, t = pair[q], d(pair[q])
            else:
                v = pair[q].astype(np.float32)
                t = d(v)
            hold.append(t)
            vals[q] = v
            args += [t.data_ptr(), kd]
        keep = torch.full((k, C), 7, dtype=torch.uint8, device="cuda")
        _lib.check(lib.illico_filter_marker_pairs(d_gene.data_ptr(), d_rows.data_ptr(), k, C, S, *args, *bounds, compare_abs,
                                                  keep.data_ptr(), torch.cuda.current_stream().cuda_stream), "filter")
        fc = np.abs(vals["fc"]) if compare_abs else vals["fc"]
        with np.errstate(invalid="ignore"):
            want = (vals["in"] > bounds[0]) & (vals["out"] < bounds[1]) & (fc > bounds[2]) & (gene >= 0)
        np.testing.assert_array_equal(keep.cpu().numpy(), want.astype(np.uint8), err_msg=str(kind))
    # no plane source: group_rows may be NULL; a plane source without it is refused
    keep = torch.empty((k, C), dtype=torch.uint8, device="cuda")
    t = d(pair["in"])
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.illico_filter_marker_pairs(d_gene.data_ptr(), None, k, C, 0, t.data_ptr(), 1, t.data_ptr(), 1, t.data_ptr(), 1,
                                              *bounds, 0, keep.data_ptr(), st), "filter")
    assert lib.illico_filter_marker_pairs(d_gene.data_ptr(), None, k, C, S, t.data_ptr(), 0, t.data_ptr(), 1, t.data_ptr(), 1,
                                          *bounds, 0, keep.data_ptr(), st) == 1
