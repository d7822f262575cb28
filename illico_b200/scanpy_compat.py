"""``rank_genes_groups``: a drop-in for scanpy 1.10's ``sc.tl.rank_genes_groups``, computed on the GPU.

The result goes where scanpy puts it, ``adata.uns[key_added]``, in scanpy's layout (record arrays of length ``n_genes`` with
one field per group), so ``sc.get.rank_genes_groups_df``, ``sc.pl.rank_genes_groups*`` and
``sc.tl.filter_rank_genes_groups`` read it as they read scanpy's own.  The tests are those of ``asymptotic_wilcoxon`` /
``ttest`` with scanpy's settings (no continuity correction, two-sided); scanpy's log fold change comes from the group means
(``illico_group_sums_*`` or the t-test's moments, then ``illico_log_fold_changes``); the adjustment (``illico_bh_adjust`` /
``illico_bonferroni_adjust``) and the per-group selection in scanpy's column layout (``illico_top_genes_columns``) run on the
device, so only the ``n_genes`` records of each group cross PCIe.

``filter_rank_genes_groups``: scanpy 1.10's ``sc.tl.filter_rank_genes_groups`` over such a result (ours or scanpy's).
Fractions and fold changes come from ``uns`` when the result is one-versus-rest on the same ``groupby`` and ``use_raw``;
otherwise from one pass over the listed genes' columns of ``X`` (``illico_group_sums_*`` / ``illico_count_nonzero_*``, then
``illico_log_fold_changes`` and ``illico_nonzero_fractions``, one-versus-rest).  The criteria are evaluated on the device
(``illico_filter_marker_pairs``), so only a ``[k, groups]`` keep mask comes back.
"""
from __future__ import annotations

from typing import Literal

import numpy as np
import numpy.lib.recfunctions as rfn
import pandas as pd
import torch

from . import _lib
from .asymptotic_wilcoxon import _device_list, _run_tests, check_flag, nonzero_fractions
from .ranking import _bh_on_device

__all__ = ["filter_rank_genes_groups", "rank_genes_groups"]

METHODS = ("t-test", "t-test_overestim_var", "wilcoxon")
CORR_METHODS = ("benjamini-hochberg", "bonferroni")
KEY = "rank_genes_groups"


class _RawView:
    """What the tests read of ``adata.raw``: its matrix, genes and ``var``, with the object's ``obs``."""

    def __init__(self, adata):
        raw = adata.raw
        self.X, self.var_names, self.var = raw.X, raw.var_names, getattr(raw, "var", None)
        self.obs, self.layers = adata.obs, {}


def resolve_use_raw(adata, use_raw, layer) -> bool:
    """scanpy's ``use_raw``: None means "``adata.raw`` when there is one and no ``layer``"."""
    raw = getattr(adata, "raw", None)
    if use_raw is None:
        return raw is not None and layer is None
    check_flag("use_raw", use_raw)
    if use_raw and layer is not None:
        raise ValueError("Cannot specify `layer` and have `use_raw=True`.")
    if use_raw and raw is None:
        raise ValueError("Received `use_raw=True`, but `adata.raw` is empty.")
    return bool(use_raw)


def group_order(labels, groups, reference) -> list:
    """scanpy's ``groups_order``: the categories of the ``groupby`` column (a non-categorical column: its sorted unique labels,
    what anndata makes of it), or the labels of ``groups`` in the user's order with the reference appended when it is missing.
    Refuses, as scanpy does, ``groups`` given as one label, a ``reference`` that is not a category and any group of the order
    with fewer than 2 cells (empty categories included); an unknown label of ``groups`` is a ``ValueError`` too."""
    col = labels if isinstance(labels.dtype, pd.CategoricalDtype) else pd.Series(pd.Categorical(labels.to_numpy()))
    cats = list(col.cat.categories)
    known = set(cats)
    if isinstance(groups, (str, int, np.integer)) and not (isinstance(groups, str) and groups == "all"):
        raise ValueError("Specify a sequence of groups")
    if reference != "rest" and reference not in known:
        raise ValueError(f"reference = {reference} needs to be one of groupby = {cats}.")
    if isinstance(groups, str):
        order = cats
    else:
        order = list(pd.unique(pd.Series(list(groups), dtype=object)))
        if not order:
            raise ValueError("groups selects no group: pass 'all' or at least one label")
        if isinstance(order[0], (int, np.integer)):
            order = [str(n) for n in order]
        if reference != "rest" and reference not in set(order):
            order.append(reference)
    unknown = [g for g in order if g not in known]
    if unknown:
        raise ValueError(f"groups: {unknown} are not categories of groupby = {cats}")
    sizes = col.value_counts().to_dict()
    small = [g for g in order if sizes.get(g, 0) < 2]
    if small:
        raise ValueError(f"Could not calculate statistics for groups {', '.join(map(str, small))} since they only contain one "
                         "sample.")
    return order


def log1p_scale(adata) -> float:
    """ln of ``adata.uns["log1p"]["base"]``, or 1 when no base is set (scanpy's ``expm1(x · ln base)``)."""
    uns = getattr(adata, "uns", {})
    base = uns.get("log1p", {}).get("base") if "log1p" in uns else None
    return float(np.log(base)) if base is not None else 1.0


def records(planes: np.ndarray, fields: list) -> np.recarray:
    """A C-contiguous ``[k, C]`` array as a length-``k`` record array with one field per column, without a copy."""
    k, C = planes.shape
    dtype = np.dtype([(f, planes.dtype) for f in fields])
    return planes.view(dtype).reshape(k).view(np.recarray)


def name_records(gene: np.ndarray, var_names, fields: list) -> np.recarray:
    """The ``names`` record array: column c of the ``[k, C]`` gene indices as gene names (object fields)."""
    k = gene.shape[0]
    names = np.asarray(var_names, dtype=object)
    out = np.recarray(k, dtype=[(f, object) for f in fields])
    for c, f in enumerate(fields):
        out[f] = names[gene[:, c]]
    return out


def rank_genes_groups(
    adata,
    groupby: str,
    *,
    mask_var=None,
    use_raw: bool | None = None,
    groups="all",
    reference: str = "rest",
    n_genes: int | None = None,
    rankby_abs: bool = False,
    pts: bool = False,
    key_added: str | None = None,
    copy: bool = False,
    method: str | None = None,
    corr_method: str = "benjamini-hochberg",
    tie_correct: bool = False,
    layer: str | None = None,
    device=None,
    devices=None,
    n_threads: int = 1,
    batch_size: int | Literal["auto"] = "auto",
):
    """Ranks the genes of each group as ``scanpy.tl.rank_genes_groups`` (scanpy 1.10) does, and writes scanpy's result to
    ``adata.uns[key_added or "rank_genes_groups"]``.  Returns None, or with ``copy=True`` the ``adata.copy()`` that holds it.

    The result is a dict with ``params`` (``groupby``, ``reference``, ``method``, ``use_raw``, ``layer``, ``corr_method``, as
    resolved) and the record arrays ``names`` (object), ``scores`` (float32), ``pvals``, ``pvals_adj`` (float64) and
    ``logfoldchanges`` (float32), of length ``min(n_genes, genes tested)`` (``n_genes=None``: every gene) with one field
    ``str(group)`` per tested group.  Row ``r`` of a field is the group's ``r``-th gene by score, descending (by ``|score|``
    with ``rankby_abs``; the stored score keeps its sign).  ``pts=True`` adds ``pts``, the fraction of each group's cells
    with a non-zero value (a DataFrame indexed by the tested genes, one column per group, the reference included), and for
    ``reference="rest"`` ``pts_rest``, the same fraction among all other cells.

    Groups follow the categories of ``adata.obs[groupby]`` (a column that is not categorical: its sorted unique labels), or
    the order of ``groups``, the reference appended when it is missing; the record arrays leave the reference out.
    ``method`` is ``"t-test"`` (None, scanpy's default), ``"t-test_overestim_var"`` or ``"wilcoxon"`` (no continuity
    correction, ``tie_correct`` as given; its score is the z of the normal approximation and its p-value
    ``2 * norm.sf(|z|)``); ``"logreg"`` is not provided.  ``corr_method`` is ``"benjamini-hochberg"`` or ``"bonferroni"``
    (``min(p * genes tested, 1)``).  ``logfoldchanges`` is ``log2((expm1(mean_g) + 1e-9) / (expm1(mean_rest) + 1e-9))`` of
    the float64 group means, ``expm1(x * ln(base))`` when ``adata.uns["log1p"]["base"]`` is set.  ``use_raw=None`` reads
    ``adata.raw`` when there is one and no ``layer``; ``mask_var`` then names a column of ``adata.raw.var``.

    Errors are scanpy's, raised before any device work: ``groups`` given as one label, a ``reference`` that is not a
    category, a group of the order with fewer than 2 cells, an unknown ``method`` or ``corr_method``, ``use_raw=True`` with
    a ``layer`` or without ``adata.raw``.  An unknown label in ``groups`` is a ``ValueError`` too.

    Where it differs from scanpy: genes with equal scores are ordered by gene index (scanpy's order among ties is
    ``argpartition``'s, unspecified); ``pts`` counts values ``!= 0``, so a sparse matrix's explicitly stored zeros do not count
    (scanpy counts stored entries); scanpy's warnings (raw counts, groups of 25 cells or fewer) are not given.
    ``device``, ``devices``, ``n_threads`` and ``batch_size`` are those of ``asymptotic_wilcoxon``.
    """
    if method is None:
        method = "t-test"
    if not isinstance(method, str) or method not in METHODS:
        raise ValueError(f"Method must be one of {METHODS}, got {method!r} ('logreg' is not provided).")
    if not isinstance(corr_method, str) or corr_method not in CORR_METHODS:
        raise ValueError(f"corr_method must be one of {CORR_METHODS}, got {corr_method!r}.")
    if n_genes is not None and (isinstance(n_genes, bool) or not isinstance(n_genes, (int, np.integer)) or n_genes <= 0):
        raise ValueError(f"n_genes must be a positive integer or None, got {n_genes!r}")
    for name, flag in (("rankby_abs", rankby_abs), ("pts", pts), ("copy", copy), ("tie_correct", tie_correct)):
        check_flag(name, flag)
    if copy:
        adata = adata.copy()
    use_raw = resolve_use_raw(adata, use_raw, layer)
    order = group_order(adata.obs[groupby], groups, reference)
    log_scale = log1p_scale(adata)
    target = _RawView(adata) if use_raw else adata
    ref = None if reference == "rest" else reference
    run = _run_tests(target, False, groupby, ref, n_threads, batch_size, "two-sided", False, tie_correct, layer, device, devices,
                     score=True, on_device=True, pts=pts, method=method, groups=None if isinstance(groups, str) else order,
                     mask_var=mask_var, lfc=True, log_scale=log_scale)
    rows = pd.Index(np.asarray(run.groups, dtype=object)).get_indexer(pd.Index(order, dtype=object))
    assert (rows >= 0).all()
    tested = [g for g in order if g != ref]
    fields = [str(g) for g in tested]
    test_rows = rows[[i for i, g in enumerate(order) if g != ref]]
    res, scores, lfc = run.results, run.scores, run.lfc
    G, N = int(res.shape[0]), int(res.shape[1])
    k = N if n_genes is None else min(int(n_genes), N)
    gene, planes = top_columns(res, scores, lfc, test_rows, k, rankby_abs, corr_method)
    out = {"params": dict(groupby=groupby, reference=reference, method=method, use_raw=use_raw, layer=layer,
                          corr_method=corr_method)}
    if pts:
        pct_group, pct_rest = (p.cpu().numpy() for p in nonzero_fractions(run.nnz, run.grpc))
        var_index = pd.Index(run.var_names)
        names = [str(g) for g in order]
        out["pts"] = pd.DataFrame(pct_group[rows].T, index=var_index, columns=names)
        if ref is None:
            out["pts_rest"] = pd.DataFrame(pct_rest[rows].T, index=var_index, columns=names)
    out["names"] = name_records(gene, run.var_names, fields)
    for key, plane in planes.items():
        out[key] = records(plane, fields)
    adata.uns[key_added or KEY] = out
    return adata if copy else None


def top_columns(results: torch.Tensor, scores: torch.Tensor, lfc: torch.Tensor, group_rows, k: int, by_abs: bool,
                corr_method: str):
    """The adjustment over each group's genes and the first ``k`` genes of the groups ``group_rows`` (rows of the planes, in
    output order), on the planes' GPU (``illico_bh_adjust`` / ``illico_bonferroni_adjust``, ``illico_top_genes_columns``).
    Returns host arrays: the gene indices ``[k, C]`` int32 and ``{"scores", "pvals", "pvals_adj", "logfoldchanges"}`` ``[k, C]``
    planes, float32 / float64 / float64 / float32."""
    lib = _lib.load()
    G, N = int(results.shape[0]), int(results.shape[1])
    C = len(group_rows)
    dev = results.device
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        if corr_method == "benjamini-hochberg":
            padj, ws = _bh_on_device(results, scores, k)
        else:
            padj = torch.empty((G, N), dtype=torch.float64, device=dev)
            _lib.check(lib.illico_bonferroni_adjust(results.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), st),
                       "illico_bonferroni_adjust")
            ws = None
        need = int(lib.illico_top_genes_workspace_bytes(max(C, 1), N))
        if ws is None or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
        rows = torch.from_numpy(np.ascontiguousarray(group_rows, dtype=np.int32)).to(dev)
        gene = torch.empty((k, C), dtype=torch.int32, device=dev)
        planes = {"scores": torch.empty((k, C), dtype=torch.float32, device=dev),
                  "pvals": torch.empty((k, C), dtype=torch.float64, device=dev),
                  "pvals_adj": torch.empty((k, C), dtype=torch.float64, device=dev),
                  "logfoldchanges": torch.empty((k, C), dtype=torch.float32, device=dev)}
        if C > 0 and k > 0:
            _lib.check(lib.illico_top_genes_columns(scores.data_ptr(), N, results.data_ptr(), 3 * N, padj.data_ptr(), lfc.data_ptr(), N,
                                                    G, N, rows.data_ptr(), C, k, int(bool(by_abs)), gene.data_ptr(),
                                                    planes["scores"].data_ptr(), planes["logfoldchanges"].data_ptr(),
                                                    planes["pvals"].data_ptr(), planes["pvals_adj"].data_ptr(), ws.data_ptr(),
                                                    ws.numel(), st), "illico_top_genes_columns")
        return gene.cpu().numpy(), {key: p.cpu().numpy() for key, p in planes.items()}



FILTER_KEY = "rank_genes_groups_filtered"


def filter_rank_genes_groups(
    adata,
    *,
    key: str | None = None,
    groupby: str | None = None,
    use_raw: bool | None = None,
    key_added: str = FILTER_KEY,
    min_in_group_fraction: float = 0.25,
    min_fold_change: float = 1,
    max_out_group_fraction: float = 0.5,
    compare_abs: bool = False,
    device=None,
    devices=None,
    n_threads: int = 1,
    batch_size: int | Literal["auto"] = "auto",
):
    """Filters the marker genes of a stored ranking as ``scanpy.tl.filter_rank_genes_groups`` (scanpy 1.10) does, and
    writes the result to ``adata.uns[key_added]``.  Returns None.

    ``adata.uns[key]`` (``key=None``: ``"rank_genes_groups"``) is a result in scanpy's layout, written by
    ``rank_genes_groups`` or by scanpy.  ``groupby`` and ``use_raw`` default to its ``params``.  A listed gene of group
    ``cluster`` (a field of ``names``) is kept when its fraction of expressing cells in the group is ``>
    min_in_group_fraction``, that among all other cells is ``< max_out_group_fraction`` and its log fold change (``|lfc|`` with
    ``compare_abs``) is ``> min_fold_change``; NaN fails every criterion.  ``adata.uns[key_added]`` is a shallow copy of
    ``adata.uns[key]`` whose ``names`` has ``nan`` in place of every dropped gene; ``adata.uns[key]`` is left as it is.

    When the result is one-versus-rest (``reference="rest"``) on the same ``groupby`` and ``use_raw``, the fold change is its
    ``logfoldchanges`` (float32, compared in float32) and the fractions its ``pts`` / ``pts_rest``; with both present the
    matrix is not read at all.  Otherwise the missing quantities come from ``X`` (``adata.raw.X`` with ``use_raw``; never a
    layer): one pass over the columns of the listed genes only, one-versus-rest over every cell, giving the fractions
    (``illico_nonzero_fractions``) and ``log2((f(mean_in) + 1e-9) / (f(mean_out) + 1e-9))`` with ``f = expm1(x · ln base)``
    (``adata.uns["log1p"]["base"]``, else ``expm1``) from float64 group sums (``illico_log_fold_changes``).

    Errors, raised before any device work: ``key`` not in ``adata.uns`` or ``groupby`` not in ``adata.obs``
    (``KeyError``); a bound that is not a real number, ``compare_abs`` not a bool, ``use_raw=True`` without ``adata.raw``,
    non-unique gene names (``ValueError``); a listed name not among the genes (``KeyError``).  When ``X`` is read: a field
    that matches no group of ``groupby`` by ``str``, two groups with the same ``str``, or a cell with a missing label
    (``ValueError``).

    Where it differs from scanpy: a recomputed fold change comes from float64 sums (scanpy averages in the matrix's dtype; on
    integer counts both are the same double, otherwise they can differ in the last bits); fractions count values ``!= 0``,
    not a sparse matrix's stored entries; a field is matched to a group by ``str(group)`` (scanpy's ``obs[groupby] ==
    field`` matches nothing in a column that is not of strings and drops the whole group); a missing label is refused; a name
    that is already ``nan`` (a filtered result filtered again) stays ``nan`` (scanpy raises).  scanpy's log message is not
    given.  ``device``, ``devices``, ``n_threads`` and ``batch_size`` are those of ``asymptotic_wilcoxon``.
    """
    key = KEY if key is None else key
    if key not in adata.uns:
        raise KeyError(f"{key!r} is not in adata.uns: run rank_genes_groups first")
    stored = adata.uns[key]
    params = stored["params"]
    groupby = params["groupby"] if groupby is None else groupby
    use_raw = params["use_raw"] if use_raw is None else use_raw
    bounds = {"min_in_group_fraction": min_in_group_fraction, "min_fold_change": min_fold_change,
              "max_out_group_fraction": max_out_group_fraction}
    for name, value in bounds.items():
        if isinstance(value, (bool, np.bool_)) or not isinstance(value, (int, float, np.integer, np.floating)):
            raise ValueError(f"{name} must be a real number, got {value!r}")
    check_flag("compare_abs", compare_abs)
    check_flag("use_raw", use_raw)
    if groupby not in adata.obs:
        raise KeyError(f"groupby = {groupby!r} is not a column of adata.obs")
    if use_raw and getattr(adata, "raw", None) is None:
        raise ValueError("Received `use_raw=True`, but `adata.raw` is empty.")
    var_names = pd.Index(adata.raw.var_names if use_raw else adata.var_names)
    if not var_names.is_unique:
        raise ValueError("filter_rank_genes_groups needs unique gene names")
    same = params.get("groupby") == groupby and params.get("reference") == "rest" and params.get("use_raw") == use_raw
    use_logfolds, use_fraction = same and "logfoldchanges" in stored, same and "pts_rest" in stored

    names = stored["names"]
    fields = list(names.dtype.names)
    k, C = len(names), len(fields)
    plain = np.asarray(names)                       # (field access on a plain structured array, not a recarray)
    listed = np.empty((k, C), dtype=object)
    for c, f in enumerate(fields):
        listed[:, c] = plain[f]
    flat = listed.reshape(-1)
    gene = var_names.get_indexer(pd.Index(flat, dtype=object)).reshape(k, C)
    missing = pd.isna(listed)
    absent = (gene < 0) & ~missing
    if absent.any():
        raise KeyError(f"{listed[absent][0]!r} is not among the genes of {'adata.raw' if use_raw else 'adata'}")

    sources = {}      # quantity -> [k, C] host plane taken from uns (the others come from the device planes)
    if use_fraction:
        for q, frame in (("in", stored["pts"]), ("out", stored["pts_rest"])):
            sources[q] = _pairs_plane(frame, listed, missing, fields)
    if use_logfolds:
        fc = _field_plane(stored["logfoldchanges"], fields)
        sources["fc"] = fc if fc.dtype == np.float32 else fc.astype(np.float64)
    read = not (use_logfolds and use_fraction)
    rows = None
    if read:
        from .groups import _factorize_sorted

        groups, _ = _factorize_sorted(adata.obs[groupby])     # (the run's np.unique order; missing labels are refused)
        strs = [str(g) for g in groups]
        if len(set(strs)) != len(strs):
            raise ValueError(f"groupby = {groupby!r} has two groups with the same str: {strs}")
        row_of = {s: i for i, s in enumerate(strs)}
        missing = [f for f in fields if f not in row_of]
        if missing:
            raise ValueError(f"fields {missing} of {key!r} are not groups of groupby = {groupby!r}")
        rows = np.array([row_of[f] for f in fields], dtype=np.int32)

    dev = _device_list(device, devices)[0]
    keep = np.zeros((k, C), dtype=np.uint8)
    union = np.unique(gene[gene >= 0])
    if k and C and union.size:
        to_col = np.full(len(var_names), -1, dtype=np.int32)
        to_col[union] = np.arange(union.size, dtype=np.int32)
        col = np.where(gene >= 0, to_col[gene], -1).astype(np.int32)     # gene -> column of the run (over U)
        planes = {}
        if read:
            mask = np.zeros(len(var_names), dtype=bool)
            mask[union] = True
            target = _RawView(adata) if use_raw else adata
            run = _run_tests(target, False, groupby, None, n_threads, batch_size, "two-sided", False, False, None, device, devices,
                             score=False, on_device=True, pts=not use_fraction, mask_var=mask, lfc=not use_logfolds,
                             log_scale=log1p_scale(adata), stats_only=True)
            dev = run.device
            if not use_fraction:
                planes["in"], planes["out"] = nonzero_fractions(run.nnz, run.grpc)
            if not use_logfolds:
                planes["fc"] = run.lfc
        keep = _filter_pairs(col, rows, sources, planes, union.size, min_in_group_fraction, max_out_group_fraction,
                             min_fold_change, compare_abs, dev)
    kept = np.where(keep.astype(bool), listed, np.nan)
    out = np.empty(k, dtype=[(f, object) for f in fields])
    for c, f in enumerate(fields):
        out[f] = kept[:, c]
    out = out.view(np.recarray)
    result = stored.copy()
    result["names"] = out
    adata.uns[key_added] = result


def _field_plane(rec: np.ndarray, fields: list) -> np.ndarray:
    """The numeric fields ``fields`` of a record array as the columns of a ``[k, C]`` array (a view where numpy can make
    one: a result's float32 ``logfoldchanges`` in field order)."""
    if not fields:
        return np.empty((len(rec), 0), dtype=np.float32)
    return rfn.structured_to_unstructured(np.asarray(rec)[fields])


def _pairs_plane(frame: pd.DataFrame, listed: np.ndarray, missing: np.ndarray, fields: list) -> np.ndarray:
    """``frame[field].loc[name]`` for every listed (rank, field) pair as a ``[k, C]`` plane (float32 if the frame is, else
    float64); a ``nan`` name gives NaN, a field or name missing from the frame is a ``KeyError``."""
    k, C = listed.shape
    at = frame.index.get_indexer(pd.Index(listed.reshape(-1), dtype=object)).reshape(k, C)
    absent = (at < 0) & ~missing
    if absent.any():
        raise KeyError(f"{listed[absent][0]!r} is not in the index of the stored fractions")
    cols = frame.columns.get_indexer(pd.Index(fields, dtype=object))
    if (cols < 0).any():
        raise KeyError(f"{fields[int(np.argmax(cols < 0))]!r} is not a column of the stored fractions")
    values = frame.to_numpy()
    dtype = np.float32 if values.dtype == np.float32 else np.float64
    out = values[np.maximum(at, 0), cols[None, :]].astype(dtype, copy=False)
    out[at < 0] = np.nan
    return out


def _filter_pairs(col: np.ndarray, rows, sources: dict, planes: dict, stride: int, min_in: float, max_out: float,
                  min_fc: float, compare_abs: bool, dev) -> np.ndarray:
    """``illico_filter_marker_pairs`` on the listed pairs: each quantity from its device plane (``planes``, ``[G, stride]``
    float64) or from its host ``[k, C]`` plane (``sources``).  Returns the host ``keep`` mask ``[k, C]`` uint8."""
    lib = _lib.load()
    k, C = col.shape
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        hold = []

        def arg(q):
            if q in planes:
                p = planes[q]
                assert p.dtype == torch.float64 and p.is_contiguous() and p.shape[1] == stride
                return p.data_ptr(), _lib.PAIRS_PLANE
            t = torch.from_numpy(np.ascontiguousarray(sources[q])).to(dev)
            hold.append(t)
            return t.data_ptr(), _lib.PAIRS_F32 if t.dtype == torch.float32 else _lib.PAIRS_F64

        d_col = torch.from_numpy(np.ascontiguousarray(col)).to(dev)
        d_rows = torch.from_numpy(rows).to(dev) if rows is not None else None
        keep = torch.empty((k, C), dtype=torch.uint8, device=dev)
        (pi, ki), (po, ko), (pf, kf) = arg("in"), arg("out"), arg("fc")
        _lib.check(lib.illico_filter_marker_pairs(d_col.data_ptr(), d_rows.data_ptr() if d_rows is not None else None, k, C, stride,
                                                  pi, ki, po, ko, pf, kf, float(min_in), float(max_out), float(min_fc),
                                                  int(bool(compare_abs)), keep.data_ptr(), st), "illico_filter_marker_pairs")
        return keep.cpu().numpy()
