"""``rank_genes_groups``: a drop-in for scanpy 1.10's ``sc.tl.rank_genes_groups``, computed on the GPU.

The result goes where scanpy puts it, ``adata.uns[key_added]``, in scanpy's layout (record arrays of length ``n_genes`` with
one field per group), so ``sc.get.rank_genes_groups_df``, ``sc.pl.rank_genes_groups*`` and
``sc.tl.filter_rank_genes_groups`` read it as they read scanpy's own.  The tests are those of ``asymptotic_wilcoxon`` /
``ttest`` with scanpy's settings (no continuity correction, two-sided); scanpy's log fold change comes from the group means
(``illico_group_sums_*`` or the t-test's moments, then ``illico_log_fold_changes``); the adjustment (``illico_bh_adjust`` /
``illico_bonferroni_adjust``) and the per-group selection in scanpy's column layout (``illico_top_genes_columns``) run on the
device, so only the ``n_genes`` records of each group cross PCIe.
"""
from __future__ import annotations

from typing import Literal

import numpy as np
import pandas as pd
import torch

from . import _lib
from .asymptotic_wilcoxon import _run_tests, check_flag, nonzero_fractions
from .ranking import _bh_on_device

__all__ = ["rank_genes_groups"]

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
    uns = getattr(adata, "uns", {})
    base = uns.get("log1p", {}).get("base") if "log1p" in uns else None
    log_scale = float(np.log(base)) if base is not None else 1.0
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

