"""``rank_genes``: for each group, its genes ranked strongest first, with adjusted p-values (what
``scanpy.tl.rank_genes_groups`` reports), selected on the device.

The tests run exactly as in ``asymptotic_wilcoxon`` (same upload, plan, shards and backed streaming), with the score plane
on, but the results stay on the GPU: Benjamini-Hochberg (``illico_bh_adjust``) and the per-group sort
(``illico_top_genes``) run there, and only the ``G x n_genes`` selected records cross PCIe.  With ``pts`` or a marker
filter, the cells expressing each gene are counted on the GPU too (``illico_count_nonzero_*``, ``illico_nonzero_fractions``)
and scanpy's ``filter_rank_genes_groups`` criteria are applied there, before the selection
(``illico_top_genes_filtered``).
"""
from __future__ import annotations

import math
from typing import Literal

import numpy as np
import pandas as pd
import torch

from . import _lib
from .asymptotic_wilcoxon import _run_tests, check_flag, nonzero_fractions
from .engine import check_method

__all__ = ["rank_genes"]

COLUMNS = ["feature", "score", "p_value", "p_adj", "statistic", "fold_change", "log2_fold_change"]
PTS_COLUMNS = ["pct_nz_group", "pct_nz_reference"]


def _bound(name: str, value, upper: float | None):
    """A filter threshold: None (not given), or a real number in [0, upper] (NaN and bools refused)."""
    if value is None:
        return None
    if isinstance(value, (bool, np.bool_)) or not isinstance(value, (int, float, np.integer, np.floating)) \
            or not (value >= 0 and (upper is None or value <= upper)):
        raise ValueError(f"{name} must be a real number in [0, {upper if upper is not None else 'inf'}] or None, got {value!r}")
    return float(value)


def rank_genes(
    adata,
    is_log1p: bool,
    group_keys: str,
    reference: str | None = None,
    n_genes: int | None = 100,
    rankby_abs: bool = False,
    n_threads: int = 1,
    batch_size: int | Literal["auto"] = "auto",
    alternative: str = "two-sided",
    use_continuity: bool = True,
    tie_correct: bool = True,
    layer: str | None = None,
    device=None,
    devices=None,
    pts: bool = False,
    min_in_group_fraction: float | None = None,
    max_out_group_fraction: float | None = None,
    min_fold_change: float | None = None,
    method: str = "wilcoxon",
    groups=None,
    mask_var=None,
) -> pd.DataFrame:
    """The ``n_genes`` strongest genes of every group, by Wilcoxon score (or Welch's t with ``method="t-test"``).

    The tests are those of ``asymptotic_wilcoxon`` (same arguments, same checks and errors).  Each group's genes are
    sorted by ``score`` descending -- the signed z of the normal approximation, ``(n_r n_t / 2 - U) / sigma``, positive
    when the group ranks above the reference / rest -- or by ``|score|`` with ``rankby_abs``; equal scores keep the gene
    order of ``var_names`` and NaN scores come last.  ``n_genes=None`` ranks every gene; larger values are clipped to the
    number of genes.

    Returns a ``pd.DataFrame`` indexed by ``MultiIndex (pert, rank)`` (groups in ``np.unique`` order, the reference group
    left out, ``rank = 0 .. n_genes - 1``) with columns ``feature`` (categorical over ``var_names`` when they are
    unique), ``score``, ``p_value``, ``p_adj`` (Benjamini-Hochberg
    over all genes of the group, not only the ones shown), ``statistic`` (U), ``fold_change`` and ``log2_fold_change``.

    ``pts`` adds the columns ``pct_nz_group`` (fraction of the group's cells with a non-zero value) and ``pct_nz_reference``
    (the same in the reference group, or in all other cells for one-versus-rest), as ``scanpy.tl.rank_genes_groups(pts=True)``.
    ``min_in_group_fraction`` / ``max_out_group_fraction`` / ``min_fold_change`` keep only the genes with
    ``pct_nz_group >= min_in_group_fraction``, ``pct_nz_reference <= max_out_group_fraction`` and
    ``fold_change >= min_fold_change`` (with ``rankby_abs``: or ``fold_change <= 1 / min_fold_change``), each criterion
    only when given, a NaN failing it (scanpy's ``filter_rank_genes_groups`` defaults are 0.25, 0.5 and 1).  The filter
    runs before the selection: a group has ``min(n_genes, genes kept)`` rows (none when nothing is kept) and ``p_adj``
    stays over all of its genes.  A filter implies ``pts``.

    ``method`` is scanpy's: ``"wilcoxon"`` (the default), ``"t-test"`` or ``"t-test_overestim_var"`` (Welch's t-test, as
    ``illico_b200.ttest``).  For a t-test ``score`` and ``statistic`` are t (``score`` with NaN replaced by 0, the p-value
    NaN replaced by 1), the fold change is the Wilcoxon call's, and ``use_continuity`` / ``tie_correct`` are ignored.

    ``groups`` is scanpy's (see ``asymptotic_wilcoxon``): only the selected groups are tested and shown, each with the rows
    it has in the same call without ``groups``.

    ``mask_var`` is scanpy's (see ``asymptotic_wilcoxon``): only the selected genes are tested and ranked -- ``n_genes`` is
    clipped to their number, ``feature`` is categorical over their names, and ``p_adj`` is over the selected genes of each
    group.
    """
    check_method(method)
    if n_genes is not None:
        if isinstance(n_genes, bool) or not isinstance(n_genes, (int, np.integer)):
            raise ValueError(f"n_genes must be a positive integer or None, got {n_genes!r}")
        if n_genes <= 0:
            raise ValueError(f"n_genes must be a positive integer or None, got {n_genes}")
    check_flag("pts", pts)
    min_in = _bound("min_in_group_fraction", min_in_group_fraction, 1.0)
    max_out = _bound("max_out_group_fraction", max_out_group_fraction, 1.0)
    fc_min = _bound("min_fold_change", min_fold_change, None)
    with_pts = bool(pts) or any(v is not None for v in (min_in, max_out, fc_min))
    run = _run_tests(adata, is_log1p, group_keys, reference, n_threads, batch_size, alternative, use_continuity,
                     tie_correct, layer, device, devices, score=True, on_device=True, pts=with_pts, method=method, groups=groups,
                     mask_var=mask_var)
    res, scores = run.results, run.scores
    G, N = int(res.shape[0]), int(res.shape[1])
    k = N if n_genes is None else min(int(n_genes), N)
    var_names = np.asarray(run.var_names)
    keep = np.arange(G)
    if reference is not None:
        keep = keep[keep != run.grpc.encoded_ref_group]
    width = 7 if with_pts else 5
    rows = np.full(G, k)                                   # rows shown per group
    if N == 0 or keep.size == 0:
        gene, rec = np.zeros((G, 0), np.int32), np.zeros((G, 0, width))
        k, rows[:] = 0, 0
    elif with_pts:
        pct = tuple(p[:G] for p in nonzero_fractions(run.nnz, run.grpc))     # (one-versus-rest pseudo-groups dropped)
        fc_max = (1.0 / fc_min if fc_min > 0 else math.inf) if rankby_abs and fc_min is not None else None
        gene, rec, kept = top_genes_filtered(res, scores, pct, k, rankby_abs, min_in, max_out, fc_min, fc_max)
        rows = np.minimum(rows, kept)
    else:
        gene, rec = top_genes(res, scores, k, rankby_abs)
    rows = rows[keep]
    shown = np.arange(k)[None, :] < rows[:, None]
    gene, rec = gene[keep][shown], rec[keep][shown]
    # index and feature column from codes: building them from G k strings would cost more than the ranking itself
    starts = np.cumsum(rows) - rows
    index = pd.MultiIndex(levels=[pd.Index(np.asarray(run.groups)[keep]), pd.RangeIndex(k)],
                          codes=[np.repeat(np.arange(keep.size), rows), np.arange(gene.size) - np.repeat(starts, rows)],
                          names=["pert", "rank"], verify_integrity=False)
    names = pd.Index(var_names)
    feature = pd.Categorical.from_codes(gene, categories=names) if names.is_unique else var_names[gene]
    with np.errstate(divide="ignore", invalid="ignore"):
        log2fc = np.log2(rec[:, 3])
    cols = {"feature": feature, "score": rec[:, 0], "p_value": rec[:, 1], "p_adj": rec[:, 4], "statistic": rec[:, 2],
            "fold_change": rec[:, 3], "log2_fold_change": log2fc}
    if with_pts:
        cols.update(pct_nz_group=rec[:, 5], pct_nz_reference=rec[:, 6])
    return pd.DataFrame(cols, index=index, columns=COLUMNS + (PTS_COLUMNS if with_pts else []), copy=False)


def top_genes(results: torch.Tensor, scores: torch.Tensor, k: int, by_abs: bool = False):
    """Benjamini-Hochberg over each group's genes, then its first ``k`` genes by score, on the tensors' GPU
    (``illico_bh_adjust`` + ``illico_top_genes``).  ``results``: ``[G, N, 3]``, ``scores``: ``[G, N]`` float64, contiguous,
    same device.  Returns host arrays ``(gene [G, k] int32, record [G, k, 5] float64)``, a record being
    ``(score, p_value, statistic, fold_change, p_adj)``."""
    lib = _lib.load()
    G, N = int(results.shape[0]), int(results.shape[1])
    dev = results.device
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        padj, ws = _bh_on_device(results, scores, k)
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 5), dtype=torch.float64, device=dev)
        _lib.check(lib.illico_top_genes(scores.data_ptr(), N, results.data_ptr(), 3 * N, padj.data_ptr(), G, N, k, int(bool(by_abs)),
                                        gene.data_ptr(), rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "illico_top_genes")
        return gene.cpu().numpy(), rec.cpu().numpy()


def _bh_on_device(results: torch.Tensor, scores: torch.Tensor, k: int):
    """``(p_adj [G, N], workspace)``: Benjamini-Hochberg over each group's genes, enqueued on the current stream, and a
    workspace large enough for the selection that follows."""
    lib = _lib.load()
    G, N = int(results.shape[0]), int(results.shape[1])
    dev = results.device
    assert results.dtype == scores.dtype == torch.float64 and results.is_contiguous() and scores.is_contiguous()
    assert tuple(scores.shape) == (G, N) and scores.device == dev and 1 <= k <= N
    st = torch.cuda.current_stream(dev).cuda_stream
    padj = torch.empty((G, N), dtype=torch.float64, device=dev)
    ws = torch.empty(int(max(lib.illico_bh_workspace_bytes(G, N), lib.illico_top_genes_workspace_bytes(G, N))),
                     dtype=torch.uint8, device=dev)
    _lib.check(lib.illico_bh_adjust(results.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), ws.data_ptr(), ws.numel(), st),
               "illico_bh_adjust")
    return padj, ws


def top_genes_filtered(results: torch.Tensor, scores: torch.Tensor, pct, k: int, by_abs: bool = False, min_in=None,
                       max_out=None, fc_min=None, fc_max=None):
    """``top_genes`` with the expressing-cell fractions ``pct = (pct_group, pct_ref)`` (``[G, N]`` float64 on the same
    device) in the record and the marker filter applied first (``illico_top_genes_filtered``; a bound of None is not
    given).  Returns host arrays ``(gene [G, k] int32, record [G, k, 7] float64, kept [G] int32)``, a record being
    ``(score, p_value, statistic, fold_change, p_adj, pct_group, pct_ref)``; row g holds ``min(k, kept[g])`` genes, then
    gene -1 and NaN records."""
    lib = _lib.load()
    G, N = int(results.shape[0]), int(results.shape[1])
    dev = results.device
    pg, pr = pct
    assert pg.dtype == pr.dtype == torch.float64 and pg.is_contiguous() and pr.is_contiguous()
    assert tuple(pg.shape) == tuple(pr.shape) == (G, N) and pg.device == pr.device == dev
    nan = lambda v: math.nan if v is None else float(v)  # noqa: E731
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        padj, ws = _bh_on_device(results, scores, k)
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 7), dtype=torch.float64, device=dev)
        kept = torch.empty(G, dtype=torch.int32, device=dev)
        _lib.check(lib.illico_top_genes_filtered(scores.data_ptr(), N, results.data_ptr(), 3 * N, padj.data_ptr(), pg.data_ptr(),
                                                 pr.data_ptr(), G, N, k, int(bool(by_abs)), nan(min_in), nan(max_out), nan(fc_min),
                                                 nan(fc_max), gene.data_ptr(), rec.data_ptr(), kept.data_ptr(), ws.data_ptr(),
                                                 ws.numel(), st), "illico_top_genes_filtered")
        return gene.cpu().numpy(), rec.cpu().numpy(), kept.cpu().numpy()
