"""``rank_genes``: for each group, its genes ranked strongest first, with adjusted p-values (what
``scanpy.tl.rank_genes_groups`` reports), selected on the device.

The tests run exactly as in ``asymptotic_wilcoxon`` (same upload, plan, shards and backed streaming), with the score plane
on, but the results stay on the GPU: Benjamini-Hochberg (``illico_bh_adjust``) and the per-group sort
(``illico_top_genes``) run there, and only the ``G x n_genes`` selected records cross PCIe.
"""
from __future__ import annotations

from typing import Literal

import numpy as np
import pandas as pd
import torch

from . import _lib
from .asymptotic_wilcoxon import _run_tests

__all__ = ["rank_genes"]

COLUMNS = ["feature", "score", "p_value", "p_adj", "statistic", "fold_change", "log2_fold_change"]


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
) -> pd.DataFrame:
    """The ``n_genes`` strongest genes of every group, by Wilcoxon score.

    The tests are those of ``asymptotic_wilcoxon`` (same arguments, same checks and errors).  Each group's genes are
    sorted by ``score`` descending -- the signed z of the normal approximation, ``(n_r n_t / 2 - U) / sigma``, positive
    when the group ranks above the reference / rest -- or by ``|score|`` with ``rankby_abs``; equal scores keep the gene
    order of ``var_names`` and NaN scores come last.  ``n_genes=None`` ranks every gene; larger values are clipped to the
    number of genes.

    Returns a ``pd.DataFrame`` indexed by ``MultiIndex (pert, rank)`` (groups in ``np.unique`` order, the reference group
    left out, ``rank = 0 .. n_genes - 1``) with columns ``feature`` (categorical over ``var_names`` when they are
    unique), ``score``, ``p_value``, ``p_adj`` (Benjamini-Hochberg
    over all genes of the group, not only the ones shown), ``statistic`` (U), ``fold_change`` and ``log2_fold_change``.
    """
    if n_genes is not None:
        if isinstance(n_genes, bool) or not isinstance(n_genes, (int, np.integer)):
            raise ValueError(f"n_genes must be a positive integer or None, got {n_genes!r}")
        if n_genes <= 0:
            raise ValueError(f"n_genes must be a positive integer or None, got {n_genes}")
    run = _run_tests(adata, is_log1p, group_keys, reference, n_threads, batch_size, alternative, use_continuity,
                     tie_correct, layer, device, devices, score=True, on_device=True)
    res, scores = run.results, run.scores
    G, N = int(res.shape[0]), int(res.shape[1])
    k = N if n_genes is None else min(int(n_genes), N)
    var_names = np.asarray(adata.var_names)
    keep = np.arange(G)
    if reference is not None:
        keep = keep[keep != run.grpc.encoded_ref_group]
    if N == 0 or keep.size == 0:
        gene, rec = np.zeros((G, 0), np.int32), np.zeros((G, 0, 5))
        k = 0
    else:
        gene, rec = top_genes(res, scores, k, rankby_abs)
    gene, rec = gene[keep].reshape(-1), rec[keep].reshape(-1, 5)
    # index and feature column from codes: building them from G k strings would cost more than the ranking itself
    index = pd.MultiIndex(levels=[pd.Index(np.asarray(run.groups)[keep]), pd.RangeIndex(k)],
                          codes=[np.repeat(np.arange(keep.size), k), np.tile(np.arange(k), keep.size)], names=["pert", "rank"],
                          verify_integrity=False)
    names = pd.Index(var_names)
    feature = pd.Categorical.from_codes(gene, categories=names) if names.is_unique else var_names[gene]
    with np.errstate(divide="ignore", invalid="ignore"):
        log2fc = np.log2(rec[:, 3])
    return pd.DataFrame({"feature": feature, "score": rec[:, 0], "p_value": rec[:, 1], "p_adj": rec[:, 4],
                         "statistic": rec[:, 2], "fold_change": rec[:, 3], "log2_fold_change": log2fc}, index=index,
                        columns=COLUMNS, copy=False)


def top_genes(results: torch.Tensor, scores: torch.Tensor, k: int, by_abs: bool = False):
    """Benjamini-Hochberg over each group's genes, then its first ``k`` genes by score, on the tensors' GPU
    (``illico_bh_adjust`` + ``illico_top_genes``).  ``results``: ``[G, N, 3]``, ``scores``: ``[G, N]`` float64, contiguous,
    same device.  Returns host arrays ``(gene [G, k] int32, record [G, k, 5] float64)``, a record being
    ``(score, p_value, statistic, fold_change, p_adj)``."""
    lib = _lib.load()
    G, N = int(results.shape[0]), int(results.shape[1])
    dev = results.device
    assert results.dtype == scores.dtype == torch.float64 and results.is_contiguous() and scores.is_contiguous()
    assert tuple(scores.shape) == (G, N) and scores.device == dev and 1 <= k <= N
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        padj = torch.empty((G, N), dtype=torch.float64, device=dev)
        ws = torch.empty(int(max(lib.illico_bh_workspace_bytes(G, N), lib.illico_top_genes_workspace_bytes(G, N))),
                         dtype=torch.uint8, device=dev)
        _lib.check(lib.illico_bh_adjust(results.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), ws.data_ptr(), ws.numel(), st),
                   "illico_bh_adjust")
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 5), dtype=torch.float64, device=dev)
        _lib.check(lib.illico_top_genes(scores.data_ptr(), N, results.data_ptr(), 3 * N, padj.data_ptr(), G, N, k, int(bool(by_abs)),
                                        gene.data_ptr(), rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "illico_top_genes")
        return gene.cpu().numpy(), rec.cpu().numpy()
