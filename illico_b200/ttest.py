"""``ttest``: Welch's t-test for every (group, gene) on the GPU -- scanpy's ``rank_genes_groups(method="t-test")`` and
``method="t-test_overestim_var"`` -- in ``asymptotic_wilcoxon``'s result layout.

The matrix is read once per gene batch for the per-(group, gene) cell count, sum and sum of squares
(``illico_group_moments_*``, csrc/counts.cu); the means, variances, Welch's t, its degrees of freedom and the Student t
p-value follow in a float64 epilogue (``illico_welch_ttest``, csrc/ttest.cu).  No ranks, no sort, no recoding of float64
values.  Upload, group plan, gene shards over ``devices``, backed streaming and the CSR repartition are those of
``asymptotic_wilcoxon``.
"""
from __future__ import annotations

from typing import Literal

import numpy as np

from .asymptotic_wilcoxon import _bh_adjust, _host_fractions, _result_frame, _run_tests, check_flag
from .engine import WILCOXON, check_method

__all__ = ["ttest"]


def ttest(
    adata,
    group_keys: str,
    reference: str | None = None,
    *,
    method: str = "t-test",
    is_log1p: bool = False,
    alternative: str = "two-sided",
    n_threads: int = 1,
    batch_size: int | Literal["auto"] = "auto",
    layer: str | None = None,
    device=None,
    devices=None,
    return_array: bool = False,
    p_adjust: bool = False,
    log2_fold_change: bool = False,
    score: bool = False,
    pts: bool = False,
    groups=None,
    mask_var=None,
):
    """Welch's t-test of every group against ``reference`` (or, when it is None, against all other cells) in every gene.

    ``method`` is ``"t-test"`` or ``"t-test_overestim_var"`` (scanpy's hack for small groups: the comparison sample's
    variance is divided by the group's size instead of its own).  Per group and gene, with ``n`` cells:
    ``mean = sum x / n``, ``var = (sum x^2 / n - mean^2) * n / (n - 1)`` (unless ``n == 1``), accumulated in float64 (scanpy
    1.10's ``_get_mean_var``, one pass), then ``scipy.stats.ttest_ind_from_stats(..., equal_var=False, alternative)``.

    Returns the ``(pert, feature)`` DataFrame of ``asymptotic_wilcoxon`` with ``p_value`` (NaN replaced by 1, as scanpy
    does), ``statistic`` (Welch's t as computed: NaN when both samples are constant and equal, +-inf when both are constant
    and differ) and ``fold_change`` (the Wilcoxon call's expression: mean of the group over mean of the comparison sample,
    of ``expm1(x)`` when ``is_log1p``; ``inf`` where the comparison mean is 0).  The reference group's rows are
    ``(1, 0, fold change of the control with itself)``.  ``is_log1p`` affects only the fold change.
    ``score`` adds t with NaN replaced by 0 (scanpy's ``scores``); ``p_adjust``, ``log2_fold_change``, ``pts``,
    ``return_array``, ``device``, ``devices``, ``n_threads``, ``batch_size``, ``layer``, ``groups`` and ``mask_var`` are
    those of ``asymptotic_wilcoxon``.
    """
    if check_method(method) == WILCOXON:
        raise ValueError("ttest runs the t-tests; method='wilcoxon' is asymptotic_wilcoxon")
    check_flag("pts", pts)
    run = _run_tests(adata, is_log1p, group_keys, reference, n_threads, batch_size, alternative, True, True, layer, device,
                     devices, score=score, on_device=False, pts=pts, method=method, groups=groups,
                     mask_var=mask_var)
    out = run.results
    extra = {}
    if p_adjust:
        extra["p_adj"] = _bh_adjust(out, run.device)
    if log2_fold_change:
        with np.errstate(divide="ignore", invalid="ignore"):
            extra["log2_fold_change"] = np.log2(out[:, :, 2])
    if score:
        extra["score"] = run.scores
    if pts:
        extra["pct_nz_group"], extra["pct_nz_reference"] = _host_fractions(run)
    if return_array:
        if extra:
            return run.groups, np.asarray(run.var_names), out, extra
        return run.groups, np.asarray(run.var_names), out
    return _result_frame(run.groups, run.var_names, out, extra)
