"""Group encoding and the device "plan" derived from it.

``encode_and_count_groups`` mirrors the reference (``illico/utils/groups.py:18-58``): same
``GroupContainer`` fields, same lexicographic group order (``np.unique``), same ``ValueError``
when the reference label is absent, ``encoded_ref_group == -1`` for one-versus-rest.  The
reference's per-label Python dict loop (0.33 s at 300k cells) is replaced by a vectorised
factorisation; the result is identical.

``build_plan`` turns a GroupContainer into the tables the CUDA kernels read
(``illico_plan_t`` in ``include/illico_b200.h``): cells permuted to group-contiguous order and every
group cut into segments of at most ``seg_max`` cells.
"""
from __future__ import annotations

from collections import namedtuple
from typing import Any

import os

import numpy as np

GroupContainer = namedtuple(
    "GroupContainer",
    ["encoded_groups", "counts", "indices", "indptr", "encoded_ref_group"],
)

SEG_MAX_DEFAULT = 512
# Longest segment a plan may have: the kernels count a segment's cells in 16-bit counters (the staging kernels' count
# tiles, the one-versus-rest table bins, the fused CSR pass's control histogram).
SEG_MAX_LIMIT = 65535
SEG_MAX_ENV = "ILLICO_B200_SEG_MAX"
# Slots start on, and are padded to, a multiple of this many floats (a multiple of 8 = one 32-byte sector).  32 floats
# = one 128-byte line: a typical slot (~15 non-zeros of a ~150-cell group) then lies in ONE line / 64-byte fetch
# granule instead of straddling two (measured: staging 2.10 -> 2.01 ms at the K562 shape).
SLOT_ALIGN = max(8, int(os.environ.get("ILLICO_B200_SLOT_ALIGN", "32")) // 8 * 8)


def _factorize_sorted(groups):
    """``(unique_sorted, inverse)`` with ``np.unique``'s ordering.  Strings go through a hash-based
    factorisation (12 ms instead of 170 ms at 300k labels); the sorted uniques are the same."""
    import pandas as pd

    if isinstance(groups, (pd.Series, pd.Index)) and isinstance(groups.dtype, pd.CategoricalDtype):
        # AnnData keeps obs columns categorical: the codes are already there (1 ms instead of 20 ms at 300k cells);
        # only the categories in use count, in np.unique's (sorted) order
        cat = groups.cat if isinstance(groups, pd.Series) else groups
        codes = np.asarray(cat.codes)
        if (codes < 0).any():
            raise ValueError("group labels contain missing values")
        cats = np.asarray(cat.categories)
        used = np.flatnonzero(np.bincount(codes, minlength=len(cats)) > 0)
        uniq = cats[used]
        if uniq.dtype == object and all(isinstance(x, str) for x in uniq):
            uniq = uniq.astype(str)
        order = np.argsort(uniq, kind="stable")
        remap = np.full(len(cats), -1, dtype=np.int64)
        remap[used[order]] = np.arange(used.size)
        return uniq[order], remap[codes]
    if isinstance(groups, (pd.Series, pd.Index)):
        arr = groups.to_numpy()
    else:
        arr = np.asarray(groups)
    if arr.ndim != 1:
        raise ValueError("group labels must be one-dimensional")
    if arr.dtype.kind in "OUS":
        codes, uniq = pd.factorize(arr, sort=True)
        if (codes < 0).any():
            raise ValueError("group labels contain missing values")
        uniq = np.asarray(uniq)
        if uniq.dtype == object and all(isinstance(x, str) for x in uniq):
            uniq = uniq.astype(str)  # what np.unique returns for a list of str
        return uniq, codes
    uniq, inverse = np.unique(arr, return_inverse=True)
    return uniq, inverse.reshape(-1)


def encode_and_count_groups(groups, ref_group: Any):
    """Returns ``(unique_groups, GroupContainer)`` exactly like the reference."""
    unique_groups, inverse = _factorize_sorted(groups)
    if ref_group is not None:
        hit = np.nonzero(unique_groups == ref_group)[0]
        if hit.size == 0:
            raise ValueError(f"Reference group `{ref_group}` is not present in the group labels.")
        encoded_ref = int(hit[0])
    else:
        encoded_ref = -1
    return unique_groups, _container(inverse, len(unique_groups), encoded_ref)


def _container(codes, G: int, encoded_ref: int) -> GroupContainer:
    encoded = np.ascontiguousarray(codes, dtype=np.int64)
    counts = np.bincount(encoded, minlength=G).astype(np.int64)
    small = encoded.astype(np.int16) if G < 2**15 else encoded  # 16-bit keys take numpy's radix sort
    indices = np.argsort(small, kind="stable").astype(np.int64)
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return GroupContainer(encoded, counts, indices, indptr, encoded_ref)


# ---- groups= : the groups a call tests ----------------------------------------------------------------------------------
# Cells of a one-versus-rest pseudo-group (the cells of the groups not tested, collapsed): below the fused path's 65 536-cell
# group limit (DESIGN.md section 2.2), so that collapsing them never moves a batch off that path.
PSEUDO_GROUP_MAX = 65535


def select_groups(unique_groups, groups, encoded_ref: int):
    """Indices into ``unique_groups`` (ascending: ``np.unique`` order) of the groups ``groups`` asks for, the reference group
    added when it is missing; None when that is every group.  ``groups``: None or ``"all"`` (every group), one label
    (a ``str``) or an iterable of labels, duplicates collapsed.  An unknown label or an empty selection is a ``ValueError``."""
    import pandas as pd

    if groups is None or (isinstance(groups, str) and groups == "all"):
        return None
    labels = [groups] if isinstance(groups, str) else list(groups)
    if not labels:
        raise ValueError("groups selects no group: pass None or 'all' for every group, or at least one label")
    hit = pd.Index(unique_groups).get_indexer(pd.Index(labels, dtype=object))
    if (hit < 0).any():
        missing = [lab for lab, h in zip(labels, hit) if h < 0]
        raise ValueError(f"groups: {missing} not found in the group labels")
    sel = np.unique(np.concatenate([hit, [encoded_ref]]) if encoded_ref >= 0 else hit)
    return None if sel.size == len(unique_groups) else sel.astype(np.int64)


def subset_for_reference(grpc: GroupContainer, sel: np.ndarray):
    """One-versus-reference on the selected groups ``sel``: ``(rows, GroupContainer)`` -- the rows of their cells, ascending,
    and the container of the matrix made of those rows (groups renumbered ``0 .. sel.size - 1`` in the same order, the
    reference among them).  Every selected group keeps its cells in their order, so the plan gives it the segments of the
    full call."""
    remap = np.full(grpc.counts.size, -1, dtype=np.int64)
    remap[sel] = np.arange(sel.size)
    codes = remap[grpc.encoded_groups]
    rows = np.flatnonzero(codes >= 0)
    return rows, _container(codes[rows], sel.size, int(remap[grpc.encoded_ref_group]))


def collapse_unselected(grpc: GroupContainer, sel: np.ndarray) -> GroupContainer:
    """One-versus-rest on the selected groups ``sel``: every cell stays (the rest of a group is every other cell).  The
    selected groups become groups ``0 .. sel.size - 1``; the other cells, in ascending row order, are cut into
    ``ceil(n / PSEUDO_GROUP_MAX)`` runs of near-equal size, the pseudo-groups ``sel.size ..``, whose rows of every output are
    dropped."""
    remap = np.full(grpc.counts.size, -1, dtype=np.int64)
    remap[sel] = np.arange(sel.size)
    codes = remap[grpc.encoded_groups]
    rest = np.flatnonzero(codes < 0)
    P = -(-rest.size // PSEUDO_GROUP_MAX)
    codes[rest] = sel.size + np.arange(rest.size, dtype=np.int64) * P // rest.size
    return _container(codes, sel.size + P, -1)


def _is_stable_group_order(enc, perm) -> bool:
    e = enc[perm]
    if np.any(np.diff(e) < 0):
        return False
    same = np.diff(e) == 0
    return bool(np.all(np.diff(perm)[same] > 0))


def check_seg_max(seg_max) -> int:
    """``seg_max`` as an int, or a ``ValueError`` naming ``ILLICO_B200_SEG_MAX`` unless it is an integer in
    ``[1, SEG_MAX_LIMIT]``."""
    if isinstance(seg_max, (bool, np.bool_)) or not isinstance(seg_max, (int, np.integer)):
        raise ValueError(f"{SEG_MAX_ENV} (plan segment length) must be an integer, got {seg_max!r}")
    if not 1 <= seg_max <= SEG_MAX_LIMIT:
        raise ValueError(f"{SEG_MAX_ENV} (plan segment length) must be in [1, {SEG_MAX_LIMIT}], got {seg_max}")
    return int(seg_max)


def seg_max_from_env() -> int:
    """The plan segment length: ``ILLICO_B200_SEG_MAX`` if set, else 512.  An invalid value is an error."""
    raw = os.environ.get(SEG_MAX_ENV)
    if raw is None:
        return SEG_MAX_DEFAULT
    try:
        value = int(raw.strip())
    except ValueError:
        raise ValueError(f"{SEG_MAX_ENV} (plan segment length) must be an integer, got {raw!r}") from None
    return check_seg_max(value)


class HostPlan:
    """numpy form of ``illico_plan_t``.  ``seg_max`` (default: :func:`seg_max_from_env`) must lie in
    ``[1, SEG_MAX_LIMIT]``."""

    def __init__(self, grpc: GroupContainer, seg_max: int | None = None):
        seg_max = seg_max_from_env() if seg_max is None else check_seg_max(seg_max)
        enc = np.asarray(grpc.encoded_groups, dtype=np.int64)
        counts = np.asarray(grpc.counts, dtype=np.int64)
        n, G = enc.size, counts.size
        if n >= 2**31 - 1:
            raise ValueError("more than 2^31 cells are not supported")
        if G == 0 or n == 0:
            raise ValueError("empty input")
        if counts.sum() != n or counts.min() < 1:
            raise ValueError("inconsistent GroupContainer")
        self.n_cells, self.n_groups = int(n), int(G)
        self.ref_group = int(grpc.encoded_ref_group)
        self.seg_max = int(seg_max)
        perm = np.asarray(grpc.indices)  # stable argsort of the codes: ascending cell index inside a group
        if perm.size != n or not _is_stable_group_order(enc, perm):
            small = enc.astype(np.int16) if G < 2**15 else enc
            perm = np.argsort(small, kind="stable")
        group_off = np.concatenate([[0], np.cumsum(counts)])
        nseg = np.maximum(1, -(-counts // seg_max))
        group_seg = np.concatenate([[0], np.cumsum(nseg)])
        S = int(group_seg[-1])
        seg_group = np.repeat(np.arange(G), nseg)
        k = np.arange(S) - group_seg[seg_group]
        seg_start = group_off[seg_group] + k * seg_max
        seg_len = np.minimum(seg_max, counts[seg_group] - k * seg_max)
        seg_pos = np.concatenate([seg_start, [n]])
        al = SLOT_ALIGN  # slots start on (and are padded to) whole sectors / fetch granules
        seg_base = np.concatenate([[0], np.cumsum((seg_len + al - 1) // al * al)])
        if seg_base[-1] >= 2**31 - 1:
            raise ValueError("slot space exceeds 2^31")
        pos_seg = np.repeat(np.arange(S), seg_len)  # segment of each position
        cell_seg = np.empty(n, dtype=np.int64)
        cell_seg[perm] = pos_seg
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)  # noqa: E731
        self.n_segments = S
        self.max_group_size = int(counts.max())
        self.ref_group_size = int(counts[self.ref_group]) if self.ref_group >= 0 else 0
        others = np.delete(counts, self.ref_group) if self.ref_group >= 0 else counts
        self.max_target_group_size = int(others.max()) if others.size else 0
        self.slot_cap = int(seg_base[-1])
        self.ref_seg_begin = int(group_seg[self.ref_group]) if self.ref_group >= 0 else 0
        self.ref_seg_end = int(group_seg[self.ref_group + 1]) if self.ref_group >= 0 else 0
        self.perm, self.cell_seg = i32(perm), i32(cell_seg)
        self.seg_pos, self.seg_base, self.seg_group = i32(seg_pos), i32(seg_base), i32(seg_group)
        self.group_seg, self.group_size = i32(group_seg), i32(counts)

    TABLES = ("perm", "cell_seg", "seg_pos", "seg_base", "seg_group", "group_seg", "group_size")


def build_plan(grpc: GroupContainer, seg_max: int | None = None) -> HostPlan:
    return HostPlan(grpc, seg_max)
