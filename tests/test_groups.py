"""``groups=`` (scanpy's ``rank_genes_groups(groups=...)``) for ``asymptotic_wilcoxon``, ``ttest`` and ``rank_genes``.

The defining property: every selected group's rows equal its rows in the same call without ``groups``.  One-versus-reference
runs on the rows of the selected groups' cells only (``illico_select_rows_*``, the row-list host pack, the staging threads'
gather); one-versus-rest runs on every cell with the other groups collapsed into pseudo-groups of fewer than 65 536 cells.
The selection kernels are checked against numpy / scipy slicing, and small cases against the CPU oracle and
``scipy.stats.mannwhitneyu``: one-versus-reference on the subset a user would cut by hand, one-versus-rest on the full matrix
(its rest holds the cells of the groups not tested)."""
import numpy as np
import pytest
from scipy import sparse, stats

from tests.util import FakeAnnData

CONTROL = "ctrl"


def labelled_counts(seed, n_cells, n_genes, n_groups, control_share=0.3, density=0.15):
    """Integer counts (every sum exact in any order) and labels: a control group of ``control_share`` of the cells, the rest
    spread over ``n_groups`` perturbations of uneven size."""
    rng = np.random.RandomState(seed)
    X = (rng.poisson(2.0, (n_cells, n_genes)) * (rng.rand(n_cells, n_genes) < density)).astype(np.float32)
    names = np.array([f"p{k:03d}" for k in range(n_groups)])
    w = rng.rand(n_groups) + 0.2
    labels = rng.choice(names, size=n_cells, p=w / w.sum()).astype(object)
    labels[rng.rand(n_cells) < control_share] = CONTROL
    X[:, 0] = 0.0                                                    # an all-zero gene
    X[labels == names[1], 1] += 5.0                                  # a marker
    return X, labels.astype(str)


# ---- CPU: selection, containers, plan, pseudo-groups, host pack -------------------------------------------------------------

def test_select_groups_validation():
    from illico_b200.groups import select_groups

    uniq = np.array(["a", "b", "c", "ctrl"])
    assert select_groups(uniq, None, 3) is None
    assert select_groups(uniq, "all", 3) is None
    np.testing.assert_array_equal(select_groups(uniq, "b", 3), [1, 3])            # one str = one label; reference added
    np.testing.assert_array_equal(select_groups(uniq, ["c", "a", "c"], -1), [0, 2])  # duplicates collapsed, np.unique order
    np.testing.assert_array_equal(select_groups(uniq, ("ctrl", "a"), 3), [0, 3])
    assert select_groups(uniq, ["a", "b", "c"], 3) is None                          # every group: the call without groups
    with pytest.raises(ValueError, match="'zz'"):
        select_groups(uniq, ["a", "zz"], 3)
    with pytest.raises(ValueError, match="no group"):
        select_groups(uniq, [], 3)
    with pytest.raises(ValueError, match="no group"):
        select_groups(uniq, np.array([], dtype=str), -1)
    np.testing.assert_array_equal(select_groups(np.array([1, 5, 9]), [9], -1), [2])  # non-string labels


def test_bad_groups_fail_before_device_work():
    """The selection is refused while the labels are encoded, before a device is looked for (so it runs without a GPU too)."""
    from illico_b200 import asymptotic_wilcoxon, rank_genes, ttest

    X, labels = labelled_counts(0, 200, 8, 4)
    ad = FakeAnnData(X, labels)
    for call in (lambda g: asymptotic_wilcoxon(ad, False, "pert", CONTROL, groups=g),
                 lambda g: ttest(ad, "pert", None, groups=g), lambda g: rank_genes(ad, False, "pert", None, groups=g)):
        with pytest.raises(ValueError, match="nope"):
            call(["p001", "nope"])
        with pytest.raises(ValueError, match="no group"):
            call([])


def test_subset_container_and_plan_keep_every_group_s_segments():
    from illico_b200.groups import HostPlan, encode_and_count_groups, select_groups, subset_for_reference

    _, labels = labelled_counts(1, 5000, 2, 30)
    uniq, grpc = encode_and_count_groups(labels, CONTROL)
    sel = select_groups(uniq, ["p003", "p017", "p004"], grpc.encoded_ref_group)
    rows, sub = subset_for_reference(grpc, sel)
    assert np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(sub.counts, grpc.counts[sel])
    assert uniq[sel][sub.encoded_ref_group] == CONTROL
    np.testing.assert_array_equal(uniq[sel][sub.encoded_groups], labels[rows])
    for seg_max in (512, 37):
        full, part = HostPlan(grpc, seg_max), HostPlan(sub, seg_max)
        for k, g in enumerate(sel):
            fs = range(full.group_seg[g], full.group_seg[g + 1])
            ps = range(part.group_seg[k], part.group_seg[k + 1])
            assert len(fs) == len(ps)
            for a, b in zip(fs, ps):        # the same cells, in the same order, segment by segment
                cells_full = full.perm[full.seg_pos[a]:full.seg_pos[a + 1]]
                cells_part = rows[part.perm[part.seg_pos[b]:part.seg_pos[b + 1]]]
                np.testing.assert_array_equal(cells_full, cells_part)
        assert part.ref_group_size == full.ref_group_size


def test_one_versus_rest_pseudo_groups_stay_below_the_fused_limit():
    from illico_b200.groups import PSEUDO_GROUP_MAX, HostPlan, collapse_unselected, encode_and_count_groups, select_groups

    rng = np.random.RandomState(2)
    n = 200_000
    labels = np.where(rng.rand(n) < 0.5, "big", rng.choice(["a", "b", "c", "d"], size=n))   # "big": 100k cells
    uniq, grpc = encode_and_count_groups(labels, None)
    sel = select_groups(uniq, ["b", "d"], -1)
    col = collapse_unselected(grpc, sel)
    S = sel.size
    assert col.encoded_ref_group == -1 and col.counts.sum() == n
    np.testing.assert_array_equal(col.counts[:S], grpc.counts[sel])
    for k, g in enumerate(sel):
        np.testing.assert_array_equal(np.flatnonzero(col.encoded_groups == k), np.flatnonzero(grpc.encoded_groups == g))
    pseudo = col.counts[S:]
    unselected = n - grpc.counts[sel].sum()
    assert unselected > 65536 and pseudo.sum() == unselected
    assert pseudo.size == -(-unselected // PSEUDO_GROUP_MAX) and pseudo.max() < 65536 and pseudo.min() >= 1
    HostPlan(col)          # a valid plan


def test_host_row_list_pack_matches_contiguous_pack():
    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(3)
    n, N, b = 300, 173, 141                       # a column shard (row stride N) of b columns; b not a multiple of 32
    X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) < 0.2)).astype(np.float32)
    X[4, 5], X[9, 6] = -0.0, np.nan
    rows = np.ascontiguousarray(np.sort(rng.choice(n, 77, replace=False)), dtype=np.int64)
    W = (b + 31) // 32

    def pack(fn, *args, nr):
        mask = np.zeros((nr, W), np.uint32)
        off = np.zeros(nr + 1, np.uint32)
        vals = np.zeros(nr * b + 16, np.float32)
        cnt = fn(*args, nr, b, mask.ctypes.data, off.ctypes.data, vals.ctypes.data, vals.size)
        return cnt, mask, off, vals[:max(cnt, 0)]

    shard = X[:, 10:10 + b]
    got = pack(lib.illico_host_pack_row_list_f32, shard.ctypes.data, N, rows.ctypes.data, nr=rows.size)
    contiguous = np.ascontiguousarray(shard[rows])
    want = pack(lib.illico_host_pack_rows_f32, contiguous.ctypes.data, b, nr=rows.size)
    assert got[0] == want[0] > 0
    for g, w in zip(got[1:], want[1:]):
        np.testing.assert_array_equal(g.view(np.uint32), w.view(np.uint32))
    mask, off, vals = np.zeros((rows.size, W), np.uint32), np.zeros(rows.size + 1, np.uint32), np.zeros(b, np.float32)
    assert lib.illico_host_pack_row_list_f32(shard.ctypes.data, N, rows.ctypes.data, rows.size, b, mask.ctypes.data,
                                                              off.ctypes.data, vals.ctypes.data, b) == -1   # does not fit


# ---- GPU: the selection kernels ------------------------------------------------------------------------------------------

def _dev_select(kind, M, rows_np, dtype):
    """Calls the C entry points directly and returns host arrays."""
    import torch

    from illico_b200 import _lib

    lib = _lib.load()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    code = _lib.DTYPE_F32 if dtype == np.float32 else _lib.DTYPE_F64
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    rows = torch.from_numpy(rows_np.astype(np.int32)).to(dev)
    n_sel = rows_np.size
    if kind == "dense":
        X, n_cols = M
        src = torch.from_numpy(X).to(dev)
        out_ld = (n_cols + 3) & ~3
        out = torch.full((max(n_sel, 1), out_ld), 7.0, dtype=tdt, device=dev)
        _lib.check(lib.illico_select_rows_dense(src.data_ptr(), code, X.shape[1], n_cols, rows.data_ptr(), n_sel, out.data_ptr(),
                                                out_ld, st), "select dense")
        return out.cpu().numpy()[:n_sel]
    A = M
    data = torch.from_numpy(A.data.astype(dtype)).to(dev)
    idx = torch.from_numpy(A.indices.astype(np.int32)).to(dev)
    ptr = torch.from_numpy(A.indptr.astype(np.int64)).to(dev)
    if kind == "csr":
        n_out = n_sel
        indptr = torch.empty(n_out + 1, dtype=torch.int64, device=dev)
        _lib.check(lib.illico_select_rows_csr_indptr(ptr.data_ptr(), rows.data_ptr(), n_sel, indptr.data_ptr(), st), "csr indptr")
    else:
        n_out = A.shape[1]
        new_row = np.full(A.shape[0], -1, np.int32)
        new_row[rows_np] = np.arange(n_sel)
        nr = torch.from_numpy(new_row).to(dev)
        indptr = torch.empty(n_out + 1, dtype=torch.int64, device=dev)
        _lib.check(lib.illico_select_rows_csc_indptr(idx.data_ptr(), ptr.data_ptr(), n_out, nr.data_ptr(), indptr.data_ptr(), st),
                   "csc indptr")
    nnz = int(indptr[-1].item())
    od = torch.full((max(nnz, 1),), 7.0, dtype=tdt, device=dev)
    oi = torch.full((max(nnz, 1),), -7, dtype=torch.int32, device=dev)
    if kind == "csr":
        _lib.check(lib.illico_select_rows_csr(data.data_ptr(), code, idx.data_ptr(), ptr.data_ptr(), rows.data_ptr(), n_sel,
                                              indptr.data_ptr(), od.data_ptr(), oi.data_ptr(), st), "csr copy")
    else:
        _lib.check(lib.illico_select_rows_csc(data.data_ptr(), code, idx.data_ptr(), ptr.data_ptr(), n_out, nr.data_ptr(),
                                              indptr.data_ptr(), od.data_ptr(), oi.data_ptr(), st), "csc compact")
    return indptr.cpu().numpy(), od.cpu().numpy()[:nnz], oi.cpu().numpy()[:nnz]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("which", ["some", "one", "all"])
def test_selection_kernels_match_numpy_and_scipy(dtype, which):
    rng = np.random.RandomState(5)
    n, N = 3000, 1500
    X = (rng.rand(n, N) < 0.05) * rng.standard_normal((n, N))
    X[rng.rand(n) < 0.2] = 0.0                                     # empty rows
    X[:, rng.rand(N) < 0.3] *= (rng.rand(n, 1) < 0.02)              # columns with few entries
    X = X.astype(dtype)
    rows = {"some": np.sort(rng.choice(n, 1234, replace=False)), "one": np.array([n - 1]), "all": np.arange(n)}[which]
    # dense: a source of ld = N read for its first 1029 columns (output padded to 1032, the padding zeroed)
    got = _dev_select("dense", (X, 1029), rows, dtype)
    np.testing.assert_array_equal(got[:, :1029], X[rows, :1029])
    assert got.shape[1] == 1032 and not got[:, 1029:].any()
    Xr = sparse.csr_matrix(X)
    ptr, d, i = _dev_select("csr", Xr, rows, dtype)
    want = Xr[rows]
    assert (np.diff(Xr.indptr)[rows] == 0).any() or which != "some"
    np.testing.assert_array_equal(ptr, want.indptr)
    np.testing.assert_array_equal(i, want.indices)
    np.testing.assert_array_equal(d, want.data)
    Xc = sparse.csc_matrix(X)
    ptr, d, i = _dev_select("csc", Xc, rows, dtype)
    want = sparse.csc_matrix(Xc[rows])                                 # scipy keeps each column's rows ascending
    want.sort_indices()
    np.testing.assert_array_equal(ptr, want.indptr)
    np.testing.assert_array_equal(i, want.indices)
    np.testing.assert_array_equal(d, want.data)
    if which != "all":
        assert (np.diff(want.indptr) == 0).sum() > (np.diff(Xc.indptr) == 0).sum()      # columns that lost every entry


@pytest.mark.gpu
def test_row_list_upload_packed_and_staged(monkeypatch):
    """hostio.h2d_2d with a row list: the packed upload (illico_host_pack_row_list_f32) and the staging threads' gather
    deliver exactly X[rows], and only those rows cross PCIe."""
    import torch

    from illico_b200 import hostio

    monkeypatch.setenv("ILLICO_STAGE_CHUNK_MB", "4")
    monkeypatch.setattr(hostio, "CHUNK_BYTES", 4 << 20)
    rng = np.random.RandomState(6)
    n, N = 10000, 2117
    X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) < 0.12)).astype(np.float32)
    rows = np.sort(rng.choice(n, 8600, replace=False)).astype(np.int64)
    dev = torch.device("cuda", 0)
    for mode in ("1", "0"):
        monkeypatch.setenv("ILLICO_PACK_UPLOAD", mode)
        hostio.LAST_UPLOAD.clear()
        dst = torch.full((rows.size, N), 7.0, dtype=torch.float32, device=dev)
        hostio.h2d_2d(dst, X, rows=rows).finish()
        torch.cuda.synchronize()
        np.testing.assert_array_equal(dst.cpu().numpy(), X[rows])
        if mode == "1":
            st = hostio.LAST_UPLOAD
            assert st["raw"] == 0 and st["packed"] == -(-rows.size // ((4 << 20) // (N * 4)))
            assert st["bytes"] < 0.35 * rows.size * N * 4


# ---- GPU: the equivalence property ---------------------------------------------------------------------------------------

ROUTES = ["dense_pinned", "dense_pageable", "dense_packed", "cuda_tensor", "csr", "csc", "backed_csc", "backed_dense", "float64"]
METHODS = ["wilcoxon", "t-test", "t-test_overestim_var"]


def _route_input(route, X, monkeypatch, tmp_path):
    """(matrix as the route takes it, call kwargs, integer data?)"""
    import torch

    from illico_b200 import hostio

    monkeypatch.setenv("ILLICO_PACK_UPLOAD", "0")
    if route == "dense_pinned":
        hp = torch.empty(X.shape, dtype=torch.float32, pin_memory=True)
        hp.copy_(torch.from_numpy(X))
        return hp.numpy(), {}, True
    if route == "dense_pageable":
        monkeypatch.setattr(hostio, "CHUNK_BYTES", 1 << 20)          # several chunks over several staging threads
        return X, {}, True
    if route == "dense_packed":
        monkeypatch.setenv("ILLICO_PACK_UPLOAD", "1")
        monkeypatch.setattr(hostio, "CHUNK_BYTES", 4 << 20)
        return X, {}, True
    if route == "cuda_tensor":
        return torch.from_numpy(X).to("cuda:0"), {}, True
    if route == "csr":
        return sparse.csr_matrix(X), {}, True
    if route == "csc":
        return sparse.csc_matrix(X), {}, True
    if route == "backed_csc":
        from illico_b200.backed import MemmapCSC, save_csc

        Xc = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
        return MemmapCSC(str(tmp_path / "csc")), dict(batch_size=16, n_threads=2), True
    if route == "backed_dense":
        from illico_b200.backed import MemmapDense, save_dense

        save_dense(str(tmp_path / "d.bin"), X)
        return MemmapDense(str(tmp_path / "d.bin")), dict(batch_size=24, n_threads=3), True
    assert route == "float64"
    return X.astype(np.float64) / 3.0, {}, False             # values float32 cannot hold: the recode path


def _call(method, Xin, labels, reference, groups, pts, kw):
    from illico_b200 import asymptotic_wilcoxon, ttest

    ad = FakeAnnData(Xin, labels)
    common = dict(return_array=True, score=True, pts=pts, p_adjust=True, groups=groups, **kw)
    if method == "wilcoxon":
        return asymptotic_wilcoxon(ad, False, "pert", reference, **common)
    return ttest(ad, "pert", reference, method=method, **common)


def assert_rows_of_full_call(sub, full, method, integer, what):
    """sub: (groups, var, results, extra) of a call with groups=; full: the same call without.  Every selected group's rows
    are its rows in the full call."""
    g_sub, _, res_sub, ex_sub = sub
    g_full, _, res_full, ex_full = full
    idx = np.searchsorted(g_full, g_sub)
    np.testing.assert_array_equal(g_full[idx], g_sub, err_msg=what)
    want, want_ex = res_full[idx], {k: v[idx] for k, v in ex_full.items()}
    assert set(ex_sub) == set(want_ex)
    exact = integer
    # U (Wilcoxon) / p_value: bit for bit; off integer data the t-test's p and t within 1e-10 and the fold change within 1e-14:
    # its float64 group sums are added in another order (the recode pass adds them with atomics, in no fixed order even
    # between two identical calls; one-versus-rest totals run over other groups) -- measured up to 3e-15
    cols = {0: 0.0 if (method == "wilcoxon" or exact) else 1e-10, 1: 0.0 if (method == "wilcoxon" or exact) else 1e-10,
            2: 0.0 if exact else 1e-14}
    for c, rtol in cols.items():
        if rtol == 0.0:
            np.testing.assert_array_equal(res_sub[:, :, c], want[:, :, c], err_msg=f"{what}: column {c}")
        else:
            # (t: also 1e-12 absolute -- where the two means cancel, t is rounding noise around 0)
            atol = 1e-12 if c == 1 else 0.0
            np.testing.assert_allclose(res_sub[:, :, c], want[:, :, c], rtol=rtol, atol=atol, err_msg=f"{what}: column {c}")
    for k in ("pct_nz_group", "pct_nz_reference"):
        if k in want_ex:
            np.testing.assert_array_equal(ex_sub[k], want_ex[k], err_msg=f"{what}: {k}")
    t_like = method != "wilcoxon" and not exact
    for k in ("score", "p_adj"):
        if t_like:
            np.testing.assert_allclose(ex_sub[k], want_ex[k], rtol=1e-10, atol=1e-12 if k == "score" else 0.0, err_msg=f"{what}: {k}")
        else:
            np.testing.assert_array_equal(ex_sub[k], want_ex[k], err_msg=f"{what}: {k}")


def _subsets(labels):
    names = sorted(set(labels) - {CONTROL})
    return [[names[3]], [names[1], names[6], names[-1], names[1]], names]   # one group, a few (one duplicated), all


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("test", ["ovo", "ovr"])
@pytest.mark.parametrize("route", ROUTES)
def test_selected_rows_equal_the_full_call(route, test, method, monkeypatch, tmp_path):
    if route == "dense_packed":      # the packed upload squeezes matrices of 64 MB and more: a large control group
        X, labels = labelled_counts(7, 10000, 2117, 12, control_share=0.8)
    else:
        X, labels = labelled_counts(7, 5000, 320, 12, control_share=0.75)
    Xin, kw, integer = _route_input(route, X, monkeypatch, tmp_path)
    reference = CONTROL if test == "ovo" else None
    for pts in (False, True):
        full = _call(method, Xin, labels, reference, None, pts, kw)
        for groups in _subsets(labels):
            if route == "dense_packed":
                from illico_b200 import hostio
                hostio.LAST_UPLOAD.clear()
            sub = _call(method, Xin, labels, reference, groups, pts, kw)
            want_groups = sorted(set(groups) | ({CONTROL} if reference else set()))
            assert list(sub[0]) == want_groups
            assert_rows_of_full_call(sub, full, method, integer, f"{route} {test} {method} pts={pts} groups={groups}")
            if route == "dense_packed" and test == "ovo" and len(groups) == 1:
                from illico_b200 import hostio
                n_sel = int(np.isin(labels, want_groups).sum())
                assert hostio.LAST_UPLOAD.get("packed", 0) > 0
                assert hostio.LAST_UPLOAD["bytes"] < 0.35 * n_sel * X.shape[1] * 4 < 0.35 * X.nbytes


@pytest.mark.gpu
def test_rank_genes_groups_equal_the_full_call(monkeypatch, tmp_path):
    from illico_b200 import rank_genes

    X, labels = labelled_counts(8, 4000, 200, 10, control_share=0.5)
    for route in ("dense_pageable", "csc", "cuda_tensor"):
        Xin, kw, _ = _route_input(route, X, monkeypatch, tmp_path)
        ad = FakeAnnData(Xin, labels)
        for reference in (CONTROL, None):
            for method in METHODS:
                for filt in ({}, dict(pts=True), dict(min_in_group_fraction=0.1, max_out_group_fraction=0.5, min_fold_change=1.0)):
                    args = dict(n_genes=25, method=method, **filt, **kw)
                    full = rank_genes(ad, False, "pert", reference, **args)
                    for groups in _subsets(labels):
                        sub = rank_genes(ad, False, "pert", reference, groups=groups, **args)
                        shown = sorted(set(groups))
                        want = full.loc[full.index.get_level_values("pert").isin(shown)]
                        what = f"{route} ref={reference} {method} {filt} {groups}"
                        assert list(sub.index) == list(want.index), what
                        np.testing.assert_array_equal(np.asarray(sub["feature"]), np.asarray(want["feature"]), err_msg=what)
                        for col in sub.columns[1:]:
                            np.testing.assert_array_equal(sub[col].to_numpy(), want[col].to_numpy(), err_msg=f"{what} {col}")


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
def test_one_versus_rest_with_more_than_65536_unselected_cells(method):
    """80 000 cells: the unselected ones fill two pseudo-groups; ranks, tie sums and the rest's totals are those of the
    full call (and the batch stays on the fused path: integer counts)."""
    X, labels = labelled_counts(9, 80_000, 24, 6, control_share=0.9)
    for pts in (False, True):
        full = _call(method, X, labels, None, None, pts, {})
        for groups in (["p002"], ["p000", "p004", CONTROL]):
            sub = _call(method, X, labels, None, groups, pts, {})
            assert_rows_of_full_call(sub, full, method, True, f"ovr big {method} {groups} pts={pts}")


@pytest.mark.gpu
def test_groups_on_every_gpu():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    X, labels = labelled_counts(10, 5000, 333, 12, control_share=0.6)
    for Xin in (X, sparse.csr_matrix(X), sparse.csc_matrix(X), torch.from_numpy(X).to("cuda:0")):
        for reference in (CONTROL, None):
            for method in ("wilcoxon", "t-test"):
                full = _call(method, Xin, labels, reference, None, True, dict(devices="all"))
                for groups in _subsets(labels):
                    sub = _call(method, Xin, labels, reference, groups, True, dict(devices="all"))
                    assert_rows_of_full_call(sub, full, method, True, f"devices=all {type(Xin)} {reference} {method} {groups}")


# ---- GPU: against independent answers --------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_against_the_oracle_and_scipy():
    """One-versus-reference equals the oracle on the subset a user cuts by hand; one-versus-rest equals the oracle on the
    full matrix -- not on that subset: the rest of a selected group holds the cells of the groups not tested."""
    import oracle
    from illico_b200 import asymptotic_wilcoxon
    from tests.parity import assert_parity

    X, labels = labelled_counts(11, 2500, 30, 8, control_share=0.4)
    groups = ["p002", "p005"]
    ad = FakeAnnData(X, labels)
    # one-versus-reference: the subset
    g, _, res = asymptotic_wilcoxon(ad, False, "pert", CONTROL, groups=groups, return_array=True)
    mask = np.isin(labels, groups + [CONTROL])
    og, p, U, fc = oracle.run(X[mask], labels[mask], CONTROL)
    assert list(g) == list(og)
    assert_parity((res[:, :, 0], res[:, :, 1], res[:, :, 2]), (p, U, fc), ref_row=list(og).index(CONTROL), what="ovo subset")
    # one-versus-rest: the full matrix
    g, _, res = asymptotic_wilcoxon(ad, False, "pert", None, groups=groups, return_array=True)
    og, p, U, fc = oracle.run(X, labels, None)
    idx = np.searchsorted(og, g)
    assert_parity((res[:, :, 0], res[:, :, 1], res[:, :, 2]), (p[idx], U[idx], fc[idx]), what="ovr full")
    og_sub, p_sub, U_sub, _ = oracle.run(X[np.isin(labels, groups)], labels[np.isin(labels, groups)], None)
    assert not np.array_equal(U_sub, res[:, :, 1])            # the hand-cut subset's "rest" is another test
    # scipy on the raw arrays: U of the rest sample and the p-value, gene by gene
    for k, name in enumerate(g):
        inside = labels == name
        u, pv = stats.mannwhitneyu(X[~inside].astype(np.float64), X[inside].astype(np.float64), axis=0, method="asymptotic",
                                   use_continuity=True, alternative="two-sided")
        live = np.isfinite(pv)
        np.testing.assert_array_equal(res[k, live, 1], u[live])
        np.testing.assert_allclose(res[k, live, 0], pv[live], rtol=1e-9, atol=1e-300)
