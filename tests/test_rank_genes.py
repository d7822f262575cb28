"""The score plane (``score=True``) and per-group ranking (``rank_genes``, ``illico_top_genes``).

The score is checked bit for bit against a numpy restatement of its definition, ``(mu - U) / sigma`` with the p-value's
sigma, computed from the oracle's exact U and tie sums; the ranking against ``np.lexsort`` of the full score frame."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from tests.golden import cases as C
from tests.util import FakeAnnData

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- numpy restatements ----------------------------------------------------------------------------------------------

def score_reference(U, ties, counts, ref_row, n_cells, tie_correct):
    """(mu - U) / sigma in float64, in the kernels' operation order; 0 where the tie correction is <= 1e-9 and on the
    control row.  ``ties``: [G, N] (one-versus-reference) or [N] (one-versus-rest), as ``oracle.run(want_ties=True)``."""
    n_t = np.asarray(counts, dtype=np.int64)[:, None]
    n_r = np.int64(counts[ref_row]) if ref_row is not None else np.int64(n_cells) - n_t
    n = n_r + n_t
    tie = np.where(np.isnan(ties), 0.0, ties) if tie_correct else np.zeros_like(ties)
    with np.errstate(divide="ignore", invalid="ignore"):
        tie_corr = 1.0 - tie / (n * (n - 1) * (n + 1)).astype(np.float64)
        prod12 = (n_r * n_t * (n_r + n_t + 1)).astype(np.float64) / 12.0
        mu = (n_r * n_t).astype(np.float64) / 2.0
        z = (mu - U) / np.sqrt(prod12 * tie_corr)
    z = np.where(tie_corr > 1e-9, z, 0.0)
    z = np.broadcast_to(z, U.shape).copy()
    if ref_row is not None:
        z[ref_row] = 0.0
    return z


def bh_reference(p):
    """statsmodels multipletests(method="fdr_bh") per row (the restatement of test_optional_columns_p_adj_and_log2fc)."""
    G, N = p.shape
    want = np.empty_like(p)
    for g in range(G):
        order = np.argsort(p[g], kind="stable")
        raw = p[g][order] / (np.arange(1, N + 1) / float(N))
        adj = np.minimum.accumulate(raw[::-1])[::-1]
        adj[adj > 1] = 1
        want[g, order] = adj
    return want


def rank_order(s, by_abs):
    key = -np.abs(s) if by_abs else -s
    return np.lexsort((np.arange(s.size), key))


# ---- CPU -------------------------------------------------------------------------------------------------------------

def test_flags_layout_matches_header(tmp_path):
    """ctypes' Flags has the size and field offsets of illico_flags_t in include/illico_b200.h."""
    from illico_b200 import _lib

    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "illico_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(illico_flags_t), offsetof(illico_flags_t, group_sums),'
                   ' offsetof(illico_flags_t, scores), offsetof(illico_flags_t, score_group_stride)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    F = _lib.Flags
    assert got == [ctypes.sizeof(F), F.group_sums.offset, F.scores.offset, F.score_group_stride.offset]
    assert _lib.ABI_VERSION == 3


def test_public_names_are_functions_whatever_the_import_order():
    code = ("import illico_b200 as m; from illico_b200 import rank_genes; from illico_b200 import asymptotic_wilcoxon; "
            "assert callable(rank_genes) and callable(asymptotic_wilcoxon) and callable(m.asymptotic_wilcoxon)")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


def test_rank_genes_without_gpu_raises(monkeypatch):
    import torch

    from illico_b200 import _lib, rank_genes, synth

    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    X, labels = synth.k562_like(seed=3, n_cells=200, n_genes=8, n_perts=3)
    with pytest.raises(_lib.IllicoCudaError):
        rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=synth.CONTROL)


@pytest.mark.parametrize("n_genes", [0, -3, 2.5, True])
def test_rank_genes_rejects_bad_n_genes(n_genes):
    from illico_b200 import rank_genes, synth

    X, labels = synth.k562_like(seed=3, n_cells=200, n_genes=8, n_perts=3)
    with pytest.raises(ValueError):
        rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", n_genes=n_genes)


# ---- GPU: the score plane --------------------------------------------------------------------------------------------

def _scored(X, labels, reference, **kw):
    """(groups, results [G, N, 3], score [G, N]) of asymptotic_wilcoxon(score=True, return_array=True)."""
    from illico_b200 import asymptotic_wilcoxon

    groups, _, out, extra = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=reference, score=True,
                                                return_array=True, **kw)
    assert list(extra) == ["score"]
    return groups, out, extra["score"]


def _want_score(X, labels, reference, is_log1p=False, use_continuity=True, tie_correct=True, alternative="two-sided"):
    from illico_b200.groups import encode_and_count_groups

    _, grpc = encode_and_count_groups(labels, reference)
    groups, p, U, fc, ties = oracle.run(X, labels, reference, is_log1p=is_log1p, use_continuity=use_continuity,
                                        tie_correct=tie_correct, alternative=alternative, want_ties=True)
    ref_row = grpc.encoded_ref_group if reference is not None else None
    return score_reference(U, ties, grpc.counts, ref_row, X.shape[0], tie_correct)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(C.CASES))
def test_score_plane_is_exact_on_golden_cases(name):
    """Every golden case x format x flag combination: the score equals the numpy restatement bit for bit; p-values and U
    are bit-identical to the same call without the score, and so are the fold changes of integer counts."""
    from illico_b200 import asymptotic_wilcoxon

    builder, grid, batch_size = C.CASES[name]
    X, labels, reference = builder()
    integer_counts = bool(np.array_equal(X, np.round(X)))
    for fmt, test, cc, tc, alt, log1p in grid:
        ref = reference if test == "ovo" else None
        kw = dict(is_log1p=log1p, batch_size=batch_size, alternative=alt, use_continuity=cc, tie_correct=tc)
        Xf = C.to_format(X, fmt)
        groups, out, score = _scored(Xf, labels, ref, **kw)
        _, _, base = asymptotic_wilcoxon(FakeAnnData(Xf, labels), group_keys="pert", reference=ref, return_array=True, **kw)
        what = f"{name}:{fmt}:{test}:cc{cc}:tc{tc}:{alt}:log{log1p}"
        np.testing.assert_array_equal(out[:, :, :2], base[:, :, :2], err_msg=what)
        if integer_counts and not log1p:
            np.testing.assert_array_equal(out[:, :, 2], base[:, :, 2], err_msg=what)
        else:
            # table slots claimed and values staged with atomics, in arrival order: the fold change's sum of non-integer
            # values may be added in another order -- and differ in the last bit -- between any two calls, score or not
            np.testing.assert_allclose(out[:, :, 2], base[:, :, 2], rtol=1e-14, atol=0, err_msg=what)
        want = _want_score(Xf, labels, ref, log1p, cc, tc, alt)
        np.testing.assert_array_equal(score, want, err_msg=what)
        if ref is not None:
            assert not score[int(np.searchsorted(groups, ref))].any()


def _route_case():
    """Count-like matrix whose genes take every route of the fused paths (table, wide table, handed back) next to
    continuous, all-zero and high-count genes."""
    rng = np.random.RandomState(31)
    n, N = 6000, 72
    X = (rng.poisson(1.0, size=(n, N)) * (rng.rand(n, N) >= 0.7)).astype(np.float32)
    sizes = rng.randint(3, 400, size=14)
    codes = np.concatenate([np.repeat(np.arange(sizes.size), sizes), rng.randint(0, sizes.size, size=n - sizes.sum())])
    rng.shuffle(codes)
    labels = [f"g{c:02d}" for c in codes]
    X[:, 1] = 0.0                                                   # all-zero gene
    X[:, 2] = rng.poisson(30.0, n)                                  # many distinct values: wide table or handed back
    X[:, 3] = np.round(rng.gamma(2.0, 2.0, n), 3)                   # continuous: handed back
    X[:, 10] = rng.poisson(12.0, n)
    X[:, 12] = rng.poisson(45.0, n)                                 # past the wide table's 64
    X[:, 40:44] = rng.poisson(30.0, (n, 4))
    return X, labels, "g06"


ROUTES = {
    "fused_narrow": {"ILLICO_FUSED_WIDE": "0", "ILLICO_FUSED_LIST_SHARE": "1.0"},
    "fused_wide": {"ILLICO_FUSED_WIDE": "1", "ILLICO_FUSED_LIST_SHARE": "1.0"},
    "hand_back_list": {"ILLICO_FUSED_LIST_SHARE": "1.0"},
    "hand_back_all": {"ILLICO_FUSED_LIST_SHARE": "0.0"},
    "general": {"ILLICO_OVO_FUSED": "0", "ILLICO_OVR_FUSED": "0", "ILLICO_CSR_FUSED": "0"},
}


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("fmt", ["dense", "csr"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_score_plane_every_kernel_route(monkeypatch, route, fmt, test):
    """The fused epilogues (narrow, wide), the hand-back list and whole-batch hand-back, and the general path all write
    the same, exact scores."""
    from illico_b200 import _lib

    for k, v in ROUTES[route].items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    X, labels, ref = _route_case()
    reference = ref if test == "ovo" else None
    Xf = C.to_format(X, fmt)
    _lib.profile_report()
    _, _, score = _scored(Xf, labels, reference, is_log1p=False)
    ran = _lib.profile_report()
    if route == "general":
        assert "fused_epilogue_kernel" not in ran
    else:
        assert "fused_epilogue_kernel" in ran
    if route == "fused_wide" and fmt == "dense" and test == "ovo":
        assert "fused_wide_epilogue_kernel" in ran
    np.testing.assert_array_equal(score, _want_score(Xf, labels, reference), err_msg=f"{route} {fmt} {test}")


class _Backed:
    def __init__(self, X):
        self._X = X
        self.shape = X.shape

    def __getitem__(self, key):
        return self._X[key]


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["csc", "float64", "backed_dense", "backed_csc", "device_tensor", "devices_all"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_score_plane_every_input_route(tmp_path, source, test):
    """CSC, float64 input recoded on the device, backed streaming, a device-resident tensor and devices="all"."""
    import torch
    from scipy import sparse

    from illico_b200 import synth
    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense

    X, labels = synth.k562_like(seed=7, n_cells=5000, n_genes=67, n_perts=9)
    X[:, 11] = np.random.RandomState(2).poisson(25.0, X.shape[0])
    reference = synth.CONTROL if test == "ovo" else None
    kw = {}
    if source == "csc":
        Xin = Xo = sparse.csc_matrix(X)
    elif source == "float64":
        Xin = Xo = X.astype(np.float64) * (1.0 + 1e-12)                  # values float32 cannot hold: recoded
    elif source == "backed_dense":
        save_dense(str(tmp_path / "d.bin"), X)
        Xin, Xo, kw = MemmapDense(str(tmp_path / "d.bin")), X, dict(batch_size=16, n_threads=3)
    elif source == "backed_csc":
        Xc = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
        Xin, Xo, kw = MemmapCSC(str(tmp_path / "csc")), Xc, dict(batch_size=20, n_threads=2)
    elif source == "device_tensor":
        Xin, Xo = torch.from_numpy(X).cuda(), X
    else:
        Xin, Xo, kw = X, X, dict(devices="all")
    _, out, score = _scored(Xin, labels, reference, is_log1p=False, **kw)
    np.testing.assert_array_equal(score, _want_score(Xo, labels, reference), err_msg=source)


# ---- GPU: rank_genes --------------------------------------------------------------------------------------------------

def check_ranking(df, X, labels, reference, n_genes, by_abs=False, **kw):
    """rank_genes' frame against the full score=True frame: order, every column bit for bit, BH over all genes."""
    from illico_b200 import asymptotic_wilcoxon

    kw.setdefault("is_log1p", False)
    var_names = [f"gene_{i}" for i in range(X.shape[1])]
    groups, _, out, extra = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=reference, score=True,
                                                p_adjust=True, return_array=True, **kw)
    G, N = out.shape[:2]
    k = N if n_genes is None else min(n_genes, N)
    kept = [g for g in range(G) if reference is None or groups[g] != reference]
    assert list(df.columns) == ["feature", "score", "p_value", "p_adj", "statistic", "fold_change", "log2_fold_change"]
    assert df.index.names == ["pert", "rank"] and len(df) == len(kept) * k
    assert list(df.index.get_level_values("pert")) == list(np.repeat(np.asarray(groups)[kept], k))
    assert list(df.index.get_level_values("rank")) == list(np.tile(np.arange(k), len(kept)))
    padj = bh_reference(out[:, :, 0])
    np.testing.assert_array_equal(extra["p_adj"], padj)
    got = df.to_numpy()
    for i, g in enumerate(kept):
        sel = rank_order(extra["score"][g], by_abs)[:k]
        rows = got[i * k:(i + 1) * k]
        assert list(rows[:, 0]) == [var_names[j] for j in sel], f"group {groups[g]}"
        np.testing.assert_array_equal(rows[:, 1].astype(float), extra["score"][g, sel])
        np.testing.assert_array_equal(rows[:, 2].astype(float), out[g, sel, 0])
        np.testing.assert_array_equal(rows[:, 3].astype(float), extra["p_adj"][g, sel])
        np.testing.assert_array_equal(rows[:, 4].astype(float), out[g, sel, 1])
        np.testing.assert_array_equal(rows[:, 5].astype(float), out[g, sel, 2])
        with np.errstate(divide="ignore", invalid="ignore"):
            np.testing.assert_array_equal(rows[:, 6].astype(float), np.log2(out[g, sel, 2]))
    return extra["score"]


@pytest.mark.gpu
@pytest.mark.parametrize("n_genes", [None, 1, 100, 5000])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_rank_genes_against_full_frame(n_genes, test):
    from illico_b200 import rank_genes, synth

    X, labels = synth.k562_like(seed=91, n_cells=4000, n_genes=700, n_perts=6)
    X[:, :20] *= (np.asarray(labels) == "p0001")[:, None] * 3 + 1         # a few real effects
    X[:, 30:60] = 0.0                                                      # all-zero genes: score 0, ranked in index order
    reference = synth.CONTROL if test == "ovo" else None
    df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=reference, n_genes=n_genes)
    score = check_ranking(df, X, labels, reference, n_genes)
    assert (score[:, 30:60] == 0).all()
    if reference is not None:
        assert reference not in set(df.index.get_level_values("pert"))
    else:
        assert len(set(df.index.get_level_values("pert"))) == len(set(labels))


@pytest.mark.gpu
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_rank_genes_by_abs_and_options(test):
    from illico_b200 import rank_genes, synth

    X, labels = synth.k562_like(seed=92, n_cells=3000, n_genes=300, n_perts=5)
    reference = synth.CONTROL if test == "ovo" else None
    kw = dict(alternative="less", use_continuity=False, tie_correct=False, batch_size=64)
    df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=reference, n_genes=40,
                    rankby_abs=True, **kw)
    check_ranking(df, X, labels, reference, 40, by_abs=True, **kw)


@pytest.mark.gpu
def test_rank_genes_wide_matrix():
    from illico_b200 import rank_genes, synth

    X, labels = synth.k562_like(seed=93, n_cells=1500, n_genes=40_000, n_perts=3, masked=0.97)
    df = rank_genes(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference=synth.CONTROL, n_genes=100)
    check_ranking(df, X, labels, synth.CONTROL, 100)


@pytest.mark.gpu
def test_rank_genes_many_groups():
    from illico_b200 import rank_genes

    X, labels, reference = C.CASES["c5_many_groups"][0]()
    Xf = C.to_format(X, "csr")
    assert len(set(labels)) > 10_000
    for ref in (reference, None):
        df = rank_genes(FakeAnnData(Xf, labels), is_log1p=False, group_keys="pert", reference=ref, n_genes=4)
        check_ranking(df, Xf, labels, ref, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_rank_genes_devices_and_backed_match_single_gpu(tmp_path, test):
    import pandas as pd
    from scipy import sparse

    from illico_b200 import rank_genes, synth
    from illico_b200.backed import MemmapCSC, save_csc

    X, labels = synth.k562_like(seed=94, n_cells=5000, n_genes=131, n_perts=9)
    X[:, 11] = np.random.RandomState(2).poisson(25.0, X.shape[0])
    reference = synth.CONTROL if test == "ovo" else None
    kw = dict(is_log1p=False, group_keys="pert", reference=reference, n_genes=25)
    want = rank_genes(FakeAnnData(X, labels), **kw)
    check_ranking(want, X, labels, reference, 25)
    same = lambda a, b: pd.testing.assert_frame_equal(a, b, check_exact=True)  # noqa: E731
    same(rank_genes(FakeAnnData(X, labels), devices="all", **kw), want)
    Xs = sparse.csr_matrix(X)
    same(rank_genes(FakeAnnData(Xs, labels), devices="all", **kw), want)
    Xc = sparse.csc_matrix(X)
    save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
    same(rank_genes(FakeAnnData(MemmapCSC(str(tmp_path / "csc")), labels), batch_size=32, n_threads=2, **kw), want)


@pytest.mark.gpu
@pytest.mark.parametrize("by_abs", [False, True])
def test_top_genes_entry_point_on_planted_scores(by_abs):
    """illico_top_genes directly: NaN after every number, -0.0 equal to +0.0, runs of equal values in index order,
    k = 1 .. N, records gathered from the planes (p_adj NULL -> NaN)."""
    import torch

    from illico_b200 import _lib

    rng = np.random.RandomState(5)
    G, N = 4, 3000
    s = np.round(rng.randn(G, N) * 3, 1)                                  # many runs of equal values
    s[:, rng.choice(N, 200, replace=False)] = np.nan
    s[:, rng.choice(N, 150, replace=False)] = 0.0
    s[:, rng.choice(N, 150, replace=False)] = -0.0
    s[0, :40] = np.inf
    s[1, :40] = -np.inf
    s[2] = 0.0                                                             # a group of ties only
    s[3, ::2] = -0.0
    res = rng.rand(G, N, 3)
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    ds, dr = torch.from_numpy(s).to(dev), torch.from_numpy(res).to(dev)
    ws = torch.empty(int(lib.illico_top_genes_workspace_bytes(G, N)), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    for k in (1, 17, N):
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 5), dtype=torch.float64, device=dev)
        _lib.check(lib.illico_top_genes(ds.data_ptr(), N, dr.data_ptr(), 3 * N, None, G, N, k, int(by_abs), gene.data_ptr(),
                                        rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "illico_top_genes")
        gene, rec = gene.cpu().numpy(), rec.cpu().numpy()
        for g in range(G):
            sel = rank_order(s[g], by_abs)[:k]
            np.testing.assert_array_equal(gene[g], sel, err_msg=f"group {g} k {k}")
            np.testing.assert_array_equal(rec[g, :, 0], s[g, sel])
            np.testing.assert_array_equal(rec[g, :, 1:4], res[g, sel])
            assert np.isnan(rec[g, :, 4]).all()
    bad = torch.empty((G, 1), dtype=torch.int32, device=dev)
    for k in (0, N + 1):                                                   # k outside [1, N]: refused, nothing enqueued
        assert lib.illico_top_genes(ds.data_ptr(), N, dr.data_ptr(), 3 * N, None, G, N, k, 0, bad.data_ptr(), dr.data_ptr(),
                                    ws.data_ptr(), ws.numel(), st) != 0
