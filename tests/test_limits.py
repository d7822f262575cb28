"""The kernels at their limits: the plan's segment length and the caps their shared tables, 16-bit counters and tier
switches are built on.  Every planted size below is derived from the `constexpr` caps parsed out of the CUDA sources,
so that a changed cap moves the tests with it; every run is compared with the CPU oracle, including the exact 2U and
tie sums of the debug outputs (a dispatcher called with ``debug=`` always takes the general path)."""
import os
import re

import numpy as np
import pytest

import oracle
from tests.golden import cases as C
from tests.parity import P_ATOL, assert_parity
from tests.util import FakeAnnData, planes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "illico_b200", "csrc")
CAP_NAMES = {
    "rank_ovo.cu": ("REF_CAP", "DT_CAP", "NE_CAP", "ST_CAP", "STREAM_MAX", "WARP_CAP"),
    "rank_ovr.cu": ("T_CAP", "T_MULTI", "MAX_DISTINCT", "HASH_CAP"),
    "fused.cu": ("DCAP",),
}
_CONSTEXPR = re.compile(r"^\s*constexpr\s+int\s+([A-Z][A-Z0-9_]*)\s*=\s*(\d+)\s*;", re.M)
U8_MAX = 255        # ovr_table_kernel's 8-bit segment records
U16_MAX = 65535     # the 16-bit per-segment / per-group counters
PAIR_MAX = 208063   # one-versus-reference pairs up to this many cells: tie sums below 2^53


def _parse_caps() -> dict:
    caps = {}
    for fname, names in CAP_NAMES.items():
        with open(os.path.join(CSRC, fname)) as f:
            found = dict(_CONSTEXPR.findall(f.read()))
        caps.update({n: int(found[n]) if n in found else None for n in names})
    return caps


CAPS = _parse_caps()


def cap(name: str) -> int:
    value = CAPS[name]
    if value is None:
        pytest.fail(f"constexpr int {name} is no longer defined in {CSRC}")
    return value


# ============================================ CPU ==============================================================

def test_caps_come_from_the_source():
    missing = [n for n, v in CAPS.items() if v is None]
    assert not missing, f"caps no longer defined as `constexpr int NAME = N;`: {missing}"
    # the planted sizes below rely on these orderings
    assert 0 < cap("STREAM_MAX") < cap("WARP_CAP") // 2 < cap("WARP_CAP") < cap("REF_CAP")
    assert cap("DT_CAP") < cap("ST_CAP") < cap("REF_CAP") and cap("NE_CAP") >= 1
    assert cap("T_CAP") < cap("MAX_DISTINCT") < cap("HASH_CAP") < U16_MAX and cap("DCAP") >= 2


BAD_SEG_MAX = [0, -1, U16_MAX + 1, 1.5, "7", True]


@pytest.mark.parametrize("bad", BAD_SEG_MAX)
def test_segment_length_is_validated(bad):
    from illico_b200.engine import Engine
    from illico_b200.groups import build_plan, encode_and_count_groups

    _, grpc = encode_and_count_groups(np.array(["a", "b", "a", "c"]), "a")
    with pytest.raises(ValueError, match="ILLICO_B200_SEG_MAX"):
        build_plan(grpc, bad)
    with pytest.raises(ValueError, match="ILLICO_B200_SEG_MAX"):
        Engine(grpc, seg_max=bad)


@pytest.mark.parametrize("bad", ["0", "-1", str(U16_MAX + 1), "1.5", "abc", ""])
def test_segment_length_from_the_environment_is_validated(monkeypatch, bad):
    from illico_b200 import asymptotic_wilcoxon
    from illico_b200.groups import seg_max_from_env

    monkeypatch.setenv("ILLICO_B200_SEG_MAX", bad)
    with pytest.raises(ValueError, match="ILLICO_B200_SEG_MAX"):
        seg_max_from_env()
    X = np.arange(12, dtype=np.float32).reshape(4, 3)
    with pytest.raises(ValueError, match="ILLICO_B200_SEG_MAX"):
        asymptotic_wilcoxon(FakeAnnData(X, ["a", "b", "a", "c"]), is_log1p=False, group_keys="pert", reference="a")


@pytest.mark.parametrize("good", [1, U16_MAX])
def test_segment_length_limits_are_accepted(monkeypatch, good):
    from illico_b200.groups import build_plan, encode_and_count_groups, seg_max_from_env

    labels = np.repeat(np.array(["a", "b", "c"]), [U16_MAX + 2, 3, 1])
    _, grpc = encode_and_count_groups(labels, "a")
    p = build_plan(grpc, good)
    seg_len = np.diff(p.seg_pos)
    assert seg_len.max() == min(good, U16_MAX) and seg_len.min() >= 1
    monkeypatch.setenv("ILLICO_B200_SEG_MAX", str(good))
    assert seg_max_from_env() == good
    assert build_plan(grpc).seg_max == good


def test_engine_cache_keys_on_the_segment_length(monkeypatch):
    from illico_b200 import dispatch
    from illico_b200.groups import encode_and_count_groups

    built = []

    class FakeEngine:
        def __init__(self, grpc, device=None, seg_max=None):
            built.append(seg_max)

    monkeypatch.setattr(dispatch, "Engine", FakeEngine)
    _, grpc = encode_and_count_groups(np.array(["a", "b", "a", "c"]), "a")
    dispatch.clear_caches()
    try:
        monkeypatch.delenv("ILLICO_B200_SEG_MAX", raising=False)
        e512 = dispatch.engine_for(grpc, "cuda:0")
        assert dispatch.engine_for(grpc, "cuda:0") is e512
        monkeypatch.setenv("ILLICO_B200_SEG_MAX", "7")
        e7 = dispatch.engine_for(grpc, "cuda:0")
        assert e7 is not e512 and built == [512, 7]
        monkeypatch.setenv("ILLICO_B200_SEG_MAX", "512")
        assert dispatch.engine_for(grpc, "cuda:0") is e512
    finally:
        dispatch.clear_caches()


# ============================================ GPU ==============================================================

@pytest.fixture
def cuda_lib():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from illico_b200 import _lib

    lib = _lib.load()
    before = _lib.launch_count()
    yield lib
    assert _lib.launch_count() > before, "no kernel of libillico_b200.so was launched"


def _run(X, labels, reference, **kw):
    from illico_b200 import asymptotic_wilcoxon

    groups = np.unique(np.asarray(labels))
    df = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=reference, is_log1p=False, **kw)
    return planes(df, len(groups), X.shape[1])


def _debug(fmt, test, Xf, labels, reference):
    """(p, U, fc) and the debug integers {u2, tie_sum, tie_exact} of the dispatcher (general path)."""
    from illico_b200 import dispatch
    from illico_b200.groups import encode_and_count_groups

    _, grpc = encode_and_count_groups(labels, reference)
    fn = getattr(dispatch, f"{fmt}_{test}_mwu_kernel_over_contiguous_col_chunk")
    dbg = {}
    got = fn(Xf, 0, Xf.shape[1], grpc, False, True, True, "two-sided", debug=dbg)
    return got, {k: v.cpu().numpy() for k, v in dbg.items()}


def _assert_exact(dbg, U, ties, ref_row, what, exact_ties=None):
    """debug 2U and f64 tie sums bit for bit against the oracle; the exact tie sum equals the f64 one below 2^53 and
    ``exact_ties`` (Python ints, wrapped to 64 bits like the int64 output) above."""
    rows = np.ones(U.shape[0], bool)
    if ref_row is not None:
        rows[ref_row] = False
    np.testing.assert_array_equal(dbg["u2"][rows], (2 * U[rows]).astype(np.int64), err_msg=f"{what}: 2U")
    tie, te = (dbg["tie_sum"][rows], dbg["tie_exact"][rows]) if ref_row is not None else (dbg["tie_sum"], dbg["tie_exact"])
    want = ties[rows] if ref_row is not None else ties
    np.testing.assert_array_equal(tie, want, err_msg=f"{what}: f64 tie sum")
    small = (want >= 0) & (want < 2.0 ** 53)   # (the reference's int64 Z^3 - Z wraps for pairs of > 2 097 151 zeros)
    np.testing.assert_array_equal(te[small].astype(np.float64), want[small], err_msg=f"{what}: exact tie sum")
    if exact_ties is not None:
        ex = np.array([int(v) % (1 << 64) for v in np.ravel(exact_ties[rows] if ref_row is not None else exact_ties)],
                      dtype=np.uint64)
        np.testing.assert_array_equal(te.view(np.uint64).ravel(), ex, err_msg=f"{what}: exact tie sum (mod 2^64)")
    else:
        assert small.all(), f"{what}: tie sums above 2^53 need exact_ties"


def _check_against_oracle(fmt, test, X, labels, reference, want=None, what=""):
    """Default route (asymptotic_wilcoxon) and debug integers (general path) against the oracle."""
    Xf = C.to_format(X, fmt)
    ref = reference if test == "ovo" else None
    groups, p, U, fc, ties = want if want is not None else oracle.run(Xf, labels, ref, want_ties=True)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    assert_parity(_run(Xf, labels, ref), (p, U, fc), ref_row=ref_row, what=f"{what} default route")
    got, dbg = _debug(fmt, test, Xf, labels, ref)
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{what} debug call")
    _assert_exact(dbg, U, ties, ref_row, what)


# ---------------------------------------------------------------------------------------------------------------
# 3. results do not depend on the segment length

SEG_LENGTHS = [1, 7, 255, 256, 511, 513, 4096, U16_MAX]


def _mixed_case(fmt):
    """~10k cells x 40 genes: K562-like counts, Poisson(30) genes, continuous genes, a negative gene (dense only), a gene
    that is zero everywhere; a 5 600-cell control (5 600 segments at length 1) and skewed group sizes."""
    rng = np.random.RandomState(2024)
    sizes = {"ctrl": 5600, "big": 1500, "mid0": 400, "mid1": 400}
    sizes.update({f"s{i:02d}": 50 for i in range(40)})
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n, N = labels.size, 40
    X = np.zeros((n, N), np.float32)
    X[:, :20] = rng.poisson(0.3, (n, 20)) * (rng.rand(n, 20) < 0.6)             # K562-like counts
    X[:, 20:24] = rng.poisson(30.0, (n, 4))                                       # high counts
    X[:, 24:34] = rng.lognormal(0.0, 1.0, (n, 10)) * (rng.rand(n, 10) < 0.5)      # continuous, half zeros
    X[:, 34:38] = rng.lognormal(0.0, 1.0, (n, 4))                                 # continuous, dense
    X[:, 38] = rng.randn(n)                                                       # negative values
    if fmt != "dense":
        X[:, 38] = np.abs(X[:, 38])      # (the sparse kernels assume stored values > 0)
    assert not X[:, 39].any()
    assert sizes["ctrl"] > 4142 and sizes["ctrl"] <= 6000
    return X, labels


def _close(a, b, rtol, atol, what):
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b), err_msg=what)
    np.testing.assert_array_equal(np.isposinf(a), np.isposinf(b), err_msg=what)
    fin = np.isfinite(b)
    np.testing.assert_allclose(a[fin], b[fin], rtol=rtol, atol=atol, err_msg=what)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_results_do_not_depend_on_the_segment_length(cuda_lib, monkeypatch, fmt, test):
    from illico_b200 import dispatch

    X, labels = _mixed_case(fmt)
    Xf = C.to_format(X, fmt)
    ref = "ctrl" if test == "ovo" else None
    groups, p, U, fc, ties = oracle.run(Xf, labels, ref, want_ties=True)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    routes = ("default", "general")

    def run_all(seg):
        monkeypatch.setenv("ILLICO_B200_SEG_MAX", str(seg))
        dispatch.clear_caches()
        out = {}
        for route in routes:
            for var in ("ILLICO_OVO_FUSED", "ILLICO_OVR_FUSED", "ILLICO_CSR_FUSED"):
                monkeypatch.setenv(var, "0" if route == "general" else "1")
            out[route] = _run(Xf, labels, ref)
        monkeypatch.delenv("ILLICO_OVO_FUSED")
        monkeypatch.delenv("ILLICO_OVR_FUSED")
        monkeypatch.delenv("ILLICO_CSR_FUSED")
        out["debug"] = _debug(fmt, test, Xf, labels, ref)
        return out

    base = run_all(512)
    for seg in [512] + SEG_LENGTHS:
        got = base if seg == 512 else run_all(seg)
        what = f"{fmt}:{test}:seg={seg}"
        for route in routes:
            gp, gU, gfc = got[route]
            assert_parity((gp, gU, gfc), (p, U, fc), ref_row=ref_row, what=f"{what}:{route} vs oracle")
            bp, bU, bfc = base[route]
            np.testing.assert_array_equal(gU, bU, err_msg=f"{what}:{route}: U differs from length 512")
            _close(gp, bp, 1e-13, P_ATOL, f"{what}:{route}: p")
            _close(gfc, bfc, 1e-14, 0.0, f"{what}:{route}: fold change")   # (CSR staging adds with atomics)
        (dp, dU, dfc), dbg = got["debug"]
        assert_parity((dp, dU, dfc), (p, U, fc), ref_row=ref_row, what=f"{what}:debug vs oracle")
        _assert_exact(dbg, U, ties, ref_row, what)
    dispatch.clear_caches()


# ---------------------------------------------------------------------------------------------------------------
# 4. a control of 2.3 M cells at the default segment length

def _exact_pair_ties(X, labels, ref):
    """[G, N] exact tie sums (Python ints) of every (group, control) pair: sum over the pair's distinct values (the
    zeros one block) of t^3 - t."""
    groups = np.unique(labels)
    out = np.zeros((groups.size, X.shape[1]), dtype=object)
    ctrl = labels == ref
    for j in range(X.shape[1]):
        cv, cc = np.unique(X[ctrl, j], return_counts=True)
        base = dict(zip(cv.tolist(), cc.tolist()))
        for gi, g in enumerate(groups):
            if g == ref:
                continue
            m = dict(base)
            gv, gc = np.unique(X[labels == g, j], return_counts=True)
            for v, c in zip(gv.tolist(), gc.tolist()):
                m[v] = m.get(v, 0) + c
            out[gi, j] = sum(t ** 3 - t for t in m.values())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "dense"])
def test_two_million_cell_control_at_the_default_segment_length(cuda_lib, monkeypatch, fmt):
    """4 493 control segments: more than ovo_kernel's 2 048-word offset table.  The pairs exceed PAIR_MAX cells, so the
    general path runs and the f64 tie sums are the ordered replay."""
    import time

    from illico_b200 import dispatch

    monkeypatch.delenv("ILLICO_B200_SEG_MAX", raising=False)
    rng = np.random.RandomState(5)
    n_ctrl = 2_300_000
    sizes = {"ctrl": n_ctrl, **{f"p{i}": 200 + 50 * i for i in range(6)}}
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    assert -(-n_ctrl // 512) == 4493
    X = np.zeros((n, 4), np.float32)
    X[:, 0] = np.where(rng.rand(n) < 0.7, rng.lognormal(0, 1, n), 0)     # continuous
    X[:, 1] = rng.poisson(0.8, n)                                         # counts
    other = labels != "ctrl"
    X[other, 2] = rng.poisson(2.0, other.sum())                           # zero in the control
    Xf = C.to_format(X, fmt)
    t0 = time.perf_counter()
    groups, p, U, fc, ties = oracle.run(Xf, labels, "ctrl", want_ties=True, n_threads=oracle.max_threads())
    print(f"oracle, {n} cells x 4 genes ({fmt}): {time.perf_counter() - t0:.1f} s")
    ref_row = int(np.searchsorted(groups, "ctrl"))
    assert_parity(_run(Xf, labels, "ctrl"), (p, U, fc), ref_row=ref_row, what=f"{fmt} 2.3M control")
    got, dbg = _debug(fmt, "ovo", Xf, labels, "ctrl")
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{fmt} 2.3M control, debug call")
    _assert_exact(dbg, U, ties, ref_row, f"{fmt} 2.3M control", exact_ties=_exact_pair_ties(X, labels, "ctrl"))
    dispatch.clear_caches()


# ---------------------------------------------------------------------------------------------------------------
# 5. the 65 535 / 65 536 boundary of the 16-bit counters

BIG_CTRL = PAIR_MAX - U16_MAX     # 142 528: with a 65 535-cell group the pair has exactly PAIR_MAX cells


def _boundary_case(test, big):
    """A big group of `big` cells (OVO: next to a BIG_CTRL-cell control); 8 genes (dense rows stay 16-byte aligned)."""
    rng = np.random.RandomState(big)
    if test == "ovo":
        sizes = {"ctrl": BIG_CTRL, "big": big, "a": 300, "b": 40}
    else:
        sizes = {"big": big, "a": 20000, "b": 3000, "c": 40}
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    in_big = labels == "big"
    X = np.zeros((n, 8), np.float32)
    X[:, 0] = rng.poisson(0.5, n)
    X[in_big, 0] = 3.0                                       # one value in every cell of the big group
    # genes 1, 2: the control (OVO) / the whole column (OVR) holds the value 1 exactly 65 535 / 65 536 times, among
    # >= 13 distinct integer values (the fused wide table keeps 16-bit multiplicities)
    host = np.flatnonzero(labels == "ctrl") if test == "ovo" else np.arange(n)
    for j, k in ((1, U16_MAX), (2, U16_MAX + 1)):
        X[:, j] = rng.randint(0, 20, n)
        X[host, j] = rng.randint(2, 20, host.size)
        X[rng.choice(host, k, replace=False), j] = 1.0
        assert np.count_nonzero(X[host, j] == 1.0) == k and np.unique(X[host, j]).size - 1 >= cap("DCAP") + 1
    X[:, 3] = rng.lognormal(0, 1, n) * (rng.rand(n) < 0.5)   # continuous
    X[:, 4] = rng.poisson(1.5, n)
    X[:, 5:] = rng.poisson(0.2, (n, 3))
    assert np.count_nonzero(X[in_big, 0]) == big and np.unique(X[in_big, 0]).size == 1
    if test == "ovo":   # gene 0 of the big group: ovo_kernel's table path (group < 65 536 cells) with a capped, recounted m
        c0 = X[labels == "ctrl", 0]
        assert np.unique(c0[c0 > 0]).size <= cap("DT_CAP")
    return X, labels


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
@pytest.mark.parametrize("big", [U16_MAX, U16_MAX + 1])
def test_sixteen_bit_counter_boundary(cuda_lib, monkeypatch, fmt, test, big):
    from illico_b200 import dispatch

    X, labels = _boundary_case(test, big)
    Xf = C.to_format(X, fmt)
    ref = "ctrl" if test == "ovo" else None
    want = oracle.run(Xf, labels, ref, want_ties=True)
    fused_var = "ILLICO_CSR_FUSED" if fmt == "csr" else f"ILLICO_{test.upper()}_FUSED"
    for seg in (512, U16_MAX):           # at U16_MAX the big group (65 535 cells) is one segment
        monkeypatch.setenv("ILLICO_B200_SEG_MAX", str(seg))
        monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
        dispatch.clear_caches()
        what = f"{fmt}:{test}:big={big}:seg={seg}"
        if fmt != "csc":
            monkeypatch.setenv(fused_var, "1")
            _run(Xf, labels, ref)
            ran = cuda_lib.illico_last_fused_ms() >= 0
            assert ran == (big <= U16_MAX), f"{what}: fused path ran={ran}"
        _check_against_oracle(fmt, test, X, labels, "ctrl", want=want, what=what)
        monkeypatch.setenv(fused_var, "0")
        Xg = _run(Xf, labels, ref)
        groups, p, U, fc, _ = want
        assert_parity(Xg, (p, U, fc), ref_row=int(np.searchsorted(groups, ref)) if ref else None,
                      what=f"{what} general path")
        monkeypatch.delenv(fused_var)
    dispatch.clear_caches()


# ---------------------------------------------------------------------------------------------------------------
# 6. rank-kernel tiers: one planted gene on each side of each cap (general path, debug integers against the oracle)

def _pool(k, seed):
    """k distinct positive float32 values (exact multiples of 1/16, in random order)."""
    v = (np.arange(1, k + 1) / 16.0 + 0.5).astype(np.float32)
    return np.random.RandomState(seed).permutation(v)


def _plant(col, cells, k, values, rng):
    """k of `cells` get `values` (cycled so that every value is used when k >= len(values)); the others stay 0."""
    pick = rng.choice(cells, k, replace=False)
    vals = np.resize(values, k) if k >= len(values) else rng.choice(values, k, replace=False)
    col[pick] = rng.permutation(vals)


def _ovo_tier_case():
    """control 4 000 cells, groups P (1 100 cells), Q (300) and 20 of 40.  One planted gene per (cap, side)."""
    rng = np.random.RandomState(606)
    sizes = {"ctrl": 4000, "P": 1100, "Q": 300, **{f"s{i:02d}": 40 for i in range(20)}}
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    ctrl, P, Q = (np.flatnonzero(labels == x) for x in ("ctrl", "P", "Q"))
    others = np.flatnonzero(labels != "ctrl")
    genes, names = [], []

    def gene(name, ctrl_nnz, ctrl_distinct, check):
        col = np.zeros(n, np.float32)
        pool = _pool(ctrl_distinct, len(genes))
        _plant(col, ctrl, ctrl_nnz, pool, rng)
        # other groups: values of the control's pool (ties with it) and some it lacks, a few non-zeros each
        extra = pool[-1] + 0.25 + np.arange(1, 9, dtype=np.float32) / 4
        for g in np.unique(labels[others]):
            cells = np.flatnonzero(labels == g)
            k = min(cells.size, 6)
            _plant(col, cells, k, np.concatenate([pool[:3], extra[:1]]), rng)
        check(col)
        genes.append(col)
        names.append(name)
        return col

    def distinct(v):
        return np.unique(v[v != 0]).size

    REF_CAP, DT_CAP, NE_CAP, ST_CAP = cap("REF_CAP"), cap("DT_CAP"), cap("NE_CAP"), cap("ST_CAP")
    for k in (REF_CAP, REF_CAP + 1):          # control non-zeros: sorted in shared memory / in the CTA's slab
        gene(f"REF_CAP:{k}", k, k, lambda c, k=k: (np.count_nonzero(c[ctrl]) == k and distinct(c[ctrl]) == k) or
             pytest.fail("REF_CAP gene"))
    for d in (DT_CAP, DT_CAP + 1):            # distinct control values: table path or not
        gene(f"DT_CAP:{d}", 3000, d, lambda c, d=d: distinct(c[ctrl]) == d or pytest.fail("DT_CAP gene"))
    for e in (NE_CAP, NE_CAP + 1):            # values of group Q the control lacks, on the table path
        col = gene(f"NE_CAP:{e}", 3000, 10, lambda c: None)
        col[Q] = 0
        absent = (_pool(10, 99)[:e] + 100.0).astype(np.float32)
        _plant(col, Q, 60, np.concatenate([absent, col[ctrl][col[ctrl] > 0][:5]]), rng)
        assert distinct(col[ctrl]) <= DT_CAP
        assert np.setdiff1d(col[Q][col[Q] > 0], col[ctrl]).size == e, "NE_CAP gene"
    for d in (ST_CAP, ST_CAP + 1):            # distinct control values of the search table: hashed (> REF_CAP nnz) ...
        gene(f"ST_CAP:hashed:{d}", REF_CAP + 1000, d, lambda c, d=d: (distinct(c[ctrl]) == d and
             np.count_nonzero(c[ctrl]) > REF_CAP) or pytest.fail("ST_CAP hashed gene"))
    for d in (ST_CAP, ST_CAP + 1):            # ... and sorted (<= REF_CAP non-zeros) branch
        gene(f"ST_CAP:sorted:{d}", REF_CAP - 100, d, lambda c, d=d: (distinct(c[ctrl]) == d and
             np.count_nonzero(c[ctrl]) <= REF_CAP) or pytest.fail("ST_CAP sorted gene"))
    W = cap("WARP_CAP")
    for m in (cap("STREAM_MAX"), cap("STREAM_MAX") + 1, W // 2, W // 2 + 1, W, W + 1):   # non-zeros of group P
        col = gene(f"group_nnz:{m}", 2000, 200, lambda c: None)
        col[P] = 0
        _plant(col, P, m, np.concatenate([col[ctrl][col[ctrl] > 0][:150], _pool(400, 7) + 50]), rng)
        assert np.count_nonzero(col[P]) == m and distinct(col[ctrl]) > DT_CAP
        assert max(np.count_nonzero(col[labels == g]) for g in np.unique(labels) if g not in ("ctrl", "P")) <= cap("STREAM_MAX")
    return np.stack(genes, axis=1), labels, names


def _ovr_tier_case():
    """70 000 cells in 30 groups; a 300-cell group W.  One planted gene per (cap, side)."""
    rng = np.random.RandomState(707)
    sizes = {"W": 300, **{f"g{i:02d}": 2323 for i in range(29)}}
    sizes["g00"] += 70000 - sum(sizes.values())
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    W = np.flatnonzero(labels == "W")
    genes, names = [], []
    T_CAP, MD, HC = cap("T_CAP"), cap("MAX_DISTINCT"), cap("HASH_CAP")
    for d in (T_CAP, T_CAP + 1):              # distinct values of a gene: table kernel or not
        col = np.zeros(n, np.float32)
        _plant(col, np.arange(n), 30000, _pool(d, d), rng)
        assert np.unique(col[col > 0]).size == d
        genes.append(col), names.append(f"T_CAP:{d}")
    for k in (U8_MAX, U8_MAX + 1):            # stored values in one segment (group W = one segment at length 512)
        col = np.zeros(n, np.float32)
        _plant(col, np.flatnonzero(labels != "W"), 5000, _pool(6, 1), rng)
        _plant(col, W, k, _pool(6, 1), rng)
        assert np.count_nonzero(col[W]) == k and np.unique(col[col > 0]).size <= T_CAP
        genes.append(col), names.append(f"seg_records:{k}")
    for d in (MD, MD + 1):                    # distinct values: histogram path or path S
        col = np.zeros(n, np.float32)
        _plant(col, np.arange(n), 3 * d, _pool(d, d), rng)
        assert np.unique(col[col > 0]).size == d
        genes.append(col), names.append(f"MAX_DISTINCT:{d}")
    for k in (HC, HC + 1, U16_MAX, U16_MAX + 1):   # gene non-zeros (all distinct): shared sort / slab / bucket index
        col = np.zeros(n, np.float32)
        _plant(col, np.arange(n), k, _pool(k, k), rng)
        assert np.count_nonzero(col) == k and np.unique(col[col > 0]).size == k > MD
        genes.append(col), names.append(f"gene_nnz:{k}")
    return np.stack(genes, axis=1), labels, names


def _tier_check(monkeypatch, fmt, test, X, labels, ref, names, seg=512):
    from illico_b200 import dispatch

    monkeypatch.setenv("ILLICO_B200_SEG_MAX", str(seg))
    for var in ("ILLICO_OVO_FUSED", "ILLICO_OVR_FUSED", "ILLICO_CSR_FUSED"):
        monkeypatch.setenv(var, "0")
    dispatch.clear_caches()
    Xf = C.to_format(X, fmt)
    r = ref if test == "ovo" else None
    groups, p, U, fc, ties = oracle.run(Xf, labels, r, want_ties=True)
    ref_row = int(np.searchsorted(groups, r)) if r is not None else None
    got, dbg = _debug(fmt, test, Xf, labels, r)
    for j, name in enumerate(names):
        sl = (slice(None), slice(j, j + 1))
        assert_parity(tuple(a[sl] for a in got), (p[sl], U[sl], fc[sl]), ref_row=ref_row, what=f"{test} {name}")
        d = {k: v[..., j:j + 1] for k, v in dbg.items()}
        _assert_exact(d, U[sl], ties[..., j:j + 1], ref_row, f"{fmt}:{test}:seg={seg} {name}")
    assert_parity(_run(Xf, labels, r), (p, U, fc), ref_row=ref_row, what=f"{fmt}:{test} general path")
    dispatch.clear_caches()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_ovo_kernel_tiers_at_their_caps(cuda_lib, monkeypatch, fmt):
    X, labels, names = _ovo_tier_case()
    _tier_check(monkeypatch, fmt, "ovo", X, labels, "ctrl", names)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_ovr_kernels_at_their_caps(cuda_lib, monkeypatch, fmt):
    X, labels, names = _ovr_tier_case()
    _tier_check(monkeypatch, fmt, "ovr", X, labels, None, names)


@pytest.mark.gpu
@pytest.mark.parametrize("n_multi", ["T_MULTI", "T_MULTI+1"])
def test_ovr_table_kernel_multi_segment_groups(cuda_lib, monkeypatch, n_multi):
    """At segment length 7 every group of 8 cells has two segments: T_MULTI of them go to whole warps, more are ranked
    inline by their thread."""
    rng = np.random.RandomState(808)
    k = cap("T_MULTI") + (1 if n_multi.endswith("+1") else 0)
    sizes = {**{f"m{i:03d}": 8 for i in range(k)}, **{f"s{i:02d}": 5 for i in range(20)}}
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    X = np.stack([rng.poisson(lam, n) * (rng.rand(n) < 0.7) for lam in (0.5, 2.0, 6.0)], axis=1).astype(np.float32)
    assert all(np.unique(X[:, j][X[:, j] > 0]).size <= cap("T_CAP") for j in range(X.shape[1]))
    assert sum(1 for g, s in sizes.items() if s > 7) == k
    _tier_check(monkeypatch, "dense", "ovr", X, labels, None, ["lam0.5", "lam2", "lam6"], seg=7)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_fused_narrow_table_cap(cuda_lib, monkeypatch, fmt, test):
    """Genes whose control (OVO) / whole column (OVR) has DCAP or DCAP + 1 distinct values: the fused pass runs, and
    its results match the general path and the oracle."""
    from illico_b200 import dispatch

    rng = np.random.RandomState(909)
    sizes = {"ctrl": 3000, **{f"p{i:02d}": 100 for i in range(30)}}
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    n = labels.size
    D = cap("DCAP")
    X = np.zeros((n, 8), np.float32)
    for j, d in enumerate((D, D + 1, D, D + 1)):
        X[:, j] = (rng.randint(0, d + 1, n) * (1 if j < 2 else 1.5)).astype(np.float32)   # integers (wide) / not
    X[:, 4:] = rng.poisson(0.4, (n, 4))
    host = labels == "ctrl" if test == "ovo" else np.ones(n, bool)
    for j, d in enumerate((D, D + 1, D, D + 1)):
        assert np.unique(X[host, j][X[host, j] > 0]).size == d
    Xf = C.to_format(X, fmt)
    ref = "ctrl" if test == "ovo" else None
    groups, p, U, fc = oracle.run(Xf, labels, ref)
    ref_row = int(np.searchsorted(groups, ref)) if ref else None
    var = "ILLICO_CSR_FUSED" if fmt == "csr" else f"ILLICO_{test.upper()}_FUSED"
    monkeypatch.delenv("ILLICO_B200_SEG_MAX", raising=False)
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
    monkeypatch.setenv(var, "1")
    fused = _run(Xf, labels, ref)
    assert cuda_lib.illico_last_fused_ms() >= 0, "the fused pass did not run"
    monkeypatch.setenv(var, "0")
    general = _run(Xf, labels, ref)
    for got, route in ((fused, "fused"), (general, "general")):
        assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{fmt}:{test} {route}")
    dispatch.clear_caches()
