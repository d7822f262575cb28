"""Input that is not float32, on every kernel route, against the float64 oracle.

Every real dtype is converted on upload (``illico_convert_values``); a matrix that float32 cannot hold exactly keeps a
float64 copy, and each of its gene batches is recoded on the device to order-preserving float32 codes, with the fold
change taken from float64 group sums (``illico_flags_t::group_sums``).  The tests below plant values at the edges of that
conversion and run the recoded codes through every route of the dispatchers: the dense fused narrow and wide passes, the
CSR fused pass, genes handed back one by one or as a whole batch, the general rank kernels, and the sub-batches of
``Engine._run_batch_wide``.  Every run is compared with ``oracle.run`` on the same values widened to float64: U bit for
bit, p within 1e-12, the fold change within 1e-10 (also with ``is_log1p``: the oracle takes ``expm1`` in float64), and,
through the debug outputs, the exact 2U and tie sums."""
import numpy as np
import pytest

import oracle
from tests.golden import cases as C
from tests.parity import assert_parity
from tests.test_limits import _assert_exact
from tests.test_rank_genes import score_reference
from tests.util import FakeAnnData, planes

FLT_MAX = float(np.finfo(np.float32).max)
DCAP, DW = 12, 64          # fused.cu: narrow table slots per gene, largest count of the wide table


def _widen(Xf):
    """The same matrix with float64 values (what the oracle is given)."""
    if isinstance(Xf, np.ndarray):
        return Xf.astype(np.float64)
    Y = Xf.copy()
    Y.data = Y.data.astype(np.float64)
    return Y


def _inexact(a) -> bool:
    """float32 changes some (non-NaN) value of ``a``."""
    x = np.asarray(a, dtype=np.float64).ravel()
    x = x[~np.isnan(x)]
    with np.errstate(over="ignore"):
        return bool(np.any(x.astype(np.float32).astype(np.float64) != x))


def _labels(sizes, rng):
    labels = np.repeat(np.array(list(sizes)), list(sizes.values()))
    rng.shuffle(labels)
    return labels


# ============================================ CPU ==============================================================

def test_host_widens_dtypes_torch_cannot_hold():
    from illico_b200.engine import _uploadable

    a = np.array([0, 1, 7, 200], dtype=np.uint8)
    for dt, want in ((np.uint16, np.int64), (np.uint32, np.int64), (np.uint64, np.float64), (np.bool_, np.float64)):
        w = _uploadable(a.astype(dt))
        assert w.dtype == want, dt
        np.testing.assert_array_equal(w, a.astype(dt).astype(want))
    for dt in (np.float32, np.float64, np.float16, np.int8, np.uint8, np.int16, np.int32, np.int64):
        x = a.astype(dt)
        assert _uploadable(x) is x, dt


# ---------------------------------------------------------------------------------------------------------------
# the planted route matrix: one gene column per route of the fused and general paths

N_ROUTE_GENES = 256
WHOLE_BATCH_FROM = 224      # genes 224 .. 255 are continuous: a batch holding them is handed back whole


def _route_case(fmt):
    """3 000 cells x 256 genes of float64 values float32 cannot hold (log1p(k), k / 10).  Per block of 16 genes:
    r 0-5, 13, 14: <= 12 distinct positive values (narrow table; r 13: values the control lacks);
    r 6-10, 15: 13-64 distinct positive values (wide table);
    r 11: an edge gene, rotating over all zero / constant / a single non-zero / control all zero;
    r 12: continuous (> 64 distinct values) or, dense only, signed -- handed back one by one (1 gene in 16).
    Genes 224-255 are continuous, so any batch holding them is handed back whole.  Continuous values stay below 3:
    with log1p, no group holds nearly all of a gene's expm1 sum (one-versus-rest takes the rest as total - sum)."""
    rng = np.random.RandomState(4242)
    labels = _labels({"ctrl": 1200, **{f"p{i:02d}": 150 for i in range(12)}}, rng)
    n = labels.size
    ctrl = labels == "ctrl"
    X = np.zeros((n, N_ROUTE_GENES))
    kinds = []
    for j in range(N_ROUTE_GENES):
        r, blk = j % 16, j // 16
        val = np.log1p if j % 2 == 0 else (lambda k: k / 10.0)
        mask = rng.rand(n)
        if j >= WHOLE_BATCH_FROM:
            kind, col = "continuous", rng.uniform(0.05, 3.0, n) * (mask < 0.7)
        elif r in (0, 1, 2, 3, 4, 5, 13, 14):
            kind = "narrow"
            k = rng.randint(1, 9, n) * (mask < 0.4) if r != 14 else np.minimum(rng.poisson(0.5, n), 8)
            if r == 13:
                k[ctrl] = np.minimum(k[ctrl], 5)
            col = val(k.astype(np.float64))
        elif r in (6, 7, 8, 9, 10, 15):
            kind = "wide"
            k = rng.randint(1, 41, n) * (mask < 0.6) if r != 15 else np.minimum(rng.poisson(14.0, n), DW)
            col = val(k.astype(np.float64))
        elif r == 11:
            kind = ("zero", "constant", "single", "ctrl_zero")[blk % 4]
            col = np.zeros(n)
            if kind == "constant":
                col[:] = 0.3
            elif kind == "single":
                col[(blk * 7) % n] = 0.7
            elif kind == "ctrl_zero":
                col = val(rng.randint(1, 6, n) * (mask < 0.5).astype(np.float64))
                col[ctrl] = 0.0
        elif blk % 2 == 0 or fmt != "dense":
            kind, col = "continuous", rng.uniform(0.05, 3.0, n) * (mask < 0.6)
        else:
            kind = "signed"
            col = np.log1p(rng.randint(1, 9, n) * (mask < 0.5).astype(np.float64))
            neg = rng.rand(n) < 0.05
            col[neg] = -np.log1p(rng.randint(1, 4, neg.sum()).astype(np.float64))
        X[:, j] = col
        kinds.append(kind)
    return X, labels, kinds


@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_route_case_plants_what_it_claims(fmt):
    X, labels, kinds = _route_case(fmt)
    ctrl = labels == "ctrl"
    assert _inexact(X) and X.dtype == np.float64
    assert fmt == "dense" or (X >= 0).all()
    for j, kind in enumerate(kinds):
        x = X[:, j]
        d = np.unique(x[x > 0]).size
        if kind == "narrow":
            assert 1 <= d <= DCAP and _inexact(x), j
        elif kind == "wide":
            assert DCAP < d <= DW and np.unique(x[ctrl & (x > 0)]).size > DCAP and _inexact(x), j
        elif kind == "continuous":
            assert np.unique(x[x != 0]).size > DW, j
        elif kind == "signed":
            assert (x < 0).any() and x[x > 0].sum() > -5 * x[x < 0].sum(), j   # (group sums far from 0)
        elif kind == "zero":
            assert not x.any()
        elif kind == "constant":
            assert np.unique(x).size == 1 and x[0] != 0
        elif kind == "single":
            assert np.count_nonzero(x) == 1
        else:
            assert not x[ctrl].any() and x[~ctrl].any()
    # every batch of 64 / 86 genes below gene 224 hands back fewer than an eighth of its genes one by one
    flagged = np.array([k in ("continuous", "signed") for k in kinds])
    for width in (64, 86):
        for lb in range(0, N_ROUTE_GENES, width):
            share = flagged[lb:lb + width].mean()
            assert share > 1 / 8 if lb + width > WHOLE_BATCH_FROM else share < 1 / 8, (width, lb)
    assert {"narrow", "wide", "continuous", "zero", "constant", "single", "ctrl_zero"} <= set(kinds)
    assert fmt != "dense" or "signed" in kinds


def _f64_only_case(fmt):
    """Values that are distinct only in float64 (float32 would tie them), 1 400 cells x 6 genes:
    0, 1: pairs x / nextafter(x, inf) split across groups, near 1 and near 2^30;
    2: subnormal doubles in group a, where the other groups have zeros;
    3: values above FLT_MAX (1e39, 1e300, the double after FLT_MAX) and +inf;
    4: -0.0 and negative subnormals among zeros and positives (sparse: their absolute values);
    5: a narrow count gene (log1p)."""
    rng = np.random.RandomState(77)
    labels = _labels({"ctrl": 600, "a": 300, "b": 300, "c": 200}, rng)
    n = labels.size
    g = {k: labels == k for k in ("ctrl", "a", "b", "c")}
    X = np.zeros((n, 6))
    for j, base in ((0, 1.0), (1, 2.0 ** 30)):
        x = base + rng.randint(1, 6, n) / 3.0
        X[:, j] = np.where(g["a"], np.nextafter(x, np.inf), x)
        X[g["c"], j] = np.nextafter(x[g["c"]], -np.inf)
        X[rng.rand(n) < 0.3, j] = 0.0
    sub = np.array([5e-324, 1e-310, 2.5e-320, 2.2250738585072e-308])
    X[:, 2] = np.where(rng.rand(n) < 0.3, 1.0, 0.0)
    X[g["b"], 2] *= 2.0
    pick = g["a"] & (rng.rand(n) < 0.5)
    X[pick, 2] = rng.choice(sub, pick.sum())
    big = np.array([1e39, 1e300, np.nextafter(FLT_MAX, np.inf), 1.0])
    X[:, 3] = rng.choice(big, n) * (rng.rand(n) < 0.6)
    X[np.flatnonzero(g["a"])[:5], 3] = np.inf
    X[:, 4] = np.where(rng.rand(n) < 0.4, 0.5, 0.0)
    X[rng.rand(n) < 0.3, 4] = -0.0
    X[g["c"] & (rng.rand(n) < 0.2), 4] = -1e-310
    X[:, 5] = np.log1p(np.minimum(rng.poisson(0.8, n), 8).astype(np.float64))
    if fmt != "dense":
        X = np.abs(X)
    return X, labels


def test_float64_only_values_would_tie_in_float32():
    """The planted values matter: rounded to float32, genes 0-3 would rank differently (U changes)."""
    X, labels = _f64_only_case("dense")
    with np.errstate(over="ignore"):
        X32 = X.astype(np.float32)
    _, _, U64, _ = oracle.run(X, labels, "ctrl")
    _, _, U32, _ = oracle.run(X32, labels, "ctrl")
    for j in range(4):
        assert not np.array_equal(U64[:, j], U32[:, j]), j
    assert np.signbit(X[:, 4]).any() and (X[:, 2][X[:, 2] > 0] < 1e-300).any() and np.isposinf(X[:, 3]).any()


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


@pytest.fixture
def profile(monkeypatch, cuda_lib):
    """``report()`` -> {kernel name: (ms, launches)} of the launches since the previous ``report()``."""
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_PROFILE", "1")
    _lib.profile_report()
    return _lib.profile_report


def _run(X, labels, reference, **kw):
    from illico_b200 import asymptotic_wilcoxon

    groups = np.unique(np.asarray(labels))
    df = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=reference, **kw)
    return planes(df, len(groups), X.shape[1])


def _debug(fmt, test, Xf, labels, reference, kw):
    """(p, U, fc) and the debug integers {u2, tie_sum, tie_exact} of the dispatcher (general path)."""
    from illico_b200 import dispatch
    from illico_b200.groups import encode_and_count_groups

    _, grpc = encode_and_count_groups(labels, reference)
    fn = getattr(dispatch, f"{fmt}_{test}_mwu_kernel_over_contiguous_col_chunk")
    dbg = {}
    got = fn(Xf, 0, Xf.shape[1], grpc, kw.get("is_log1p", False), kw.get("use_continuity", True), kw.get("tie_correct", True),
             kw.get("alternative", "two-sided"), debug=dbg)
    return got, {k: v.cpu().numpy() for k, v in dbg.items()}


def _want(Xf, labels, ref, **kw):
    groups, p, U, fc, ties = oracle.run(_widen(Xf), labels, ref, want_ties=True, **kw)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    return (p, U, fc), ties, ref_row


def _check(Xf, labels, ref, fmt, test, what, kw, want=None):
    """Default route and the debug integers against the oracle."""
    kw = {"is_log1p": False, **kw}
    (p, U, fc), ties, ref_row = want or _want(Xf, labels, ref, **kw)
    assert_parity(_run(Xf, labels, ref, **kw), (p, U, fc), ref_row=ref_row, what=f"{what} default route")
    got, dbg = _debug(fmt, test, Xf, labels, ref, kw)
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{what} debug call")
    _assert_exact(dbg, U, ties, ref_row, what)


def _recoded(rep) -> bool:
    return any(k.startswith("wide_collect_") for k in rep)


# ---------------------------------------------------------------------------------------------------------------
# a. illico_convert_values against numpy

LONG = 1_000_003           # not a multiple of the 256-thread block, longer than one pass of the grid


def _convert_cases(name):
    """(case, host array) pairs of dtype `name`; specials are planted at the front, the inexact one at the very end."""
    rng = np.random.RandomState(len(name))
    dt = np.dtype(name)
    if dt.kind == "f":
        base = (rng.randint(-4000, 4000, LONG) / 4.0).astype(dt)
    else:
        info = np.iinfo(dt)
        base = rng.randint(max(info.min, -100), min(info.max, 100) + 1, LONG).astype(dt)
    out = [("plain", base)]
    if name == "float64":
        exact = base.copy()
        exact[:9] = [np.inf, -np.inf, np.nan, -0.0, FLT_MAX, -FLT_MAX, 2.0 ** -149, 2.0 ** -126, 2.0 ** 24 + 2]
        out.append(("specials_exact", exact))
        for case, v in (("inexact_last", 0.1), ("subnormal_last", 1e-310), ("neg_subnormal_last", -5e-324),
                        ("above_flt_max_last", 1e39), ("far_above_last", -1e300),
                        ("after_flt_max_last", np.nextafter(FLT_MAX, np.inf))):
            a = exact.copy()
            a[-1] = v
            out.append((case, a))
    elif name == "float32":
        a = base.copy()
        a[:6] = [np.inf, -np.inf, np.nan, -0.0, np.float32(1e-45), np.finfo(np.float32).max]
        out.append(("specials", a))
    elif name == "float16":
        a = base.copy()
        a[:7] = [np.inf, -np.inf, np.nan, -0.0, np.float16(2.0 ** -24), np.float16(-3 * 2.0 ** -24), np.finfo(np.float16).max]
        a[-1] = np.float16(5 * 2.0 ** -24)                      # float16 subnormals are exact in float32
        out.append(("specials_subnormal", a))
    elif name in ("int32", "int64"):
        a = base.copy()
        a[:2] = [2 ** 24, -(2 ** 24)]
        out.append(("two_pow_24", a))
        b = a.copy()
        b[-1] = 2 ** 24 + 1
        out.append(("two_pow_24_plus_1_last", b))
        c = a.copy()
        c[-1] = -(2 ** 24 + 1)
        out.append(("minus_two_pow_24_plus_1_last", c))
        if name == "int64":
            d = a.copy()
            d[:2] = [2 ** 40, -(2 ** 52)]
            out.append(("big_exact", d))
            d = d.copy()
            d[-1] = 2 ** 40 + 1
            out.append(("big_inexact_last", d))
    else:
        info = np.iinfo(dt)
        a = base.copy()
        a[:2] = [info.min, info.max]
        out.append(("extremes", a))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["float32", "float64", "float16", "int8", "uint8", "int16", "int32", "int64"])
def test_convert_values_matches_numpy(cuda_lib, name):
    import torch

    from illico_b200 import _lib
    from illico_b200.engine import _DTYPE_CODE

    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    for case, a in _convert_cases(name):
        src = torch.from_numpy(a).to(dev)
        code = _DTYPE_CODE[src.dtype]
        f = torch.empty(a.size, dtype=torch.float32, device=dev)
        d = torch.empty(a.size, dtype=torch.float64, device=dev)
        flag = torch.full((1,), 7, dtype=torch.int32, device=dev)
        _lib.check(cuda_lib.illico_convert_values(src.data_ptr(), code, a.size, f.data_ptr(), d.data_ptr(), flag.data_ptr(), st),
                   "illico_convert_values")
        got32, got64, verdict = f.cpu().numpy(), d.cpu().numpy(), int(flag.item())
        with np.errstate(over="ignore"):
            want32, want64 = a.astype(np.float32), a.astype(np.float64)
        what = f"{name}:{case}"
        nan = np.isnan(want64)
        np.testing.assert_array_equal(np.isnan(got32), nan, err_msg=what)
        np.testing.assert_array_equal(np.isnan(got64), nan, err_msg=what)
        np.testing.assert_array_equal(got32[~nan].view(np.uint32), want32[~nan].view(np.uint32), err_msg=f"{what}: float32 bits")
        np.testing.assert_array_equal(got64[~nan].view(np.uint64), want64[~nan].view(np.uint64), err_msg=f"{what}: float64 bits")
        assert _inexact(want64) == case.endswith("_last"), f"{what}: the case does not plant what it says"
        assert verdict == int(case.endswith("_last")), f"{what}: exactness verdict {verdict}"
    # a count of 0 converts nothing and leaves the verdict at 0
    flag = torch.full((1,), 7, dtype=torch.int32, device=dev)
    src = torch.zeros(4, dtype=torch.float64, device=dev)
    f = torch.empty(4, dtype=torch.float32, device=dev)
    _lib.check(cuda_lib.illico_convert_values(src.data_ptr(), _lib.DTYPE_F64, 0, f.data_ptr(), None, flag.data_ptr(), st),
               "illico_convert_values")
    assert int(flag.item()) == 0


# ---------------------------------------------------------------------------------------------------------------
# b. every kernel route under recoding

ROUTE_CASES = [(fmt, test, log1p) for fmt in ("dense", "csr", "csc") for test in ("ovo", "ovr") for log1p in (False, True)]


def _bitwise_same(a, b, rows, what):
    np.testing.assert_array_equal(a[1], b[1], err_msg=f"{what}: U")
    np.testing.assert_array_equal(a[0][rows], b[0][rows], err_msg=f"{what}: p")
    np.testing.assert_allclose(a[2][rows], b[2][rows], rtol=1e-13, atol=0, err_msg=f"{what}: fold change")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,test,log1p", ROUTE_CASES)
def test_every_kernel_route_under_recoding(monkeypatch, profile, fmt, test, log1p):
    """Batches of 64 genes (16-byte aligned code rows) and of 86 (padded rows: every batch, not only the last one of 84
    genes, must reach the fused pass).  Dense one-versus-reference runs the
    narrow and (without log1p) wide fused passes with genes handed back; CSR one-versus-reference the CSR fused pass;
    one-versus-rest the general path (its fused path and ovr_table_kernel do not take group sums).  Each fused run
    equals the same call with the fused path off, p and U bit for bit."""
    from illico_b200 import dispatch

    i = ROUTE_CASES.index((fmt, test, log1p))
    kw = dict(is_log1p=log1p, alternative=C.ALTERNATIVES[i % 3], use_continuity=i % 2 == 0, tie_correct=(i // 2) % 3 != 2)
    X, labels, kinds = _route_case(fmt)
    Xf = C.to_format(X, fmt)
    ref = "ctrl" if test == "ovo" else None
    want = _want(Xf, labels, ref, **kw)
    (p, U, fc), _, ref_row = want
    rows = np.arange(U.shape[0]) != (ref_row if ref_row is not None else -1)
    fused_var = "ILLICO_CSR_FUSED" if fmt == "csr" else f"ILLICO_{test.upper()}_FUSED"
    fused_kernel = {"dense": "fused_pass_kernel", "csr": "fused_csr_pass_kernel"}.get(fmt) if test == "ovo" else None
    dispatch.clear_caches()
    # default hand-back share (an eighth: the batch holding genes 224-255 goes back whole), then every flagged gene
    # handed back one by one (the CSR pass flags the 13-64 value genes, which would otherwise send every batch back)
    for batch, share in ((64, None), (86, "1.0")):
        if share is not None:
            monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", share)
        what = (f"{fmt}:{test}:log1p={log1p}:batch={batch}:share={share}:{kw['alternative']}:cc={kw['use_continuity']}"
                f":tc={kw['tie_correct']}")
        got = _run(Xf, labels, ref, batch_size=batch, **kw)
        rep = profile()
        assert_parity(got, (p, U, fc), ref_row=ref_row, what=what)
        assert f"wide_collect_{fmt}_kernel" in rep, f"{what}: not recoded: {sorted(rep)}"
        if test == "ovr":
            assert "ovr_kernel" in rep and "ovr_table_kernel" not in rep, f"{what}: {sorted(rep)}"
        if fused_kernel is None:
            continue
        n_batches = -(-N_ROUTE_GENES // batch)
        assert rep.get(fused_kernel, (0, 0))[1] == n_batches, f"{what}: {fused_kernel} did not run on every batch: {rep}"
        assert "ovo_kernel" in rep, f"{what}: no gene was handed back"
        if fmt == "dense":
            assert ("fused_wide_pass_kernel" in rep) == (not log1p), f"{what}: {sorted(rep)}"
            if not log1p:
                monkeypatch.setenv("ILLICO_FUSED_WIDE", "0")
                narrow = _run(Xf, labels, ref, batch_size=batch, **kw)
                monkeypatch.delenv("ILLICO_FUSED_WIDE")
                rep = profile()
                assert "fused_pass_kernel" in rep and "fused_wide_pass_kernel" not in rep, f"{what}: {sorted(rep)}"
                _bitwise_same(narrow, got, rows, f"{what} narrow pass only")
        monkeypatch.setenv(fused_var, "0")
        general = _run(Xf, labels, ref, batch_size=batch, **kw)
        monkeypatch.delenv(fused_var)
        rep = profile()
        assert fused_kernel not in rep, f"{what}: the fused path was not turned off"
        _bitwise_same(got, general, rows, f"{what} fused vs general path")
    if fmt == "csr" and test == "ovo":
        # The CSR pass has no wide table: it flags the 13-64 value genes, and a pass that flags more than an eighth of a
        # batch stops early and hands the whole batch back.  Without them (and the continuous genes) the pass keeps its
        # own results, which must be the oracle's and the general path's.
        monkeypatch.delenv("ILLICO_FUSED_LIST_SHARE")
        cols = [j for j, k in enumerate(kinds) if k not in ("wide", "continuous")]
        what = f"{fmt}:{test}:log1p={log1p}: narrow genes"
        got = _run(Xf[:, cols], labels, ref, batch_size=86, **kw)
        rep = profile()
        assert rep.get(fused_kernel, (0, 0))[1] == -(-len(cols) // 86), f"{what}: {rep}"
        assert_parity(got, (p[:, cols], U[:, cols], fc[:, cols]), ref_row=ref_row, what=what)
        monkeypatch.setenv(fused_var, "0")
        general = _run(Xf[:, cols], labels, ref, batch_size=86, **kw)
        monkeypatch.delenv(fused_var)
        _bitwise_same(got, general, rows, f"{what} fused vs general path")
    got, dbg = _debug(fmt, test, Xf, labels, ref, kw)
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{fmt}:{test}:log1p={log1p} debug call")
    _assert_exact(dbg, U, want[1], ref_row, f"{fmt}:{test}:log1p={log1p}")
    dispatch.clear_caches()


# ---------------------------------------------------------------------------------------------------------------
# c. float64 values distinct only in float64 must not become ties

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_values_distinct_only_in_float64(profile, fmt, test):
    X, labels = _f64_only_case(fmt)
    Xf = C.to_format(X, fmt)
    ref = "ctrl" if test == "ovo" else None
    _check(Xf, labels, ref, fmt, test, f"{fmt}:{test} float64-only values", {})
    assert f"wide_collect_{fmt}_kernel" in profile()


# ---------------------------------------------------------------------------------------------------------------
# d. every dtype end to end

DTYPE_CASES = ["float16", "int8", "uint8", "int16", "int32", "int32_above_2_24", "int64", "uint16", "uint32", "uint64", "bool",
               "float64_exact", "float64_one_inexact"]
RECODED = {"int32_above_2_24", "float64_one_inexact"}


def _dtype_case(name):
    """2 500 cells x 12 genes of dtype `name`; gene 0 holds the dtype's edge values."""
    rng = np.random.RandomState(DTYPE_CASES.index(name))
    labels = _labels({"ctrl": 700, **{f"p{i}": 300 for i in range(6)}}, rng)
    n = labels.size
    k = rng.poisson(1.5, (n, 12)) * (rng.rand(n, 12) < 0.6)
    if name == "float16":
        X = (k * 0.5).astype(np.float16)
        X[:, 0] = (k[:, 0] * 2.0 ** -24).astype(np.float16)                  # float16 subnormals
        assert np.all(np.abs(X[:, 0][X[:, 0] != 0]) < np.finfo(np.float16).tiny)
    elif name == "int8":
        X = (k - 2 * (rng.rand(n, 12) < 0.1)).astype(np.int8)                # a few negative values (dense only)
        X[:3, 0] = [-128, 127, -1]
    elif name == "uint8":
        X = np.minimum(k * 40, 255).astype(np.uint8)
    elif name == "int16":
        X = (k * 1000).astype(np.int16)
        X[0, 0] = 32767
    elif name == "int32":
        X = (k * 3).astype(np.int32)
    elif name == "int32_above_2_24":
        X = np.where(k > 0, 2 ** 24 + k, 0).astype(np.int32)                 # 2^24 + odd: float32 cannot hold them
    elif name == "int64":
        X = (k * 7).astype(np.int64)
        X[0, 0] = 2 ** 24
    elif name == "uint16":
        X = (k * 300).astype(np.uint16)
    elif name == "uint32":
        X = (k * 70000).astype(np.uint32)
    elif name == "uint64":
        X = (k * 11).astype(np.uint64)
    elif name == "bool":
        X = k > 0
    else:
        X = k * 0.25
        if name == "float64_one_inexact":
            X[np.flatnonzero(X[:, 5])[0], 5] = 0.1                           # one value flips the matrix to recoding
    assert _inexact(X) == (name in RECODED)
    return X, labels


@pytest.mark.gpu
@pytest.mark.parametrize("name", DTYPE_CASES)
def test_every_dtype_end_to_end(profile, name):
    from illico_b200 import dispatch

    X, labels = _dtype_case(name)
    formats = ["dense"] if name in ("float16", "int8") else ["dense", "csr", "csc"]
    for fmt in formats:
        Xf = C.to_format(X, fmt)
        assert Xf.dtype == X.dtype
        for test in ("ovo", "ovr"):
            ref = "ctrl" if test == "ovo" else None
            dispatch.clear_caches()
            _check(Xf, labels, ref, fmt, test, f"{name}:{fmt}:{test}", {})
            rep = profile()
            assert "convert_values_kernel" in rep, f"{name}:{fmt}:{test}: no conversion"
            assert _recoded(rep) == (name in RECODED), f"{name}:{fmt}:{test}: recoded={_recoded(rep)}"
    dispatch.clear_caches()


# ---------------------------------------------------------------------------------------------------------------
# e. input routes: device-resident tensors, backed streaming (the verdict per batch), devices="all"

def _partly_inexact(rng, labels, n_genes, inexact_batches, width):
    """Counts as float64; the gene batches in `inexact_batches` (of `width` genes) hold k / 10 instead of k / 4."""
    n = labels.size
    k = (rng.poisson(2.0, (n, n_genes)) * (rng.rand(n, n_genes) < 0.5)).astype(np.float64)
    X = k / 4.0
    for bi in inexact_batches:
        X[:, bi * width:(bi + 1) * width] = k[:, bi * width:(bi + 1) * width] / 10.0
    return X


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["torch_float64", "torch_int32", "backed_dense", "backed_csc", "devices_all"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_input_routes_of_other_dtypes(tmp_path, profile, route, test):
    import torch
    from scipy import sparse

    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense

    rng = np.random.RandomState(31)
    labels = _labels({"ctrl": 900, **{f"p{i}": 250 for i in range(8)}}, rng)
    ref = "ctrl" if test == "ovo" else None
    width, n_genes = 16, 64
    X = _partly_inexact(rng, labels, n_genes, (1, 3), width)
    kw, recodes = {}, None
    if route == "torch_float64":
        Xin, Xo, recodes = torch.from_numpy(X).cuda(), X, ("wide_collect_dense_kernel", 1)
    elif route == "torch_int32":
        Xo = np.rint(X * 40).astype(np.int32)            # 10 k and 4 k: exact in float32
        Xin = torch.from_numpy(Xo).cuda()
    elif route == "backed_dense":
        save_dense(str(tmp_path / "d.bin"), X)
        Xin, Xo, kw, recodes = MemmapDense(str(tmp_path / "d.bin")), X, dict(batch_size=width, n_threads=3), ("wide_collect_dense_kernel", 2)
        assert Xin.dtype == np.float64
    elif route == "backed_csc":
        Xc = sparse.csc_matrix(X)
        save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
        Xin, Xo, kw, recodes = MemmapCSC(str(tmp_path / "csc")), Xc, dict(batch_size=width, n_threads=2), ("wide_collect_csc_kernel", 2)
    else:
        Xin, Xo, kw, recodes = X, X, dict(devices="all"), ("wide_collect_dense_kernel", None)
    (p, U, fc), _, ref_row = _want(Xo, labels, ref)
    got = _run(Xin, labels, ref, is_log1p=False, **kw)
    rep = profile()
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{route}:{test}")
    if recodes is None:
        assert not _recoded(rep), f"{route}: {sorted(rep)}"
    else:
        name, launches = recodes
        assert name in rep, f"{route}: not recoded: {sorted(rep)}"
        if launches is not None:   # backed: only the batches holding inexact values are recoded
            assert rep[name][1] == launches, f"{route}: {rep[name][1]} recoded batches"


# ---------------------------------------------------------------------------------------------------------------
# f. more than one sub-batch in Engine._run_batch_wide (2^26 keys per sub-batch)

@pytest.mark.gpu
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_recoded_dense_sub_batches(monkeypatch, profile, test):
    """70 000 cells x 1 000 genes of float64 log1p counts (560 MB): 2^26 // 70 000 = 958 genes per sub-batch, rounded
    down to 956, so every sub-batch starts on a 16-byte boundary and the dense fused path takes the recoded codes."""
    from illico_b200 import asymptotic_wilcoxon, dispatch
    from illico_b200.engine import DENSE, Engine
    from illico_b200.groups import encode_and_count_groups

    rng = np.random.RandomState(2026)
    n, N = 70_000, 1_000
    labels = _labels({"ctrl": 20_000, **{f"p{i:02d}": 1_250 for i in range(40)}}, rng)
    assert labels.size == n and ((1 << 26) // n) % 4 != 0
    X = np.log1p(np.minimum(rng.poisson(0.5, (n, N)), 8).astype(np.float64))
    X[:, 7] = rng.lognormal(0.0, 1.0, n) * (rng.rand(n) < 0.5)                # a gene handed back
    ref = "ctrl" if test == "ovo" else None
    groups, p, U, fc, ties = oracle.run(X, labels, ref, want_ties=True, n_threads=oracle.max_threads())
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None

    subs = []
    run_batch = Engine.run_batch

    def spy(self, M, lb, ub, *args, **kwargs):
        if M.fmt == DENSE and M.raw is None and M.unconverted is None and not M.pending:   # (a recoded sub-batch)
            subs.append((ub - lb, M.ld))
        return run_batch(self, M, lb, ub, *args, **kwargs)

    monkeypatch.setattr(Engine, "run_batch", spy)
    dispatch.clear_caches()
    g, _, out, extra = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=ref, is_log1p=False,
                                           score=True, return_array=True)
    rep = profile()
    what = f"{test}: sub-batches {subs}"
    assert len(subs) >= 2 and sum(w for w, _ in subs) == N, what
    assert all(w % 4 == 0 for w, _ in subs[:-1]) and all(ld % 4 == 0 and ld - w < 4 for w, ld in subs), what
    assert rep["wide_sort_kernel"][1] == len(subs), what
    if test == "ovo":
        assert "fused_pass_kernel" in rep, f"{what}: the fused pass did not run: {sorted(rep)}"
    assert_parity((out[:, :, 0], out[:, :, 1], out[:, :, 2]), (p, U, fc), ref_row=ref_row, what=what)
    _, grpc = encode_and_count_groups(labels, ref)
    np.testing.assert_array_equal(extra["score"], score_reference(U, ties, grpc.counts, ref_row, n, True), err_msg=what)
    subs.clear()
    got, dbg = _debug("dense", test, X, labels, ref, {})
    assert len(subs) >= 2, f"debug call: sub-batches {subs}"
    assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{what} debug call")
    _assert_exact(dbg, U, ties, ref_row, f"{test}: sub-batches put together")
    dispatch.clear_caches()
