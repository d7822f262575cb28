"""GPU parity tests: the CUDA path (through the public API and the C ABI) against the reference's golden
vectors and the CPU oracle.  Bars (BASELINE.json north_star): U and tie sums bit-exact, p-values within
relative 1e-12 (absolute 2.3e-308 for sub-normal p), fold change within relative 1e-10."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle  # noqa: E402
from tests.golden import cases as C  # noqa: E402
from tests.parity import FC_RTOL, FC_RTOL_LOG1P_F32, assert_parity  # noqa: E402
from tests.util import FakeAnnData, planes  # noqa: E402


@pytest.fixture(scope="module", autouse=True)
def _cuda_library_loaded():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from illico_b200 import _lib

    _lib.load()
    before = _lib.launch_count()
    yield
    assert _lib.launch_count() > before, "no kernel of libillico_b200.so was launched: native path not exercised"


def _run(X, labels, reference, **kw):
    from illico_b200 import asymptotic_wilcoxon

    groups = np.unique(np.asarray(labels))
    df = asymptotic_wilcoxon(FakeAnnData(X, labels), group_keys="pert", reference=reference, **kw)
    assert list(df.columns) == ["p_value", "statistic", "fold_change"]
    assert df.index.names == ["pert", "feature"] and len(df) == len(groups) * X.shape[1]
    return groups, planes(df, len(groups), X.shape[1])


@pytest.mark.parametrize("name", list(C.CASES))
def test_cuda_matches_reference_golden(golden_dir, name):
    builder, grid, batch_size = C.CASES[name]
    X, labels, reference = builder()
    gold = np.load(os.path.join(golden_dir, f"{name}.npz"))
    groups = gold["groups"]
    for fmt, test, cc, tc, alt, log1p in grid:
        ref = reference if test == "ovo" else None
        kw = dict(is_log1p=log1p, batch_size=batch_size, alternative=alt, use_continuity=cc, tie_correct=tc)
        g, got = _run(C.to_format(X, fmt), labels, ref, **kw)
        assert list(g) == list(groups)
        want = gold[C.combo_key(fmt, test, cc, tc, alt, log1p)]
        ref_row = int(np.searchsorted(groups, reference)) if test == "ovo" else None
        fc_rtol = FC_RTOL_LOG1P_F32 if (log1p and X.dtype == np.float32) else FC_RTOL
        assert_parity(got, (want[0], want[1], want[2]), ref_row=ref_row, fc_rtol=fc_rtol,
                      what=f"{name}:{fmt}:{test}:cc{cc}:tc{tc}:{alt}")


@pytest.mark.parametrize("name", ["conftest", "k562_mini", "k562_mini_cont", "bign", "edge"])
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovr", "ovo"])
def test_dispatchers_exact_integers_and_tie_sums(name, fmt, test):
    """The six dispatchers behind the reference's plug-in signature, called on gene sub-ranges, with the
    debug outputs of the C ABI: 2U as an exact integer and the f64 tie sum, both bit-exact vs the oracle."""
    import torch

    from illico_b200.groups import encode_and_count_groups
    from illico_b200.registry import dispatcher_registry

    X, labels, reference = C.CASES[name][0]()
    ref = reference if test == "ovo" else None
    _, grpc = encode_and_count_groups(labels, ref)
    Xf = C.to_format(X, fmt)
    n_genes = X.shape[1]
    lb, ub = (1, n_genes - 1) if n_genes > 3 else (0, n_genes)
    groups, p, U, fc, ties = oracle.run(Xf, labels, ref, want_ties=True)
    disp = dispatcher_registry.get(test, fmt)
    dbg = {}
    gp, gU, gfc = disp(Xf, lb, ub, grpc, False, True, True, "two-sided", debug=dbg)
    assert gp.shape == (len(groups), ub - lb) and gp.flags.c_contiguous and gp.dtype == np.float64
    ref_row = grpc.encoded_ref_group if test == "ovo" else None
    assert_parity((gp, gU, gfc), (p[:, lb:ub], U[:, lb:ub], fc[:, lb:ub]), ref_row=ref_row, what=f"{name}:{fmt}:{test}")
    u2 = dbg["u2"].cpu().numpy()
    tie = dbg["tie_sum"].cpu().numpy()
    rows = np.ones(len(groups), bool)
    if ref_row is not None:
        rows[ref_row] = False
    np.testing.assert_array_equal(u2[rows], (2 * U[:, lb:ub][rows]).astype(np.int64))
    want_t = ties[:, lb:ub] if test == "ovo" else ties[lb:ub]
    if test == "ovo":
        # bit-exact also for pairs above 208 063 cells, whose f64 tie sum depends on the accumulation order
        np.testing.assert_array_equal(tie[rows], want_t[rows])
    else:
        np.testing.assert_array_equal(tie, want_t)
    torch.cuda.synchronize()


def test_error_behaviour_matches_reference():
    from scipy import sparse

    from illico_b200 import asymptotic_wilcoxon

    X, labels, reference = C.CASES["conftest"][0]()
    # reference not among the labels -> ValueError (reference utils/groups.py:40-41)
    with pytest.raises(ValueError, match="is not present in the group labels"):
        asymptotic_wilcoxon(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", reference="non-targeting")
    # unsorted CSR indices -> ValueError (reference asymptotic_wilcoxon.py:185-193)
    csr = sparse.csr_matrix(X)
    perm = np.arange(X.shape[1])[::-1]
    bad = sparse.csr_matrix((csr.data.copy(), perm[csr.indices].astype(np.int32), csr.indptr.copy()), shape=csr.shape)
    assert not bad.has_sorted_indices
    with pytest.raises(ValueError, match="indices are not sorted"):
        asymptotic_wilcoxon(FakeAnnData(bad, labels), is_log1p=False, group_keys="pert", reference=reference)
    # unsupported container -> KeyError with the reference's message (utils/registry.py:54-58)
    with pytest.raises(KeyError, match="Support for data type .* is not implemented."):
        asymptotic_wilcoxon(FakeAnnData(sparse.coo_matrix(X), labels), is_log1p=False, group_keys="pert")
    with pytest.raises(ValueError, match="Invalid batch_size value"):
        asymptotic_wilcoxon(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", batch_size="big")
    with pytest.raises(ValueError, match="Unsupported alternative"):
        asymptotic_wilcoxon(FakeAnnData(X, labels), is_log1p=False, group_keys="pert", alternative="both")


@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_input_not_mutated_and_layer_and_batching(fmt):
    """reference tests/test_asymptotic_wilcoxon.py:187-194; `layer=`; results independent of batch size."""
    X, labels, reference = C.CASES["batched"][0]()
    Xf = C.to_format(X, fmt)
    keep = Xf.copy()
    from illico_b200 import asymptotic_wilcoxon

    ad = FakeAnnData(np.zeros((X.shape[0], X.shape[1]), np.float32), labels, layers={"counts": Xf})
    outs = [asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference=reference, layer="counts", batch_size=bs)
            for bs in (7, 128, "auto")]
    for o in outs[1:]:
        np.testing.assert_array_equal(o.to_numpy(), outs[0].to_numpy())
    assert list(outs[0].index.get_level_values("feature")[: X.shape[1]]) == [f"gene_{i}" for i in range(X.shape[1])]
    if fmt == "dense":
        np.testing.assert_array_equal(Xf, keep)
    else:
        np.testing.assert_array_equal(Xf.toarray(), keep.toarray())


class _BackedDense:
    """Duck-typed out-of-core dense container (h5py.Dataset protocol: shape, dtype, obj[:, lb:ub])."""

    def __init__(self, path, shape):
        self._mm = np.memmap(path, dtype=np.float32, mode="r", shape=shape)
        self.shape, self.dtype, self.reads = shape, np.dtype(np.float32), 0

    def __getitem__(self, key):
        self.reads += 1
        return np.asarray(self._mm[key])


class _BackedCSC:
    """Duck-typed backed CSC (anndata _CSCDataset protocol): obj[:, lb:ub] -> scipy CSC."""

    def __init__(self, csc):
        self._m, self.shape = csc, csc.shape

    def __getitem__(self, key):
        return self._m[key]


@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_backed_streaming_matches_in_ram(tmp_path, test):
    """Config 4 path: disk-backed dense / CSC streamed in gene batches through reader threads."""
    from scipy import sparse

    from illico_b200 import asymptotic_wilcoxon
    from illico_b200.registry import BackedCSCDataHandler, BackedDenseDataHandler, data_handler_registry

    data_handler_registry.register(_BackedDense)(BackedDenseDataHandler)
    data_handler_registry.register(_BackedCSC)(BackedCSCDataHandler)
    X, labels, reference = C.CASES["batched"][0]()
    ref = reference if test == "ovo" else None
    path = tmp_path / "x.f32"
    X.tofile(path)
    # the ORACLE is the yardstick (VERDICT r1 weak #1(i)), and the committed golden vectors of this case
    g, po, Uo, fco = oracle.run(X, labels, ref, is_log1p=False)
    ref_row = int(np.searchsorted(g, ref)) if ref is not None else None
    G = len(g)
    bd = _BackedDense(path, X.shape)
    got = asymptotic_wilcoxon(FakeAnnData(bd, labels), is_log1p=False, group_keys="pert", reference=ref, batch_size=64,
                              n_threads=3)
    assert bd.reads == -(-X.shape[1] // 64)
    assert_parity(planes(got, G, X.shape[1]), (po, Uo, fco), ref_row=ref_row, what="backed dense vs oracle")
    got = asymptotic_wilcoxon(FakeAnnData(_BackedCSC(sparse.csc_matrix(X)), labels), is_log1p=False, group_keys="pert",
                              reference=ref, batch_size=50, n_threads=2)
    assert_parity(planes(got, G, X.shape[1]), (po, Uo, fco), ref_row=ref_row, what="backed CSC vs oracle")
    # the package's own on-disk containers (np.memmap behind obj[:, lb:ub]; BASELINE config 4 on boxes without h5py)
    from illico_b200.backed import MemmapCSC, MemmapDense, save_csc, save_dense

    Xc = sparse.csc_matrix(X)
    save_csc(str(tmp_path / "csc"), Xc.data, Xc.indices, Xc.indptr, Xc.shape)
    save_dense(str(tmp_path / "dense.bin"), X)
    for cont in (MemmapCSC(str(tmp_path / "csc")), MemmapDense(str(tmp_path / "dense.bin"))):
        got = asymptotic_wilcoxon(FakeAnnData(cont, labels), is_log1p=False, group_keys="pert", reference=ref, batch_size=96,
                                  n_threads=4)
        assert_parity(planes(got, G, X.shape[1]), (po, Uo, fco), ref_row=ref_row, what=f"{type(cont).__name__} vs oracle")
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "batched.npz"))
    want = gold[C.combo_key("csc", test, True, True, "two-sided", False)]
    assert_parity(planes(got, G, X.shape[1]), (want[0], want[1], want[2]), ref_row=ref_row, what="backed vs golden")


def test_k562_shape_properties_and_oracle_sample():
    """BASELINE config-2/3 shape (300k cells, 2000 perturbations + control) on a gene subset: size-independent
    checks at full column length plus oracle parity on sampled genes.
      OVR: sum_g R_g = n(n+1)/2 exactly, with R_g = n_ref n_g + n_g(n_g+1)/2 - U_g.
      dense == CSR == CSC bit for bit in U; p in [0, 1]."""
    from scipy import sparse

    from illico_b200 import asymptotic_wilcoxon, synth

    n, N, perts = 300_000, 96, 2_000
    X, labels = synth.k562_like(seed=21, n_cells=n, n_genes=N, n_perts=perts)
    groups, counts = np.unique(np.asarray(labels), return_counts=True)
    G = len(groups)
    res = {}
    for fmt, Xf in (("dense", X), ("csr", sparse.csr_matrix(X)), ("csc", sparse.csc_matrix(X))):
        for ref in (None, synth.CONTROL):
            _, _, arr = asymptotic_wilcoxon(FakeAnnData(Xf, labels), is_log1p=False, group_keys="pert", reference=ref,
                                            return_array=True)
            res[fmt, ref] = arr.copy()
    for ref in (None, synth.CONTROL):
        np.testing.assert_array_equal(res["csr", ref][:, :, 1], res["dense", ref][:, :, 1])
        np.testing.assert_array_equal(res["csc", ref][:, :, 1], res["dense", ref][:, :, 1])
        np.testing.assert_allclose(res["csr", ref][:, :, 0], res["dense", ref][:, :, 0], rtol=1e-12, atol=2.3e-308)
        assert np.all((res["dense", ref][:, :, 0] >= 0) & (res["dense", ref][:, :, 0] <= 1))
    U = res["dense", None][:, :, 1]
    n_g = counts[:, None].astype(np.float64)
    R = (n - n_g) * n_g + n_g * (n_g + 1) / 2 - U
    np.testing.assert_array_equal(R.sum(axis=0), np.full(N, n * (n + 1) / 2))
    # oracle parity on a few genes (the oracle needs ~1 s per dense gene at this size)
    sample = [0, 17, 95]
    for ref in (None, synth.CONTROL):
        g, p, Uo, fc = oracle.run(np.ascontiguousarray(X[:, sample]), labels, ref, n_threads=3, batch_size=1)
        got = res["dense", ref][:, sample, :]
        ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
        assert_parity((got[:, :, 0], got[:, :, 1], got[:, :, 2]), (p, Uo, fc), ref_row=ref_row, what=f"k562 ref={ref}")
    assert G == perts + 1


def test_two_million_cells_csr_against_oracle():
    """BASELINE config-5 column length (2 M cells, control + 1000 perturbations) on a handful of genes:
    int64-sized tie terms (n0^3 ~ 6e18), ordered tie sums, multi-segment control."""
    from scipy import sparse

    from illico_b200 import asymptotic_wilcoxon, synth

    n, N, perts = 2_000_000, 6, 1_000
    rng = np.random.RandomState(31)
    labels, _ = synth.perturbation_labels(rng, n, perts)
    X = rng.poisson(1.0, size=(n, N)).astype(np.float32)
    X[rng.rand(n, N) < 0.9] = 0
    X[:, 5] = (rng.rand(n) < 0.1) * rng.gamma(2.0, 2.0, n).astype(np.float32)  # continuous non-zeros: path S
    csr = sparse.csr_matrix(X)
    groups = np.unique(np.asarray(labels))
    for ref in (synth.CONTROL, None):
        _, _, got = asymptotic_wilcoxon(FakeAnnData(csr, labels), is_log1p=False, group_keys="pert", reference=ref,
                                        return_array=True)
        g, p, U, fc = oracle.run(csr, labels, ref, n_threads=6, batch_size=1)
        ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
        assert_parity((got[:, :, 0], got[:, :, 1], got[:, :, 2]), (p, U, fc), ref_row=ref_row, what=f"2M cells ref={ref}")


@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovr", "ovo"])
def test_float64_and_integer_inputs(fmt, test):
    """Values float32 cannot hold (float64 noise, large integers) are ranked exactly through order-preserving
    recoding; dtypes that float32 holds exactly (int32 counts) take the normal path."""
    X, labels, reference = C.CASES["conftest"][0]()
    ref = reference if test == "ovo" else None
    rng = np.random.RandomState(8)
    noise = rng.rand(*X.shape) * 1e-9                      # differences far below float32 resolution
    X64 = np.where(X > 0, X.astype(np.float64) + noise, 0.0)
    X64[:, 3] = np.where(X[:, 3] > 0, X[:, 3].astype(np.float64) + 2.0**40, 0.0)  # big integers
    Xi = X.astype(np.int32)
    for arr in (X64, Xi):
        Xf = C.to_format(arr, fmt)
        groups, got = _run(Xf, labels, ref, is_log1p=False, batch_size=4)
        g, p, U, fc = oracle.run(Xf, labels, ref)
        ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
        assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"{arr.dtype}:{fmt}:{test}")


def _random_case(seed):
    """Random shapes, sparsity, value kinds and group structures: exercises every tier of the rank kernels."""
    rng = np.random.RandomState(seed)
    n = int(rng.choice([37, 300, 1500, 6000, 20000]))
    N = int(rng.choice([1, 3, 9, 33]))
    kind = rng.choice(["counts", "bigcounts", "continuous", "signed", "constant", "empty"])
    dens = float(rng.choice([0.02, 0.1, 0.5, 1.0]))
    if kind == "counts":
        X = rng.poisson(1.5, size=(n, N)).astype(np.float32)
    elif kind == "bigcounts":
        X = rng.poisson(40.0, size=(n, N)).astype(np.float32)       # > 20 distinct values: general paths
    elif kind == "continuous":
        X = rng.gamma(2.0, 2.0, size=(n, N)).astype(np.float32)
    elif kind == "signed":
        X = np.round(rng.randn(n, N) * 3, 1).astype(np.float32)
    elif kind == "constant":
        X = np.full((n, N), 2.0, dtype=np.float32)
    else:
        X = np.zeros((n, N), dtype=np.float32)
    X[rng.rand(n, N) >= dens] = 0
    structure = rng.choice(["many_small", "few_big", "skewed", "two"])
    if structure == "many_small":
        codes = rng.randint(0, max(2, n // 7), size=n)
    elif structure == "few_big":
        codes = rng.randint(0, 4, size=n)
    elif structure == "skewed":
        codes = np.minimum(rng.geometric(0.3, size=n), 12)
    else:
        codes = (rng.rand(n) < 0.5).astype(int)
    codes[0], codes[-1] = codes.min(), codes.max()
    labels = [f"g{c:05d}" for c in codes]
    return X, labels, kind, structure


@pytest.mark.parametrize("seed", range(24))
def test_random_inputs_against_oracle(seed):
    from scipy import sparse

    X, labels, kind, structure = _random_case(seed)
    rng = np.random.RandomState(1000 + seed)
    fmt = ["dense", "csr", "csc"][seed % 3]
    if kind == "signed":
        fmt = "dense"  # the sparse reference kernels assume stored values > 0
    Xf = C.to_format(X, fmt)
    uniq = sorted(set(labels))
    ref = uniq[int(rng.randint(len(uniq)))] if seed % 2 == 0 else None
    alt = C.ALTERNATIVES[seed % 3]
    kw = dict(is_log1p=bool(seed % 5 == 0), use_continuity=bool(seed % 4 != 1), tie_correct=bool(seed % 7 != 3), alternative=alt)
    groups, got = _run(Xf, labels, ref, batch_size=int(rng.choice([1, 4, 64])), **kw)
    g, p, U, fc = oracle.run(Xf, labels, ref, **kw)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    fc_rtol = FC_RTOL_LOG1P_F32 if kw["is_log1p"] else FC_RTOL
    # all-zero genes / groups: the oracle and the kernels both give inf or nan fold changes in the same places
    assert_parity(got, (p, U, fc), ref_row=ref_row, fc_rtol=fc_rtol, what=f"seed {seed}: {kind}/{structure}/{fmt}/ref={ref}")
    assert sparse is not None


@pytest.mark.parametrize("n_genes,batch", [(1028, "auto"), (1030, 1026), (520, 260), (6, 4), (1001, "auto")])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_dense_staging_tma_and_plain_paths_agree(monkeypatch, n_genes, batch, test):
    """The TMA staging kernel (16-byte aligned batches) and the plain-load kernel (anything else) give the same
    answer bit for bit, on shapes that exercise partial CTAs, row pieces rounded up to 16 bytes and the unaligned
    fall-back; one of them is checked against the oracle."""
    from illico_b200 import synth

    X, labels = synth.k562_like(seed=21, n_cells=3001, n_genes=n_genes, n_perts=12)
    X[:, 3] = 0.0                       # an all-zero gene
    X[:, 5] = 1.0 + (np.arange(X.shape[0]) % 3)  # a gene without zeros (lane buffer flushes every stage)
    ref = synth.CONTROL if test == "ovo" else None
    monkeypatch.setenv("ILLICO_STAGE_TMA", "1")
    groups, tma = _run(X, labels, ref, is_log1p=False, batch_size=batch)
    monkeypatch.setenv("ILLICO_STAGE_TMA", "0")
    _, plain = _run(X, labels, ref, is_log1p=False, batch_size=batch)
    # p and U bit for bit; the fold change to rounding (the fused path, which only TMA-capable batches take, multiplies
    # by reciprocals of the group sizes where the general path divides)
    np.testing.assert_array_equal(tma[0], plain[0])
    np.testing.assert_array_equal(tma[1], plain[1])
    np.testing.assert_allclose(tma[2], plain[2], rtol=1e-14, atol=0)
    g, p, U, fc = oracle.run(X, labels, ref, is_log1p=False)
    ref_row = int(np.searchsorted(groups, ref)) if ref is not None else None
    assert_parity(tma, (p, U, fc), ref_row=ref_row, what=f"tma staging {n_genes}/{batch}/{test}")


def _fused_case(kind, n_cells=6000, n_genes=72, seed=31):
    """Count-like matrix whose genes exercise every route of the fused one-versus-reference path."""
    rng = np.random.RandomState(seed)
    X = (rng.poisson(1.0, size=(n_cells, n_genes)) * (rng.rand(n_cells, n_genes) >= 0.7)).astype(np.float32)
    sizes = rng.randint(3, 400, size=14)
    codes = np.repeat(np.arange(sizes.size), sizes)
    codes = np.concatenate([codes, rng.randint(0, sizes.size, size=n_cells - codes.size)])
    rng.shuffle(codes)
    labels = [f"g{c:02d}" for c in codes]
    ref_code = {"first": 0, "last": sizes.size - 1, "middle": 6}[kind.split(":")[0]]
    ctrl = codes == ref_code
    X[:, 1] = 0.0                                                   # all-zero gene
    X[:, 2] = rng.poisson(30.0, n_cells)                            # > 10 distinct control values: handed back
    X[:, 3] = np.round(rng.gamma(2.0, 2.0, n_cells), 3)             # continuous: handed back
    X[~ctrl, 4] = rng.poisson(3.0, (~ctrl).sum()) + 20.0            # every perturbation value is absent from the control
    X[ctrl, 5] = 0.0                                                # control all zero, perturbations not
    X[:, 6] = rng.poisson(0.5, n_cells) - 1.0 * (rng.rand(n_cells) < 0.05)   # a few negative values
    X[0, 7] = np.nan if False else 1.0e30                           # one huge value in some group
    X[~ctrl, 8] = (rng.poisson(4.0, (~ctrl).sum()) * 7.0)           # more than 10 distinct values outside the control
    X[:, 40:44] = rng.poisson(30.0, (n_cells, 4))                   # a run of handed-back genes
    return X, labels, f"g{ref_code:02d}"


@pytest.mark.parametrize("kind", ["first", "middle", "last", "middle:log1p", "middle:less"])
def test_fused_ovo_routes_match_general_path_and_oracle(monkeypatch, kind):
    """fused.cu: table genes, extras, handed-back genes (merged runs), control position, log1p, alternatives:
    identical U to the general path and to the oracle; p / fold change within tolerance."""
    X, labels, ref = _fused_case(kind)
    log1p = kind.endswith("log1p")
    if log1p:
        X = np.log1p(np.abs(X)).astype(np.float32)
    kw = dict(is_log1p=log1p, alternative="less" if kind.endswith("less") else "two-sided")
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_OVO_FUSED", "1")
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")     # hand the flagged genes back one by one however many there are
    groups, fused = _run(X, labels, ref, batch_size="auto", **kw)
    assert _lib.load().illico_last_fused_ms() >= 0, "the fused kernel did not run"
    monkeypatch.setenv("ILLICO_OVO_FUSED", "0")
    _, general = _run(X, labels, ref, batch_size="auto", **kw)
    ref_row = int(np.searchsorted(groups, ref))
    rows = np.arange(len(groups)) != ref_row
    np.testing.assert_array_equal(fused[1], general[1])
    np.testing.assert_allclose(fused[0][rows], general[0][rows], rtol=1e-13, atol=2.3e-308)
    g, p, U, fc = oracle.run(X, labels, ref, **kw)
    fc_rtol = FC_RTOL_LOG1P_F32 if log1p else FC_RTOL
    assert_parity(fused, (p, U, fc), ref_row=ref_row, fc_rtol=fc_rtol, what=f"fused ovo {kind}")


@pytest.mark.parametrize("kind", ["first", "middle", "last:less", "middle:batched"])
def test_fused_ovo_wide_table_matches_general_path_and_oracle(monkeypatch, kind):
    """fused.cu, wide table (integer counts up to 64 indexed by value, histogram folded against the control at the end
    of each group): dense high-count genes next to sparse ones, values the control lacks, the largest value the table
    holds and one beyond it, fractional / negative genes in the same tile -- identical U to the general path and to the
    oracle, with and without the wide pass."""
    from illico_b200 import _lib

    X, labels, ref = _fused_case(kind)
    rng = np.random.RandomState(5)
    n = X.shape[0]
    ctrl = np.array(labels) == ref
    X[:, 10] = rng.poisson(12.0, n)                                   # dense, ~30 distinct values
    X[:, 11] = rng.poisson(12.0, n) * (rng.rand(n) < 0.5)             # the reference's fixture: masked Poisson
    X[:, 12] = rng.poisson(45.0, n)                                   # reaches past 64 somewhere: handed back during the pass
    X[:, 13] = np.minimum(rng.poisson(50.0, n), 64)                   # the largest value the table holds, heavily tied
    X[:, 14] = rng.poisson(20.0, n); X[ctrl, 14] = np.minimum(X[ctrl, 14], 18)   # values above every control value
    X[:, 15] = rng.poisson(20.0, n); X[np.flatnonzero(~ctrl)[7], 15] = 2.5   # one fractional value outside the control
    X[:, 17] = rng.poisson(20.0, n); X[np.flatnonzero(~ctrl)[9], 17] = -3.0  # one negative value outside the control
    X[:, 16] = rng.poisson(9.0, n)                                    # 11+ distinct control values: goes wide by choice
    kw = dict(is_log1p=False, alternative="less" if kind.endswith("less") else "two-sided",
              batch_size=40 if kind.endswith("batched") else "auto")
    monkeypatch.setenv("ILLICO_OVO_FUSED", "1")
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
    _lib.profile_report()
    groups, wide = _run(X, labels, ref, **kw)
    assert "fused_wide_pass_kernel" in _lib.profile_report(), "the wide pass did not run"
    monkeypatch.setenv("ILLICO_FUSED_WIDE", "0")
    _, narrow = _run(X, labels, ref, **kw)
    assert "fused_wide_pass_kernel" not in _lib.profile_report()
    monkeypatch.setenv("ILLICO_OVO_FUSED", "0")
    _, general = _run(X, labels, ref, **kw)
    ref_row = int(np.searchsorted(groups, ref))
    rows = np.arange(len(groups)) != ref_row
    for got, what in ((wide, "wide"), (narrow, "narrow")):
        np.testing.assert_array_equal(got[1], general[1], err_msg=what)
        np.testing.assert_allclose(got[0][rows], general[0][rows], rtol=1e-13, atol=2.3e-308, err_msg=what)
        np.testing.assert_allclose(got[2][rows], general[2][rows], rtol=1e-13, atol=0, err_msg=what)
    g, p, U, fc = oracle.run(X, labels, ref, is_log1p=False, alternative=kw["alternative"])
    assert_parity(wide, (p, U, fc), ref_row=ref_row, what=f"fused ovo wide {kind}")


def test_fused_ovo_debug_integers_and_continuous_batches(monkeypatch):
    """Exact 2U / tie sums through the fused path's debug outputs; a mostly continuous batch skips the fused path."""
    import ctypes as Ct

    import torch

    from illico_b200 import _lib, synth
    from illico_b200.engine import DeviceMatrix, Engine, make_flags
    from illico_b200.groups import encode_and_count_groups

    X, labels = synth.k562_like(seed=41, n_cells=5000, n_genes=64, n_perts=25)
    uniq, grpc = encode_and_count_groups(labels, synth.CONTROL)
    eng = Engine(grpc, torch.device("cuda", 0))
    flags = make_flags(False, True, True, "two-sided", "dense")
    out = {}
    for fused in ("1", "0"):
        monkeypatch.setenv("ILLICO_OVO_FUSED", fused)
        M = DeviceMatrix("dense", X.shape, torch.from_numpy(X).cuda())
        res = torch.zeros((eng.n_groups, X.shape[1], 3), dtype=torch.float64, device="cuda")
        dbg = {}
        eng.run_batch(M, 0, X.shape[1], flags, res, 0, dbg)
        torch.cuda.synchronize()
        out[fused] = (res.cpu().numpy(), {k: v.cpu().numpy() for k, v in dbg.items()})
    ref_row = int(np.searchsorted(uniq, synth.CONTROL))
    rows = np.arange(len(uniq)) != ref_row
    for k in ("u2", "tie_sum", "tie_exact"):
        np.testing.assert_array_equal(out["1"][1][k][rows], out["0"][1][k][rows], err_msg=k)
    np.testing.assert_array_equal(out["1"][0][:, :, 1], out["0"][0][:, :, 1])
    # continuous data: the table kernel flags (almost) every gene and the dispatcher takes the general path
    Xc, labels_c = synth.k562_like(seed=42, n_cells=4000, n_genes=32, n_perts=10, continuous=True)
    monkeypatch.setenv("ILLICO_OVO_FUSED", "1")
    groups, got = _run(Xc, labels_c, synth.CONTROL, is_log1p=False)
    g, p, U, fc = oracle.run(Xc, labels_c, synth.CONTROL, is_log1p=False)
    assert_parity(got, (p, U, fc), ref_row=int(np.searchsorted(groups, synth.CONTROL)), what="continuous via dispatcher")
    assert Ct is not None and _lib is not None


@pytest.mark.parametrize("kind", ["first", "middle:log1p", "middle:less"])
def test_fused_ovr_routes_match_general_path_and_oracle(monkeypatch, kind):
    """One-versus-rest through the fused pass (sample table, count extension, handed-back genes) against the general
    path and the oracle."""
    X, labels, _ = _fused_case(kind)
    X[:, 6] = np.abs(X[:, 6])
    log1p = kind.endswith("log1p")
    if log1p:
        X = np.log1p(np.abs(X)).astype(np.float32)
    kw = dict(is_log1p=log1p, alternative="less" if kind.endswith("less") else "two-sided")
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_OVR_FUSED", "1")
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
    groups, fused = _run(X, labels, None, batch_size="auto", **kw)
    assert _lib.load().illico_last_fused_ms() >= 0, "the fused kernel did not run"
    monkeypatch.setenv("ILLICO_OVR_FUSED", "0")
    _, general = _run(X, labels, None, batch_size="auto", **kw)
    np.testing.assert_array_equal(fused[1], general[1])
    np.testing.assert_allclose(fused[0], general[0], rtol=1e-13, atol=2.3e-308)
    g, p, U, fc = oracle.run(X, labels, None, **kw)
    assert_parity(fused, (p, U, fc), fc_rtol=FC_RTOL_LOG1P_F32 if log1p else FC_RTOL, what=f"fused ovr {kind}")


def test_fused_ovr_tie_sum_above_2_53(monkeypatch):
    """300k cells, 90 % zeros: the zero block's t^3 - t alone passes 2^53, so the f64 tie sum is order dependent;
    the fused path's per-gene kernel must reproduce the dense kernels' order (golden case `bign`, reference output)."""
    X, labels, reference = C.CASES["bign"][0]()
    monkeypatch.setenv("ILLICO_OVR_FUSED", "1")
    groups, fused = _run(X, labels, None, is_log1p=False)
    monkeypatch.setenv("ILLICO_OVR_FUSED", "0")
    _, general = _run(X, labels, None, is_log1p=False)
    for a, b in zip(fused[:2], general[:2]):
        np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("test", ["ovo", "ovr"])
@pytest.mark.parametrize("kind", ["first", "middle:log1p", "last:less"])
def test_fused_csr_routes_match_general_path_and_oracle(monkeypatch, test, kind):
    """CSR input through the shared-memory histogram pass (fused.cu): count genes, genes handed back, multi-segment
    groups (atomically accumulated records), log1p tables claimed while streaming -- against the general CSR path
    and the oracle."""
    from scipy import sparse

    X, labels, ref = _fused_case(kind, n_cells=9000)
    X = np.abs(X)
    X[X > 1e20] = 3.0
    log1p = "log1p" in kind
    if log1p:
        X = np.log1p(X).astype(np.float32)
    # one big group (cut into several 512-cell segments) next to the small ones
    labels = list(labels)
    for i in range(0, 2400):
        labels[i] = "g05"
    Xs = sparse.csr_matrix(X)
    reference = ref if test == "ovo" else None
    kw = dict(is_log1p=log1p, alternative="less" if kind.endswith("less") else "two-sided")
    from illico_b200 import _lib

    monkeypatch.setenv("ILLICO_CSR_FUSED", "1")
    monkeypatch.setenv("ILLICO_PROFILE", "1")
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
    groups, fused = _run(Xs, labels, reference, batch_size="auto", **kw)
    assert _lib.load().illico_last_fused_ms() >= 0, "the fused CSR pass did not run"
    monkeypatch.setenv("ILLICO_CSR_FUSED", "0")
    _, general = _run(Xs, labels, reference, batch_size="auto", **kw)
    ref_row = int(np.searchsorted(groups, reference)) if reference is not None else None
    rows = np.ones(len(groups), bool)
    if ref_row is not None:
        rows[ref_row] = False
    np.testing.assert_array_equal(fused[1], general[1])
    np.testing.assert_allclose(fused[0][rows], general[0][rows], rtol=1e-13, atol=2.3e-308)
    g, p, U, fc = oracle.run(Xs, labels, reference, **kw)
    assert_parity(fused, (p, U, fc), ref_row=ref_row, fc_rtol=FC_RTOL_LOG1P_F32 if log1p else FC_RTOL,
                  what=f"fused csr {test} {kind}")


@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_fused_gate_falls_back_when_many_genes_are_handed_back(monkeypatch, fmt):
    """Default policy, decided on the device: when more than an eighth of a batch is flagged the whole batch goes through
    the general path (hand-back mode ALL); the answer is the same either way."""
    X, labels, ref = _fused_case("middle")
    X = np.abs(X)
    X[X > 1e20] = 3.0
    Xf = C.to_format(X, fmt)
    from illico_b200 import _lib

    before = _lib.launch_count()
    groups, got = _run(Xf, labels, ref, is_log1p=False)
    assert _lib.launch_count() > before
    g, p, U, fc = oracle.run(Xf, labels, ref, is_log1p=False)
    assert_parity(got, (p, U, fc), ref_row=int(np.searchsorted(groups, ref)), what=f"gate {fmt}")


def test_cuda_array_interface_input():
    """A device array of another library (CuPy, numba): anything exposing ``__cuda_array_interface__`` is ranked in
    place, like a CUDA tensor (SURVEY.md section 8f.3).  CuPy is not in this image: a minimal stand-in carries the
    interface of a CUDA buffer."""
    import torch

    from illico_b200 import synth

    X, labels = synth.k562_like(seed=12, n_cells=3000, n_genes=40, n_perts=8)
    dev = torch.from_numpy(X).cuda()

    class DeviceArray:                      # what cupy.ndarray looks like from outside
        def __init__(self, t):
            self._keep = t
            self.shape = tuple(t.shape)
            self.__cuda_array_interface__ = t.__cuda_array_interface__

    groups, got = _run(DeviceArray(dev), labels, synth.CONTROL, is_log1p=False)
    g, p, U, fc = oracle.run(X, labels, synth.CONTROL, is_log1p=False)
    assert_parity(got, (p, U, fc), ref_row=int(np.searchsorted(groups, synth.CONTROL)), what="cuda array interface")


def test_device_resident_torch_input():
    """SURVEY 8f.3: a CUDA tensor is used where it is (no host round trip); same answer as the ndarray path."""
    import torch

    from illico_b200 import synth

    X, labels = synth.k562_like(seed=51, n_cells=3000, n_genes=40, n_perts=8)
    _, want = _run(X, labels, synth.CONTROL, is_log1p=False)
    _, got = _run(torch.from_numpy(X).cuda(), labels, synth.CONTROL, is_log1p=False)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)
    _, got64 = _run(torch.from_numpy(X.astype(np.float64)).cuda(), labels, None, is_log1p=False)
    _, want64 = _run(X, labels, None, is_log1p=False)
    np.testing.assert_array_equal(got64[1], want64[1])


@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_dispatchers_called_from_concurrent_threads(fmt):
    """The reference drives its dispatchers from joblib threads (ctypes releases the GIL): concurrent calls on one
    engine must give the same chunks as sequential ones (illico/asymptotic_wilcoxon.py:212-249)."""
    from concurrent.futures import ThreadPoolExecutor

    from illico_b200 import dispatch, synth
    from illico_b200.groups import encode_and_count_groups

    X, labels = synth.k562_like(seed=61, n_cells=4000, n_genes=96, n_perts=15)
    X[:, 7] = np.random.RandomState(1).poisson(25.0, X.shape[0])      # a gene the fused path hands back
    Xf = C.to_format(X, fmt)
    if fmt != "dense":
        Xf = dispatch.CSRMatrix(Xf.data, Xf.indices, Xf.indptr, Xf.shape)
    uniq, grpc = encode_and_count_groups(labels, synth.CONTROL)
    fn = getattr(dispatch, f"{fmt}_ovo_mwu_kernel_over_contiguous_col_chunk")
    chunks = [(lb, min(96, lb + 16)) for lb in range(0, 96, 16)]
    seq = [fn(Xf, lb, ub, grpc, False, True, True, "two-sided") for lb, ub in chunks]
    with ThreadPoolExecutor(max_workers=6) as ex:
        par = list(ex.map(lambda c: fn(Xf, c[0], c[1], grpc, False, True, True, "two-sided"), chunks * 3))
    for k, got in enumerate(par):
        want = seq[k % len(chunks)]
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
    dispatch.clear_caches()


@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_fused_dense_compacted_hand_back(monkeypatch, test):
    """Scattered handed-back genes (here 7 of 72), listed on the device: staged one by one from the matrix and ranked by
    the general path with the device-side count (mode LIST); same answer when the whole batch is redone (mode ALL) and
    from the general path alone."""
    X, labels, ref = _fused_case("middle")
    X = np.abs(X)
    X[X > 1e20] = 3.0
    reference = ref if test == "ovo" else None
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "1.0")
    groups, compact = _run(X, labels, reference, is_log1p=False)
    monkeypatch.setenv("ILLICO_FUSED_LIST_SHARE", "0.0")
    _, merged = _run(X, labels, reference, is_log1p=False)
    monkeypatch.setenv("ILLICO_OVO_FUSED", "0")
    monkeypatch.setenv("ILLICO_OVR_FUSED", "0")
    _, general = _run(X, labels, reference, is_log1p=False)
    for a, b in zip(merged, general):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(compact, general):
        np.testing.assert_array_equal(a, b)
    g, p, U, fc = oracle.run(X, labels, reference, is_log1p=False)
    ref_row = int(np.searchsorted(groups, reference)) if reference is not None else None
    assert_parity(compact, (p, U, fc), ref_row=ref_row, what=f"compacted hand-back {test}")


@pytest.mark.parametrize("fmt", ["dense", "csr"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_hand_back_modes_on_the_device(monkeypatch, fmt, test):
    """The three device-side hand-back modes of the fused dispatchers (none / listed genes / whole batch) on one matrix:
    count genes with 0, 3 and 40 % high-count genes scattered among them; dense and CSR; against the oracle."""
    from illico_b200 import synth

    for frac in (0.0, 0.03, 0.4):
        X, labels = synth.k562_like(seed=95, n_cells=5000, n_genes=200, n_perts=14)
        rng = np.random.RandomState(3)
        for j in rng.choice(200, size=int(200 * frac), replace=False):
            X[:, j] = rng.poisson(25.0, X.shape[0]) * (rng.rand(X.shape[0]) < 0.6)
        reference = synth.CONTROL if test == "ovo" else None
        Xf = C.to_format(X, fmt)
        groups, got = _run(Xf, labels, reference, is_log1p=False)
        g, p, U, fc = oracle.run(Xf, labels, reference, is_log1p=False, n_threads=4)
        ref_row = int(np.searchsorted(groups, reference)) if reference is not None else None
        assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"hand-back {fmt} {test} frac={frac}")


@pytest.mark.parametrize("fmt", ["dense", "csr"])
def test_dispatcher_cache_sees_in_place_changes(fmt):
    """ADVICE r1 / VERDICT r1 weak #9: a matrix transformed in place between two dispatcher calls (normalise, log1p -- the
    standard scanpy flow) is uploaded again instead of being served from the cached device copy."""
    from illico_b200 import dispatch, synth
    from illico_b200.groups import encode_and_count_groups

    X, labels = synth.k562_like(seed=71, n_cells=3000, n_genes=32, n_perts=6)
    uniq, grpc = encode_and_count_groups(labels, synth.CONTROL)
    fn = getattr(dispatch, f"{fmt}_ovo_mwu_kernel_over_contiguous_col_chunk")

    def host(Xd):
        Xf = C.to_format(Xd, fmt)
        return Xf if fmt == "dense" else dispatch.CSRMatrix(Xf.data, Xf.indices, Xf.indptr, Xf.shape)

    Xf = host(X.copy())
    first = fn(Xf, 0, 32, grpc, False, True, True, "two-sided")
    g, p, U, fc = oracle.run(X, labels, synth.CONTROL, is_log1p=False)
    ref_row = int(np.searchsorted(g, synth.CONTROL))
    assert_parity(first, (p, U, fc), ref_row=ref_row, what="before the in-place change")
    arr = Xf if fmt == "dense" else Xf.data
    np.log1p(arr, out=arr)                               # same buffer, same address, new content
    second = fn(Xf, 0, 32, grpc, True, True, True, "two-sided")
    Xl = np.log1p(X)
    g, p, U, fc = oracle.run(Xl, labels, synth.CONTROL, is_log1p=True)
    assert_parity(second, (p, U, fc), ref_row=ref_row, fc_rtol=FC_RTOL_LOG1P_F32, what="after the in-place change")
    dispatch.clear_caches()


def test_torch_tensor_on_another_device_is_moved_not_read_remotely():
    import torch

    from illico_b200 import synth

    X, labels = synth.k562_like(seed=72, n_cells=500, n_genes=8, n_perts=3)
    t = torch.from_numpy(X).cuda()
    groups, got = _run(t, labels, None, is_log1p=False)           # device defaults to the tensor's
    assert got[1].shape == (len(groups), 8)
    if torch.cuda.device_count() > 1:                             # the shard is peer-copied to the GPU that ranks it
        _, other = _run(t, labels, None, is_log1p=False, device="cuda:1")
        for a, b in zip(other, got):
            np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_pageable_pinned_and_strided_uploads_agree(fmt, test):
    """The three host-to-device routes of hostio (pinned 2-D copy, pageable input through the staging ring with several
    worker threads and chunks, strided column shards) deliver the same matrix: results identical to the oracle's."""
    import torch

    from illico_b200 import hostio, synth

    n, N = 70_000, 48                                             # 13 MB dense: above the direct-copy threshold
    X, labels = synth.k562_like(seed=81, n_cells=n, n_genes=N, n_perts=12)
    reference = synth.CONTROL if test == "ovo" else None
    g, p, U, fc = oracle.run(X, labels, reference, is_log1p=False, n_threads=4)
    ref_row = int(np.searchsorted(g, reference)) if reference is not None else None
    old = hostio.CHUNK_BYTES
    hostio.CHUNK_BYTES = 1 << 20                                  # many chunks per worker thread
    try:
        Xf = C.to_format(X, fmt)
        _, got = _run(Xf, labels, reference, is_log1p=False)      # pageable: staged
        assert_parity(got, (p, U, fc), ref_row=ref_row, what=f"pageable {fmt}")
        if fmt == "dense":
            pin = torch.from_numpy(X).pin_memory()
            _, got = _run(pin.numpy(), labels, reference, is_log1p=False)
            assert_parity(got, (p, U, fc), ref_row=ref_row, what="pinned dense")
            wide = np.zeros((n, N + 16), dtype=np.float32)
            wide[:, 8:8 + N] = X
            _, got = _run(wide[:, 8:8 + N], labels, reference, is_log1p=False)   # strided pageable view
            assert_parity(got, (p, U, fc), ref_row=ref_row, what="strided dense")
            pw = torch.from_numpy(wide).pin_memory()
            _, got = _run(pw.numpy()[:, 8:8 + N], labels, reference, is_log1p=False)   # strided pinned view: 2-D DMA
            assert_parity(got, (p, U, fc), ref_row=ref_row, what="strided pinned dense")
    finally:
        hostio.CHUNK_BYTES = old


@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
@pytest.mark.parametrize("test", ["ovo", "ovr"])
def test_devices_argument_shards_genes(fmt, test):
    """`devices=`: one host thread per GPU, contiguous gene shards, slabs delivered into one array -- identical to the
    single-GPU call (with one GPU present the same device is used for a single shard; with more, for real)."""
    import torch

    from illico_b200 import asymptotic_wilcoxon, synth

    X, labels = synth.k562_like(seed=82, n_cells=5000, n_genes=67, n_perts=9)
    X[:, 11] = np.random.RandomState(2).poisson(25.0, X.shape[0])          # one gene for the general path
    reference = synth.CONTROL if test == "ovo" else None
    Xf = C.to_format(X, fmt)
    _, want = _run(Xf, labels, reference, is_log1p=False)
    n_dev = torch.cuda.device_count()
    for devices in (["cuda:0"], "all", n_dev):
        _, got = _run(Xf, labels, reference, is_log1p=False, devices=devices)
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
    with pytest.raises(ValueError):
        asymptotic_wilcoxon(FakeAnnData(Xf, labels), is_log1p=False, group_keys="pert", reference=reference, device="cuda:0",
                            devices="all")


def test_device_compute_pval_known_answers(golden_dir):
    """VERDICT r1 weak #1(iii): the 1 300 known answers of the reference's `compute_pval` (illico/utils/math.py:64-118,
    incl. huge z and the tie_corr cut-off) against the DEVICE epilogue code (epilogue.cuh), not only against the oracle."""
    import torch

    from illico_b200 import _lib

    rows = np.load(os.path.join(golden_dir, "primitives.npz"))["pval_rows"]
    n_ref, n_tgt = rows[:, 0].astype(np.int64), rows[:, 1].astype(np.int64)
    alt_names = list(C.ALTERNATIVES)
    alt = np.array([_lib.ALTERNATIVES[alt_names[int(a)]] for a in rows[:, 5]], dtype=np.int32)
    dev = torch.device("cuda", torch.cuda.current_device())
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    args = [t(n_ref), t(n_tgt), t(n_ref + n_tgt), t(rows[:, 2]), t(rows[:, 3]), t(n_ref * n_tgt / 2.0), t(rows[:, 4]), t(alt)]
    out = torch.empty(rows.shape[0], dtype=torch.float64, device=dev)
    lib = _lib.load()
    rc = lib.illico_compute_pval_batch(*[a.data_ptr() for a in args], out.data_ptr(), rows.shape[0],
                                       torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "illico_compute_pval_batch")
    np.testing.assert_allclose(out.cpu().numpy(), rows[:, 6], rtol=1e-12, atol=2.3e-308)


def test_optional_columns_p_adj_and_log2fc():
    """SURVEY 8f.4: Benjamini-Hochberg `p_adj` per group (statsmodels fdr_bh semantics, restated in numpy here) and
    `log2_fold_change`; the default call returns the reference's three columns only."""
    from illico_b200 import asymptotic_wilcoxon, synth

    X, labels = synth.k562_like(seed=91, n_cells=4000, n_genes=700, n_perts=6)
    X[:, :20] *= (np.asarray(labels) == "p0001")[:, None] * 3 + 1          # a few real effects
    ad = FakeAnnData(X, labels)
    base = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference=synth.CONTROL)
    assert list(base.columns) == ["p_value", "statistic", "fold_change"]
    df = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference=synth.CONTROL, p_adjust=True, log2_fold_change=True)
    assert list(df.columns) == ["p_value", "statistic", "fold_change", "p_adj", "log2_fold_change"]
    np.testing.assert_array_equal(df[["p_value", "statistic", "fold_change"]].to_numpy(), base.to_numpy())
    G, N = len(set(labels)), X.shape[1]
    p = df["p_value"].to_numpy().reshape(G, N)
    want = np.empty_like(p)
    for g in range(G):                                    # statsmodels.stats.multitest.multipletests(method="fdr_bh")
        order = np.argsort(p[g], kind="stable")
        raw = p[g][order] / (np.arange(1, N + 1) / float(N))
        adj = np.minimum.accumulate(raw[::-1])[::-1]
        adj[adj > 1] = 1
        want[g, order] = adj
    np.testing.assert_array_equal(df["p_adj"].to_numpy().reshape(G, N), want)
    with np.errstate(divide="ignore", invalid="ignore"):
        np.testing.assert_array_equal(df["log2_fold_change"].to_numpy(), np.log2(df["fold_change"].to_numpy()))


@pytest.mark.parametrize("fmt", ["dense", "csr"])
@pytest.mark.parametrize("log1p", [False, True])
def test_ovo_stream_tier_with_repeated_values(fmt, log1p):
    """ovo_kernel's stream tier (control with more than 64 distinct values, groups of at most 28 non-zeros): values that
    repeat inside a group and values shared with the control -- the telescoped per-element tie terms and the private
    occurrence hash against the oracle (U and tie sums bit-exact)."""
    import torch

    from illico_b200 import dispatch, synth
    from illico_b200.groups import encode_and_count_groups

    rng = np.random.RandomState(77)
    n, N = 9000, 40
    labels, _ = synth.perturbation_labels(rng, n, 110, p_control=0.25)
    X = (np.round(rng.gamma(2.0, 2.0, size=(n, N)) * 8) / 8).astype(np.float32)      # ~150 distinct values per gene
    X[rng.rand(n, N) < 0.7] = 0
    X[:, 3] = np.where(rng.rand(n) < 0.3, rng.gamma(2.0, 2.0, n), 0).astype(np.float32)   # no repeats at all
    if fmt == "dense":
        X[:, 4] = -X[:, 4]                 # negative values (dense only: the sparse kernels assume stored values > 0)
    if log1p:
        X = np.log1p(np.abs(X)).astype(np.float32)
    Xf = C.to_format(X, fmt)
    groups, got = _run(Xf, labels, synth.CONTROL, is_log1p=log1p)
    g, p, U, fc = oracle.run(Xf, labels, synth.CONTROL, is_log1p=log1p)
    ref_row = int(np.searchsorted(groups, synth.CONTROL))
    assert_parity(got, (p, U, fc), ref_row=ref_row, fc_rtol=FC_RTOL_LOG1P_F32 if log1p else FC_RTOL, what="stream tier")
    # exact integers and tie sums through the dispatcher's debug outputs
    uniq, grpc = encode_and_count_groups(labels, synth.CONTROL)
    fn = getattr(dispatch, f"{fmt}_ovo_mwu_kernel_over_contiguous_col_chunk")
    Xd = Xf if fmt == "dense" else dispatch.CSRMatrix(Xf.data, Xf.indices, Xf.indptr, Xf.shape)
    dbg = {}
    fn(Xd, 0, N, grpc, log1p, True, True, "two-sided", debug=dbg)
    _, _, _, _, ties = oracle.run(Xf, labels, synth.CONTROL, is_log1p=log1p, want_ties=True)
    rows = np.arange(len(groups)) != ref_row
    np.testing.assert_array_equal(dbg["tie_sum"].cpu().numpy()[rows], ties[rows])
    np.testing.assert_array_equal(dbg["u2"].cpu().numpy()[rows], (2 * U[rows]).astype(np.int64))
    dispatch.clear_caches()
    assert torch.cuda.is_available()


@pytest.mark.gpu
@pytest.mark.parametrize("n_shards", [1, 3, 8])
def test_csr_repartition_matches_host_slicing(n_shards):
    """repartition.py / csrc/repart.cu (rows -> genes repartition of a CSR matrix; csr_get_contig_cols_into_csr,
    illico/utils/sparse/csr.py:144-196, across GPUs): row blocks cut on the device and scattered into the shards' arrays
    give exactly the column slices scipy gives -- empty rows, empty shards' pieces, explicit zeros included.  (All shards
    live on cuda:0 here; the stores are the same instructions when the arrays are another GPU's.)"""
    import torch
    from scipy import sparse

    from illico_b200 import repartition

    rng = np.random.RandomState(3)
    n, N = 5000, 700
    X = sparse.random(n, N, density=0.07, format="csr", dtype=np.float32, random_state=rng)
    X.data[:] = rng.poisson(2.0, X.nnz).astype(np.float32)          # some stored zeros
    X = sparse.csr_matrix(X)
    X[17] = 0                                                        # (keeps explicit zeros: an all-zero row of stored values)
    X.sort_indices()
    edges = np.linspace(0, N, n_shards + 1).astype(int)
    edges[1:-1] += rng.randint(-20, 20, size=n_shards - 1) if n_shards > 1 else 0
    dev = torch.device("cuda", 0)
    shards = repartition.repartition_csr(X, [dev] * n_shards, list(edges))
    torch.cuda.synchronize()
    for j, M in enumerate(shards):
        want = X[:, edges[j]:edges[j + 1]]
        assert M.shape == want.shape and M.gene_offset == edges[j]
        np.testing.assert_array_equal(M.indptr.cpu().numpy(), want.indptr)
        np.testing.assert_array_equal(M.indices.cpu().numpy(), want.indices)
        np.testing.assert_array_equal(M.data.cpu().numpy(), want.data)
    # unsorted rows are refused with the reference's error (asymptotic_wilcoxon.py:185-193)
    Y = X.copy()
    r = int(np.argmax(np.diff(Y.indptr) > 3))
    a = Y.indptr[r]
    Y.indices[a], Y.indices[a + 1] = Y.indices[a + 1], Y.indices[a]
    with pytest.raises(ValueError, match="indices are not sorted"):
        repartition.repartition_csr(Y, [dev] * n_shards, list(edges))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["dense", "csr", "csc"])
def test_native_recoding_of_float64_values(fmt):
    """csrc/recode.cu (illico_recode_*): float64 values become, per gene, float32 codes that keep order, ties, zero and
    sign -- in the input's own layout -- and the float64 group sums of the original values come with them."""
    import ctypes as Ct

    import torch
    from scipy import sparse

    from illico_b200 import _lib

    lib = _lib.load()
    rng = np.random.RandomState(0)
    n, N, G = 3000, 9, 7
    X = np.round(rng.randn(n, N) * 3, 1)
    X[rng.rand(n, N) < 0.4] = 0.0
    X[:, 1] = np.abs(X[:, 1]) + 1.0          # no zeros, all positive
    X[:, 2] = -np.abs(X[:, 2]) - 1.0         # all negative
    X[:, 3] += 2.0**40 * (X[:, 3] > 0)       # beyond float32 resolution
    X[:, 4] = 0.0                            # nothing stored
    X[0, 5] = -0.0
    X[:, 6] = rng.randn(n) * 1e-3            # all distinct
    groups = rng.randint(0, G, n).astype(np.int32)
    lb, ub = 1, 8                            # a window of the genes
    b = ub - lb
    dev = torch.device("cuda", 0)
    enc = torch.from_numpy(groups).to(dev)
    sums = torch.empty((G, b), dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    if fmt == "dense":
        d = torch.from_numpy(X).to(dev)
        codes = torch.empty((n, b), dtype=torch.float32, device=dev)
        ws = torch.empty(int(lib.illico_recode_workspace_bytes(n * b, b)), dtype=torch.uint8, device=dev)
        rc = lib.illico_recode_dense(d.data_ptr(), _lib.DTYPE_F64, N, lb, b, n, enc.data_ptr(), G, 0, codes.data_ptr(), sums.data_ptr(),
                                     ws.data_ptr(), ws.numel(), st)
        _lib.check(rc, "illico_recode_dense")
        got = codes.cpu().numpy()
    else:
        S = (sparse.csr_matrix if fmt == "csr" else sparse.csc_matrix)(X)
        S.sort_indices()
        data = torch.from_numpy(S.data.astype(np.float64)).to(dev)
        idx = torch.from_numpy(S.indices.astype(np.int32)).to(dev)
        ptr = torch.from_numpy(S.indptr.astype(np.int64)).to(dev)
        codes = torch.zeros(S.nnz, dtype=torch.float32, device=dev)
        keys = n * b if fmt == "csr" else int(S.indptr[ub] - S.indptr[lb])
        ws = torch.empty(int(lib.illico_recode_workspace_bytes(keys, b)), dtype=torch.uint8, device=dev)
        if fmt == "csr":
            rc = lib.illico_recode_csr(data.data_ptr(), _lib.DTYPE_F64, idx.data_ptr(), ptr.data_ptr(), n, lb, b, enc.data_ptr(), G, 0,
                                       codes.data_ptr(), sums.data_ptr(), ws.data_ptr(), ws.numel(), st)
        else:
            rc = lib.illico_recode_csc(data.data_ptr(), _lib.DTYPE_F64, idx.data_ptr(), ptr.data_ptr(), lb, b, keys, enc.data_ptr(), G, 0,
                                       codes.data_ptr(), sums.data_ptr(), ws.data_ptr(), ws.numel(), st)
        _lib.check(rc, f"illico_recode_{fmt}")
        C_ = (sparse.csr_matrix if fmt == "csr" else sparse.csc_matrix)((codes.cpu().numpy(), S.indices, S.indptr), shape=S.shape)
        got = np.asarray(C_[:, lb:ub].todense(), dtype=np.float32)
    torch.cuda.synchronize()
    assert got.dtype == np.float32 and Ct is not None
    for j in range(b):
        x, c = X[:, lb + j], got[:, j]
        assert np.array_equal(np.sign(c), np.sign(x)), j
        order = np.argsort(x, kind="stable")
        assert np.all(np.diff(c[order]) >= 0), j
        assert np.array_equal(np.diff(c[order]) == 0, np.diff(x[order]) == 0), j
    want = np.zeros((G, b))
    np.add.at(want, groups, X[:, lb:ub])
    np.testing.assert_allclose(sums.cpu().numpy(), want, rtol=1e-12, atol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["pageable", "pinned", "shard", "mixed"])
def test_packed_upload_rebuilds_the_matrix(monkeypatch, source):
    """hostio._h2d_2d_packed (csrc/hostpack.c + unpack_rows_kernel): a mostly-zero float32 matrix squeezed on the host
    (bit mask + values), sent packed and rebuilt in HBM is the matrix, bit for bit -- NaN kept, -0.0 a zero; pinned
    sources, column shards of a wider matrix, and chunks too dense to squeeze (sent as they are)."""
    import torch

    from illico_b200 import hostio

    monkeypatch.setenv("ILLICO_STAGE_CHUNK_MB", "4")
    monkeypatch.setattr(hostio, "CHUNK_BYTES", 4 << 20)
    monkeypatch.setenv("ILLICO_PACK_UPLOAD", "1")
    rng = np.random.RandomState(4)
    n, N = 9000, 2117
    X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) < 0.12)).astype(np.float32)
    X[5, 7] = -0.0
    X[6, 8] = np.nan
    X[:, -1] = 3.0
    if source == "mixed":
        X[2000:4500] = rng.rand(2500, N).astype(np.float32) + 1.0        # chunks that do not squeeze
    if source == "pinned":
        hp = torch.empty((n, N), dtype=torch.float32, pin_memory=True)
        hp.copy_(torch.from_numpy(X))
        src = hp.numpy()
    elif source == "shard":
        src = X[:, 100:2050]
    else:
        src = X
    dev = torch.device("cuda", 0)
    dst = torch.full(src.shape, 7.0, dtype=torch.float32, device=dev)
    hostio.h2d_2d(dst, src).finish()
    torch.cuda.synchronize()
    got = dst.cpu().numpy()
    want = np.where(src == 0, np.float32(0.0), src)                       # (-0.0 arrives as +0.0)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    st = hostio.LAST_UPLOAD
    assert st["packed"] + st["raw"] == -(-n // ((4 << 20) // (src.shape[1] * 4)))
    if source == "mixed":
        assert st["raw"] >= 2
    if source in ("pageable", "shard"):
        assert st["raw"] == 0 and st["bytes"] < 0.35 * src.size * 4


def test_bench_steps_and_dumped_outputs(tmp_path):
    """bench.py: `--steps K` times K steps (K times the launches of one), and `--dump-outputs` writes what the last timed
    step computed -- on the benchmark's own seeded inputs, the oracle's results."""
    import json
    import subprocess
    import sys

    import torch

    import bench

    root = os.path.dirname(os.path.abspath(bench.__file__))
    cells, genes, perts = 3000, 40, 10
    args = [sys.executable, os.path.join(root, "bench.py"), "--cells", str(cells), "--genes", str(genes), "--perts",
            str(perts), "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--others", "none"]
    lines = {}
    for steps in (1, 3):
        out = subprocess.check_output(args + ["--steps", str(steps), "--dump-outputs", str(tmp_path / str(steps))],
                                      text=True, cwd=root)
        lines[steps] = json.loads(out.strip().splitlines()[-1])
    assert lines[3]["steps"] == 3 and lines[1]["gpu_launches"] > 0
    assert lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"]

    labels, reference = bench.make_labels(0, cells, perts, bench.WORKLOADS["dense_ovo"])
    X = bench.gen_dense("counts", 17, cells, genes, torch.device("cuda", 0)).cpu().numpy()
    groups, p, U, fc = oracle.run(X, labels, reference)
    for steps in (1, 3):
        d = tmp_path / str(steps)
        got = [np.load(d / f"{k}.npy") for k in ("p_value", "statistic", "fold_change", "test_index")]
        assert all(a.dtype == np.float64 and a.shape == (len(groups) * genes,) for a in got)
        np.testing.assert_array_equal(got[3], np.arange(len(groups) * genes))
        assert_parity(tuple(a.reshape(len(groups), genes) for a in got[:3]), (p, U, fc),
                      ref_row=int(np.searchsorted(groups, reference)), what=f"bench --dump-outputs, {steps} steps")
