"""CPU tests of the host logic, the oracle wiring and the C-ABI surface (no compute calls without a GPU)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_build_and_exported_symbols():
    """The CUDA library builds for sm_100a here (no GPU needed) and exports every symbol the header declares."""
    from illico_b200 import _lib, build

    path = build.build()
    assert os.path.exists(path)
    header = open(os.path.join(ROOT, "include", "illico_b200.h")).read()
    declared = set(re.findall(r"\b(illico_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    out = subprocess.check_output(["nm", "-D", "--defined-only", path], text=True)
    exported = set(re.findall(r" T (illico_[a-z0-9_]+)", out))
    assert declared <= exported, declared - exported
    lib = _lib.load()
    assert lib.illico_abi_version() == _lib.ABI_VERSION
    assert lib.illico_launch_count() == 0
    sass = subprocess.run(["cuobjdump", "-lelf", path], capture_output=True, text=True).stdout
    assert "sm_100a" in sass


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "illico_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", src, re.M), f
                assert "liboracle" not in src, f


def test_environment_switches_match_design_table():
    """Every environment variable the package reads is listed in DESIGN.md's switch table, and the table lists no
    variable the package no longer reads."""
    read = set()
    for dirpath, _, files in os.walk(os.path.join(ROOT, "illico_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                read |= set(re.findall(r"[\"'](ILLICO_[A-Z0-9_]+)[\"']", open(os.path.join(dirpath, f)).read()))
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    table = design.split("### Environment switches", 1)[1].split("\n#", 1)[0]
    rows = [line.split("|")[1] for line in table.splitlines() if line.startswith("| `")]
    listed = set(re.findall(r"`(ILLICO_[A-Z0-9_]+)`", "".join(rows)))
    assert read == listed, f"read but not listed: {sorted(read - listed)}; listed but not read: {sorted(listed - read)}"

def test_no_gpu_means_loud_failure():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from illico_b200 import _lib, asymptotic_wilcoxon
    from tests.util import FakeAnnData

    X = np.ones((8, 3), dtype=np.float32)
    with pytest.raises(_lib.IllicoCudaError):
        asymptotic_wilcoxon(FakeAnnData(X, list("aabbccdd")), is_log1p=False, group_keys="pert")


def test_encode_and_count_groups_matches_reference_semantics():
    import oracle
    from illico_b200.groups import encode_and_count_groups

    rng = np.random.RandomState(0)
    labels = [f"pert_{v}" for v in rng.randint(0, 12, size=500)] + ["non-targeting"] * 7
    uniq, g = encode_and_count_groups(labels, "non-targeting")
    o_uniq, o_enc, o_counts, o_idx, o_ptr, o_ref = oracle.encode_groups(labels, "non-targeting")
    assert list(uniq) == list(o_uniq) == sorted(set(labels))
    np.testing.assert_array_equal(g.encoded_groups, o_enc)
    np.testing.assert_array_equal(g.counts, o_counts)
    np.testing.assert_array_equal(g.indptr, o_ptr)
    assert g.encoded_ref_group == o_ref == list(uniq).index("non-targeting")
    # indices: cells sorted by group (reference utils/groups.py:47)
    assert sorted(g.indices.tolist()) == list(range(len(labels)))
    assert all(g.encoded_groups[g.indices[g.indptr[k]:g.indptr[k + 1]]].tolist() == [k] * g.counts[k] for k in range(len(uniq)))
    _, g2 = encode_and_count_groups(labels, None)
    assert g2.encoded_ref_group == -1
    with pytest.raises(ValueError, match="is not present in the group labels"):
        encode_and_count_groups(labels, "missing")
    # numeric labels sort numerically like np.unique
    uniq, g3 = encode_and_count_groups([10, 2, 2, 33, 10], 2)
    assert list(uniq) == [2, 10, 33] and g3.encoded_ref_group == 0


@pytest.mark.parametrize("seg_max", [1, 7, 512])
def test_plan_invariants(seg_max):
    from illico_b200.groups import build_plan, encode_and_count_groups

    rng = np.random.RandomState(1)
    labels = rng.randint(0, 9, size=1000).tolist() + [99]
    _, g = encode_and_count_groups(labels, 3)
    p = build_plan(g, seg_max)
    n = len(labels)
    assert sorted(p.perm.tolist()) == list(range(n))
    assert np.all(np.diff(g.encoded_groups[p.perm]) >= 0)  # groups contiguous
    for k in range(p.n_groups):  # stable inside a group
        rows = p.perm[g.indptr[k]:g.indptr[k + 1]]
        assert np.all(np.diff(rows) > 0)
    assert p.seg_pos[0] == 0 and p.seg_pos[-1] == n and np.all(np.diff(p.seg_pos) >= 1)
    assert np.all(np.diff(p.seg_pos) <= seg_max)
    assert np.all(p.seg_base % 8 == 0) and p.slot_cap == p.seg_base[-1]
    assert np.all(np.diff(p.seg_base) >= np.diff(p.seg_pos))
    assert p.group_seg[0] == 0 and p.group_seg[-1] == p.n_segments
    for s in range(p.n_segments):
        cells = p.perm[p.seg_pos[s]:p.seg_pos[s + 1]]
        assert np.all(p.cell_seg[cells] == s)
        assert np.all(g.encoded_groups[cells] == p.seg_group[s])
        assert p.group_seg[p.seg_group[s]] <= s < p.group_seg[p.seg_group[s] + 1]
    assert p.max_group_size == g.counts.max() and p.ref_group_size == g.counts[g.encoded_ref_group]


def test_registries_mirror_the_reference():
    from scipy import sparse

    from illico_b200.registry import (KernelDataFormat, Test, data_handler_registry, dispatcher_registry)

    assert {k for k in dispatcher_registry} == {(t, f) for t in Test for f in KernelDataFormat}
    X = np.zeros((4, 3), dtype=np.float32)
    assert data_handler_registry.get(X).kernel_data_format() is KernelDataFormat.DENSE
    assert data_handler_registry.get(sparse.csr_matrix(X)).kernel_data_format() is KernelDataFormat.CSR
    assert data_handler_registry.get(sparse.csc_matrix(X)).kernel_data_format() is KernelDataFormat.CSC
    h = data_handler_registry.get(X)
    assert h.fetch(1, 2) == (X, (1, 2)) or h.fetch(1, 2)[1] == (1, 2)

    class Backed:  # e.g. an anndata _CSRDataset: not supported, same KeyError text as the reference
        shape = (4, 3)

    with pytest.raises(KeyError, match="Support for data type .* is not implemented."):
        data_handler_registry.get(Backed())
    with pytest.raises(KeyError, match="No dispatcher registered"):
        dispatcher_registry.get("ovo", "dense") if False else dispatcher_registry.__class__().get("ovo", "dense")


def test_gene_shards_cover_all_genes():
    from illico_b200.parallel import gene_shard

    for n, w in ((8000, 8), (15, 4), (3, 8), (20000, 3)):
        shards = [gene_shard(n, r, w) for r in range(w)]
        assert shards[0][0] == 0 and shards[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(shards, shards[1:]))
        assert max(u - l for l, u in shards) - min(u - l for l, u in shards) <= 1
    wts = np.r_[np.full(100, 10.0), np.full(900, 1.0)]
    shards = [gene_shard(1000, r, 2, wts) for r in range(2)]
    assert shards[0][0] == 0 and shards[1][1] == 1000 and shards[0][1] == shards[1][0]
    assert abs(wts[: shards[0][1]].sum() - wts[shards[0][1]:].sum()) <= 20.0


def _gather_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    from illico_b200.parallel import gather_results, gene_shard

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    G, N = 5, 11
    full = torch.arange(G * N * 3, dtype=torch.float64).reshape(G, N, 3)
    lb, ub = gene_shard(N, rank, world)
    out = gather_results(full[:, lb:ub].contiguous(), N)
    q.put((rank, bool(torch.equal(out, full))))
    dist.destroy_process_group()


def test_gather_results_world_size_2_gloo():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert got == [(0, True), (1, True)]


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` times the reference's CPU path on the host cores and prints one JSON line."""
    import json

    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cells", "3000",
                                   "--genes", "32", "--perts", "10", "--steps", "1", "--warmup", "0"], text=True, cwd=ROOT)
    line = json.loads(out.strip().splitlines()[-1])
    # the unmodified numba reference when it is importable here (/root/reference or baseline/_ref), else the C port
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["config"]["workload"].startswith("dense_ovo") and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0


def test_categorical_labels_encode_like_strings():
    """AnnData obs columns are categorical: the fast path gives the same groups / codes as the string path,
    drops unused categories and keeps np.unique's order even when the categories are not sorted."""
    import pandas as pd

    from illico_b200.groups import encode_and_count_groups

    rng = np.random.RandomState(3)
    names = np.array(["zeta", "alpha", "non-targeting", "beta", "unused", "Gamma"])
    labels = names[rng.choice([0, 1, 2, 3, 5], size=5000)]
    ser = pd.Series(pd.Categorical(labels, categories=names))
    u1, g1 = encode_and_count_groups(ser, "non-targeting")
    u2, g2 = encode_and_count_groups(list(labels), "non-targeting")
    assert list(u1) == list(u2) == sorted(set(labels))
    np.testing.assert_array_equal(g1.encoded_groups, g2.encoded_groups)
    np.testing.assert_array_equal(g1.counts, g2.counts)
    assert g1.encoded_ref_group == g2.encoded_ref_group
    import pytest

    with pytest.raises(ValueError, match="not present"):
        encode_and_count_groups(ser, "unused")


def test_register_into_reference_registry(monkeypatch):
    """INTEGRATION.md section 2: the six GPU dispatchers replace the numba ones in the reference's own registry (a
    stand-in of the reference's registry module: the reference is not part of this repository); without the reference,
    registering reports False."""
    import illico_b200
    from illico_b200 import dispatch as gpu
    from tests.util import reference_registry_standin

    monkeypatch.setitem(sys.modules, "illico", None)          # not importable
    assert illico_b200.register_into_reference() is False
    mods = reference_registry_standin()
    for name, mod in mods.items():
        monkeypatch.setitem(sys.modules, name, mod)
    ref = mods["illico.utils.registry"]
    assert illico_b200.register_into_reference() is True
    assert len(ref.dispatcher_registry) == 6
    for fmt in ref.KernelDataFormat:
        for test in ref.Test:
            fn = ref.dispatcher_registry[(test, fmt)]
            assert fn is getattr(gpu, f"{fmt.value}_{test.value}_mwu_kernel_over_contiguous_col_chunk")


def test_torch_tensor_handler_registered():
    import torch

    from illico_b200.registry import TorchDenseDataHandler, data_handler_registry

    h = data_handler_registry.get(torch.zeros((4, 3)))
    assert isinstance(h, TorchDenseDataHandler) and h.kernel_data_format().value == "dense"


def test_result_frame_matches_from_product():
    """The fast DataFrame assembly gives exactly what the reference builds (asymptotic_wilcoxon.py:252-256)."""
    import pandas as pd

    from illico_b200.asymptotic_wilcoxon import _result_frame

    rng = np.random.RandomState(0)
    groups = np.array(["b", "non-targeting", "a10", "a2"])
    var_names = pd.Index([f"g{i}" for i in range(7)])
    out = rng.rand(len(groups), len(var_names), 3)
    got = _result_frame(groups, var_names, out)
    want = pd.DataFrame(
        data=out.reshape(-1, 3),
        index=pd.MultiIndex.from_product([pd.Series(groups, name="pert", dtype=str), pd.Series(var_names, name="feature", dtype=str)],
                                         names=["pert", "feature"]),
        columns=["p_value", "statistic", "fold_change"])
    pd.testing.assert_frame_equal(got, want)
    assert got.index.names == ["pert", "feature"]
    assert got.loc[("a10", "g3"), "statistic"] == out[2, 3, 1]
    # duplicated gene names: from_product's semantics are kept
    dup = pd.Index(["g0", "g1", "g0"])
    got = _result_frame(groups, dup, out[:, :3])
    want = pd.DataFrame(out[:, :3].reshape(-1, 3), index=pd.MultiIndex.from_product(
        [pd.Series(groups, name="pert", dtype=str), pd.Series(dup, name="feature", dtype=str)], names=["pert", "feature"]),
        columns=["p_value", "statistic", "fold_change"])
    pd.testing.assert_frame_equal(got, want)


def test_dispatch_cache_keys_follow_content_not_addresses():
    """ADVICE r1: a matrix transformed in place, or a relabelled GroupContainer, must never hit a stale cache entry."""
    from illico_b200 import dispatch

    rng = np.random.RandomState(3)
    X = rng.poisson(1.0, size=(500, 40)).astype(np.float32)
    fp0 = dispatch._fingerprint(X)
    assert dispatch._fingerprint(X) == fp0
    np.log1p(X, out=X)                                # the standard in-place scanpy step
    assert dispatch._fingerprint(X) != fp0
    big = np.zeros(3_000_000, dtype=np.float32)       # sampled fingerprint: both ends and the strided sample are covered
    f = dispatch._fingerprint(big)
    big[-1] = 1.0
    assert dispatch._fingerprint(big) != f
    assert dispatch._fingerprint(np.asfortranarray(X)) == dispatch._fingerprint(np.asfortranarray(X))
    assert isinstance(dispatch._fingerprint(X[::2, ::3]), int)   # non-contiguous views are sampled too


def test_host_pack_rows_matches_numpy():
    """csrc/hostpack.c (the host half of the packed upload; no GPU involved): bit masks, row offsets and the values in
    order, for full and ragged widths, strided rows, NaN and -0.0, and the no-room answer."""
    import ctypes as C

    from illico_b200 import _lib

    lib = _lib.load()
    assert lib.illico_host_pack_isa() in (0, 1, 2)
    rng = np.random.RandomState(2)
    for n, N, lo, hi in ((37, 96, 0, 96), (50, 203, 5, 198), (11, 64, 0, 33), (3, 40, 1, 2)):
        X = (rng.poisson(1.0, (n, N)) * (rng.rand(n, N) < 0.3)).astype(np.float32)
        X[0, lo] = -0.0
        X[n - 1, hi - 1] = np.nan
        view = X[:, lo:hi]
        b = hi - lo
        W = (b + 31) // 32
        mask = np.full((n, W), 0xFFFFFFFF, dtype=np.uint32)
        off = np.zeros(n + 1, dtype=np.uint32)
        vals = np.full(n * b + 16, -1.0, dtype=np.float32)
        nnz = lib.illico_host_pack_rows_f32(view.ctypes.data, N, n, b, mask.ctypes.data, off.ctypes.data, vals.ctypes.data, vals.size)
        nz = view != 0
        assert nnz == int(nz.sum())
        bits = np.unpackbits(mask.view(np.uint8).reshape(n, -1), axis=1, bitorder="little")[:, :b].astype(bool)
        assert np.array_equal(bits, nz)
        assert np.array_equal(np.diff(off.astype(np.int64)), nz.sum(1))
        assert np.array_equal(vals[:nnz].view(np.uint32), view[nz].view(np.uint32))
        # padding bits of the last word stay clear
        if b % 32:
            assert not (mask[:, -1] >> np.uint32(b % 32)).any()
        assert lib.illico_host_pack_rows_f32(view.ctypes.data, N, n, b, mask.ctypes.data, off.ctypes.data, vals.ctypes.data, b) == -1
    assert C is not None


def test_row_blocks_balance_stored_values():
    """repartition.row_blocks: contiguous row ranges that cover every row once and hold about the same number of stored
    values (what each GPU uploads before the rows -> genes exchange)."""
    from illico_b200.repartition import row_blocks

    rng = np.random.RandomState(0)
    counts = rng.poisson(700, 10_000)
    counts[2000:2500] = 0                                  # a stretch of empty rows
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    for k in (1, 2, 3, 8):
        blocks = row_blocks(indptr, k)
        assert len(blocks) == k and blocks[0][0] == 0 and blocks[-1][1] == counts.size
        assert all(blocks[i][1] == blocks[i + 1][0] for i in range(k - 1))
        nnz = [indptr[b] - indptr[a] for a, b in blocks]
        assert max(nnz) - min(nnz) <= 2 * counts.max()
    empty = row_blocks(np.zeros(6, dtype=np.int64), 3)      # a matrix without stored values: the rows are still covered once
    assert empty[0][0] == 0 and empty[-1][1] == 5 and sum(b - a for a, b in empty) == 5


def test_pack_decision_samples_the_density(monkeypatch):
    """hostio._pack_wanted: only large float32 matrices whose sampled rows are mostly zeros are squeezed."""
    from illico_b200 import hostio

    monkeypatch.delenv("ILLICO_PACK_UPLOAD", raising=False)
    rng = np.random.RandomState(1)
    n, b = 20_000, 1024                                     # 82 MB
    sparse_x = (rng.rand(n, b) < 0.1).astype(np.float32)
    dense_x = rng.rand(n, b).astype(np.float32)
    assert hostio._pack_wanted(sparse_x, n, b)
    assert not hostio._pack_wanted(dense_x, n, b)
    assert not hostio._pack_wanted(sparse_x.astype(np.float64), n, b)
    assert not hostio._pack_wanted(sparse_x[:1000], 1000, b)          # small: not worth the threads
    monkeypatch.setenv("ILLICO_PACK_UPLOAD", "0")
    assert not hostio._pack_wanted(sparse_x, n, b)
