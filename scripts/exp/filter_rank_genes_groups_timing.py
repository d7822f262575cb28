"""Cost of scanpy's marker filter, filter_rank_genes_groups, on one GPU, after rank_genes_groups(method="wilcoxon",
reference="non-targeting", n_genes=100) at the K562 shape (300 000 x 8 000, 2 000 perturbations + control):

  1. the union |U| of the listed genes and the bytes that cross PCIe for a dense host matrix (its columns only);
  2. each device step alone on the U columns of the matrix (CUDA events, medians): the stats pass (illico_group_sums_dense
     with its count plane), illico_nonzero_fractions, illico_log_fold_changes and illico_filter_marker_pairs;
  3. the filter end to end from a pinned dense host matrix, from host CSR and from a CUDA tensor, next to the
     rank_genes_groups call it follows (alternated, medians), and the branch that reads no matrix (a reference="rest",
     pts=True result);
  4. the test file's numpy / pandas restatement of scanpy's loop on 20 groups, per group.  It stands in for scanpy (which
     is not installed) and is not scanpy.

Usage: python scripts/exp/filter_rank_genes_groups_timing.py [--reps 9] [--e2e-reps 3] [--out results.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts", "exp"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402
from scipy import sparse  # noqa: E402

from rank_genes_timing import card, stats, timed  # noqa: E402

CELLS, GENES, PERTS = 300_000, 8_000, 2_000


class Ad:
    def __init__(self, X, labels):
        self.X, self.raw, self.uns, self.layers = X, None, {}, {}
        self.obs = pd.DataFrame({"pert": pd.Categorical(labels)})
        self.var_names = pd.Index([f"g{i}" for i in range(GENES)])
        self.var = pd.DataFrame(index=self.var_names)


def wall(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def main():
    import bench
    from illico_b200 import _lib, filter_rank_genes_groups, rank_genes_groups
    from illico_b200.asymptotic_wilcoxon import nonzero_fractions
    from illico_b200.engine import DeviceMatrix, Engine
    from illico_b200.groups import encode_and_count_groups

    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("filter_rank_genes_groups_timing.py measures on a GPU; none found")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    dev = torch.device("cuda", 0)
    labels, ref = bench.make_labels(0, CELLS, PERTS, {"test": "ovo"})
    Xd = bench.gen_dense("counts", 17, CELLS, GENES, dev)
    pinned = torch.empty((CELLS, GENES), dtype=torch.float32, pin_memory=True)
    pinned.copy_(Xd)
    csr_d = Xd.to_sparse_csr()
    csr = sparse.csr_matrix((csr_d.values().cpu().numpy(), csr_d.col_indices().cpu().numpy().astype(np.int32),
                             csr_d.crow_indices().cpu().numpy()), shape=(CELLS, GENES))
    del csr_d
    torch.cuda.empty_cache()
    inputs = {"dense_pinned": pinned.numpy(), "csr": csr, "cuda_tensor": Xd}

    # 1. the listed genes
    ad = Ad(inputs["dense_pinned"], labels)
    rank_genes_groups(ad, "pert", method="wilcoxon", reference=ref, n_genes=100)
    names = ad.uns["rank_genes_groups"]["names"]
    fields = list(names.dtype.names)
    listed = np.column_stack([ad.var_names.get_indexer(pd.Index(names[f], dtype=object)) for f in fields]).astype(np.int32)
    U = np.unique(listed)
    res["shape"] = {"cells": CELLS, "genes": GENES, "groups": len(fields), "k": len(names), "union": int(U.size),
                    "dense_pcie_bytes": int(CELLS * U.size * 4), "dense_full_bytes": int(CELLS * GENES * 4)}
    print("shape", json.dumps(res["shape"]), flush=True)

    # 2. the device steps alone, on the U columns
    uniq, grpc = encode_and_count_groups(ad.obs["pert"], None)
    eng = Engine(grpc, dev)
    G, N = eng.n_groups, int(U.size)
    M = DeviceMatrix("dense", (CELLS, N), Xd[:, torch.from_numpy(U).long().to(dev)].contiguous())
    lib = _lib.load()
    st = torch.cuda.current_stream(dev).cuda_stream
    sums = torch.empty((G, N), dtype=torch.float64, device=dev)
    nnz = torch.empty((G, N), dtype=torch.int32, device=dev)
    lfc = torch.empty((G, N), dtype=torch.float64, device=dev)
    sizes = torch.from_numpy(np.asarray(grpc.counts, dtype=np.int32)).to(dev)
    row_of = {str(g): i for i, g in enumerate(uniq)}
    rows = torch.from_numpy(np.array([row_of[f] for f in fields], dtype=np.int32)).to(dev)
    col = torch.from_numpy(np.searchsorted(U, listed).astype(np.int32)).to(dev)
    keep = torch.empty(col.shape, dtype=torch.uint8, device=dev)
    k, Cn = col.shape

    def stats_pass():
        _lib.check(lib.illico_group_sums_dense(M.data.data_ptr(), _lib.DTYPE_F32, N, 0, N, C.byref(eng.plan), sums.data_ptr(),
                                               nnz.data_ptr(), N, N, st), "sums")

    planes = {}

    def fractions():
        planes["in"], planes["out"] = nonzero_fractions(nnz, grpc)

    def lfc_pass():
        _lib.check(lib.illico_log_fold_changes(sums.data_ptr(), N, sizes.data_ptr(), G, N, -1, CELLS, 1.0, lfc.data_ptr(), N, st),
                   "lfc")

    def pairs():
        _lib.check(lib.illico_filter_marker_pairs(col.data_ptr(), rows.data_ptr(), k, Cn, N, planes["in"].data_ptr(), 0,
                                                  planes["out"].data_ptr(), 0, lfc.data_ptr(), 0, 0.25, 0.5, 1.0, 0,
                                                  keep.data_ptr(), st), "pairs")

    steps = {"stats_pass": stats_pass, "nonzero_fractions": fractions, "log_fold_changes": lfc_pass,
             "filter_marker_pairs": pairs}
    for _ in range(3):
        for f in steps.values():
            f()
    torch.cuda.synchronize()
    t = {name: [] for name in steps}
    for _ in range(a.reps):
        for name, f in steps.items():
            t[name].append(timed(f))
    res["kernels"] = {name: stats(v) for name, v in t.items()}
    print("kernels", json.dumps(res["kernels"]), flush=True)
    del M, sums, nnz, lfc, planes
    torch.cuda.empty_cache()

    # 3. end to end
    e2e = {}
    for name, X in inputs.items():
        ad = Ad(X, labels)
        runs = {"rank_genes_groups": lambda ad=ad: rank_genes_groups(ad, "pert", method="wilcoxon", reference=ref, n_genes=100),
                "filter_rank_genes_groups": lambda ad=ad: filter_rank_genes_groups(ad)}
        for f in runs.values():
            f()
        tt = {key: [] for key in runs}
        for _ in range(a.e2e_reps):
            for key, f in runs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                tt[key].append((time.perf_counter() - t0) * 1e3)
        e2e[name] = {key: stats(v) for key, v in tt.items()}
        print("end_to_end", name, json.dumps(e2e[name]), flush=True)
    ad = Ad(inputs["dense_pinned"], labels)
    rank_genes_groups(ad, "pert", method="wilcoxon", n_genes=100, pts=True)
    ad.X = None                                  # the no-read branch never touches it
    e2e["no_read_rest_pts"] = {"filter_rank_genes_groups": stats(wall(lambda: filter_rank_genes_groups(ad), a.e2e_reps))}
    print("end_to_end no_read", json.dumps(e2e["no_read_rest_pts"]), flush=True)
    res["end_to_end"] = e2e

    # 4. the test file's host restatement (a stand-in for scanpy's loop, not scanpy) on 20 groups
    sys.path.insert(0, ROOT)
    from tests.test_filter_rank_genes_groups import oracle_quantities

    ad = Ad(inputs["dense_pinned"], labels)
    rank_genes_groups(ad, "pert", method="wilcoxon", reference=ref, n_genes=100)
    st_ = ad.uns["rank_genes_groups"]
    sub = pd.DataFrame({f: st_["names"][f] for f in list(st_["names"].dtype.names)[:20]}).to_records(index=False)
    ad.uns["sub"] = dict(st_, names=sub)
    t0 = time.perf_counter()
    oracle_quantities(ad, key="sub")
    ms = (time.perf_counter() - t0) * 1e3
    res["host_restatement_20_groups"] = {"ms": ms, "per_group_ms": ms / 20,
                                         "label": "numpy/pandas restatement from the tests, not scanpy"}
    print("host restatement", json.dumps(res["host_restatement_20_groups"]), flush=True)
    res["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
