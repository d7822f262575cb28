"""Cost of scanpy's call, rank_genes_groups, on one GPU: the kernels it adds and the call end to end.

  1. the group sums pass (illico_group_sums_*) against the count pass (illico_count_nonzero_*) and the moments pass
     (illico_group_moments_*) on the same batches of bench.py's K562-shape inputs (dense and CSR, OVO and OVR); then
     illico_log_fold_changes and illico_bonferroni_adjust on a whole [G, N] plane, and illico_top_genes_columns against
     illico_top_genes (k = 100 and k = N); CUDA events, variants alternated, medians;
  2. rank_genes_groups(method="wilcoxon", n_genes=100) end to end from host memory (dense pinned, K562 shape, OVO) against
     rank_genes(n_genes=100), alternated, medians; then n_genes=None, with the host record-array assembly timed on its own.

Usage: python scripts/exp/rank_genes_groups_timing.py [--reps 9] [--e2e-reps 3] [--out results.json]
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
import torch  # noqa: E402

from rank_genes_timing import card, stats, timed  # noqa: E402

WORKLOADS = ("dense_ovo", "dense_ovr", "csr_ovo", "csr_ovr")


def kernels(reps):
    import bench
    from illico_b200 import _lib

    class A:
        seed, cells, genes, perts = 0, 0, 0, 0

    lib = _lib.load()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    for name in WORKLOADS:
        w = bench.Workload(name, A(), dev, 0, 1)
        M, eng, hp = w.M, w.eng, w.eng.host_plan
        G, N = w.G, w.genes
        nnz = torch.empty((G, N), dtype=torch.int32, device=dev)
        step = eng.max_batch_genes(N, "t-test")
        batches = [(lb, min(N, lb + step)) for lb in range(0, N, step)]
        bmax = max(ub - lb for lb, ub in batches)
        mom = torch.empty((3, G, bmax), dtype=torch.float64, device=dev)
        s1, s2, sf = (mom[k].data_ptr() for k in range(3))
        head = lambda lb, ub: ([M.data.data_ptr(), _lib.DTYPE_F32] +  # noqa: E731
                               ([M.ld] if M.fmt == "dense" else [M.indices.data_ptr(), M.indptr.data_ptr()]) +
                               [lb, ub - lb, C.byref(eng.plan)])

        def count():
            for lb, ub in batches:
                eng.count_nonzero(M, lb, ub, nnz, lb)

        def sums():
            for lb, ub in batches:
                _lib.check(getattr(lib, f"illico_group_sums_{M.fmt}")(*head(lb, ub), s1, None, 0, bmax, st), "sums")

        def sums_counts():
            for lb, ub in batches:
                _lib.check(getattr(lib, f"illico_group_sums_{M.fmt}")(*head(lb, ub), s1, nnz.data_ptr() + lb * 4, N, bmax, st),
                           "sums")

        def moments():
            for lb, ub in batches:
                _lib.check(getattr(lib, f"illico_group_moments_{M.fmt}")(*head(lb, ub), 0, s1, s2, sf, None, 0, bmax, st), "moments")

        lfc = torch.empty((G, N), dtype=torch.float64, device=dev)
        padj = torch.empty((G, N), dtype=torch.float64, device=dev)
        scores = torch.randn((G, N), dtype=torch.float64, device=dev)
        w.results[:, :, 0].uniform_()

        def lfc_pass():
            for lb, ub in batches:
                _lib.check(lib.illico_log_fold_changes(s1, bmax, eng._tables["group_size"].data_ptr(), G, ub - lb, hp.ref_group,
                                                       hp.n_cells, 1.0, lfc.data_ptr() + lb * 8, N, st), "lfc")

        def bonferroni():
            _lib.check(lib.illico_bonferroni_adjust(w.results.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), st), "bonferroni")

        ws = torch.empty(int(lib.illico_top_genes_workspace_bytes(G, N)), dtype=torch.uint8, device=dev)
        rows = torch.arange(G, dtype=torch.int32, device=dev)
        sel = {}
        for k in (100, N):
            gene = torch.empty((G, k), dtype=torch.int32, device=dev)
            rec = torch.empty((G, k, 5), dtype=torch.float64, device=dev)
            cg = torch.empty((k, G), dtype=torch.int32, device=dev)
            cs, cl = (torch.empty((k, G), dtype=torch.float32, device=dev) for _ in range(2))
            cp, cq = (torch.empty((k, G), dtype=torch.float64, device=dev) for _ in range(2))

            def top(k=k, gene=gene, rec=rec):
                _lib.check(lib.illico_top_genes(scores.data_ptr(), N, w.results.data_ptr(), 3 * N, padj.data_ptr(), G, N, k, 0,
                                                gene.data_ptr(), rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "top")

            def cols(k=k, cg=cg, cs=cs, cl=cl, cp=cp, cq=cq):
                _lib.check(lib.illico_top_genes_columns(scores.data_ptr(), N, w.results.data_ptr(), 3 * N, padj.data_ptr(),
                                                        lfc.data_ptr(), N, G, N, rows.data_ptr(), G, k, 0, cg.data_ptr(), cs.data_ptr(),
                                                        cl.data_ptr(), cp.data_ptr(), cq.data_ptr(), ws.data_ptr(), ws.numel(), st),
                           "cols")

            sel[f"top_genes_k{k}"], sel[f"top_genes_columns_k{k}"] = top, cols
        runs = {"count": count, "sums": sums, "sums_with_counts": sums_counts, "moments": moments, "lfc": lfc_pass,
                "bonferroni": bonferroni, **sel}
        for _ in range(3):
            for f in runs.values():
                f()
        torch.cuda.synchronize()
        t = {k: [] for k in runs}
        for _ in range(reps):
            for k, f in runs.items():
                t[k].append(timed(f))
        res = {k: stats(v) for k, v in t.items()}
        out[name] = {"G": G, "cells": w.cells, "genes": N, "batches": len(batches), "fmt": M.fmt, **res,
                     "sums_over_count": res["sums"]["median_ms"] / res["count"]["median_ms"],
                     "sums_over_moments": res["sums"]["median_ms"] / res["moments"]["median_ms"]}
        print(name, json.dumps(out[name]), flush=True)
        del w, M, eng, nnz, mom, lfc, padj, scores, ws, sel, runs
        torch.cuda.empty_cache()
    return out


def end_to_end(reps):
    import pandas as pd

    import bench
    from illico_b200 import rank_genes, rank_genes_groups, scanpy_compat

    dev = torch.device("cuda", 0)
    cells, genes, perts = 300_000, 8_000, 2_000
    labels, ref = bench.make_labels(0, cells, perts, {"test": "ovo"})
    Xd = bench.gen_dense("counts", 17, cells, genes, dev)
    pinned = torch.empty((cells, genes), dtype=torch.float32, pin_memory=True)
    pinned.copy_(Xd)
    del Xd
    torch.cuda.empty_cache()
    ad = bench.Ad(pinned.numpy(), labels, genes)
    ad.obs = pd.DataFrame({"pert": pd.Categorical(labels)})
    ad.uns, ad.raw = {}, None
    runs = {"rank_genes_n100": lambda: rank_genes(ad, is_log1p=False, group_keys="pert", reference=ref, n_genes=100),
            "rank_genes_groups_n100": lambda: rank_genes_groups(ad, "pert", method="wilcoxon", reference=ref, n_genes=100),
            "rank_genes_groups_all": lambda: rank_genes_groups(ad, "pert", method="wilcoxon", reference=ref)}
    # the host record-array assembly on its own, on [k, G] planes of the n_genes=None shape
    k, C = genes, perts
    rng = np.random.RandomState(0)
    gene = rng.randint(0, genes, size=(k, C)).astype(np.int32)
    planes = {"scores": rng.randn(k, C).astype(np.float32), "pvals": rng.rand(k, C)}
    fields = [f"p{i}" for i in range(C)]
    names = pd.Index([f"g{i}" for i in range(genes)])
    runs["host_names_records_all"] = lambda: scanpy_compat.name_records(gene, names, fields)
    runs["host_numeric_records_all"] = lambda: [scanpy_compat.records(p, fields) for p in planes.values()]
    for f in runs.values():
        f()
    t = {k: [] for k in runs}
    for _ in range(reps):
        for key, f in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = f()
            torch.cuda.synchronize()
            t[key].append((time.perf_counter() - t0) * 1e3)
            del r
    out = {k: stats(v) for k, v in t.items()}
    print("end_to_end", json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_genes_groups_timing.py measures on a GPU; none found")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    res["kernels"] = kernels(a.reps)
    res["end_to_end"] = end_to_end(a.e2e_reps)
    res["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
