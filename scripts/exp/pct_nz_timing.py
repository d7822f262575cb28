"""Cost of counting the cells that express each gene (pts) and of the marker filter, on one GPU.

  1. the count pass (illico_count_nonzero_*) on bench.py's K562 dense OVO, CSR OVO and dense continuous OVO inputs, the
     config-5 shard (CSR) and the config-4 CSC shape, each next to the dispatcher step and the staging kernel
     (illico_stage_*_f32) on the same batches; CUDA events, medians.  The count pass's bytes (every value it reads, plus
     the column indices for CSR / CSC) over its time, as a fraction of a device-to-device copy peak measured in the same
     call (read + write bytes over time, 4 GiB buffers);
  2. rank_genes(n_genes=100) end to end from host memory (dense pinned, K562 shape): pts off, pts on, and scanpy's default
     filter (0.25 / 0.5 / 1), alternated, medians;
  3. asymptotic_wilcoxon(pts=True) against the same call without it, alternated, medians.

Usage: python scripts/exp/pct_nz_timing.py [--reps 9] [--e2e-reps 3] [--out results.json]
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


def copy_peak_gbs(reps):
    n = 1 << 32
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    ms = stats([timed(lambda: b.copy_(a)) for _ in range(reps)])["median_ms"]
    del a, b
    torch.cuda.empty_cache()
    return 2 * n / (ms * 1e-3) / 1e9


def count_passes(reps, peak):
    import bench
    from illico_b200 import _lib

    class A:
        seed, cells, genes, perts = 0, 0, 0, 0

    lib = _lib.load()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    for name in ("dense_ovo", "csr_ovo", "dense_ovo_continuous", "c5_shard", "backed_csc_ovr"):
        w = bench.Workload(name, A(), dev, 0, 1)
        M, eng, plan = w.M, w.eng, C.byref(w.eng.plan)
        nnz = torch.empty((w.G, w.genes), dtype=torch.int32, device=dev)

        def count():
            for lb, ub in w.batches:
                eng.count_nonzero(M, lb, ub, nnz, lb)

        def stage():
            for lb, ub in w.batches:
                t = eng._ensure_buffers(ub - lb)
                if M.fmt == "dense":
                    rc = lib.illico_stage_dense_f32(M.data.data_ptr(), M.ld, lb, ub - lb, plan, t.ir_vals.data_ptr(),
                                                    t.ir_cnt.data_ptr(), st)
                elif M.fmt == "csr":
                    rc = lib.illico_stage_csr_f32(M.data.data_ptr(), M.indices.data_ptr(), M.indptr.data_ptr(), lb, ub - lb, plan,
                                                  t.ir_vals.data_ptr(), t.ir_cnt.data_ptr(), t.ws.data_ptr(), t.ws.numel(), st)
                else:
                    _lib.check(lib.illico_zero_counts(t.ir_cnt.data_ptr(), ub - lb, plan, st), "illico_zero_counts")
                    rc = lib.illico_stage_csc_f32(M.data.data_ptr(), M.indices.data_ptr(), M.indptr.data_ptr(), lb, ub - lb, plan,
                                                  t.ir_vals.data_ptr(), t.ir_cnt.data_ptr(), st)
                _lib.check(rc, "illico_stage")

        runs = {"count": count, "stage": stage, "dispatcher_step": w.step}
        for _ in range(3):
            for f in runs.values():
                f()
        torch.cuda.synchronize()
        t = {k: [] for k in runs}
        for _ in range(reps):
            for k, f in runs.items():
                t[k].append(timed(f))
        if M.fmt == "dense":
            nbytes = w.cells * w.genes * 4
        else:
            nbytes = int(M.indptr[-1].item()) * 8 + int(M.indptr.numel()) * 8
        ms = stats(t["count"])["median_ms"]
        out[name] = {"G": w.G, "cells": w.cells, "genes": w.genes, "batches": len(w.batches), "fmt": M.fmt,
                     **{k: stats(v) for k, v in t.items()}, "count_bytes": nbytes,
                     "count_gbs": nbytes / (ms * 1e-3) / 1e9, "count_frac_of_copy_peak": nbytes / (ms * 1e-3) / 1e9 / peak}
        print(name, json.dumps(out[name]), flush=True)
        del w, M, eng, nnz
        torch.cuda.empty_cache()
    return out


def end_to_end(reps):
    import pandas as pd

    import bench
    from illico_b200 import asymptotic_wilcoxon, rank_genes

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
    kw = dict(is_log1p=False, group_keys="pert", reference=ref)
    scanpy_filter = dict(min_in_group_fraction=0.25, max_out_group_fraction=0.5, min_fold_change=1)
    runs = {"rank_genes_100": lambda: rank_genes(ad, n_genes=100, **kw),
            "rank_genes_100_pts": lambda: rank_genes(ad, n_genes=100, pts=True, **kw),
            "rank_genes_100_filtered": lambda: rank_genes(ad, n_genes=100, **scanpy_filter, **kw),
            "asymptotic_wilcoxon": lambda: asymptotic_wilcoxon(ad, return_array=True, **kw),
            "asymptotic_wilcoxon_pts": lambda: asymptotic_wilcoxon(ad, return_array=True, pts=True, **kw)}
    rows = {k: f() for k, f in runs.items()}
    rows = {k: (len(v) if hasattr(v, "index") else None) for k, v in rows.items()}
    t = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = f()
            torch.cuda.synchronize()
            t[k].append((time.perf_counter() - t0) * 1e3)
            del r
    out = {k: stats(v) for k, v in t.items()}
    out["frame_rows"] = rows
    print("end_to_end", json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pct_nz_timing.py measures on a GPU; none found")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    res["copy_peak_gbs"] = copy_peak_gbs(a.reps)
    print("copy_peak_gbs", res["copy_peak_gbs"], flush=True)
    res["count_pass"] = count_passes(a.reps, res["copy_peak_gbs"])
    res["end_to_end"] = end_to_end(a.e2e_reps)
    res["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
