"""Cost of Welch's t-test (method="t-test") on one GPU, next to the Wilcoxon path on the same inputs.

  1. the moments pass (illico_group_moments_*) against the count pass (illico_count_nonzero_*) on the same batches of
     bench.py's inputs: K562 dense OVO, dense continuous OVO and OVR, CSR OVO, the config-5 shard (CSR) and the config-4 CSC
     shape; CUDA events, medians.  Bytes read (every value, plus the column indices for CSR / CSC) over the moments pass's
     time, as a fraction of a device-to-device copy peak measured in the same call (read + write bytes over time, 4 GiB);
  2. the epilogue (illico_welch_ttest) alone on those moment planes;
  3. the t-test step (moments + epilogue, Engine.run_batch(method="t-test")) against the Wilcoxon dispatcher step;
  4. rank_genes(n_genes=100, method="t-test") end to end from host memory (dense pinned, K562 shape) against
     rank_genes(n_genes=100), alternated, medians.

Usage: python scripts/exp/ttest_timing.py [--reps 9] [--e2e-reps 3] [--out results.json]
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

from pct_nz_timing import copy_peak_gbs  # noqa: E402
from rank_genes_timing import card, stats, timed  # noqa: E402

WORKLOADS = ("dense_ovo", "dense_ovo_continuous", "dense_ovr_continuous", "csr_ovo", "c5_shard", "backed_csc_ovr")


def passes(reps, peak):
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
        nnz = torch.empty((w.G, w.genes), dtype=torch.int32, device=dev)
        scores = torch.empty((w.G, w.genes), dtype=torch.float64, device=dev)
        tbatches = [(lb, min(w.genes, lb + eng.max_batch_genes(w.genes, "t-test")))
                    for lb in range(0, w.genes, eng.max_batch_genes(w.genes, "t-test"))]
        bmax = max(ub - lb for lb, ub in tbatches)
        mom = torch.empty((3, w.G, bmax), dtype=torch.float64, device=dev)
        s1, s2, sf = (mom[k].data_ptr() for k in range(3))

        def count():
            for lb, ub in tbatches:
                eng.count_nonzero(M, lb, ub, nnz, lb)

        def moments():
            for lb, ub in tbatches:
                if M.fmt == "dense":
                    rc = lib.illico_group_moments_dense(M.data.data_ptr(), _lib.DTYPE_F32, M.ld, lb, ub - lb, C.byref(eng.plan), 0, s1,
                                                        s2, sf, None, 0, bmax, st)
                else:
                    rc = getattr(lib, f"illico_group_moments_{M.fmt}")(M.data.data_ptr(), _lib.DTYPE_F32, M.indices.data_ptr(),
                                                                       M.indptr.data_ptr(), lb, ub - lb, C.byref(eng.plan), 0, s1,
                                                                       s2, sf, None, 0, bmax, st)
                _lib.check(rc, "illico_group_moments")

        def epilogue():
            lb, ub = tbatches[0]
            _lib.check(lib.illico_welch_ttest(s1, s2, None, bmax, eng._tables["group_size"].data_ptr(), w.G, ub - lb, hp.ref_group,
                                              hp.n_cells, 0, 0, w.results.data_ptr(), w.genes * 3, scores.data_ptr(), w.genes, st),
                       "illico_welch_ttest")

        def ttest_step():
            for lb, ub in tbatches:
                eng.run_batch(M, lb, ub, w.flags, w.results, lb, scores=scores, method="t-test")

        def wilcoxon_step():
            for lb, ub in w.batches:
                eng.run_batch(M, lb, ub, w.flags, w.results, lb, scores=scores)

        runs = {"count": count, "moments": moments, "epilogue": epilogue, "ttest_step": ttest_step, "wilcoxon_step": wilcoxon_step}
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
        res = {k: stats(v) for k, v in t.items()}
        ms = res["moments"]["median_ms"]
        out[name] = {"G": w.G, "cells": w.cells, "genes": w.genes, "ttest_batches": len(tbatches), "fmt": M.fmt, **res,
                     "moments_bytes": nbytes, "moments_gbs": nbytes / (ms * 1e-3) / 1e9,
                     "moments_frac_of_copy_peak": nbytes / (ms * 1e-3) / 1e9 / peak,
                     "moments_over_count": ms / res["count"]["median_ms"],
                     "epilogue_tests": w.G * (tbatches[0][1] - tbatches[0][0]),
                     "ttest_over_wilcoxon": res["ttest_step"]["median_ms"] / res["wilcoxon_step"]["median_ms"]}
        print(name, json.dumps(out[name]), flush=True)
        del w, M, eng, nnz, scores, mom
        torch.cuda.empty_cache()
    return out


def end_to_end(reps):
    import pandas as pd

    import bench
    from illico_b200 import rank_genes

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
    kw = dict(is_log1p=False, group_keys="pert", reference=ref, n_genes=100)
    runs = {"rank_genes_wilcoxon": lambda: rank_genes(ad, **kw), "rank_genes_ttest": lambda: rank_genes(ad, method="t-test", **kw)}
    for f in runs.values():
        f()
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
    print("end_to_end", json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ttest_timing.py measures on a GPU; none found")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    res["copy_peak_gbs"] = copy_peak_gbs(a.reps)
    print("copy_peak_gbs", res["copy_peak_gbs"], flush=True)
    res["passes"] = passes(a.reps, res["copy_peak_gbs"])
    res["end_to_end"] = end_to_end(a.e2e_reps)
    res["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
