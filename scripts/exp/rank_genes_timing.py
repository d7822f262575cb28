"""Cost of the score plane and of ranking on the device (rank_genes), on one GPU.

  1. kernel step of the K562-shape dense OVO, CSR OVO and dense continuous OVO workloads (bench.py's inputs) with the score
     plane off and on, alternating, CUDA events; the results of both must be bit-identical;
  2. illico_bh_adjust + illico_top_genes at K562 (k = 100 and k = N), at the config-5 shard and at 50 x 40 000, next to
     the device-to-host copy of the [G, N, 3] result they replace;
  3. end to end from host memory (dense pinned, CSR): rank_genes(n_genes=100) against asymptotic_wilcoxon(...) returning
     its DataFrame, alternating (and with devices="all" when there are several GPUs).

Usage: python scripts/exp/rank_genes_timing.py [--reps 9] [--e2e-reps 3] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def stats(ms):
    ms = sorted(ms)
    return {"median_ms": ms[len(ms) // 2], "min_ms": ms[0], "max_ms": ms[-1], "n": len(ms)}


def kernel_steps(reps):
    import bench

    class A:
        seed, cells, genes, perts = 0, 0, 0, 0

    out = {}
    dev = torch.device("cuda", 0)
    for name in ("dense_ovo", "csr_ovo", "dense_ovo_continuous"):
        w = bench.Workload(name, A(), dev, 0, 1)
        sc = torch.empty((w.G, w.genes), dtype=torch.float64, device=dev)
        res_off = torch.empty_like(w.results)

        def off():
            for lb, ub in w.batches:
                w.eng.run_batch(w.M, lb, ub, w.flags, res_off, lb)

        def on():
            for lb, ub in w.batches:
                w.eng.run_batch(w.M, lb, ub, w.flags, w.results, lb, scores=sc)

        for _ in range(3):
            off(), on()
        torch.cuda.synchronize()
        t_off, t_on = [], []
        for _ in range(reps):
            t_off.append(timed(off))
            t_on.append(timed(on))
        same = bool(torch.equal(res_off.view(torch.int64), w.results.view(torch.int64)))
        out[name] = {"G": w.G, "N": w.genes, "score_off": stats(t_off), "score_on": stats(t_on), "results_identical": same,
                     "score_plane_mb": w.G * w.genes * 8 / 1e6}
        print(name, json.dumps(out[name]), flush=True)
        del w, sc, res_off
        torch.cuda.empty_cache()
    return out


def selection(reps):
    from illico_b200 import _lib

    lib = _lib.load()
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    for G, N, k in ((2001, 8000, 100), (2001, 8000, 8000), (10001, 2500, 100), (50, 40000, 100)):
        g = torch.Generator(device=dev).manual_seed(G + N)
        res = torch.rand((G, N, 3), dtype=torch.float64, device=dev, generator=g)
        sc = torch.randn((G, N), dtype=torch.float64, device=dev, generator=g) * 5
        padj = torch.empty((G, N), dtype=torch.float64, device=dev)
        ws = torch.empty(max(int(lib.illico_bh_workspace_bytes(G, N)), int(lib.illico_top_genes_workspace_bytes(G, N))),
                         dtype=torch.uint8, device=dev)
        gene = torch.empty((G, k), dtype=torch.int32, device=dev)
        rec = torch.empty((G, k, 5), dtype=torch.float64, device=dev)
        host = torch.empty((G, N, 3), dtype=torch.float64, pin_memory=True)

        def bh():
            _lib.check(lib.illico_bh_adjust(res.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), ws.data_ptr(), ws.numel(), st), "bh")

        def top():
            _lib.check(lib.illico_top_genes(sc.data_ptr(), N, res.data_ptr(), 3 * N, padj.data_ptr(), G, N, k, 0, gene.data_ptr(),
                                            rec.data_ptr(), ws.data_ptr(), ws.numel(), st), "top")

        def d2h():
            host.copy_(res, non_blocking=True)

        for _ in range(2):
            bh(), top(), d2h()
        torch.cuda.synchronize()
        t_bh, t_top, t_d2h = [], [], []
        for _ in range(reps):
            t_bh.append(timed(bh))
            t_top.append(timed(top))
            t_d2h.append(timed(d2h))
        out[f"G{G}_N{N}_k{k}"] = {"bh_adjust": stats(t_bh), "top_genes": stats(t_top), "d2h_results": stats(t_d2h),
                                  "results_mb": G * N * 24 / 1e6}
        print(G, N, k, json.dumps(out[f"G{G}_N{N}_k{k}"]), flush=True)
        del res, sc, padj, ws, gene, rec, host
        torch.cuda.empty_cache()
    return out


def end_to_end(reps):
    import pandas as pd
    from scipy import sparse

    import bench
    from illico_b200 import asymptotic_wilcoxon, rank_genes
    from illico_b200.asymptotic_wilcoxon import _run_tests

    dev = torch.device("cuda", 0)
    cells, genes, perts = 300_000, 8_000, 2_000
    labels, ref = bench.make_labels(0, cells, perts, {"test": "ovo"})
    Xd = bench.gen_dense("counts", 17, cells, genes, dev)
    pinned = torch.empty((cells, genes), dtype=torch.float32, pin_memory=True)
    pinned.copy_(Xd)
    v, c, p = bench.gen_csr("counts", 17, cells, genes, dev)
    Xcsr = sparse.csr_matrix((v.cpu().numpy(), c.cpu().numpy(), p.cpu().numpy()), shape=(cells, genes))
    del Xd, v, c, p
    torch.cuda.empty_cache()
    out = {}
    device_sets = [None] + (["all"] if torch.cuda.device_count() > 1 else [])
    for fmt, X in (("dense_pinned", pinned.numpy()), ("csr", Xcsr)):
        ad = bench.Ad(X, labels, genes)
        ad.obs = pd.DataFrame({"pert": pd.Categorical(labels)})
        for devices in device_sets:
            kw = dict(is_log1p=False, group_keys="pert", reference=ref, devices=devices)
            runs = {"asymptotic_wilcoxon_frame": lambda: asymptotic_wilcoxon(ad, **kw),
                    "rank_genes_100": lambda: rank_genes(ad, n_genes=100, **kw),
                    # rank_genes' first phase alone: the tests with the score plane, results left on the device
                    "tests_on_device": lambda: _run_tests(ad, False, "pert", ref, 1, "auto", "two-sided", True, True, None, None,
                                                          devices, score=True, on_device=True)}
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
            key = f"{fmt}_devices_{devices or 'one'}"
            out[key] = {k: stats(v) for k, v in t.items()}
            print(key, json.dumps(out[key]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_genes_timing.py measures on a GPU; none found")
    res = {"card": card()}
    print(json.dumps(res["card"]), flush=True)
    res["kernel_step"] = kernel_steps(a.reps)
    res["selection"] = selection(a.reps)
    res["end_to_end"] = end_to_end(a.e2e_reps)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
