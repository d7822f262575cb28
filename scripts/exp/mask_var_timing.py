"""Cost of ``mask_var=`` on one GPU, at the K562 shape (300 000 cells x 8 000 genes, 2 000 perturbations plus the control,
~9.5 % non-zero integer counts), one-versus-reference, with 2 000 of the 8 000 genes selected, scattered.

  1. end to end, from a pinned host matrix, a pageable host matrix, a host CSR matrix and a CUDA tensor: the full call,
     the call with ``mask_var``, and a host subset ``X[:, mask]`` (numpy / scipy; torch indexing for the CUDA tensor)
     followed by the full call on it; variants alternated, medians;
  2. bytes that crossed PCIe: the packed upload's count (``hostio.LAST_UPLOAD``; -1 when the upload did not pack) for
     dense host input, the stored arrays for CSR (it goes up whole with ``mask_var``), none for the CUDA tensor;
  3. the device column cuts alone: the dense gather (``illico_select_cols_dense`` through ``select.select_cols``) on the
     CUDA tensor, and the CSR compaction on the matrix in HBM: CUDA events, medians, and their bytes (read + write) over a
     device-to-device copy rate measured in the same call; for the gather also the bytes of the 32-byte sectors its reads
     touch, which is what DRAM moves.
The card's name and power limit are read in the same call.

Usage: python scripts/exp/mask_var_timing.py [--reps 5] [--out results.json]
"""
from __future__ import annotations

import argparse
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

from pct_nz_timing import copy_peak_gbs  # noqa: E402
from rank_genes_timing import card, stats, timed  # noqa: E402

CELLS, GENES, PERTS, SELECTED = 300_000, 8_000, 2_000, 2_000


class AD:
    def __init__(self, X, labels, mask):
        self.X, self.layers = X, {}
        self.obs = pd.DataFrame({"pert": pd.Categorical(labels)})
        self.var_names = pd.Index([f"g{i}" for i in range(X.shape[1])])
        self.var = pd.DataFrame({"highly_variable": mask}, index=self.var_names) if mask is not None else pd.DataFrame(index=self.var_names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    from illico_b200 import _lib, asymptotic_wilcoxon, hostio, synth
    from illico_b200.engine import DENSE, DeviceMatrix
    from illico_b200.registry import CSRDataHandler
    from illico_b200.select import ColumnSelection, compact, select_cols

    out = {"card": card(), "shape": [CELLS, GENES, PERTS], "selected_genes": SELECTED}
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.RandomState(0)
    labels, _ = synth.perturbation_labels(rng, CELLS, PERTS)
    labels = np.asarray(labels)
    mask = np.zeros(GENES, bool)
    mask[np.sort(rng.choice(GENES, SELECTED, replace=False))] = True
    cols = np.flatnonzero(mask)
    Xd = synth.k562_like_torch(0, CELLS, GENES, device=dev)
    torch.cuda.synchronize()
    pageable = Xd.cpu().numpy()
    pinned = torch.empty((CELLS, GENES), dtype=torch.float32, pin_memory=True)
    pinned.copy_(Xd)
    csr_d = Xd.to_sparse_csr()
    csr = sparse.csr_matrix((csr_d.values().cpu().numpy(), csr_d.col_indices().cpu().numpy().astype(np.int32),
                             csr_d.crow_indices().cpu().numpy()), shape=(CELLS, GENES))
    del csr_d
    torch.cuda.empty_cache()
    inputs = {"dense_pinned": pinned.numpy(), "dense_pageable": pageable, "csr": csr, "cuda_tensor": Xd}
    d_cols = torch.from_numpy(cols).to(dev)

    def subset(X):
        if isinstance(X, torch.Tensor):
            return X[:, d_cols]
        return X[:, mask]

    def call(X, variant):
        t0 = time.perf_counter()
        if variant == "host_subset":
            X = subset(X)
        asymptotic_wilcoxon(AD(X, labels, mask if variant == "masked" else None), False, "pert", synth.CONTROL,
                            mask_var="highly_variable" if variant == "masked" else None, return_array=True)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    variants = ("full", "masked", "host_subset")
    e2e, pcie = {}, {}
    for name, X in inputs.items():
        for v in variants:                               # warm-up of every shape
            call(X, v)
        times = {v: [] for v in variants}
        for _ in range(a.reps):
            for v in variants:                           # alternated
                hostio.LAST_UPLOAD.clear()
                times[v].append(call(X, v))
                if name.startswith("dense"):
                    pcie[f"{name}/{v}"] = int(hostio.LAST_UPLOAD.get("bytes", -1))
        e2e[name] = {v: stats(t) for v, t in times.items()}
        for v in variants:
            e2e[name][v]["vs_full"] = e2e[name][v]["median_ms"] / e2e[name]["full"]["median_ms"]
        print(name, {v: round(s["median_ms"], 1) for v, s in e2e[name].items()}, flush=True)
    whole = csr.data.nbytes + csr.indices.nbytes + (CELLS + 1) * 8
    sub = csr[:, mask]
    pcie["csr/full"] = pcie["csr/masked"] = int(whole)
    pcie["csr/host_subset"] = int(sub.data.nbytes + sub.indices.nbytes + (CELLS + 1) * 8)
    for v in variants:
        pcie[f"cuda_tensor/{v}"] = 0
    out["e2e_ms"], out["pcie_bytes"] = e2e, pcie

    peak = copy_peak_gbs(a.reps)
    out["copy_peak_gbs"] = peak
    sel = ColumnSelection(cols, GENES)
    kern = {}
    M_dense = DeviceMatrix(DENSE, (CELLS, GENES), Xd)
    for _ in range(2):
        select_cols(M_dense, (0, GENES), sel, 0, SELECTED)
    ms = stats([timed(lambda: select_cols(M_dense, (0, GENES), sel, 0, SELECTED)) for _ in range(a.reps)])
    ms["bytes"] = 2 * CELLS * SELECTED * 4 + SELECTED * 4          # the selected values read and written, the column list
    ms["gbs"] = ms["bytes"] / (ms["median_ms"] * 1e-3) / 1e9
    ms["of_copy_peak"] = ms["gbs"] / peak
    # what DRAM has to move: memory is read in 32-byte sectors, and a row's scattered selected columns touch most of them
    sectors = np.unique(cols // 8).size
    ms["sector_bytes"] = CELLS * (sectors * 32 + SELECTED * 4)
    ms["sector_gbs"] = ms["sector_bytes"] / (ms["median_ms"] * 1e-3) / 1e9
    ms["sector_of_copy_peak"] = ms["sector_gbs"] / peak
    kern["dense_gather"] = ms
    print("dense gather", ms, flush=True)
    M_csr, _ = CSRDataHandler(csr).upload_shard(0, GENES, dev)
    M_csr.ready()
    new_col = torch.from_numpy(sel.new_col()).to(dev)

    def compact_csr():
        return compact(M_csr.data, _lib.DTYPE_F32, M_csr.indices, M_csr.indptr.data_ptr(), CELLS, new_col)

    for _ in range(2):
        kept = int(compact_csr()[0][-1].item())
    ms = stats([timed(compact_csr) for _ in range(a.reps)])
    nnz = csr.nnz
    # count pass: row pointers and column indices read; compaction: values and indices read, kept entries written, the
    # new row pointer written twice (lengths, then their scan)
    ms["bytes"] = (CELLS + 1) * 8 + nnz * 4 + nnz * 8 + kept * 8 + 2 * (CELLS + 1) * 8
    ms["gbs"] = ms["bytes"] / (ms["median_ms"] * 1e-3) / 1e9
    ms["of_copy_peak"] = ms["gbs"] / peak
    kern["csr_compaction"] = ms
    print("csr compaction", ms, flush=True)
    out["select_kernels"] = kern
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
