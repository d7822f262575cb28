"""Cost of ``groups=`` one-versus-reference on one GPU, at the K562 shape (300 000 cells x 8 000 genes, 2 000 perturbations
plus the control, ~9.5 % non-zero integer counts).

  1. end to end: ``asymptotic_wilcoxon(..., reference=control, groups=...)`` with 20, 200 and 2 000 (every) perturbations
     against the same call without ``groups``, from a pinned host matrix, a pageable host matrix, a CUDA tensor and a host
     CSR matrix; variants alternated, medians;
  2. bytes that crossed PCIe: the packed upload's count (``hostio.LAST_UPLOAD``) for dense host input, the stored arrays
     of the selected rows for CSR, none for the CUDA tensor;
  3. the device selection kernels alone (``select.select_rows`` on the CUDA tensor and on the CSR matrix in HBM): CUDA
     events, medians, and their bytes (read + write) over a device-to-device copy peak measured in the same call.
The card's name and power limit are read in the same call.

Usage: python scripts/exp/groups_timing.py [--reps 5] [--out results.json]
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

CELLS, GENES, PERTS = 300_000, 8_000, 2_000


class AD:
    def __init__(self, X, labels):
        self.X, self.layers = X, {}
        self.obs = pd.DataFrame({"pert": pd.Categorical(labels)})
        self.var_names = pd.Index([f"g{i}" for i in range(X.shape[1])])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    a = ap.parse_args()
    from illico_b200 import asymptotic_wilcoxon, hostio, synth
    from illico_b200.groups import encode_and_count_groups, select_groups, subset_for_reference
    from illico_b200.registry import CSRDataHandler
    from illico_b200.select import RowSelection, select_rows

    out = {"card": card(), "shape": [CELLS, GENES, PERTS]}
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rng = np.random.RandomState(0)
    labels, _ = synth.perturbation_labels(rng, CELLS, PERTS)
    labels = np.asarray(labels)
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
    perts = sorted(set(labels) - {synth.CONTROL})
    picks = {"none": None, "20": perts[::PERTS // 20][:20], "200": perts[::PERTS // 200][:200], "2000": perts}
    uniq, grpc = encode_and_count_groups(labels, synth.CONTROL)
    share = {}
    for k, g in picks.items():
        sel = select_groups(uniq, g, grpc.encoded_ref_group) if g is not None else None
        share[k] = 1.0 if sel is None else float(np.isin(grpc.encoded_groups, sel).mean())
    out["selected_cell_share"] = share
    inputs = {"dense_pinned": pinned.numpy(), "dense_pageable": pageable, "cuda_tensor": Xd, "csr": csr}

    def call(X, groups):
        t0 = time.perf_counter()
        asymptotic_wilcoxon(AD(X, labels), False, "pert", synth.CONTROL, groups=groups, return_array=True)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    e2e, pcie = {}, {}
    for name, X in inputs.items():
        for k, g in picks.items():                      # warm-up of every shape
            call(X, g)
        times = {k: [] for k in picks}
        for _ in range(a.reps):
            for k, g in picks.items():                  # alternated
                hostio.LAST_UPLOAD.clear()
                times[k].append(call(X, g))
                if name.startswith("dense"):
                    pcie[f"{name}/{k}"] = int(hostio.LAST_UPLOAD.get("bytes", -1))
        e2e[name] = {k: stats(v) for k, v in times.items()}
        for k in picks:
            e2e[name][k]["vs_no_groups"] = e2e[name][k]["median_ms"] / e2e[name]["none"]["median_ms"]
        print(name, {k: round(v["median_ms"], 1) for k, v in e2e[name].items()}, flush=True)
    for k, g in picks.items():
        sel = select_groups(uniq, g, grpc.encoded_ref_group) if g is not None else None
        rows = np.arange(CELLS) if sel is None else subset_for_reference(grpc, sel)[0]
        pcie[f"csr/{k}"] = int((csr.indptr[rows + 1] - csr.indptr[rows]).sum()) * 8 + (rows.size + 1) * 8
        pcie[f"cuda_tensor/{k}"] = 0
    out["e2e_ms"], out["pcie_bytes"] = e2e, pcie

    peak = copy_peak_gbs(a.reps)
    out["copy_peak_gbs"] = peak
    from illico_b200.engine import DENSE, DeviceMatrix

    M_dense = DeviceMatrix(DENSE, (CELLS, GENES), Xd)
    M_csr, _ = CSRDataHandler(csr).upload_shard(0, GENES, dev)
    M_csr.ready()
    kern = {}
    for k in ("20", "200"):
        rows, _ = subset_for_reference(grpc, select_groups(uniq, picks[k], grpc.encoded_ref_group))
        sel = RowSelection(rows, CELLS)
        for name, M in (("dense", M_dense), ("csr", M_csr)):
            for _ in range(2):
                S, _ = select_rows(M, (0, GENES), sel)
            ms = stats([timed(lambda: select_rows(M, (0, GENES), sel)) for _ in range(a.reps)])
            # read + write: the rows' values (CSR: values and column indices, and each row's two indptr entries and its new one)
            moved = 2 * rows.size * GENES * 4 if name == "dense" else 2 * int(S.indptr[-1].item()) * 8 + rows.size * 8 * 3
            ms["bytes"] = moved
            ms["gbs"] = moved / (ms["median_ms"] * 1e-3) / 1e9
            ms["of_copy_peak"] = ms["gbs"] / peak
            kern[f"{name}/{k}"] = ms
            print(name, k, ms, flush=True)
    out["select_kernels"] = kern
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
