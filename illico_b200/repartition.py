"""Rows -> genes repartition of an in-RAM CSR matrix across the GPUs of one host (SURVEY.md section 8e).

The path shards by genes, a CSR matrix is laid out by rows.  Instead of cutting gene ranges out of every row on the host
(the reference's ``csr_get_contig_cols_into_csr``, ``illico/utils/sparse/csr.py:144-196``) or sending the whole matrix to
every GPU, each GPU receives one contiguous block of ROWS -- plain slices of ``data`` / ``indices``, no host work, every
byte crosses PCIe once -- and the GPUs exchange the pieces over NVLink: the kernel that cuts a row block writes each row
piece straight into the owning GPU's shard arrays through peer memory (``csrc/repart.cu``).  No GPU ever holds more than
its row block plus its gene shard.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, hostio
from .engine import CSR, DeviceMatrix, _torch_dtype, _uploadable

UNSORTED = ("Input data matrix indices are not sorted. This is very unusual and may lead to incorrect results. "
            "This can be the result of operations like `adata[:, np.random.choice(…)]` that do not preserve sorting."
            "Please make sure that indices used to chunk the adata or the expression matrix have been sorted "
            "prior to computing DE genes.")


def peer_access_ok(devices) -> bool:
    """Every GPU of the list can map every other one's memory (NVLink / NVSwitch boxes)."""
    idx = [d.index if d.index is not None else torch.cuda.current_device() for d in devices]
    return all(a == b or torch.cuda.can_device_access_peer(a, b) for a in idx for b in idx)


def row_blocks(indptr: np.ndarray, k: int) -> list:
    """``k`` contiguous row ranges with about the same number of stored values."""
    n = indptr.size - 1
    targets = indptr[-1] * np.arange(1, k, dtype=np.float64) / k
    cuts = np.searchsorted(indptr, targets, side="left")
    edges = np.concatenate([[0], np.clip(cuts, 0, n), [n]]).astype(np.int64)
    edges = np.maximum.accumulate(edges)
    return [(int(edges[i]), int(edges[i + 1])) for i in range(k)]


def repartition_csr(X, devices, gene_bounds, cols=None) -> list:
    """``X``: scipy CSR (float32-exact values); ``devices[j]`` gets genes ``[gene_bounds[j], gene_bounds[j + 1])`` of every
    row as a :class:`DeviceMatrix` (columns rebased to the shard).  Raises ``ValueError`` for unsorted row indices.
    ``cols`` (``select.ColumnSelection``): the genes are those of the selection -- each GPU compacts its row block to the
    selected columns (``select.compact``) before it counts and cuts it, so ``gene_bounds`` are in the selected-gene space."""
    import os
    import time

    timing = os.environ.get("ILLICO_REPART_TIMING") == "1"
    t_ = [time.perf_counter()]

    def lap(what):
        if timing:
            t_.append(time.perf_counter())
            print(f"[repartition] {what}: {1e3 * (t_[-1] - t_[-2]):.1f} ms", flush=True)

    lib = _lib.load()
    S = len(devices)
    assert S == len(gene_bounds) - 1 and 1 <= S <= 32
    n, N = X.shape
    data = _uploadable(np.ascontiguousarray(X.data))
    if _torch_dtype(data) != torch.float32:
        raise TypeError("repartition_csr handles float32 values")
    indices = np.ascontiguousarray(X.indices, dtype=np.int32)
    indptr = np.ascontiguousarray(X.indptr, dtype=np.int64)
    dev_idx = [d.index if d.index is not None else torch.cuda.current_device() for d in devices]
    for a in dev_idx:
        for b in dev_idx:
            _lib.check(lib.illico_enable_peer_access(a, b), "illico_enable_peer_access")
    blocks = row_blocks(indptr, S)
    lap("host arrays, peer access, row blocks")

    # ---- phase A: row block k goes to GPU k (asynchronous copies), which counts its rows' pieces per shard
    st = []
    for k, dev in enumerate(devices):
        r0, r1 = blocks[k]
        e0, e1 = int(indptr[r0]), int(indptr[r1])
        with torch.cuda.device(dev):
            d_ptr = torch.from_numpy(indptr[r0:r1 + 1] - e0).to(dev, non_blocking=True)
            d_data = torch.empty(e1 - e0, dtype=torch.float32, device=dev)
            d_idx = torch.empty(e1 - e0, dtype=torch.int32, device=dev)
            pend = [hostio.h2d_1d(d_data, data[e0:e1]), hostio.h2d_1d(d_idx, indices[e0:e1])]
            d_bounds = torch.tensor(list(gene_bounds), dtype=torch.int32, device=dev)
            cnt = torch.empty((S, max(r1 - r0, 1)), dtype=torch.int32, device=dev)
            totals = torch.zeros(S, dtype=torch.int64, device=dev)
            flag = torch.empty(1, dtype=torch.int32, device=dev)
        st.append(dict(dev=dev, r0=r0, r1=r1, ptr=d_ptr, data=d_data, idx=d_idx, pend=pend, bounds=d_bounds, cnt=cnt, totals=totals,
                       flag=flag))
    for s in st:
        with torch.cuda.device(s["dev"]):
            for p in s["pend"]:
                p.finish()
            stream = torch.cuda.current_stream(s["dev"]).cuda_stream
            nr = s["r1"] - s["r0"]
            sorted_ = lib.illico_check_csr_sorted(s["idx"].data_ptr(), s["ptr"].data_ptr(), nr, s["flag"].data_ptr(), stream)
            if sorted_ < 0:
                _lib.check(1, "illico_check_csr_sorted")
            if sorted_ != 1:
                raise ValueError(UNSORTED)
            if cols is not None:
                from .select import compact

                new_col = torch.from_numpy(cols.new_col()).to(s["dev"], non_blocking=True)
                s["ptr"], s["data"], s["idx"] = compact(s["data"], _lib.DTYPE_F32, s["idx"], s["ptr"].data_ptr(), nr, new_col)
            _lib.check(lib.illico_csr_shard_count(s["idx"].data_ptr(), s["ptr"].data_ptr(), nr, s["bounds"].data_ptr(), S,
                                                  s["cnt"].data_ptr(), s["totals"].data_ptr(), stream), "illico_csr_shard_count")
    lap("uploads started and joined, counts enqueued")
    tot = np.stack([s["totals"].cpu().numpy() for s in st])            # [block k][shard j]; the one host read of the set-up
    lap("uploads + counts done (device)")
    before = np.concatenate([np.zeros((1, S), dtype=np.int64), np.cumsum(tot, axis=0)[:-1]])   # entries of earlier blocks

    # ---- phase B: the shards' arrays, on their owners
    out = []
    for j, dev in enumerate(devices):
        with torch.cuda.device(dev):
            nnz_j = int(tot[:, j].sum())
            out.append(dict(data=torch.empty(nnz_j, dtype=torch.float32, device=dev),
                            idx=torch.empty(nnz_j, dtype=torch.int32, device=dev),
                            rows=torch.empty(n, dtype=torch.int32, device=dev)))
    for j, dev in enumerate(devices):      # the owners' allocations must exist before anybody writes into them
        torch.cuda.current_stream(dev).synchronize()
    lap("shard arrays allocated")
    PtrArr = C.c_void_p * S
    p_data = PtrArr(*[o["data"].data_ptr() for o in out])
    p_idx = PtrArr(*[o["idx"].data_ptr() for o in out])
    p_rows = PtrArr(*[o["rows"].data_ptr() for o in out])

    # ---- phase C: every GPU cuts its rows and stores the pieces where they belong (peer stores over NVLink)
    for k, s in enumerate(st):
        with torch.cuda.device(s["dev"]):
            nr = s["r1"] - s["r0"]
            if nr == 0:
                continue
            pos = torch.cumsum(s["cnt"], dim=1, dtype=torch.int64) - s["cnt"]            # exclusive scan over the block's rows
            pos += torch.from_numpy(before[k]).to(s["dev"]).unsqueeze(1)
            s["pos"] = pos
            _lib.check(lib.illico_csr_shard_scatter(s["data"].data_ptr(), s["idx"].data_ptr(), s["ptr"].data_ptr(), nr, s["r0"],
                                                    s["bounds"].data_ptr(), S, s["cnt"].data_ptr(), pos.data_ptr(), p_data, p_idx,
                                                    p_rows, torch.cuda.current_stream(s["dev"]).cuda_stream),
                       "illico_csr_shard_scatter")
    for s in st:
        torch.cuda.current_stream(s["dev"]).synchronize()

    lap("scatter (peer stores)")
    # ---- phase D: each owner's row pointer = the scan of its row counts
    shards = []
    for j, dev in enumerate(devices):
        with torch.cuda.device(dev):
            ptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(out[j]["rows"], dim=0, dtype=torch.int64, out=ptr[1:])
            width = int(gene_bounds[j + 1] - gene_bounds[j])
            shards.append(DeviceMatrix(CSR, (n, width), out[j]["data"], out[j]["idx"], ptr, gene_offset=int(gene_bounds[j])))
    lap("row pointers")
    return shards
