"""Public entry point: ``asymptotic_wilcoxon`` with the reference's signature and output
(``illico/asymptotic_wilcoxon.py:71-258``), computed on a B200 through ``libillico_b200.so``.

What changed relative to the reference's driver (same contract, different machinery):
  * gene batches go to CUDA streams on one GPU instead of joblib threads (``n_threads`` is accepted and
    used only for host-side readers of backed data; ``precompile`` is a no-op: the kernels are built
    ahead of time);
  * ``batch_size`` is the number of genes per device batch; ``"auto"`` lets the engine size batches to
    its memory budget.  Every gene is computed (the reference's ``"auto"`` split skips one boundary gene
    per split, SURVEY.md section 0.5);
  * the one-versus-reference row of the reference group is always ``(p=1, U=-1, fc)`` (the reference's
    dense kernel leaves it uninitialised, ``ovo/dense_ovo.py:116-120``).
"""
from __future__ import annotations

import os
import threading
from queue import Empty, Queue
from typing import Literal

import numpy as np
import pandas as pd
import torch
from scipy import sparse

from . import hostio
from .engine import CSR, WILCOXON, DeviceMatrix, Engine, check_method, make_flags, require_cuda
from .groups import encode_and_count_groups, seg_max_from_env
from .registry import DataHandler, data_handler_registry

__all__ = ["asymptotic_wilcoxon"]


def _batches(lb: int, ub: int, batch_size, engine: Engine, in_ram: bool, method: str = WILCOXON):
    """Gene batches of the shard ``[lb, ub)`` (global gene indices)."""
    n_genes = ub - lb
    if isinstance(batch_size, (int, np.integer)) and not isinstance(batch_size, bool):
        if batch_size <= 0:
            raise ValueError(f"Invalid batch_size value: {batch_size}. Must be 'auto' or an integer.")
        step = min(int(batch_size), engine.max_batch_genes(n_genes, method))
    elif batch_size == "auto":
        step = engine.max_batch_genes(n_genes, method)
        if not in_ram:
            step = min(step, 256)  # backed data: stream ~256 genes at a time like the reference aims for
    else:
        raise ValueError(f"Invalid batch_size value: {batch_size}. Must be 'auto' or an integer.")
    step = max(1, step)
    bounds = list(range(lb, ub, step)) + [ub]
    return list(zip(bounds[:-1], bounds[1:]))


def operator(data_handler: DataHandler, lb: int, ub: int, engine: Engine, flags, results: torch.Tensor,
             fetched=None, result_gene0: int | None = None) -> None:
    """One gene batch: fetch -> device -> stage + rank, written into ``results[:, lb:ub, :]`` on the device
    (the reference's ``operator``, ``asymptotic_wilcoxon.py:29-68``)."""
    n_cols = data_handler.data.shape[1]
    if lb < 0 or ub > n_cols or lb > ub:
        raise ValueError(f"Invalid chunk bounds: {(lb, ub)} for data with {n_cols} columns.")
    if fetched is None:
        fetched = data_handler.fetch(lb, ub)
    data, bounds = fetched
    M = data if isinstance(data, DeviceMatrix) else data_handler.to_device(data, engine)
    engine.run_batch(M, bounds[0], bounds[1], flags, results, lb if result_gene0 is None else result_gene0)


def _device_list(device, devices) -> list:
    """``device`` (one GPU, the reference-compatible default) or ``devices`` ("all", a count, or a list)."""
    if devices is None:
        return [require_cuda(device)]
    if device is not None:
        raise ValueError("pass either device= or devices=, not both")
    require_cuda(None)
    n_all = torch.cuda.device_count()
    if isinstance(devices, str):
        if devices != "all":
            raise ValueError(f"devices must be 'all', a count or a list of devices, got {devices!r}")
        devs = list(range(n_all))
    elif isinstance(devices, (int, np.integer)):
        if not 1 <= int(devices) <= n_all:
            raise ValueError(f"devices={devices}: this host has {n_all} CUDA devices")
        devs = list(range(int(devices)))
    else:
        devs = list(devices)
    out = [require_cuda(torch.device("cuda", d) if isinstance(d, (int, np.integer)) else d) for d in devs]
    if not out or len({str(d) for d in out}) != len(out):
        raise ValueError("devices must name at least one GPU, each once")
    return out


class _Shard:
    """One GPU's share of a run: a contiguous gene range, its engine, its result slab."""

    def __init__(self, device, lb, ub):
        self.device, self.lb, self.ub = device, lb, ub
        self.error = None
        self.started = None     # (DeviceMatrix, bounds) of an upload started before the worker runs


def asymptotic_wilcoxon(
    adata,
    is_log1p: bool,
    group_keys: str,
    reference: str | None = None,
    n_threads: int = 1,
    batch_size: int | Literal["auto"] = "auto",
    alternative: str = "two-sided",
    use_continuity: bool = True,
    tie_correct: bool = True,
    layer: str | None = None,
    precompile: bool = True,
    device=None,
    devices=None,
    return_array: bool = False,
    p_adjust: bool = False,
    log2_fold_change: bool = False,
    score: bool = False,
    pts: bool = False,
):
    """Asymptotic Mann-Whitney / Wilcoxon rank-sum tests for every (group, gene) on B200 GPUs.

    Same parameters and result as ``illico.asymptotic_wilcoxon``: a ``pd.DataFrame`` indexed by
    ``MultiIndex.from_product([groups, var_names], names=["pert", "feature"])`` with float64 columns
    ``p_value``, ``statistic`` (U of the reference / rest sample) and ``fold_change``.

    Extra keyword arguments (not in the reference):
      ``device``   CUDA device (default: the current one, or where a CUDA-tensor matrix lives);
      ``devices``  ``"all"``, a count or a list: the genes are split into one contiguous shard per GPU; one host thread
                   per GPU uploads its shard, ranks it and writes its ``results[:, lb:ub]`` slab straight into the one
                   pinned result array -- no collective, no second process, one copy of ``adata`` in host memory
                   (the reference's thread pool over gene batches, ``asymptotic_wilcoxon.py:212-249``, across GPUs);
      ``return_array``  return ``(groups, var_names, results[G, N, 3])`` and skip the DataFrame;
      ``p_adjust`` / ``log2_fold_change``  add the columns ``p_adj`` (Benjamini-Hochberg over the genes of each group,
                   what ``scanpy.tl.rank_genes_groups`` reports as ``pvals_adj``) and ``log2_fold_change``;
      ``score``    add the column ``score``: the signed z of the normal approximation, ``(n_r n_t / 2 - U) / sigma`` with
                   the p-value's (tie-corrected) sigma and no continuity correction -- positive when the group ranks above
                   the reference / rest, 0 on the reference row and where p = 1 (scanpy's wilcoxon ``scores``).  Written
                   by the kernels next to the p-value;
      ``pts``      add the columns ``pct_nz_group`` (fraction of the group's cells whose value is non-zero) and
                   ``pct_nz_reference`` (the same fraction in the reference group, or in all other cells for one-versus-rest;
                   NaN when there are no other cells) -- scanpy's ``rank_genes_groups(pts=True)``.  Counted on the GPU in a
                   pass of its own; p-values, U and fold changes are those of the same call without it.
    With ``return_array`` and an optional column, the result is ``(groups, var_names, results, {name: [G, N] array})``.
    """
    del precompile  # kernels are compiled ahead of time
    check_flag("pts", pts)
    run = _run_tests(adata, is_log1p, group_keys, reference, n_threads, batch_size, alternative, use_continuity,
                     tie_correct, layer, device, devices, score=score, on_device=False, pts=pts)
    out = run.results
    extra = {}
    if p_adjust:
        extra["p_adj"] = _bh_adjust(out, run.device)
    if log2_fold_change:
        with np.errstate(divide="ignore", invalid="ignore"):
            extra["log2_fold_change"] = np.log2(out[:, :, 2])
    if score:
        extra["score"] = run.scores
    if pts:
        extra["pct_nz_group"], extra["pct_nz_reference"] = _host_fractions(run)
    if return_array:
        if extra:
            return run.groups, np.asarray(adata.var_names), out, extra
        return run.groups, np.asarray(adata.var_names), out
    return _result_frame(run.groups, adata.var_names, out, extra)


class _Run:
    """What ``_run_tests`` delivers: the groups (``np.unique`` order), the group container, the first GPU, and the results
    ``[G, N, 3]`` / score plane ``[G, N]`` / int32 count plane ``[G, N]`` of cells with a non-zero value (the planes None
    unless asked for) -- pinned host arrays, or tensors on that GPU."""

    def __init__(self, groups, grpc, device, results, scores, nnz=None):
        self.groups, self.grpc, self.device, self.results, self.scores, self.nnz = groups, grpc, device, results, scores, nnz


def check_flag(name: str, value) -> None:
    if not isinstance(value, (bool, np.bool_)):
        raise ValueError(f"{name} must be True or False, got {value!r}")


def nonzero_fractions(nnz: torch.Tensor, grpc):
    """``(pct_group, pct_ref)``, ``[G, N]`` float64 tensors on the device of the count plane ``nnz`` ``[G, N]`` int32
    (``illico_nonzero_fractions``: the one definition of the two fractions)."""
    from . import _lib

    G, N = int(nnz.shape[0]), int(nnz.shape[1])
    dev = nnz.device
    counts = np.asarray(grpc.counts, dtype=np.int64)
    with torch.cuda.device(dev):
        sizes = torch.from_numpy(counts.astype(np.int32)).to(dev)
        pg = torch.empty((G, N), dtype=torch.float64, device=dev)
        pr = torch.empty((G, N), dtype=torch.float64, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.load().illico_nonzero_fractions(nnz.data_ptr(), N, sizes.data_ptr(), G, N, int(grpc.encoded_ref_group),
                                                        int(counts.sum()), pg.data_ptr(), pr.data_ptr(), st),
                   "illico_nonzero_fractions")
    return pg, pr


def _host_fractions(run: _Run):
    """The fractions of a run whose count plane came back to the host: computed on the run's first GPU and copied back."""
    G, N = run.nnz.shape
    with torch.cuda.device(run.device):
        pg, pr = nonzero_fractions(torch.from_numpy(run.nnz).to(run.device, non_blocking=True), run.grpc)
        out = []
        for plane in (pg, pr):
            host = torch.empty((G, N), dtype=torch.float64, pin_memory=True)
            host.copy_(plane, non_blocking=True)
            out.append(host)
        torch.cuda.current_stream(run.device).synchronize()
    return out[0].numpy(), out[1].numpy()


def _run_tests(adata, is_log1p, group_keys, reference, n_threads, batch_size, alternative, use_continuity, tie_correct,
               layer, device, devices, score: bool, on_device: bool, pts: bool = False, method: str = WILCOXON) -> _Run:
    """Every (group, gene) test of ``adata``: validation, upload, group plan, one gene shard per GPU, batches, backed
    streaming.  ``on_device=False``: each shard's slabs are copied into pinned host arrays (``asymptotic_wilcoxon``).
    ``on_device=True``: they stay on the GPUs and meet in ``[G, N, 3]`` / ``[G, N]`` tensors on the first one
    (device-to-device copies; with one shard its own tensors are the result).  ``pts``: the count plane too.  ``method``:
    the Wilcoxon test or one of the t-tests (``Engine.run_batch``)."""
    check_method(method)
    X = adata.layers[layer] if layer is not None else adata.X
    if isinstance(X, (sparse.csr_array, sparse.csc_array)):
        X = sparse.csr_matrix(X) if isinstance(X, sparse.csr_array) else sparse.csc_matrix(X)
    data_handler = data_handler_registry.get(X)  # KeyError for unsupported containers, like the reference
    if devices is None and device is None and isinstance(X, torch.Tensor) and X.is_cuda:
        device = X.device          # a device-resident matrix is ranked where it lives
    seg_max = seg_max_from_env()   # an invalid ILLICO_B200_SEG_MAX fails before any device work
    devs = _device_list(device, devices)
    n_cells, n_genes = X.shape
    fmt = data_handler.kernel_data_format().value
    flags_for = lambda: make_flags(is_log1p, use_continuity, tie_correct, alternative, fmt)  # noqa: E731
    flags_for()  # validates `alternative` before any work starts
    if not (batch_size == "auto" or (isinstance(batch_size, (int, np.integer)) and not isinstance(batch_size, bool)
                                      and batch_size > 0)):
        raise ValueError(f"Invalid batch_size value: {batch_size}. Must be 'auto' or an integer.")

    from .parallel import gene_shard

    shards = [_Shard(d, *gene_shard(n_genes, r, len(devs))) for r, d in enumerate(devs)]
    shards = [sh for sh in shards if sh.ub > sh.lb] or [_Shard(devs[0], 0, n_genes)]
    plan_ready = threading.Event()
    shared: dict = {}
    # A CSR matrix on several GPUs: row blocks go up (each byte once), the GPUs cut them and exchange the pieces over
    # NVLink (repartition.py), instead of every GPU receiving the whole matrix
    prep = None
    if fmt == CSR and len(shards) > 1 and data_handler.in_ram and isinstance(X, sparse.csr_matrix) \
            and X.data.dtype == np.float32:
        from . import repartition

        if repartition.peer_access_ok([sh.device for sh in shards]):
            def _prep():
                try:
                    Ms = repartition.repartition_csr(X, [sh.device for sh in shards], [sh.lb for sh in shards] + [shards[-1].ub])
                    for sh, M in zip(shards, Ms):
                        sh.started = (M, (0, sh.ub - sh.lb))
                except BaseException as e:
                    shared["prep_error"] = e

            prep = threading.Thread(target=_prep, daemon=True)
            prep.start()

    def run_shard(sh: _Shard):
        """Everything one GPU does, on its own host thread: upload its gene shard (started before the groups are
        encoded), rank it batch by batch, deliver its slab."""
        try:
            if len(shards) > 1:
                hostio.bind_thread_to_device_node(sh.device.index if sh.device.index is not None else 0)
            if prep is not None:
                prep.join()
                if "prep_error" in shared:
                    raise shared["prep_error"]
            with torch.cuda.device(sh.device):
                M = bounds = None
                if data_handler.in_ram:
                    M, bounds = sh.started or data_handler.upload_shard(sh.lb, sh.ub, sh.device)
                plan_ready.wait()
                if "error" in shared:
                    return
                engine = Engine(shared["grpc"], sh.device, host_plan=shared["host_plan"])
                flags = flags_for()
                res = torch.empty((engine.n_groups, sh.ub - sh.lb, 3), dtype=torch.float64, device=sh.device)
                sc = torch.empty((engine.n_groups, sh.ub - sh.lb), dtype=torch.float64, device=sh.device) if score else None
                nz = torch.empty((engine.n_groups, sh.ub - sh.lb), dtype=torch.int32, device=sh.device) if pts else None
                if data_handler.in_ram:
                    M.ready()
                    if fmt == CSR and not engine.check_csr_sorted(M):
                        raise ValueError(
                            "Input data matrix indices are not sorted. This is very unusual and may lead to incorrect results. "
                            "This can be the result of operations like `adata[:, np.random.choice(…)]` that do not preserve sorting."
                            "Please make sure that indices used to chunk the adata or the expression matrix have been sorted "
                            "prior to computing DE genes."
                        )
                    off = bounds[0] - sh.lb      # gene g of the run is column g + off of the device matrix
                    for lb, ub in _batches(sh.lb, sh.ub, batch_size, engine, True, method):
                        engine.run_batch(M, lb + off, ub + off, flags, res, lb - sh.lb, scores=sc, nnz=nz, method=method)
                else:
                    _run_backed(data_handler, _batches(sh.lb, sh.ub, batch_size, engine, False, method), engine, flags, res,
                                max(1, int(n_threads)), gene0=sh.lb, scores=sc, nnz=nz, method=method)
                if on_device and len(shards) == 1:
                    shared["out"], shared["out_scores"], shared["out_nnz"] = res, sc, nz
                else:
                    kind = "d2d" if on_device else "d2h"
                    hostio.d2h_slab(shared["out"], res, sh.lb, kind)
                    if sc is not None:
                        hostio.d2h_slab(shared["out_scores"], sc, sh.lb, kind)
                    if nz is not None:
                        hostio.d2h_slab(shared["out_nnz"], nz, sh.lb, kind)
                torch.cuda.current_stream(sh.device).synchronize()
        except BaseException as e:  # re-raised on the calling thread
            sh.error = e

    workers = []
    hostio.CONCURRENT_UPLOADS = len(shards)
    if len(shards) > 1:
        workers = [threading.Thread(target=run_shard, args=(sh,), daemon=True) for sh in shards]
        for t in workers:
            t.start()
    try:
        # the reference goes through `.tolist()` + a dict loop (utils/groups.py:42-45); same encoding, vectorised.
        # With several GPUs the uploads are already running on the workers' threads while this happens.
        if len(shards) == 1 and data_handler.in_ram:
            # single GPU: start the upload from this thread, then encode while it is in flight
            with torch.cuda.device(shards[0].device):
                shards[0].started = data_handler.upload_shard(shards[0].lb, shards[0].ub, shards[0].device)
        unique_raw_groups, grpc = encode_and_count_groups(groups=adata.obs[group_keys], ref_group=reference)
        if grpc.encoded_groups.size != n_cells:
            raise ValueError(f"{grpc.encoded_groups.size} group labels for {n_cells} cells")
        from .groups import build_plan

        shared["grpc"], shared["host_plan"] = grpc, build_plan(grpc, seg_max)
        G = int(grpc.counts.size)
        if not on_device:
            shared["out"] = torch.empty((G, n_genes, 3), dtype=torch.float64, pin_memory=True)
            shared["out_scores"] = torch.empty((G, n_genes), dtype=torch.float64, pin_memory=True) if score else None
            shared["out_nnz"] = torch.empty((G, n_genes), dtype=torch.int32, pin_memory=True) if pts else None
        elif len(shards) > 1:
            shared["out"] = torch.empty((G, n_genes, 3), dtype=torch.float64, device=devs[0])
            shared["out_scores"] = torch.empty((G, n_genes), dtype=torch.float64, device=devs[0]) if score else None
            shared["out_nnz"] = torch.empty((G, n_genes), dtype=torch.int32, device=devs[0]) if pts else None
    except BaseException:
        shared["error"] = True
        plan_ready.set()
        for t in workers:
            t.join()
        raise
    plan_ready.set()
    if workers:
        for t in workers:
            t.join()
    else:
        run_shard(shards[0])
    for sh in shards:
        if sh.error is not None:
            raise sh.error
    out, scores, nnz = shared["out"], shared["out_scores"], shared.get("out_nnz")
    if not on_device:
        out, scores = out.numpy(), (scores.numpy() if scores is not None else None)
        nnz = nnz.numpy() if nnz is not None else None
    return _Run(unique_raw_groups, grpc, shards[0].device, out, scores, nnz)


def _bh_adjust(out: np.ndarray, device) -> np.ndarray:
    """Benjamini-Hochberg adjusted p-values over the genes of each group, ``[G, N]`` (needs every gene of a group, so
    it runs once on the gathered result, on one GPU: ``illico_bh_adjust``)."""
    import ctypes as C

    from . import _lib

    G, N = out.shape[0], out.shape[1]
    lib = _lib.load()
    with torch.cuda.device(device):
        res = torch.from_numpy(out).to(device, non_blocking=True)
        padj = torch.empty((G, N), dtype=torch.float64, device=device)
        ws = torch.empty(int(lib.illico_bh_workspace_bytes(G, N)), dtype=torch.uint8, device=device)
        st = torch.cuda.current_stream(device).cuda_stream
        _lib.check(lib.illico_bh_adjust(res.data_ptr(), 3 * N, 3, G, N, padj.data_ptr(), ws.data_ptr(), ws.numel(), st),
                   "illico_bh_adjust")
        host = torch.empty((G, N), dtype=torch.float64, pin_memory=True)
        host.copy_(padj, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
    del C
    return host.numpy()


def _result_frame(groups, var_names, out: np.ndarray, extra: dict | None = None) -> pd.DataFrame:
    """The reference's result (``asymptotic_wilcoxon.py:252-256``): same index as ``MultiIndex.from_product([groups,
    var_names], names=["pert", "feature"])`` and the same three float64 columns, but the index is built from its codes
    and the values are a view of the (pinned) result array: 15 ms instead of 0.2-0.45 s at 16 M rows."""
    G, N = out.shape[0], out.shape[1]
    rows = pd.Index(pd.Series(groups, dtype=str), name="pert")
    cols = pd.Index(pd.Series(var_names, dtype=str), name="feature")
    if not (rows.is_unique and cols.is_unique):   # from_product factorises duplicated labels: keep its semantics
        index = pd.MultiIndex.from_product([pd.Series(groups, name="pert", dtype=str), pd.Series(var_names, name="feature", dtype=str)],
                                           names=["pert", "feature"])
    else:
        ct = lambda n: np.int8 if n < 2**7 else np.int16 if n < 2**15 else np.int32 if n < 2**31 else np.int64  # noqa: E731
        index = pd.MultiIndex(levels=[rows, cols],
                              codes=[np.repeat(np.arange(G, dtype=ct(G)), N), np.tile(np.arange(N, dtype=ct(N)), G)],
                              names=["pert", "feature"], verify_integrity=False)
    df = pd.DataFrame(out.reshape(-1, 3), index=index, columns=["p_value", "statistic", "fold_change"], copy=False)
    for name, plane in (extra or {}).items():     # optional columns (default call: none, the reference's frame exactly)
        df[name] = plane.reshape(-1)
    return df


class _PinnedSlot:
    """One slot of the host-side ring: pinned staging arrays (grown on demand) + the event that says the device has
    finished copying out of them."""

    def __init__(self):
        self.bufs: dict = {}
        self.copied = None  # torch.cuda.Event recorded on the copy stream after the slot's H2D copies

    def stage(self, name: str, arr: np.ndarray) -> torch.Tensor:
        """Copies ``arr`` into the slot's pinned buffer ``name`` (reader thread) and returns the pinned view."""
        arr = np.ascontiguousarray(arr)
        buf = self.bufs.get(name)
        if buf is None or buf.numel() < arr.size or buf.dtype != torch.from_numpy(arr[:0]).dtype:
            buf = torch.empty(max(arr.size, 1), dtype=torch.from_numpy(arr[:0]).dtype, pin_memory=True)
            self.bufs[name] = buf
        view = buf[: arr.size]
        np.copyto(view.numpy(), arr.reshape(-1), casting="no")
        return view


def _run_backed(data_handler: DataHandler, iterator, engine: Engine, flags, results, n_readers: int, gene0: int = 0,
                scores=None, nnz=None, method: str = WILCOXON) -> None:
    """Out-of-core input (BASELINE config 4): gene batches stream disk -> pinned ring -> HBM -> kernels.

    Reader threads slice the next batches from the backed container straight into pinned staging buffers (a ring of
    ``n_readers + 2`` slots); the main thread enqueues each batch's ``cudaMemcpyAsync`` on a copy stream and the
    kernels on the compute stream, ordered by events, so the disk read and H2D copy of batch ``i + 1`` overlap the
    ranking of batch ``i`` (the reference's joblib threads overlap I/O and numba kernels the same way,
    ``asymptotic_wilcoxon.py:212-249``)."""
    from .engine import DENSE, DeviceMatrix, _to_f32_or_wide

    dev = engine.device
    order = list(iterator)
    n_slots = n_readers + 2
    free_slots: Queue = Queue()
    for _ in range(n_slots):
        free_slots.put(_PinnedSlot())
    ready: Queue = Queue(maxsize=n_slots)
    it = iter(enumerate(order))
    lock = threading.Lock()
    fmt = data_handler.kernel_data_format().value

    stop = threading.Event()

    def reader():
        while not stop.is_set():
            # the slot comes FIRST: whoever holds the lowest outstanding batch index then already owns a slot, so the
            # ring can never fill up with later batches while the batch the main thread waits for starves
            try:
                slot = free_slots.get(timeout=0.05)
            except Empty:
                continue
            with lock:
                nxt = next(it, None)
            if nxt is None:
                free_slots.put(slot)
                ready.put(None)
                return
            i, (lb, ub) = nxt
            try:
                if slot.copied is not None:
                    slot.copied.synchronize()   # the device is done reading this slot's previous batch
                data, bounds = data_handler.fetch(lb, ub)
                if fmt == DENSE:
                    staged = {"shape": data.shape, "x": slot.stage("x", data)}
                else:
                    staged = {"shape": data.shape, "data": slot.stage("data", data.data),
                              "indices": slot.stage("indices", np.asarray(data.indices, dtype=np.int32)),
                              "indptr": slot.stage("indptr", np.asarray(data.indptr, dtype=np.int64))}
                ready.put((i, lb, ub, bounds, slot, staged))
            except BaseException as e:  # surfaced on the main thread
                ready.put(e)
                return

    threads = [threading.Thread(target=reader, daemon=True) for _ in range(n_readers)]
    for t in threads:
        t.start()
    compute = torch.cuda.current_stream(dev)
    copy_stream = torch.cuda.Stream(device=dev)
    done, nxt_i, pending = 0, 0, {}
    queued = None   # (M, bounds, lb) of the batch whose copies are enqueued but whose kernels are not

    def enqueue_copies(lb, bounds, slot, staged):
        with torch.cuda.stream(copy_stream):
            # device buffers are allocated on the copy stream; the copies run while the previous batch ranks
            dv = {k: v.to(dev, non_blocking=True) for k, v in staged.items() if k != "shape"}
            slot.copied = torch.cuda.Event()
            slot.copied.record(copy_stream)
        free_slots.put(slot)
        return (dv, staged["shape"], bounds, lb, slot.copied)

    def rank(q):
        dv, shape, bounds, lb, copied = q
        compute.wait_event(copied)
        for t_ in dv.values():
            t_.record_stream(compute)   # allocated on the copy stream, consumed on the compute stream
        if fmt == DENSE:
            n, bsz = shape
            x, raw = dv["x"].view(n, bsz), None
            if x.dtype != torch.float32:
                x, raw = _to_f32_or_wide(x)
            M = DeviceMatrix(DENSE, (n, bsz), x, raw=raw)
        else:
            data, raw = dv["data"], None
            if data.dtype != torch.float32:
                data, raw = _to_f32_or_wide(data)
            M = DeviceMatrix(fmt, tuple(shape), data, dv["indices"], dv["indptr"], raw=raw)
        engine.run_batch(M, bounds[0], bounds[1], flags, results, lb - gene0, scores=scores, nnz=nnz, method=method)

    try:
        while done < n_readers:
            item = ready.get()
            if item is None:
                done += 1
                continue
            if isinstance(item, BaseException):
                raise item
            pending[item[0]] = item
            while nxt_i in pending:  # keep the gene order deterministic
                _i, lb, ub, bounds, slot, staged = pending.pop(nxt_i)
                nxt = enqueue_copies(lb, bounds, slot, staged)   # batch i + 1 starts copying ...
                if queued is not None:
                    rank(queued)                                  # ... while batch i ranks
                queued = nxt
                nxt_i += 1
        if queued is not None:
            rank(queued)
        assert nxt_i == len(order)
    finally:
        # error or not, no reader may stay blocked on a queue (they hold pinned buffers): stop them and drain
        stop.set()
        while any(t.is_alive() for t in threads):
            try:
                ready.get(timeout=0.02)
            except Empty:
                pass
        for t in threads:
            t.join()
