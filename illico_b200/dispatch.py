"""The six batch dispatchers behind the reference's plug-in signature.

    f(X, chunk_lb, chunk_ub, grpc, is_log1p, use_continuity, tie_correct, alternative)
        -> (pvalues, statistics, fold_change)        each C-contiguous float64 [n_groups, chunk_ub - chunk_lb]

(call site ``illico/asymptotic_wilcoxon.py:59-67``; registered like ``illico/utils/registry.py:193-202``).
``X`` is a host ``ndarray``, a ``CSRMatrix`` / ``CSCMatrix`` namedtuple ``(data, indices, indptr, shape)``
(``illico/utils/sparse/csc.py:10-11``), a scipy matrix, or an already resident :class:`DeviceMatrix`.
Each call stages and ranks genes ``[chunk_lb, chunk_ub)`` on the current CUDA device through the C ABI.
These functions can be dropped into the reference's own ``dispatcher_registry`` for A/B runs (INTEGRATION.md).
"""
from __future__ import annotations

import threading
import zlib
from collections import OrderedDict, namedtuple

import numpy as np
import torch

from .engine import CSC, CSR, DENSE, DeviceMatrix, Engine, make_flags
from .groups import seg_max_from_env

CSCMatrix = namedtuple("CSCMatrix", ["data", "indices", "indptr", "shape"])
CSRMatrix = namedtuple("CSRMatrix", ["data", "indices", "indptr", "shape"])

_lock = threading.RLock()
_engines: "OrderedDict[tuple, Engine]" = OrderedDict()
_matrices: "OrderedDict[tuple, tuple]" = OrderedDict()
_MAX_CACHE = 4
_FP_SAMPLES = 1 << 16


def _ptr(a) -> int:
    return int(np.asarray(a).__array_interface__["data"][0])


def _fingerprint(a) -> int:
    """Cheap content check of a host array: CRC of ~64k evenly spaced elements plus both ends.  An in-place
    transformation of the matrix (normalisation, ``log1p``) changes it; it is not a proof of equality, which is why
    :func:`clear_caches` exists and INTEGRATION.md names it."""
    a = np.asarray(a)
    if a.size == 0:
        return 0
    if a.flags.c_contiguous or a.flags.f_contiguous:
        flat = a.ravel(order="K")                      # a view
        step = max(1, flat.size // _FP_SAMPLES)
        parts = (flat[::step], flat[:1024], flat[-1024:])
    else:
        rs, cs = max(1, a.shape[0] // 256), max(1, (a.shape[1] if a.ndim > 1 else 1) // 256)
        parts = (a[::rs, ::cs] if a.ndim > 1 else a[::rs],)
    crc = 0
    for part in parts:
        crc = zlib.crc32(np.ascontiguousarray(part).view(np.uint8), crc)
    return crc


def engine_for(grpc, device=None) -> Engine:
    """One engine per (group encoding CONTENT, reference group, plan segment length, device); tiny LRU so that the
    reference's driver, which calls a dispatcher once per gene batch with the same GroupContainer, reuses the plan.
    Keyed on a checksum of the codes (2.4 MB at 300k cells, about a millisecond), not on an address: a relabelled or
    re-created array never returns a stale plan, and a changed ``ILLICO_B200_SEG_MAX`` builds a new one."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    enc = np.ascontiguousarray(grpc.encoded_groups, dtype=np.int64)
    seg_max = seg_max_from_env()
    key = (zlib.crc32(enc.view(np.uint8)), zlib.adler32(enc.view(np.uint8)), enc.size, int(grpc.encoded_ref_group), seg_max,
           str(dev))
    with _lock:
        eng = _engines.get(key)
        if eng is None:
            eng = Engine(grpc, dev, seg_max=seg_max)
            _engines[key] = eng
            while len(_engines) > _MAX_CACHE:
                _engines.popitem(last=False)
        else:
            _engines.move_to_end(key)
        return eng


def _resident(X, fmt: str, eng: Engine) -> DeviceMatrix:
    """Device copy of a host matrix handed to a dispatcher.  The reference's driver passes the WHOLE in-RAM matrix with
    every gene batch (``InRAMDataHandler.fetch``, ``illico/utils/registry.py:97-100``), so the upload is kept between
    calls -- keyed on the addresses of all the matrix's arrays, its shape and dtype, and validated on every hit by a
    content fingerprint, so that a matrix transformed in place between two runs is uploaded again.  Pass a
    :class:`DeviceMatrix` (``Engine.upload_*``) to manage residency explicitly; :func:`clear_caches` drops everything."""
    if isinstance(X, DeviceMatrix):
        return X
    arrays = (X,) if fmt == DENSE else (X.data, X.indices, X.indptr)
    key = (tuple(_ptr(a) for a in arrays), tuple(X.shape), str(np.asarray(arrays[0]).dtype), fmt, str(eng.device))
    fp = tuple(_fingerprint(a) for a in arrays)
    with _lock:
        hit = _matrices.get(key)
        if hit is not None and hit[1] == fp:
            _matrices.move_to_end(key)
            return hit[0]
        M = eng.upload_dense(X) if fmt == DENSE else eng.upload_sparse(X, fmt)
        _matrices[key] = (M, fp, X)  # the host object is kept alive so that its addresses stay unique
        while len(_matrices) > 2:
            _matrices.popitem(last=False)
        return M


def clear_caches() -> None:
    """Drops the cached plans and device copies (call it after modifying a matrix in place if in doubt)."""
    with _lock:
        _engines.clear()
        _matrices.clear()


_tls = threading.local()


def _thread_stream(device) -> torch.cuda.Stream:
    """One CUDA stream per host thread and device: the reference's joblib threads then run their batches concurrently on
    the GPU instead of queueing on the default stream (the C ABI never synchronises)."""
    streams = getattr(_tls, "streams", None)
    if streams is None:
        streams = _tls.streams = {}
    st = streams.get(str(device))
    if st is None:
        st = streams[str(device)] = torch.cuda.Stream(device=device)
    return st


def _dispatch(fmt: str, X, chunk_lb, chunk_ub, grpc, is_log1p, use_continuity, tie_correct, alternative, debug=None):
    eng = engine_for(grpc)
    lb, ub = int(chunk_lb), int(chunk_ub)
    b = ub - lb
    flags = make_flags(is_log1p, use_continuity, tie_correct, alternative, fmt)
    stream = _thread_stream(eng.device)
    with torch.cuda.device(eng.device), torch.cuda.stream(stream):
        M = _resident(X, fmt, eng)
        res = torch.empty((eng.n_groups, max(b, 0), 3), dtype=torch.float64, device=eng.device)
        eng.run_batch(M, lb, ub, flags, res, 0, debug)
        host = torch.empty(res.shape, dtype=torch.float64, pin_memory=True)
        host.copy_(res, non_blocking=True)
        stream.synchronize()          # this thread's stream only: the caller gets host arrays back
    host = host.numpy()
    return (np.ascontiguousarray(host[:, :, 0]), np.ascontiguousarray(host[:, :, 1]),
            np.ascontiguousarray(host[:, :, 2]))


def _make(fmt: str, test: str):
    def dispatcher(X, chunk_lb, chunk_ub, grpc, is_log1p, use_continuity=True, tie_correct=True,
                   alternative="two-sided", debug=None):
        is_ovo = int(grpc.encoded_ref_group) >= 0
        if is_ovo != (test == "ovo"):
            raise ValueError(f"{test} dispatcher called with encoded_ref_group={grpc.encoded_ref_group}")
        return _dispatch(fmt, X, chunk_lb, chunk_ub, grpc, is_log1p, use_continuity, tie_correct, alternative, debug)

    dispatcher.__name__ = f"{fmt}_{test}_mwu_kernel_over_contiguous_col_chunk"
    dispatcher.__qualname__ = dispatcher.__name__
    dispatcher.__doc__ = f"B200 {test.upper()} rank-sum test over a contiguous gene chunk of a {fmt} matrix."
    return dispatcher


dense_ovr_mwu_kernel_over_contiguous_col_chunk = _make(DENSE, "ovr")
dense_ovo_mwu_kernel_over_contiguous_col_chunk = _make(DENSE, "ovo")
csc_ovr_mwu_kernel_over_contiguous_col_chunk = _make(CSC, "ovr")
csc_ovo_mwu_kernel_over_contiguous_col_chunk = _make(CSC, "ovo")
csr_ovr_mwu_kernel_over_contiguous_col_chunk = _make(CSR, "ovr")
csr_ovo_mwu_kernel_over_contiguous_col_chunk = _make(CSR, "ovo")


def _register() -> None:
    from .registry import KernelDataFormat, Test, dispatcher_registry

    for fmt, kf in ((DENSE, KernelDataFormat.DENSE), (CSC, KernelDataFormat.CSC), (CSR, KernelDataFormat.CSR)):
        for test, tt in (("ovr", Test.OVR), ("ovo", Test.OVO)):
            dispatcher_registry.register(tt, kf)(globals()[f"{fmt}_{test}_mwu_kernel_over_contiguous_col_chunk"])


_register()
