"""Device engine: owns the plan tables, the batch buffers and the stream, and drives the C-ABI calls.

PyTorch is plumbing here (device memory, streams, H2D/D2H copies); every compute kernel is in
``libillico_b200.so``.  One engine per (device, group plan).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import warnings
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .groups import GroupContainer, HostPlan, build_plan, check_seg_max

DENSE, CSC, CSR = "dense", "csc", "csr"
WILCOXON = "wilcoxon"
METHODS = (WILCOXON, "t-test", "t-test_overestim_var")   # scanpy rank_genes_groups' names


def check_method(method) -> str:
    if not isinstance(method, str) or method not in METHODS:
        raise ValueError(f"method must be one of {', '.join(repr(m) for m in METHODS)}, got {method!r}")
    return method


def _env_int(name: str, default: int) -> int:
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


@dataclass
class DeviceMatrix:
    """An expression matrix (or a gene shard of one) resident in HBM, in one of the three kernel formats."""

    fmt: str
    shape: tuple
    data: torch.Tensor | None     # dense: [n, ld] float32 ; sparse: [nnz] float32
    indices: torch.Tensor | None = None   # int32 [nnz]
    indptr: torch.Tensor | None = None    # int64
    gene_offset: int = 0          # genes [gene_offset, gene_offset + shape[1]) of the caller's matrix
    raw: torch.Tensor | None = None  # values float32 cannot hold exactly (float64 / big integers), as float64:
    #                                  `data` is then unused and every batch is recoded (Engine._run_batch_wide)
    pending: list = field(default_factory=list)   # hostio.Pending uploads still in flight
    unconverted: torch.Tensor | None = None       # uploaded values of another dtype, converted once the upload is in
    _lock: object = field(default_factory=threading.Lock, repr=False, compare=False)
    _ready_event: object = field(default=None, repr=False, compare=False)

    @property
    def ld(self) -> int:
        return int(self.data.stride(0)) if self.fmt == DENSE else 0

    def ready(self) -> "DeviceMatrix":
        """Joins the uploads (the current stream then waits for their copies) and converts non-float32 values.
        Call from the thread, and under the stream, that is going to launch kernels on this matrix; any number of
        threads / streams may do so (the first one finishes the upload, the others wait for its event)."""
        with self._lock:
            if self.pending or self.unconverted is not None:
                for p in self.pending:
                    p.finish()
                self.pending = []
                if self.unconverted is not None:
                    self.data, self.raw = _to_f32_or_wide(self.unconverted)
                    self.unconverted = None
                dev = (self.data if self.data is not None else self.raw).device
                self._ready_event = torch.cuda.Event()
                self._ready_event.record(torch.cuda.current_stream(dev))
                return self
            ev = self._ready_event
        if ev is not None:
            dev = (self.data if self.data is not None else self.raw).device
            torch.cuda.current_stream(dev).wait_event(ev)
        return self


def require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.IllicoCudaError("illico_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise _lib.IllicoCudaError(f"illico_b200 runs on CUDA devices only, got {dev}")
    return dev


class Engine:
    def __init__(self, grpc: GroupContainer, device=None, seg_max: int | None = None, host_plan: HostPlan | None = None):
        if seg_max is not None:
            check_seg_max(seg_max)     # (argument errors before any device work)
        self.lib = _lib.load()
        self.device = require_cuda(device)
        self.grpc = grpc
        # the host-side plan does not depend on the device: one per run, shared by the engines of all GPUs
        # (seg_max None: ILLICO_B200_SEG_MAX, else 512; build_plan refuses a length outside [1, 65535])
        self.host_plan: HostPlan = host_plan or build_plan(grpc, seg_max)
        hp = self.host_plan
        with torch.cuda.device(self.device):
            self._tables = {k: torch.from_numpy(getattr(hp, k)).to(self.device) for k in HostPlan.TABLES}
        self.plan = _lib.Plan(
            n_cells=hp.n_cells, n_groups=hp.n_groups, n_segments=hp.n_segments, ref_group=hp.ref_group,
            max_group_size=hp.max_group_size, ref_group_size=hp.ref_group_size, ref_seg_begin=hp.ref_seg_begin,
            ref_seg_end=hp.ref_seg_end, slot_cap=hp.slot_cap, max_target_group_size=hp.max_target_group_size,
            **{k: self._tables[k].data_ptr() for k in HostPlan.TABLES})
        self._flag = torch.empty(1, dtype=torch.int32, device=self.device)   # (written by illico_check_csr_sorted itself)
        # The reference calls its dispatchers from joblib threads (ctypes drops the GIL).  The C ABI only enqueues work and
        # owns nothing, so concurrency is a matter of buffers: every host thread gets its own batch buffers (staged lists,
        # counts, workspace) and the engine needs no lock.
        self._tls = threading.local()

    # ---- sizes ---------------------------------------------------------------------------------------
    @property
    def n_groups(self) -> int:
        return self.host_plan.n_groups

    @property
    def is_ovo(self) -> bool:
        return self.host_plan.ref_group >= 0

    def max_batch_genes(self, n_genes: int, method: str = WILCOXON, lfc: bool = False) -> int:
        """Genes per device batch so that the staged lists (Wilcoxon; with ``lfc``, the float64 group sums too) or the three
        float64 moment planes (t-test) stay within the memory budget."""
        free, _total = torch.cuda.mem_get_info(self.device)
        if method == WILCOXON:
            budget = min(_env_int("ILLICO_B200_IR_BYTES", 16 << 30), int(free * 0.35))
            per_gene = self.host_plan.slot_cap * 4 + self.host_plan.n_segments * 4 + (self.host_plan.n_groups * 8 if lfc else 0)
        else:
            budget = int(free * 0.35)
            per_gene = self.host_plan.n_groups * 3 * 8
        b = max(1, budget // max(per_gene, 1))
        b = int(min(n_genes, b, _env_int("ILLICO_B200_BATCH_GENES", 1 << 30)))
        return b if b < 8 or b == n_genes else (b // 4) * 4  # multiples of 4 keep the 128-bit staging path

    def _ensure_buffers(self, b: int):
        """This thread's batch buffers, large enough for ``b`` genes."""
        t = self._tls
        if getattr(t, "buf_genes", 0) >= b:
            return t
        hp = self.host_plan
        t.ir_vals = t.ir_cnt = t.ws = None
        with torch.cuda.device(self.device):
            t.ir_vals = torch.empty(b * hp.slot_cap, dtype=torch.float32, device=self.device)
            t.ir_cnt = torch.empty(b * hp.n_segments, dtype=torch.int32, device=self.device)
            ws = int(self.lib.illico_rank_workspace_bytes(C.byref(self.plan), b))
            if ws == 0:
                raise _lib.IllicoCudaError("illico_rank_workspace_bytes failed: " + self.lib.illico_last_error().decode())
            t.ws = torch.empty(ws, dtype=torch.uint8, device=self.device)
        t.buf_genes = b
        return t

    # (bench.py's per-kernel timing and older scripts read the calling thread's buffers through these)
    @property
    def _ir_vals(self):
        return getattr(self._tls, "ir_vals", None)

    @property
    def _ir_cnt(self):
        return getattr(self._tls, "ir_cnt", None)

    @property
    def _ws(self):
        return getattr(self._tls, "ws", None)

    # ---- uploads (plumbing) -----------------------------------------------------------------------------
    def upload_dense(self, X: np.ndarray, gene_lb: int = 0, gene_ub: int | None = None) -> DeviceMatrix:
        return upload_dense(X, self.device, gene_lb, gene_ub)

    def upload_sparse(self, X, fmt: str) -> DeviceMatrix:
        return upload_sparse(X, fmt, self.device)

    def check_csr_sorted(self, M: DeviceMatrix) -> bool:
        st = torch.cuda.current_stream(self.device).cuda_stream
        rc = self.lib.illico_check_csr_sorted(M.indices.data_ptr(), M.indptr.data_ptr(), M.shape[0],
                                              self._flag.data_ptr(), st)
        if rc < 0:
            _lib.check(1, "illico_check_csr_sorted")
        return rc == 1

    # ---- one gene batch ----------------------------------------------------------------------------------
    def run_batch(self, M: DeviceMatrix, lb: int, ub: int, flags: _lib.Flags, results: torch.Tensor,
                  result_gene0: int, debug: dict | None = None, scores: torch.Tensor | None = None,
                  nnz: torch.Tensor | None = None, method: str = WILCOXON, lfc: torch.Tensor | None = None,
                  log_scale: float = 1.0, stats_only: bool = False) -> None:
        """Enqueues stage + rank for genes ``[lb, ub)`` of ``M``; writes ``results[:, result_gene0 + k, :]``.

        ``results`` is a device tensor ``[G, N_total, 3]`` float64 (contiguous).  ``scores``, a device tensor ``[G, N_total]``
        float64 (contiguous), also receives the signed score of every test at ``scores[:, result_gene0 + k]``.  ``nnz``, a
        device tensor ``[G, N_total]`` int32 (contiguous), receives at ``nnz[:, result_gene0 + k]`` how many cells of each
        group have a non-zero value (``illico_count_nonzero_*``, enqueued before the tests on the same stream).
        ``method`` "t-test" / "t-test_overestim_var": Welch's t-test instead (``_run_batch_ttest``), same outputs.
        ``lfc``, a device tensor ``[G, N_total]`` float64 (contiguous), receives scanpy's log fold change of every test at
        ``lfc[:, result_gene0 + k]`` (``illico_log_fold_changes``, ``log_scale`` = ln of the log1p base, else 1), from the
        group sums of a pass of its own (``illico_group_sums_*``, which then also writes ``nnz``) or of the t-test's moments.
        ``stats_only``: no test -- only the ``lfc`` / ``nnz`` pass is enqueued (``results`` may be None; a float64 matrix is
        summed and counted as it is, with no recoding).
        """
        b = ub - lb
        if b <= 0:
            return
        if M.shape[0] != self.host_plan.n_cells:
            raise ValueError(f"matrix has {M.shape[0]} cells, groups describe {self.host_plan.n_cells}")
        if lb < 0 or ub > M.shape[1]:
            raise ValueError(f"Invalid chunk bounds: {(lb, ub)} for data with {M.shape[1]} columns.")
        with torch.cuda.device(self.device):
            M.ready()
        if stats_only:
            if lfc is not None:
                self.log_fold_changes(M, lb, ub, lfc, result_gene0, log_scale, nnz)
            elif nnz is not None:
                self.count_nonzero(M, lb, ub, nnz, result_gene0)
            return
        if method != WILCOXON:
            return self._run_batch_ttest(M, lb, ub, flags, results, result_gene0, scores, nnz, check_method(method), lfc,
                                         log_scale)
        if lfc is not None:
            self.log_fold_changes(M, lb, ub, lfc, result_gene0, log_scale, nnz)
        elif nnz is not None:
            self.count_nonzero(M, lb, ub, nnz, result_gene0)
        if M.raw is not None:
            return self._run_batch_wide(M, lb, ub, flags, results, result_gene0, debug, scores)
        t = self._ensure_buffers(b)
        G, Ntot = results.shape[0], results.shape[1]
        assert results.dtype == torch.float64 and results.is_contiguous() and G == self.n_groups
        if scores is not None:
            assert scores.dtype == torch.float64 and scores.is_contiguous() and tuple(scores.shape) == (G, Ntot)
            flags = flags.replace(scores=scores.data_ptr() + result_gene0 * 8, score_group_stride=Ntot)
        stream = torch.cuda.current_stream(self.device)
        st = stream.cuda_stream
        for x in (t.ir_vals, t.ir_cnt, t.ws):   # a thread may enqueue on different streams over time: keep the allocator informed
            x.record_stream(stream)
        buf = _lib.BatchBuffers(t.ir_vals.data_ptr(), t.ir_cnt.data_ptr(), t.ws.data_ptr(), t.ws.numel())
        dbg = None
        if debug is not None:
            shape_t = (G, b) if self.is_ovo else (b,)
            debug["u2"] = torch.zeros((G, b), dtype=torch.int64, device=self.device)
            debug["tie_sum"] = torch.zeros(shape_t, dtype=torch.float64, device=self.device)
            debug["tie_exact"] = torch.zeros(shape_t, dtype=torch.int64, device=self.device)
            dbg = _lib.Debug(debug["u2"].data_ptr(), debug["tie_sum"].data_ptr(), debug["tie_exact"].data_ptr())
        out_ptr = results.data_ptr() + result_gene0 * 3 * 8
        gstride = Ntot * 3
        test = "ovo" if self.is_ovo else "ovr"
        dbg_ref = C.byref(dbg) if dbg is not None else None
        with torch.cuda.device(self.device):
            if M.fmt == DENSE:
                fn = getattr(self.lib, f"illico_{test}_dense_f32")
                rc = fn(M.data.data_ptr(), M.ld, lb, b, C.byref(self.plan), C.byref(flags), C.byref(buf), out_ptr,
                        gstride, dbg_ref, st)
            else:
                fn = getattr(self.lib, f"illico_{test}_{M.fmt}_f32")
                rc = fn(M.data.data_ptr(), M.indices.data_ptr(), M.indptr.data_ptr(), lb, b, C.byref(self.plan),
                        C.byref(flags), C.byref(buf), out_ptr, gstride, dbg_ref, st)
        _lib.check(rc, f"illico_{test}_{M.fmt}_f32")

    def count_nonzero(self, M: DeviceMatrix, lb: int, ub: int, nnz: torch.Tensor, result_gene0: int) -> None:
        """``nnz[:, result_gene0 + k]`` = cells of each group whose value in gene ``lb + k`` of ``M`` is non-zero, on the
        current stream.  A matrix kept as float64 (``M.raw``) is counted on those values, not on its recoded batches."""
        G, Ntot = nnz.shape
        assert nnz.dtype == torch.int32 and nnz.is_contiguous() and G == self.n_groups and nnz.device == self.device
        vals, dtype = (M.raw, _lib.DTYPE_F64) if M.raw is not None else (M.data, _lib.DTYPE_F32)
        out = nnz.data_ptr() + result_gene0 * 4
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            if M.fmt == DENSE:
                rc = self.lib.illico_count_nonzero_dense(vals.data_ptr(), dtype, int(vals.stride(0)), lb, ub - lb,
                                                         C.byref(self.plan), out, Ntot, st)
            else:
                fn = getattr(self.lib, f"illico_count_nonzero_{M.fmt}")
                rc = fn(vals.data_ptr(), dtype, M.indices.data_ptr(), M.indptr.data_ptr(), lb, ub - lb, C.byref(self.plan), out,
                        Ntot, st)
        _lib.check(rc, f"illico_count_nonzero_{M.fmt}")

    def _scratch(self, name: str, G: int, b: int) -> torch.Tensor:
        """This thread's float64 ``[G, >= b]`` scratch plane ``name`` (grown on demand), recorded on the current stream."""
        t = self._tls
        buf = getattr(t, name, None)
        if buf is None or buf.shape[-1] < b:
            setattr(t, name, None)
            with torch.cuda.device(self.device):
                buf = torch.empty((G, b), dtype=torch.float64, device=self.device)
            setattr(t, name, buf)
        buf.record_stream(torch.cuda.current_stream(self.device))
        return buf

    def log_fold_changes(self, M: DeviceMatrix, lb: int, ub: int, lfc: torch.Tensor, result_gene0: int, log_scale: float = 1.0,
                         nnz: torch.Tensor | None = None) -> None:
        """``lfc[:, result_gene0 + k]`` = scanpy's log fold change of gene ``lb + k`` of ``M`` in every group, on the current
        stream: the group sums of the batch (``illico_group_sums_*``; with ``nnz``, its count plane in the same launch, as
        ``count_nonzero``), then ``illico_log_fold_changes``.  A matrix kept as float64 (``M.raw``) is summed as it is."""
        b = ub - lb
        G, Ntot = lfc.shape
        assert lfc.dtype == torch.float64 and lfc.is_contiguous() and G == self.n_groups and lfc.device == self.device
        sums = self._scratch("sums", G, b)
        vals, dtype = (M.raw, _lib.DTYPE_F64) if M.raw is not None else (M.data, _lib.DTYPE_F32)
        cnt, cstride = (None, 0)
        if nnz is not None:
            assert nnz.dtype == torch.int32 and nnz.is_contiguous() and tuple(nnz.shape) == (G, Ntot)
            cnt, cstride = nnz.data_ptr() + result_gene0 * 4, Ntot
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            if M.fmt == DENSE:
                rc = self.lib.illico_group_sums_dense(vals.data_ptr(), dtype, int(vals.stride(0)), lb, b, C.byref(self.plan),
                                                      sums.data_ptr(), cnt, cstride, sums.shape[1], st)
            else:
                fn = getattr(self.lib, f"illico_group_sums_{M.fmt}")
                rc = fn(vals.data_ptr(), dtype, M.indices.data_ptr(), M.indptr.data_ptr(), lb, b, C.byref(self.plan), sums.data_ptr(),
                        cnt, cstride, sums.shape[1], st)
            _lib.check(rc, f"illico_group_sums_{M.fmt}")
            self._lfc_from_sums(sums.data_ptr(), sums.shape[1], b, lfc, result_gene0, log_scale, st)

    def _lfc_from_sums(self, s1: int, ms: int, b: int, lfc: torch.Tensor, result_gene0: int, log_scale: float, st) -> None:
        hp = self.host_plan
        G, Ntot = lfc.shape
        rc = self.lib.illico_log_fold_changes(s1, ms, self._tables["group_size"].data_ptr(), G, b, hp.ref_group, hp.n_cells,
                                              float(log_scale), lfc.data_ptr() + result_gene0 * 8, Ntot, st)
        _lib.check(rc, "illico_log_fold_changes")

    def _run_batch_ttest(self, M: DeviceMatrix, lb: int, ub: int, flags: _lib.Flags, results, result_gene0, scores, nnz, method,
                         lfc=None, log_scale: float = 1.0):
        """Welch's t-test of genes ``[lb, ub)``: one pass over the batch for the per-(group, gene) moments (and the count
        plane when ``nnz`` is given) -- ``illico_group_moments_*`` -- then ``illico_welch_ttest`` into the same result and
        score slabs, and ``illico_log_fold_changes`` from the same sums when ``lfc`` is given.  float64 values (``M.raw``) are read as they are: no recoding, no staged lists."""
        b = ub - lb
        G, Ntot = results.shape[0], results.shape[1]
        assert results.dtype == torch.float64 and results.is_contiguous() and G == self.n_groups
        dev = self.device
        log1p = int(bool(flags.is_log1p))
        t = self._tls
        if getattr(t, "mom_genes", 0) < b:
            t.mom = None
            with torch.cuda.device(dev):
                t.mom = torch.empty((3, G, b), dtype=torch.float64, device=dev)
            t.mom_genes = b
        mom = t.mom
        stream = torch.cuda.current_stream(dev)
        mom.record_stream(stream)
        ms = mom.shape[2]
        s1, s2, sf = (mom[k].data_ptr() for k in range(3))
        vals, dtype = (M.raw, _lib.DTYPE_F64) if M.raw is not None else (M.data, _lib.DTYPE_F32)
        cnt, cstride = (None, 0)
        if nnz is not None:
            assert nnz.dtype == torch.int32 and nnz.is_contiguous() and tuple(nnz.shape) == (G, Ntot)
            cnt, cstride = nnz.data_ptr() + result_gene0 * 4, Ntot
        if scores is not None:
            assert scores.dtype == torch.float64 and scores.is_contiguous() and tuple(scores.shape) == (G, Ntot)
        hp = self.host_plan
        with torch.cuda.device(dev):
            st = stream.cuda_stream
            if M.fmt == DENSE:
                rc = self.lib.illico_group_moments_dense(vals.data_ptr(), dtype, int(vals.stride(0)), lb, b, C.byref(self.plan), log1p,
                                                         s1, s2, sf, cnt, cstride, ms, st)
            else:
                fn = getattr(self.lib, f"illico_group_moments_{M.fmt}")
                rc = fn(vals.data_ptr(), dtype, M.indices.data_ptr(), M.indptr.data_ptr(), lb, b, C.byref(self.plan), log1p, s1, s2,
                        sf, cnt, cstride, ms, st)
            _lib.check(rc, f"illico_group_moments_{M.fmt}")
            rc = self.lib.illico_welch_ttest(s1, s2, sf if log1p else None, ms, self._tables["group_size"].data_ptr(), G, b,
                                             hp.ref_group, hp.n_cells, int(method == "t-test_overestim_var"), flags.alternative,
                                             results.data_ptr() + result_gene0 * 3 * 8, Ntot * 3,
                                             scores.data_ptr() + result_gene0 * 8 if scores is not None else None, Ntot, st)
            _lib.check(rc, "illico_welch_ttest")
            if lfc is not None:
                assert lfc.dtype == torch.float64 and lfc.is_contiguous() and tuple(lfc.shape) == (G, Ntot)
                self._lfc_from_sums(s1, ms, b, lfc, result_gene0, log_scale, st)

    def _run_batch_wide(self, M: DeviceMatrix, lb: int, ub: int, flags: _lib.Flags, results, result_gene0, debug, scores=None):
        """float64 input (values float32 cannot hold): every sub-batch is recoded on the device to order-preserving
        float32 codes in the input's own layout (exact ranks, U, ties, p) and the fold change uses float64 group sums
        computed from the original values -- ``illico_recode_{dense,csr,csc}`` (csrc/recode.cu), then the ordinary
        dispatcher.  The reference specialises its numba kernels per dtype instead (``ovr/dense_ovr.py:46-53``)."""
        n = self.host_plan.n_cells
        if n >= (1 << 24):
            raise NotImplementedError("more than 2^24 cells with values float32 cannot hold")
        dev = self.device
        enc = getattr(self, "_enc_dev", None)
        if enc is None:
            enc = self._enc_dev = torch.from_numpy(np.ascontiguousarray(self.grpc.encoded_groups, dtype=np.int32)).to(dev)
        G = self.n_groups
        st = torch.cuda.current_stream(dev).cuda_stream
        raw = M.raw
        if M.fmt != DENSE and getattr(M, "_codes", None) is None:
            M._codes = torch.empty(raw.shape, dtype=torch.float32, device=dev)     # parallel to the stored values
        # dense / CSR key lists have one slot per cell and gene: a sub-batch holds at most 2^26 of them (1 GB of keys)
        step = (ub - lb) if M.fmt == CSC else max(1, min(ub - lb, (1 << 26) // max(n, 1)))
        if M.fmt == DENSE and 4 <= step < ub - lb:
            step -= step % 4     # every sub-batch but the last starts on a 16-byte boundary of the input's rows
        for a in range(lb, ub, step):
            z = min(ub, a + step)
            b = z - a
            with torch.cuda.device(dev):
                sums = torch.empty((G, b), dtype=torch.float64, device=dev)
                if M.fmt == DENSE:
                    keys = n * b
                    codes = torch.empty((n, b), dtype=torch.float32, device=dev)   # (the recode kernel writes [n, b] rows)
                elif M.fmt == CSC:
                    keys = int(M.indptr[z]) - int(M.indptr[a])
                    codes = M._codes
                else:
                    keys = n * b
                    codes = M._codes
                ws = torch.empty(int(self.lib.illico_recode_workspace_bytes(keys, b)), dtype=torch.uint8, device=dev)
                if M.fmt == DENSE:
                    rc = self.lib.illico_recode_dense(raw.data_ptr(), _lib.DTYPE_F64, int(raw.stride(0)), a, b, n, enc.data_ptr(), G,
                                                      int(flags.is_log1p), codes.data_ptr(), sums.data_ptr(), ws.data_ptr(),
                                                      ws.numel(), st)
                    sub, sub_lb = DeviceMatrix(DENSE, (n, b), codes), 0
                elif M.fmt == CSC:
                    rc = self.lib.illico_recode_csc(raw.data_ptr(), _lib.DTYPE_F64, M.indices.data_ptr(), M.indptr.data_ptr(), a, b,
                                                    keys, enc.data_ptr(), G, int(flags.is_log1p), codes.data_ptr(), sums.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), st)
                    sub, sub_lb = DeviceMatrix(CSC, M.shape, codes, M.indices, M.indptr), a
                else:
                    rc = self.lib.illico_recode_csr(raw.data_ptr(), _lib.DTYPE_F64, M.indices.data_ptr(), M.indptr.data_ptr(), n, a, b,
                                                    enc.data_ptr(), G, int(flags.is_log1p), codes.data_ptr(), sums.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), st)
                    sub, sub_lb = DeviceMatrix(CSR, M.shape, codes, M.indices, M.indptr), a
                _lib.check(rc, f"illico_recode_{M.fmt}")
                if M.fmt == DENSE:
                    sub.data = _padded_rows(codes, st)
            f2 = flags.replace(group_sums=sums.data_ptr())
            dbg = {} if debug is not None else None
            self.run_batch(sub, sub_lb, sub_lb + b, f2, results, result_gene0 + (a - lb), dbg, scores)
            if debug is not None:
                for k, v in dbg.items():
                    debug.setdefault("_parts", {}).setdefault(k, []).append(v)
            torch.cuda.current_stream(dev).synchronize()  # sums / codes / workspace must outlive the kernels
        if debug is not None and "_parts" in debug:
            for k, parts in debug.pop("_parts").items():
                debug[k] = torch.cat(parts, dim=-1)


def _padded_rows(codes: torch.Tensor, stream: int) -> torch.Tensor:
    """A ``[n, b]`` view of ``codes`` whose rows are 16-byte aligned (stride rounded up to 4 floats, padding zeroed): the
    TMA staging kernel and the dense fused path take only such rows, so recoded batches of any width reach them."""
    n, b = codes.shape
    ld = (b + 3) & ~3
    if ld == b:
        return codes
    out = torch.empty((n, ld), dtype=torch.float32, device=codes.device)
    out[:, b:].zero_()
    _lib.check(_lib.load().illico_memcpy2d_async(out.data_ptr(), ld * 4, codes.data_ptr(), b * 4, b * 4, n, 3, stream),
               "illico_memcpy2d_async")
    return out[:, :b]


_TORCH_OK = (np.float32, np.float64, np.float16, np.int8, np.uint8, np.int16, np.int32, np.int64)


def _uploadable(a: np.ndarray) -> np.ndarray:
    """Host arrays of dtypes torch cannot hold (unsigned 16/32/64-bit, bool, ...) are widened on the host."""
    if a.dtype.type in _TORCH_OK:
        return a
    if a.dtype.kind in "ui" and a.dtype.itemsize < 8:
        return a.astype(np.int64)
    return a.astype(np.float64)


def _torch_dtype(a: np.ndarray):
    return torch.from_numpy(np.empty(0, dtype=a.dtype)).dtype


def upload_dense(X, device, gene_lb: int = 0, gene_ub: int | None = None, rows=None, cols=None) -> DeviceMatrix:
    """Starts the copy of ``X[:, gene_lb:gene_ub]`` (any real dtype) into a device matrix and returns at once: pinned
    sources go out as one strided asynchronous copy, pageable ones through the pinned staging ring of
    :mod:`illico_b200.hostio` (worker threads), so the caller keeps working on the host meanwhile.  ``rows`` (ascending
    int64, optional): only those rows go up, gathered by the staging threads.  ``cols`` (ascending int64, optional): the
    columns of ``X`` that go up, gathered the same way, in place of ``[gene_lb, gene_ub)`` (genes ``[gene_lb, gene_ub)``
    of a run over a column selection, ``gene_ub - gene_lb == len(cols)``).  ``DeviceMatrix.ready()`` joins."""
    from . import hostio

    device = require_cuda(device)
    n, N = X.shape
    if rows is not None:
        n = len(rows)
    gene_ub = N if gene_ub is None else gene_ub
    if isinstance(X, torch.Tensor):
        X = X.numpy()
    rel = None
    if cols is not None:
        c0 = int(cols[0])
        view = _uploadable(np.asarray(X[:, c0:int(cols[-1]) + 1]))
        rel = np.asarray(cols, dtype=np.int64) - c0
    else:
        view = _uploadable(np.asarray(X[:, gene_lb:gene_ub]))
    with torch.cuda.device(device):
        d = torch.empty((n, gene_ub - gene_lb), dtype=_torch_dtype(view), device=device)
        pend = hostio.h2d_2d(d, view, rows=rows, cols=rel)
    if d.dtype == torch.float32:
        return DeviceMatrix(DENSE, (n, gene_ub - gene_lb), d, gene_offset=gene_lb, pending=[pend])
    return DeviceMatrix(DENSE, (n, gene_ub - gene_lb), None, gene_offset=gene_lb, pending=[pend], unconverted=d)


def upload_sparse(X, fmt: str, device, gene_lb: int = 0, gene_ub: int | None = None) -> DeviceMatrix:
    """Starts the copies of a scipy CSR / CSC matrix (or a ``(data, indices, indptr, shape)`` namedtuple).  A CSC matrix
    can be cut to the gene shard ``[gene_lb, gene_ub)`` (its columns are contiguous); a CSR matrix always goes up whole
    (every row holds all genes) and the kernels select the gene range.  The small ``indptr`` goes first: it is
    converted (int64) into pageable memory, and a copy from pageable memory waits for everything queued before it."""
    from . import hostio

    device = require_cuda(device)
    n, N = X.shape
    data, indices, indptr = np.asarray(X.data), np.asarray(X.indices), np.asarray(X.indptr)
    offset = 0
    if fmt == CSC and (gene_lb != 0 or (gene_ub is not None and gene_ub != N)):
        gene_ub = N if gene_ub is None else gene_ub
        lo, hi = int(indptr[gene_lb]), int(indptr[gene_ub])
        data, indices, indptr = data[lo:hi], indices[lo:hi], indptr[gene_lb:gene_ub + 1] - lo
        N, offset = gene_ub - gene_lb, gene_lb
    data = _uploadable(np.ascontiguousarray(data))
    with torch.cuda.device(device):
        d_indptr = torch.from_numpy(np.ascontiguousarray(indptr, dtype=np.int64)).to(device, non_blocking=True)
        d_data = torch.empty(data.shape, dtype=_torch_dtype(data), device=device)
        d_idx = torch.empty(indices.shape, dtype=torch.int32, device=device)
        pend = [hostio.h2d_1d(d_data, data), hostio.h2d_1d(d_idx, np.ascontiguousarray(indices, dtype=np.int32))]
    if d_data.dtype == torch.float32:
        return DeviceMatrix(fmt, (n, N), d_data, d_idx, d_indptr, gene_offset=offset, pending=pend)
    return DeviceMatrix(fmt, (n, N), None, d_idx, d_indptr, gene_offset=offset, pending=pend, unconverted=d_data)


_DTYPE_CODE = {torch.float32: _lib.DTYPE_F32, torch.float64: _lib.DTYPE_F64, torch.float16: _lib.DTYPE_F16, torch.int8: _lib.DTYPE_I8,
               torch.uint8: _lib.DTYPE_U8, torch.int16: _lib.DTYPE_I16, torch.int32: _lib.DTYPE_I32, torch.int64: _lib.DTYPE_I64}


def _to_f32_or_wide(t: torch.Tensor):
    """``(float32 tensor, None)`` when float32 holds every value exactly, else ``(None, float64 tensor)``.
    Never rounds: rounding would create ties that are not in the data.  (``illico_convert_values``; one host read of
    the verdict.)"""
    lib = _lib.load()
    code = _DTYPE_CODE.get(t.dtype)
    if code is None:
        raise TypeError(f"unsupported value dtype {t.dtype}")
    src = t if t.is_contiguous() else t.contiguous()
    dev = src.device
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        f = torch.empty(src.shape, dtype=torch.float32, device=dev)
        flag = torch.empty(1, dtype=torch.int32, device=dev)
        _lib.check(lib.illico_convert_values(src.data_ptr(), code, src.numel(), f.data_ptr(), None, flag.data_ptr(), st),
                   "illico_convert_values")
        if int(flag.item()) == 0:
            return f, None
        del f
        if src.dtype == torch.float64:
            return None, src
        d = torch.empty(src.shape, dtype=torch.float64, device=dev)
        _lib.check(lib.illico_convert_values(src.data_ptr(), code, src.numel(), None, d.data_ptr(), None, st), "illico_convert_values")
        return None, d


def make_flags(is_log1p: bool, use_continuity: bool, tie_correct: bool, alternative: str, fmt: str) -> _lib.Flags:
    if alternative not in _lib.ALTERNATIVES:
        raise ValueError(f"Unsupported alternative hypothesis: {alternative}")
    return _lib.Flags(int(bool(is_log1p)), int(bool(use_continuity)), int(bool(tie_correct)),
                      _lib.ALTERNATIVES[alternative], _lib.TIES_DENSE if fmt == DENSE else _lib.TIES_SPARSE)
