"""The cells of the groups a one-versus-reference call tests (``groups=``), cut out of a device-resident matrix.

``illico_select_rows_*`` (csrc/select.cu) gather the selected rows, in ascending order, into a new matrix of the same format
and value type: the group plan built from the same rows (``groups.subset_for_reference``) then gives every selected group the
segments of the full call, and the six dispatchers run on the result unchanged.  Host input is gathered on its way up
instead where it can be (dense rows by the staging threads, CSR rows by scipy); CSC input and CUDA tensors come here.
"""
from __future__ import annotations

import threading

import numpy as np
import torch

from . import _lib
from .engine import CSC, CSR, DENSE, DeviceMatrix


class RowSelection:
    """The rows a one-versus-reference call keeps: ``rows`` (host int64, ascending) out of ``n_cells``, and per device the
    int32 row list and the ``new_row [n_cells]`` table (the row's number in the selection, -1 = dropped)."""

    def __init__(self, rows: np.ndarray, n_cells: int):
        self.rows = np.ascontiguousarray(rows, dtype=np.int64)
        self.n_cells = int(n_cells)
        self._tables: dict = {}
        self._lock = threading.Lock()

    def tables(self, device) -> tuple:
        """``(rows int32, new_row int32)`` on ``device`` (copied there once)."""
        key = str(device)
        with self._lock:
            if key not in self._tables:
                new_row = np.full(self.n_cells, -1, dtype=np.int32)
                new_row[self.rows] = np.arange(self.rows.size, dtype=np.int32)
                with torch.cuda.device(device):
                    self._tables[key] = (torch.from_numpy(self.rows.astype(np.int32)).to(device),
                                         torch.from_numpy(new_row).to(device))
            return self._tables[key]


def _values(M: DeviceMatrix):
    """The stored values (float64 when the matrix is kept as such) and their ``illico_dtype``."""
    if M.raw is not None:
        return M.raw, _lib.DTYPE_F64
    if M.data.dtype != torch.float32:
        raise TypeError(f"row selection takes float32 or float64 values, got {M.data.dtype}")
    return M.data, _lib.DTYPE_F32


def select_rows(M: DeviceMatrix, bounds: tuple, sel: RowSelection) -> tuple:
    """``(DeviceMatrix, bounds)`` of the selected rows of genes ``[bounds[0], bounds[1])`` of ``M``, enqueued on the current
    stream (a sparse selection reads its entry count back).  A matrix that already has only those rows (gathered on upload)
    is returned as it is.  Dense rows are padded to a multiple of 4 floats, which the TMA staging and the dense fused pass
    need; float64 values stay float64 (``M.raw``), to be recoded like those of the full matrix."""
    n_sel = int(sel.rows.size)
    if M.shape[0] == n_sel:
        return M, bounds
    if M.shape[0] != sel.n_cells:
        raise ValueError(f"matrix has {M.shape[0]} cells, the selection was made over {sel.n_cells}")
    dev = (M.data if M.data is not None else M.raw).device
    with torch.cuda.device(dev):
        M.ready()
        lib = _lib.load()
        st = torch.cuda.current_stream(dev).cuda_stream
        vals, code = _values(M)
        rows, new_row = sel.tables(dev)
        lb, ub = bounds
        b = ub - lb
        wide = M.raw is not None
        if M.fmt == DENSE:
            out_ld = b if wide else (b + 3) & ~3
            out = torch.empty((n_sel, max(out_ld, 1)), dtype=vals.dtype, device=dev)
            _lib.check(lib.illico_select_rows_dense(vals.data_ptr() + lb * vals.element_size(), code, int(vals.stride(0)), b,
                                                    rows.data_ptr(), n_sel, out.data_ptr(), out_ld, st), "illico_select_rows_dense")
            part = out[:, :b]
            return (DeviceMatrix(DENSE, (n_sel, b), None if wide else part, gene_offset=M.gene_offset + lb,
                                 raw=part if wide else None), (0, b))
        if M.fmt == CSR:
            indptr = torch.empty(n_sel + 1, dtype=torch.int64, device=dev)
            _lib.check(lib.illico_select_rows_csr_indptr(M.indptr.data_ptr(), rows.data_ptr(), n_sel, indptr.data_ptr(), st),
                       "illico_select_rows_csr_indptr")
            nnz = int(indptr[-1].item())
            data = torch.empty(max(nnz, 1), dtype=vals.dtype, device=dev)
            idx = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
            _lib.check(lib.illico_select_rows_csr(vals.data_ptr(), code, M.indices.data_ptr(), M.indptr.data_ptr(), rows.data_ptr(),
                                                  n_sel, indptr.data_ptr(), data.data_ptr(), idx.data_ptr(), st), "illico_select_rows_csr")
            data, idx = data[:nnz], idx[:nnz]
            return (DeviceMatrix(CSR, (n_sel, M.shape[1]), None if wide else data, idx, indptr, gene_offset=M.gene_offset,
                                 raw=data if wide else None), bounds)
        assert M.fmt == CSC
        col_ptr = M.indptr.data_ptr() + lb * 8
        indptr = torch.empty(b + 1, dtype=torch.int64, device=dev)
        _lib.check(lib.illico_select_rows_csc_indptr(M.indices.data_ptr(), col_ptr, b, new_row.data_ptr(), indptr.data_ptr(), st),
                   "illico_select_rows_csc_indptr")
        nnz = int(indptr[-1].item())
        data = torch.empty(max(nnz, 1), dtype=vals.dtype, device=dev)
        idx = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        _lib.check(lib.illico_select_rows_csc(vals.data_ptr(), code, M.indices.data_ptr(), col_ptr, b, new_row.data_ptr(),
                                              indptr.data_ptr(), data.data_ptr(), idx.data_ptr(), st), "illico_select_rows_csc")
        data, idx = data[:nnz], idx[:nnz]
        return (DeviceMatrix(CSC, (n_sel, b), None if wide else data, idx, indptr, gene_offset=M.gene_offset + lb,
                             raw=data if wide else None), (0, b))
