"""The cells of the groups a one-versus-reference call tests (``groups=``) and the genes a call tests (``mask_var=``), cut
out of a device-resident matrix.

``illico_select_rows_*`` (csrc/select.cu) gather the selected rows, in ascending order, into a new matrix of the same format
and value type: the group plan built from the same rows (``groups.subset_for_reference``) then gives every selected group the
segments of the full call, and the six dispatchers run on the result unchanged.  Host input is gathered on its way up
instead where it can be (dense rows by the staging threads, CSR rows by scipy); CSC input and CUDA tensors come here.

The selected genes (``ColumnSelection``) are a column list: gene shards and batches are ranges of the selected-gene space,
and the matrix a batch runs on holds only the selected columns, in ascending order.  Dense host matrices and CSC input are
gathered on the way up (staging threads, ``illico_host_pack_cols_f32``, scipy's CSC column index, the backed readers);
a CUDA tensor is gathered here (``illico_select_cols_dense``, its row list in the same pass), and a CSR matrix, which goes up
whole, is compacted here through a ``new_col`` table by the CSC kernels with the roles of rows and columns swapped.
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


class ColumnSelection:
    """The genes a call tests: ``cols`` (host int64, ascending) out of ``n_genes``.  Genes ``[lb, ub)`` of the run (a shard
    or a batch) are the columns ``cols[lb:ub]`` of the caller's matrix."""

    def __init__(self, cols: np.ndarray, n_genes: int):
        self.cols = np.ascontiguousarray(cols, dtype=np.int64)
        self.n_genes = int(n_genes)

    @property
    def size(self) -> int:
        return int(self.cols.size)

    def new_col(self, lb: int = 0, ub: int | None = None) -> np.ndarray:
        """``int32 [n_genes]``: column ``cols[lb + j]`` -> ``j``, every other column -> -1."""
        ub = self.size if ub is None else ub
        t = np.full(self.n_genes, -1, dtype=np.int32)
        t[self.cols[lb:ub]] = np.arange(ub - lb, dtype=np.int32)
        return t

    def runs(self, lb: int, ub: int) -> list:
        """``[(c0, c1), ...]``: the runs of consecutive columns among ``cols[lb:ub]``, as half-open column ranges."""
        c = self.cols[lb:ub]
        if c.size == 0:
            return []
        cut = np.flatnonzero(np.diff(c) != 1) + 1
        starts, ends = np.concatenate([[0], cut]), np.concatenate([cut, [c.size]])
        return [(int(c[a]), int(c[b - 1]) + 1) for a, b in zip(starts, ends)]

    def fetch(self, data_handler, lb: int, ub: int) -> tuple:
        """A backed batch of genes ``[lb, ub)``: each run of consecutive columns is read as one slice, then the pieces are
        concatenated -- ``(data, (0, ub - lb))`` like ``DataHandler.fetch``."""
        from scipy import sparse

        pieces = [data_handler.fetch(c0, c1)[0] for c0, c1 in self.runs(lb, ub)]
        if len(pieces) == 1:
            data = pieces[0]
        elif sparse.issparse(pieces[0]):
            data = sparse.hstack(pieces, format="csc")
        else:
            data = np.concatenate(pieces, axis=1)
        return data, (0, ub - lb)


def resolve_mask_var(adata, mask_var, n_genes: int):
    """scanpy's ``mask_var``: None, the name of a boolean column of ``adata.var``, or a boolean mask of length ``n_genes``
    (numpy array, list or pandas Series).  Returns the ascending int64 list of the selected genes, or None when that is every
    gene.  Integer arrays (positions), other dtypes, a wrong length, a missing column and a mask with no True are a
    ``ValueError``."""
    import pandas as pd

    if mask_var is None:
        return None
    if isinstance(mask_var, str):
        var = getattr(adata, "var", None)
        if var is None or mask_var not in getattr(var, "columns", ()):
            raise ValueError(f"mask_var: {mask_var!r} is not a column of adata.var")
        mask_var = var[mask_var]
    if isinstance(mask_var, pd.Series):
        if isinstance(mask_var.dtype, pd.BooleanDtype) and not mask_var.isna().any():
            mask_var = mask_var.to_numpy(dtype=bool)
        else:
            mask_var = mask_var.to_numpy()
    mask = np.asarray(mask_var)
    if mask.dtype != np.bool_:
        raise ValueError(f"mask_var must be a boolean mask over the genes (not positions), got dtype {mask.dtype}")
    if mask.ndim != 1 or mask.size != n_genes:
        raise ValueError(f"mask_var has shape {mask.shape}, the matrix has {n_genes} genes")
    cols = np.flatnonzero(mask).astype(np.int64)
    if cols.size == 0:
        raise ValueError("mask_var selects no gene")
    return None if cols.size == n_genes else cols


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
        indptr, data, idx = compact(vals, code, M.indices, M.indptr.data_ptr() + lb * 8, b, new_row)
        return (DeviceMatrix(CSC, (n_sel, b), None if wide else data, idx, indptr, gene_offset=M.gene_offset + lb,
                             raw=data if wide else None), (0, b))


def compact(vals: torch.Tensor, code: int, indices: torch.Tensor, indptr_ptr: int, n_major: int, new_minor: torch.Tensor) -> tuple:
    """``(indptr, values, indices)`` of a compressed matrix of ``n_major`` rows (CSR) or columns (CSC) whose minor indices
    are renumbered through ``new_minor`` (-1 = dropped; ``illico_select_rows_csc[_indptr]``, a stable compaction: each major
    slice's minor indices still ascend).  ``indptr_ptr``: the address of the first major slice's pointer (the values index
    ``vals`` / ``indices`` as they are).  Enqueued on the current stream; reads the entry count back."""
    lib = _lib.load()
    dev = vals.device
    st = torch.cuda.current_stream(dev).cuda_stream
    indptr = torch.empty(n_major + 1, dtype=torch.int64, device=dev)
    _lib.check(lib.illico_select_rows_csc_indptr(indices.data_ptr(), indptr_ptr, n_major, new_minor.data_ptr(), indptr.data_ptr(), st),
               "illico_select_rows_csc_indptr")
    nnz = int(indptr[-1].item())
    data = torch.empty(max(nnz, 1), dtype=vals.dtype, device=dev)
    idx = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    _lib.check(lib.illico_select_rows_csc(vals.data_ptr(), code, indices.data_ptr(), indptr_ptr, n_major, new_minor.data_ptr(),
                                          indptr.data_ptr(), data.data_ptr(), idx.data_ptr(), st), "illico_select_rows_csc")
    return indptr, data[:nnz], idx[:nnz]


def select_cols(M: DeviceMatrix, bounds: tuple, cols: ColumnSelection, lb: int, ub: int, rows: RowSelection | None = None) -> tuple:
    """``(DeviceMatrix, (0, ub - lb))`` holding only the columns ``cols.cols[lb:ub]`` (genes ``[lb, ub)`` of the run) of ``M``,
    enqueued on the current stream.  ``M`` holds the caller's columns ``[M.gene_offset, M.gene_offset + M.shape[1])``, a
    range that contains the selected ones; when it is exactly as wide as the selection it holds only them (the upload
    gathered them) and is returned as it is.  Dense: one gather, the row list of ``rows`` in the same pass (rows padded to a
    multiple of 4 floats, as ``select_rows`` does).  CSR: every row compacted through the ``new_col`` table.  float64 values
    stay float64 (``M.raw``)."""
    b = ub - lb
    if M.shape[1] == b:
        return M, (0, b)
    dev = (M.data if M.data is not None else M.raw).device
    with torch.cuda.device(dev):
        M.ready()
        vals, code = _values(M)
        wide = M.raw is not None
        if M.fmt == DENSE:
            lib = _lib.load()
            st = torch.cuda.current_stream(dev).cuda_stream
            d_cols = torch.from_numpy((cols.cols[lb:ub] - M.gene_offset).astype(np.int32)).to(dev, non_blocking=True)
            n_out, d_rows = M.shape[0], None
            if rows is not None:
                d_rows = rows.tables(dev)[0]
                n_out = int(rows.rows.size)
            out_ld = b if wide else (b + 3) & ~3
            out = torch.empty((n_out, max(out_ld, 1)), dtype=vals.dtype, device=dev)
            _lib.check(lib.illico_select_cols_dense(vals.data_ptr(), code, int(vals.stride(0)),
                                                    d_rows.data_ptr() if d_rows is not None else None, n_out, d_cols.data_ptr(), b,
                                                    out.data_ptr(), out_ld, st), "illico_select_cols_dense")
            part = out[:, :b]
            return DeviceMatrix(DENSE, (n_out, b), None if wide else part, gene_offset=lb, raw=part if wide else None), (0, b)
        if M.fmt != CSR:
            raise ValueError(f"column selection of a {M.fmt} matrix: its columns are cut on upload")
        new_col = cols.new_col(lb, ub)[M.gene_offset:M.gene_offset + M.shape[1]]
        d_new = torch.from_numpy(np.ascontiguousarray(new_col)).to(dev, non_blocking=True)
        indptr, data, idx = compact(vals, code, M.indices, M.indptr.data_ptr(), M.shape[0], d_new)
        return (DeviceMatrix(CSR, (M.shape[0], b), None if wide else data, idx, indptr, gene_offset=lb, raw=data if wide else None),
                (0, b))
