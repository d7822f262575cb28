"""Plug-in registries, mirroring the reference's L2 seam (``illico/utils/registry.py:15-188``).

Same names and meaning: ``Test``, ``KernelDataFormat``, ``dispatcher_registry[(Test, KernelDataFormat)]``,
``data_handler_registry[type(X)]`` with ``DataHandler.fetch(lb, ub) -> (data, (lb', ub'))``.  The numba
specific ``to_nb`` / ``input_signature`` become ``to_device`` (host arrays -> HBM); unsupported input
types raise the reference's ``KeyError("Support for data type ... is not implemented.")``.
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from enum import Enum

import numpy as np
from scipy import sparse as py_sparse

from .engine import CSC, CSR, DENSE, DeviceMatrix, Engine, upload_dense, upload_sparse


class Test(Enum):
    OVO = "ovo"
    OVR = "ovr"


class KernelDataFormat(Enum):
    DENSE = "dense"
    CSC = "csc"
    CSR = "csr"


class DispatcherRegistry(dict):
    def register(self, test: Test, data_format: KernelDataFormat):
        test, data_format = Test(test), KernelDataFormat(data_format)

        def decorator(obj):
            self[(test, data_format)] = obj
            return obj

        return decorator

    def get(self, test: Test, data_format: KernelDataFormat):
        key = (Test(test), KernelDataFormat(data_format))
        try:
            return self[key]
        except KeyError as e:
            raise KeyError(f"No dispatcher registered for test {test} and data format {data_format}.") from e


class DataHandlerRegistry(dict):
    def register(self, data_format):
        def decorator(obj):
            self[data_format] = obj
            return obj

        return decorator

    def get(self, key):
        for klass in type(key).__mro__:
            if klass in self:
                return self[klass](key)
        # device arrays of other libraries (CuPy ndarray, numba device arrays, ...): anything that exposes the CUDA array
        # interface is viewed as a torch tensor in place -- no copy, no host round trip (SURVEY.md section 8f.3)
        if hasattr(key, "__cuda_array_interface__"):
            import torch

            if torch.Tensor in self:
                return self[torch.Tensor](torch.as_tensor(key, device="cuda"))
        raise KeyError(f"Support for data type {type(key)} is not implemented.")


data_handler_registry = DataHandlerRegistry()
dispatcher_registry = DispatcherRegistry()


class DataHandler(ABC):
    """Knows how to slice gene batches out of one kind of container and put them in HBM."""

    def __init__(self, data):
        self.data = data

    @abstractmethod
    def fetch(self, lb: int, ub: int) -> tuple:
        """Returns ``(data, (lb', ub'))``: what to hand to ``to_device`` and the bounds inside it."""

    @abstractmethod
    def to_device(self, fetched, engine: Engine) -> DeviceMatrix:
        """Host container -> device-resident matrix (the reference's ``to_nb``)."""

    @abstractmethod
    def kernel_data_format(self) -> KernelDataFormat:
        pass

    @abstractmethod
    def footprint(self) -> int:
        pass

    in_ram = True


class InRAMDataHandler(DataHandler):
    """The matrix is in host (or device) memory; batches are column ranges of the resident copy
    (reference ``InRAMDataHandler.fetch``, ``registry.py:97-100``).  ``upload_shard`` puts one GPU's gene shard in its
    HBM: genes shard across GPUs with nothing exchanged between them (SURVEY.md section 8e)."""

    _resident: DeviceMatrix | None = None

    def fetch(self, lb: int, ub: int) -> tuple:
        return self.data, (lb, ub)

    def to_device(self, fetched, engine) -> DeviceMatrix:
        """Whole matrix on one device.  ``engine`` may be an :class:`Engine` or just a device."""
        if self._resident is None:
            self._resident = self.upload_shard(0, self.data.shape[1], getattr(engine, "device", engine))[0]
        return self._resident

    def upload_shard(self, lb: int, ub: int, device, rows=None, cols=None) -> tuple:
        """``(DeviceMatrix, (lb', ub'))``: genes ``[lb, ub)`` on ``device`` and their bounds inside that matrix.
        Returns as soon as the copies are started (``DeviceMatrix.ready()`` joins them).  ``rows`` (ascending int64): the
        cells a call needs; a handler that can gather them on the way up does, the others upload every row and the caller
        selects them on the device (``select.select_rows``).  ``cols`` (ascending int64, ``ub - lb`` of them): the columns
        of genes ``[lb, ub)`` of a run over a column selection; a handler that can gather them on the way up returns a
        matrix of exactly those columns, the others one holding a column range that contains them, which the caller cuts
        on the device (``select.select_cols``)."""
        raise NotImplementedError


@data_handler_registry.register(np.ndarray)
class DenseDataHandler(InRAMDataHandler):
    def upload_shard(self, lb, ub, device, rows=None, cols=None):
        return upload_dense(self.data, device, lb, ub, rows, cols), (0, ub - lb)

    def kernel_data_format(self):
        return KernelDataFormat.DENSE

    def footprint(self):
        return self.data.nbytes


@data_handler_registry.register(py_sparse.csr_matrix)
class CSRDataHandler(InRAMDataHandler):
    def upload_shard(self, lb, ub, device, rows=None, cols=None):
        # every CSR row holds all genes: the whole matrix goes to each GPU over its own link (1.9 GB at the K562 shape)
        # and the kernels select the gene range (with a column selection, the GPU compacts the rows first)
        return upload_sparse(self.data, CSR, device), (lb, ub)

    def kernel_data_format(self):
        return KernelDataFormat.CSR

    def footprint(self):
        return self.data.data.nbytes + self.data.indptr.nbytes + self.data.indices.nbytes


@data_handler_registry.register(py_sparse.csc_matrix)
class CSCDataHandler(InRAMDataHandler):
    def upload_shard(self, lb, ub, device, rows=None, cols=None):
        if cols is not None:        # the selected columns only (scipy's CSC column index copies them, indices unchanged)
            return upload_sparse(self.data[:, cols], CSC, device), (0, ub - lb)
        return upload_sparse(self.data, CSC, device, lb, ub), (0, ub - lb)

    def kernel_data_format(self):
        return KernelDataFormat.CSC

    def footprint(self):
        return self.data.data.nbytes + self.data.indptr.nbytes + self.data.indices.nbytes


class BackedDenseDataHandler(DataHandler):
    """Out-of-core dense container: anything supporting ``obj[:, lb:ub] -> ndarray`` (``h5py.Dataset``;
    reference ``H5pyDatasetDataHandler``, ``registry.py:162-168``).  Bounds are rebased to the batch."""

    in_ram = False

    def fetch(self, lb, ub):
        return np.asarray(self.data[:, lb:ub]), (0, ub - lb)

    def to_device(self, fetched, engine):
        return upload_dense(fetched, getattr(engine, "device", engine))

    def kernel_data_format(self):
        return KernelDataFormat.DENSE

    def footprint(self):
        return int(np.prod(self.data.shape)) * np.dtype(self.data.dtype).itemsize


class BackedCSCDataHandler(DataHandler):
    """Out-of-core CSC container: ``obj[:, lb:ub] -> scipy CSC`` (anndata ``_CSCDataset``;
    reference ``H5pyBackedCSCDataHandler``, ``registry.py:171-188``)."""

    in_ram = False

    def fetch(self, lb, ub):
        return py_sparse.csc_matrix(self.data[:, lb:ub]), (0, ub - lb)

    def to_device(self, fetched, engine):
        return upload_sparse(fetched, CSC, getattr(engine, "device", engine))

    def kernel_data_format(self):
        return KernelDataFormat.CSC

    def footprint(self):
        return 0


class TorchDenseDataHandler(InRAMDataHandler):
    """A 2-D ``torch.Tensor``: CUDA tensors are used where they are (no host round trip -- SURVEY section 8f.3), CPU
    tensors go through the ndarray path."""

    def upload_shard(self, lb, ub, device, rows=None, cols=None):
        import torch

        from .engine import _to_f32_or_wide

        X = self.data
        if X.ndim != 2:
            raise ValueError("expression matrix must be two-dimensional")
        if not X.is_cuda:
            return upload_dense(X.numpy(), device, lb, ub, rows, cols), (0, ub - lb)
        want = torch.device(device)
        if want.type == "cuda" and want.index is None:
            want = torch.device("cuda", torch.cuda.current_device())
        if X.device == want:
            d, raw = (X, None) if X.dtype == torch.float32 else _to_f32_or_wide(X)
            if d is not None and d.stride(1) != 1:
                d = d.contiguous()
            return DeviceMatrix(DENSE, tuple(X.shape), d, raw=raw), (lb, ub)
        # another GPU's shard of a device-resident matrix: peer copy of the columns (NVLink), never a remote read by a kernel
        # (with a column selection, the range that spans the shard's columns; the caller cuts them)
        if cols is not None:
            lb, ub = int(cols[0]), int(cols[-1]) + 1
        with torch.cuda.device(want):
            shard = X[:, lb:ub].to(want, non_blocking=True).contiguous()
        d, raw = (shard, None) if shard.dtype == torch.float32 else _to_f32_or_wide(shard)
        return DeviceMatrix(DENSE, (X.shape[0], ub - lb), d, gene_offset=lb, raw=raw), (0, ub - lb)

    def kernel_data_format(self):
        return KernelDataFormat.DENSE

    def footprint(self):
        return self.data.numel() * self.data.element_size()


def register_into_reference() -> bool:
    """Puts the six GPU dispatchers into the reference's own ``dispatcher_registry`` (``illico/utils/registry.py:61-64,
    193-202``) so that ``illico.asymptotic_wilcoxon(..., precompile=False)`` runs its batches on the B200 (INTEGRATION.md,
    section 2).  Returns False when ``illico`` is not importable."""
    try:
        from illico.utils import registry as ref
    except Exception:
        return False
    from . import dispatch as gpu

    for fmt in ref.KernelDataFormat:
        for test in ref.Test:
            ref.dispatcher_registry[(test, fmt)] = getattr(gpu, f"{fmt.value}_{test.value}_mwu_kernel_over_contiguous_col_chunk")
    return True


def _register_optional_backends() -> None:
    """h5py / anndata are optional: register their backed containers when importable."""
    try:
        import h5py

        data_handler_registry.register(h5py.Dataset)(BackedDenseDataHandler)
    except Exception:
        pass
    try:
        from anndata._core.sparse_dataset import _CSCDataset

        data_handler_registry.register(_CSCDataset)(BackedCSCDataHandler)
    except Exception:
        pass


def _register_memmap() -> None:
    from .backed import MemmapCSC, MemmapDense

    data_handler_registry.register(MemmapDense)(BackedDenseDataHandler)
    data_handler_registry.register(MemmapCSC)(BackedCSCDataHandler)


def _register_torch() -> None:
    import torch

    data_handler_registry.register(torch.Tensor)(TorchDenseDataHandler)


_register_optional_backends()
_register_memmap()
_register_torch()

from . import dispatch  # noqa: E402,F401  (registers the six GPU dispatchers)
