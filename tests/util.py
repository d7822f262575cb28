"""Test helpers: a minimal AnnData stand-in (anndata is not installed here) and result reshaping."""
import numpy as np
import pandas as pd


class FakeAnnData:
    """The four attributes ``asymptotic_wilcoxon`` reads (reference asymptotic_wilcoxon.py:178-208)."""

    def __init__(self, X, labels, var_names=None, key="pert", layers=None):
        self.X = X
        self.obs = pd.DataFrame({key: list(labels)})
        n_genes = X.shape[1]
        self.var_names = pd.Index(var_names if var_names is not None else [f"gene_{i}" for i in range(n_genes)])
        self.layers = layers or {}


def reference_registry_standin():
    """Modules shaped like the reference's plug-in seam ``illico.utils.registry`` (the ``Test`` and ``KernelDataFormat``
    enums and ``dispatcher_registry[(Test, KernelDataFormat)]``, reference utils/registry.py:15-64), holding placeholder
    dispatchers.  The reference is not part of this repository: tests put these into ``sys.modules`` in its place.
    Returns ``{module name: module}``."""
    import enum
    import types

    reg = types.ModuleType("illico.utils.registry")
    reg.Test = enum.Enum("Test", {"OVO": "ovo", "OVR": "ovr"})
    reg.KernelDataFormat = enum.Enum("KernelDataFormat", {"DENSE": "dense", "CSC": "csc", "CSR": "csr"})

    def numba_placeholder(*args, **kwargs):
        raise AssertionError("the reference's own dispatcher was called")

    reg.dispatcher_registry = {(t, f): numba_placeholder for t in reg.Test for f in reg.KernelDataFormat}
    utils = types.ModuleType("illico.utils")
    utils.registry = reg
    pkg = types.ModuleType("illico")
    pkg.utils = utils
    return {"illico": pkg, "illico.utils": utils, "illico.utils.registry": reg}


def planes(df_or_arr, n_groups, n_genes):
    arr = df_or_arr.to_numpy() if hasattr(df_or_arr, "to_numpy") else np.asarray(df_or_arr)
    arr = arr.reshape(n_groups, n_genes, 3)
    return arr[:, :, 0], arr[:, :, 1], arr[:, :, 2]
