"""SURVEY.md section 8(f3) / VERDICT r1 next #9: the six GPU dispatchers RUN the way the reference's own driver runs them.

``illico_b200.register_into_reference()`` puts them into the reference's ``dispatcher_registry``
(``illico/utils/registry.py:61-64, 193-202``); the reference's ``asymptotic_wilcoxon`` then computes every gene batch
through the registered dispatcher on its joblib threads and assembles the [G, N] result
(``illico/asymptotic_wilcoxon.py:212-249``).  The reference is not part of this repository, so a stand-in of its
registry module receives the dispatchers and ``_drive`` restates that batch loop.  The result is compared with the
committed golden vectors (the same reference with its own numba kernels) and with the oracle.
"""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle  # noqa: E402
from tests.golden import cases as C  # noqa: E402
from tests.parity import FC_RTOL, assert_parity  # noqa: E402
from tests.util import reference_registry_standin  # noqa: E402


@pytest.fixture(scope="module")
def reference_with_gpu_dispatchers():
    import illico_b200
    from illico_b200 import dispatch

    with pytest.MonkeyPatch.context() as mp:
        mods = reference_registry_standin()
        for name, mod in mods.items():
            mp.setitem(sys.modules, name, mod)
        assert illico_b200.register_into_reference() is True
        yield mods["illico.utils.registry"]
    dispatch.clear_caches()


def _drive(ref, X, labels, reference, fmt, test, batch_size, n_threads):
    """The reference's batch loop: integer gene batches (fewer than 256 genes: one batch on one thread), each computed by
    the registered dispatcher on a thread pool and written into the [G, N] result planes."""
    from illico_b200.groups import encode_and_count_groups

    groups, grpc = encode_and_count_groups(labels, reference)
    fn = ref.dispatcher_registry[(ref.Test(test), ref.KernelDataFormat(fmt))]
    n_genes = X.shape[1]
    if n_genes < 256:
        batch_size, n_threads = n_genes, 1
    out = np.full((3, len(groups), n_genes), np.nan)

    def one(lb):
        ub = min(lb + batch_size, n_genes)
        for k, plane in enumerate(fn(X, lb, ub, grpc, False, True, True, "two-sided")):
            out[k, :, lb:ub] = plane

    with ThreadPoolExecutor(max_workers=n_threads) as ex:
        list(ex.map(one, range(0, n_genes, batch_size)))
    return groups, out[0], out[1], out[2]


@pytest.mark.parametrize("name,fmt,test,n_threads,batch_size", [
    ("batched", "dense", "ovo", 3, 64),      # 300 genes: several batches on threads, concurrently
    ("batched", "csr", "ovr", 2, 128),
    ("batched", "csc", "ovo", 1, 100),
    ("k562_mini", "dense", "ovr", 1, 16),    # < 256 genes: the reference forces one batch, one thread
    ("k562_mini", "csr", "ovo", 1, 16),
    ("highcount", "dense", "ovo", 1, 16),
])
def test_reference_driver_runs_gpu_dispatchers(golden_dir, reference_with_gpu_dispatchers, name, fmt, test, n_threads, batch_size):
    from illico_b200 import _lib

    builder, grid, _bs = C.CASES[name]
    X, labels, reference = builder()
    ref = reference if test == "ovo" else None
    before = _lib.launch_count()
    groups, p, U, fc = _drive(reference_with_gpu_dispatchers, C.to_format(X, fmt), labels, ref, fmt, test, batch_size,
                              n_threads)
    assert _lib.launch_count() > before, "the driver did not reach the GPU dispatchers"
    gold = np.load(os.path.join(golden_dir, f"{name}.npz"))
    assert list(groups) == list(gold["groups"])
    want = gold[C.combo_key(fmt, test, True, True, "two-sided", False)]
    ref_row = int(np.searchsorted(groups, reference)) if test == "ovo" else None
    assert_parity((p, U, fc), (want[0], want[1], want[2]), ref_row=ref_row, fc_rtol=FC_RTOL,
                  what=f"reference driver + GPU dispatchers {name}:{fmt}:{test}")
    g, po, Uo, fco = oracle.run(C.to_format(X, fmt), labels, ref)
    assert_parity((p, U, fc), (po, Uo, fco), ref_row=ref_row, what="vs oracle")
