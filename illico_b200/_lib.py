"""ctypes binding of ``libillico_b200.so`` (declared in ``include/illico_b200.h``).

There is no CPU fallback: if the CUDA library is missing or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libillico_b200.so")

ABI_VERSION = 3
ALTERNATIVES = {"two-sided": 0, "less": 1, "greater": 2}
TIES_DENSE, TIES_SPARSE = 0, 1

_vp, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t


class Plan(C.Structure):
    """``illico_plan_t``"""

    _fields_ = [
        ("n_cells", _i32), ("n_groups", _i32), ("n_segments", _i32), ("ref_group", _i32),
        ("max_group_size", _i32), ("ref_group_size", _i32), ("ref_seg_begin", _i32), ("ref_seg_end", _i32),
        ("slot_cap", _i32), ("max_target_group_size", _i32),
        ("perm", _vp), ("cell_seg", _vp), ("seg_pos", _vp), ("seg_base", _vp), ("seg_group", _vp),
        ("group_seg", _vp), ("group_size", _vp),
    ]


class Flags(C.Structure):
    """``illico_flags_t``"""

    _fields_ = [("is_log1p", _i32), ("use_continuity", _i32), ("tie_correct", _i32), ("alternative", _i32),
                ("tie_order", _i32), ("n_cols_hint", _i32), ("group_sums", _vp), ("scores", _vp),
                ("score_group_stride", _i64)]

    def replace(self, **fields) -> "Flags":
        """A copy with some fields changed."""
        out = Flags.from_buffer_copy(self)
        for k, v in fields.items():
            setattr(out, k, v)
        return out


class Debug(C.Structure):
    """``illico_debug_t``"""

    _fields_ = [("u2", _vp), ("tie_sum", _vp), ("tie_exact", _vp)]


class BatchBuffers(C.Structure):
    """``illico_batch_buffers_t``"""

    _fields_ = [("ir_vals", _vp), ("ir_cnt", _vp), ("workspace", _vp), ("workspace_bytes", _sz)]


# name -> (restype, argtypes); every symbol include/illico_b200.h declares
_PP, _FP, _DP, _BP = C.POINTER(Plan), C.POINTER(Flags), C.POINTER(Debug), C.POINTER(BatchBuffers)
_DISPATCH_DENSE = (C.c_int, [_vp, _i64, _i32, _i32, _PP, _FP, _BP, _vp, _i64, _DP, _vp])
_DISPATCH_SPARSE = (C.c_int, [_vp, _vp, _vp, _i32, _i32, _PP, _FP, _BP, _vp, _i64, _DP, _vp])
SIGNATURES = {
    "illico_abi_version": (C.c_int, []),
    "illico_last_error": (C.c_char_p, []),
    "illico_launch_count": (_i64, []),
    "illico_last_fused_ms": (C.c_double, []),
    "illico_profile_report": (_i64, [C.c_char_p, _i64]),
    "illico_memcpy2d_async": (C.c_int, [_vp, _sz, _vp, _sz, _sz, _sz, C.c_int, _vp]),
    "illico_stage_dense_f32": (C.c_int, [_vp, _i64, _i32, _i32, _PP, _vp, _vp, _vp]),
    "illico_stage_csr_workspace_bytes": (_sz, [_PP, _i32]),
    "illico_stage_csr_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _PP, _vp, _vp, _vp, _sz, _vp]),
    "illico_stage_csc_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _PP, _vp, _vp, _vp]),
    "illico_zero_counts": (C.c_int, [_vp, _i32, _PP, _vp]),
    "illico_check_csr_sorted": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "illico_rank_workspace_bytes": (_sz, [_PP, _i32]),
    "illico_rank_ovr": (C.c_int, [_vp, _vp, _i32, _PP, _FP, _vp, _i64, _vp, _sz, _DP, _vp]),
    "illico_rank_ovo": (C.c_int, [_vp, _vp, _i32, _PP, _FP, _vp, _i64, _vp, _sz, _DP, _vp]),
    "illico_ovr_dense_f32": _DISPATCH_DENSE,
    "illico_ovo_dense_f32": _DISPATCH_DENSE,
    "illico_ovr_csr_f32": _DISPATCH_SPARSE,
    "illico_ovo_csr_f32": _DISPATCH_SPARSE,
    "illico_ovr_csc_f32": _DISPATCH_SPARSE,
    "illico_ovo_csc_f32": _DISPATCH_SPARSE,
    "illico_convert_values": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _vp, _vp]),
    "illico_recode_workspace_bytes": (_sz, [_i64, _i32]),
    "illico_recode_dense": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "illico_recode_csc": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "illico_recode_csr": (C.c_int, [_vp, _i32, _vp, _vp, _i64, _i32, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "illico_enable_peer_access": (C.c_int, [_i32, _i32]),
    "illico_csr_shard_count": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "illico_csr_shard_scatter": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "illico_host_pack_rows_f32": (C.c_long, [_vp, C.c_long, C.c_long, C.c_long, _vp, _vp, _vp, C.c_long]),
    "illico_host_pack_isa": (C.c_int, []),
    "illico_unpack_rows_f32": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _i64, _vp]),
    "illico_bh_workspace_bytes": (_sz, [_i32, _i32]),
    "illico_bh_adjust": (C.c_int, [_vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    "illico_top_genes_workspace_bytes": (_sz, [_i32, _i32]),
    "illico_top_genes": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "illico_top_genes_filtered": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _i32, _i32, _i32, _i32, C.c_double, C.c_double,
                                            C.c_double, C.c_double, _vp, _vp, _vp, _vp, _sz, _vp]),
    "illico_count_nonzero_dense": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _PP, _vp, _i64, _vp]),
    "illico_count_nonzero_csr": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _PP, _vp, _i64, _vp]),
    "illico_count_nonzero_csc": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _PP, _vp, _i64, _vp]),
    "illico_nonzero_fractions": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32, _i64, _vp, _vp, _vp]),
    "illico_group_moments_dense": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _PP, _i32, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "illico_group_moments_csr": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _PP, _i32, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "illico_group_moments_csc": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _PP, _i32, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "illico_welch_ttest": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i32, _i32, _i32, _i64, _i32, _i32, _vp, _i64, _vp, _i64, _vp]),
    "illico_student_t_batch": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "illico_compute_pval_batch": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
}

DTYPE_F32, DTYPE_F64, DTYPE_F16, DTYPE_I8, DTYPE_U8, DTYPE_I16, DTYPE_I32, DTYPE_I64 = range(8)

_lib = None


class IllicoCudaError(RuntimeError):
    pass


def load():
    """Loads the shared library (building nothing: ``__graft_entry__.build()`` / ``illico_b200.build`` do that)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IllicoCudaError(
            f"{LIB_PATH} is missing: build it with `python -m illico_b200.build` (nvcc, sm_100a). "
            "illico_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    if L.illico_abi_version() != ABI_VERSION:
        raise IllicoCudaError(f"ABI mismatch: library {L.illico_abi_version()} vs binding {ABI_VERSION}")
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().illico_last_error()
        raise IllicoCudaError(f"{what} failed: {msg.decode() if msg else rc}")


def launch_count() -> int:
    return int(load().illico_launch_count())


def profile_report() -> dict:
    """``{kernel name: (total ms, launches)}`` of the launches recorded since the last call (``ILLICO_PROFILE=1``)."""
    buf = C.create_string_buffer(1 << 16)
    load().illico_profile_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, ms, n = line.split("\t")
        out[name] = (float(ms), int(n))
    return out
