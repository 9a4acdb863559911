"""Loader + ctypes signatures of rustqip_b200/libqipb200.so (include/qipb200.h).

The product path fails loudly when the CUDA extension is missing: there is no
CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

from ._abi import QipOp
from .errors import B200Unavailable, CircuitError

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("QIPB200_LIB") or os.path.join(_HERE, "libqipb200.so")  # QIPB200_LIB: a development build
IPC_HANDLE_BYTES = 64

SCHED_DEFAULT = 0
SCHED_NO_FUSION = 1

_lib = None

# every symbol include/qipb200.h declares
EXPORTS = [
    "qipb200_abi_version", "qipb200_init", "qipb200_init_multi", "qipb200_shutdown", "qipb200_last_error",
    "qipb200_kernel_launches", "qipb200_launch_stats", "qipb200_stream_handle", "qipb200_jit_stats", "qipb200_jit_precompile", "qipb200_profile_enable", "qipb200_profile_read", "qipb200_validate_op", "qipb200_apply_op",
    "qipb200_apply_op_overwrite", "qipb200_apply_ops", "qipb200_state_new", "qipb200_state_free",
    "qipb200_state_set_basis", "qipb200_state_upload", "qipb200_state_download",
    "qipb200_state_apply_op", "qipb200_state_apply_schedule", "qipb200_state_norm2",
    "qipb200_state_sync", "qipb200_state_max_abs_diff", "qipb200_calculate_state", "qipb200_state_measure_probs",
    "qipb200_state_measure_prob", "qipb200_state_soft_measure", "qipb200_state_sample", "qipb200_state_collapse",
    "qipb200_state_new_sharded", "qipb200_state_ipc_export", "qipb200_state_ipc_import",
    "qipb200_state_qubit_map", "qipb200_state_exchange_bytes", "qipb200_plan_exchanges",
    "qipb200_state_save", "qipb200_state_load", "qipb200_schedule_parse", "qipb200_schedule_ops", "qipb200_schedule_free", "qipb200_schedule_serialise",
]


def lib():
    """Load libqipb200.so (built in-tree by `make -C rustqip_b200/csrc` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise B200Unavailable(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). rustqip_b200 has no CPU fallback." % SO_PATH)
    L = C.CDLL(SO_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    opp = C.POINTER(QipOp)
    L.qipb200_abi_version.restype = i32
    L.qipb200_init.restype, L.qipb200_init.argtypes = i32, [C.POINTER(vp), i32]
    L.qipb200_init_multi.restype, L.qipb200_init_multi.argtypes = i32, [C.POINTER(vp), i32, vp]
    L.qipb200_shutdown.restype, L.qipb200_shutdown.argtypes = None, [vp]
    L.qipb200_last_error.restype, L.qipb200_last_error.argtypes = C.c_char_p, [vp]
    L.qipb200_stream_handle.restype, L.qipb200_stream_handle.argtypes = i32, [vp, C.POINTER(vp)]
    L.qipb200_launch_stats.restype, L.qipb200_launch_stats.argtypes = i32, [vp, vp]
    L.qipb200_jit_stats.restype = i32
    L.qipb200_jit_stats.argtypes = [vp, i32, vp, C.c_char_p, C.c_size_t]
    L.qipb200_jit_precompile.restype = i32
    L.qipb200_jit_precompile.argtypes = [i32, u32, opp, C.c_size_t, vp, C.c_char_p, C.c_size_t]
    L.qipb200_profile_enable.restype, L.qipb200_profile_enable.argtypes = i32, [vp, i32]
    L.qipb200_profile_read.restype, L.qipb200_profile_read.argtypes = i32, [vp, vp]
    L.qipb200_kernel_launches.restype, L.qipb200_kernel_launches.argtypes = u64, [vp]
    L.qipb200_validate_op.restype, L.qipb200_validate_op.argtypes = i32, [vp, i32, u32, opp]
    for name in ("qipb200_apply_op", "qipb200_apply_op_overwrite"):
        f = getattr(L, name)
        f.restype, f.argtypes = i32, [vp, i32, u32, opp, vp, u64, vp, u64, u64, u64]
    L.qipb200_apply_ops.restype = i32
    L.qipb200_apply_ops.argtypes = [vp, i32, u32, opp, C.c_size_t, vp, u64, vp, u64, u64, u64]
    L.qipb200_state_new.restype, L.qipb200_state_new.argtypes = i32, [vp, i32, u32, C.POINTER(vp)]
    L.qipb200_state_free.restype, L.qipb200_state_free.argtypes = None, [vp]
    L.qipb200_state_set_basis.restype, L.qipb200_state_set_basis.argtypes = i32, [vp, u64]
    L.qipb200_state_upload.restype, L.qipb200_state_upload.argtypes = i32, [vp, vp, u64, u64]
    L.qipb200_state_download.restype, L.qipb200_state_download.argtypes = i32, [vp, vp, u64, u64]
    L.qipb200_state_apply_op.restype, L.qipb200_state_apply_op.argtypes = i32, [vp, opp]
    L.qipb200_state_apply_schedule.restype = i32
    L.qipb200_state_apply_schedule.argtypes = [vp, opp, C.c_size_t, u32]
    L.qipb200_state_norm2.restype, L.qipb200_state_norm2.argtypes = i32, [vp, C.POINTER(C.c_double)]
    L.qipb200_state_sync.restype, L.qipb200_state_sync.argtypes = i32, [vp]
    L.qipb200_state_max_abs_diff.restype = i32
    L.qipb200_state_max_abs_diff.argtypes = [vp, vp, C.POINTER(C.c_double)]
    L.qipb200_calculate_state.restype = i32
    L.qipb200_calculate_state.argtypes = [vp, i32, u32, u64, opp, C.c_size_t, u32, vp]
    L.qipb200_state_measure_probs.restype = i32
    L.qipb200_state_measure_probs.argtypes = [vp, vp, u32, vp]
    L.qipb200_state_measure_prob.restype = i32
    L.qipb200_state_measure_prob.argtypes = [vp, u64, vp, u32, C.POINTER(C.c_double)]
    L.qipb200_state_soft_measure.restype = i32
    L.qipb200_state_soft_measure.argtypes = [vp, vp, u32, C.c_double, C.POINTER(u64)]
    L.qipb200_state_sample.restype = i32
    L.qipb200_state_sample.argtypes = [vp, vp, u32, vp, u64, vp]
    L.qipb200_state_collapse.restype = i32
    L.qipb200_state_collapse.argtypes = [vp, vp, u32, u64, C.c_double]
    L.qipb200_state_new_sharded.restype = i32
    L.qipb200_state_new_sharded.argtypes = [vp, i32, u32, i32, i32, C.POINTER(vp)]
    L.qipb200_state_ipc_export.restype, L.qipb200_state_ipc_export.argtypes = i32, [vp, vp, vp]
    L.qipb200_state_ipc_import.restype, L.qipb200_state_ipc_import.argtypes = i32, [vp, vp, vp]
    L.qipb200_state_qubit_map.restype, L.qipb200_state_qubit_map.argtypes = i32, [vp, vp]
    L.qipb200_state_exchange_bytes.restype = i32
    L.qipb200_state_exchange_bytes.argtypes = [vp, C.POINTER(u64)]
    L.qipb200_plan_exchanges.restype = i32
    L.qipb200_plan_exchanges.argtypes = [i32, u32, i32, opp, C.c_size_t, vp]
    L.qipb200_state_save.restype, L.qipb200_state_save.argtypes = i32, [vp, C.c_char_p]
    L.qipb200_state_load.restype, L.qipb200_state_load.argtypes = i32, [vp, C.c_char_p]
    L.qipb200_schedule_parse.restype = i32
    L.qipb200_schedule_parse.argtypes = [vp, C.c_size_t, C.POINTER(vp), C.c_char_p, C.c_size_t]
    L.qipb200_schedule_ops.restype = opp
    L.qipb200_schedule_ops.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(u32), C.POINTER(i32)]
    L.qipb200_schedule_free.restype, L.qipb200_schedule_free.argtypes = None, [vp]
    L.qipb200_schedule_serialise.restype = C.c_size_t
    L.qipb200_schedule_serialise.argtypes = [i32, u32, opp, C.c_size_t, vp, C.c_size_t]
    _lib = L
    return L


def check(status: int, ctx=None):
    """Non-zero status -> CircuitError(msg) (the shim's mapping, SURVEY.md section 8b)."""
    if status != 0:
        msg = lib().qipb200_last_error(ctx).decode("utf-8", "replace")
        raise CircuitError(msg or ("qipb200 status %d" % status), status=status)
