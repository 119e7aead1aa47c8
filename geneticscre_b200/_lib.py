"""ctypes binding of the C ABI in include/gcre_b200.h (libgcre_b200.so, built in-tree by geneticscre_b200/build.py).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GCRE_B200_LIB") or os.path.join(PKG, "libgcre_b200.so")  # override: A/B builds during tuning

GCRE_OK, GCRE_ERR_ASSERT, GCRE_ERR_RANGE, GCRE_ERR_ARG, GCRE_ERR_CUDA, GCRE_ERR_NOMEM = 0, -1, -2, -3, -4, -5
KERNEL_AUTO, KERNEL_DENSE, KERNEL_SPARSE = 0, 1, 2


class ScoreC(C.Structure):
    _fields_ = [("score", C.c_double), ("src", C.c_int32), ("trg", C.c_int32), ("cases", C.c_int32), ("ctrls", C.c_int32)]


class UidRefC(C.Structure):
    _fields_ = [("src", C.c_int32), ("trg", C.c_int32), ("count", C.c_int32), ("location", C.c_uint32), ("path_idx", C.c_uint64)]


class ExecInfoC(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("method", "num_cases", "num_ctrls", "width_ul", "iterations", "iters_requested", "device", "sm_count")]


class DecoratedC(C.Structure):
    _fields_ = [("pvalue", C.c_double), ("score", C.c_double), ("cases1", C.c_int32), ("ctrls1", C.c_int32), ("cases2", C.c_int32), ("ctrls2", C.c_int32)]


class JoinOptsC(C.Structure):
    _fields_ = [("uid_begin", C.c_uint32), ("uid_end", C.c_uint32), ("kernel", C.c_int32), ("skip_host_perm", C.c_int32),
                ("pairs_scored", C.c_uint64), ("kernel_ms", C.c_double), ("kernel_used", C.c_int32), ("launches", C.c_int32),
                ("precounted", C.c_int32), ("split_carrier", C.c_int32), ("thresholded", C.c_int32), ("shared_masks", C.c_int32),
                ("exact_pairs", C.c_uint64), ("tail_form", C.c_int32), ("reserved2", C.c_int32)]


# every symbol include/gcre_b200.h declares: name -> (restype, argtypes)
_VP, _I, _U32 = C.c_void_p, C.c_int, C.c_uint32
SYMBOLS = {
    "gcre_last_error": (C.c_char_p, []),
    "gcre_version": (C.c_char_p, []),
    "gcre_device_count": (_I, [C.POINTER(_I)]),
    "gcre_kernel_launch_count": (_I, [C.POINTER(C.c_uint64)]),
    "gcre_release_cached_memory": (_I, []),
    "gcre_exec_create": (_I, [_I, _I, _I, _I, _I, C.POINTER(_VP)]),
    "gcre_exec_destroy": (_I, [_VP]),
    "gcre_exec_get_info": (_I, [_VP, C.POINTER(ExecInfoC)]),
    "gcre_exec_decorated_exact": (_I, [_VP, C.POINTER(C.c_uint64), _U32, C.POINTER(DecoratedC)]),
    "gcre_exec_set_stream": (_I, [_VP, _VP]),
    "gcre_exec_set_value_table": (_I, [_VP, C.POINTER(C.c_double), _I, _I]),
    "gcre_exec_generate_value_table": (_I, [_VP]),
    "gcre_log_factorial_table": (_I, [_I, C.POINTER(C.c_double)]),
    "gcre_exec_get_value_table": (_I, [_VP, C.POINTER(C.c_double), _I, _I]),
    "gcre_exec_set_permuted_cases_i32": (_I, [_VP, C.POINTER(C.c_int32), _I, _I]),
    "gcre_exec_set_permuted_masks_u64": (_I, [_VP, C.POINTER(C.c_uint64), _I]),
    "gcre_exec_set_permuted_masks_device": (_I, [_VP, _VP, _I]),
    "gcre_exec_set_permutation_strata": (_I, [_VP, C.POINTER(C.c_int32), _I]),
    "gcre_exec_generate_permuted_masks": (_I, [_VP, C.c_uint64, C.c_uint64]),
    "gcre_exec_get_permuted_masks": (_I, [_VP, C.POINTER(C.c_uint64), _I]),
    "gcre_pathset_create": (_I, [_VP, _U32, C.POINTER(_VP)]),
    "gcre_pathset_destroy": (_I, [_VP]),
    "gcre_pathset_size": (_I, [_VP, C.POINTER(_U32)]),
    "gcre_pathset_load_i32": (_I, [_VP, C.POINTER(C.c_int32), _U32, _I]),
    "gcre_pathset_load_bits": (_I, [_VP, C.POINTER(C.c_uint64), _U32, _I]),
    "gcre_pathset_load_bits_device": (_I, [_VP, _VP, _U32, _I]),
    "gcre_exec_set_value_table_device": (_I, [_VP, _VP, _I, _I]),
    "gcre_host_pack_i32": (_I, [C.POINTER(C.c_int32), _U32, _I, C.POINTER(C.c_uint64), _I]),
    "gcre_pathset_select": (_I, [_VP, C.POINTER(C.c_int32), _U32, C.POINTER(_VP)]),
    "gcre_pathset_set_row": (_I, [_VP, _U32, C.POINTER(C.c_uint64)]),
    "gcre_pathset_get_row": (_I, [_VP, _U32, C.POINTER(C.c_uint64)]),
    "gcre_pathset_download": (_I, [_VP, C.POINTER(C.c_uint64)]),
    "gcre_join": (_I, [_VP, _I, C.POINTER(UidRefC), _U32, C.POINTER(C.c_int32), _U32, _VP, _VP, _VP, _I, C.POINTER(ScoreC),
                       C.POINTER(_I), C.POINTER(C.c_double), C.POINTER(JoinOptsC)]),
    "gcre_uidset_create": (_I, [_VP, _I, C.POINTER(UidRefC), _U32, C.POINTER(C.c_int32), _U32, C.POINTER(_VP)]),
    "gcre_uidset_destroy": (_I, [_VP]),
    "gcre_join_uidset": (_I, [_VP, _VP, _VP, _VP, _VP, _I, C.POINTER(ScoreC), C.POINTER(_I), C.POINTER(C.c_double), C.POINTER(JoinOptsC)]),
    "gcre_exec_device_perm_max": (_I, [_VP, C.POINTER(_VP), C.POINTER(_I)]),
    "gcre_exec_export_perm_max": (_I, [_VP, _VP, _I]),
    "gcre_exec_import_perm_max": (_I, [_VP, _VP, _I]),
    "gcre_exec_read_perm_max": (_I, [_VP, C.POINTER(C.c_double)]),
    "gcre_merge_topk": (_I, [C.POINTER(ScoreC), C.POINTER(_I), _I, _I, C.POINTER(ScoreC), C.POINTER(_I)]),
    # test and diagnostics only
    "gcre_pathset_debug_view_info": (_I, [_VP, C.POINTER(C.c_int64)]),
    "gcre_pathset_debug_counts": (_I, [_VP, C.POINTER(C.c_uint16), C.POINTER(_U32), C.POINTER(_U32)]),
    "gcre_pathset_debug_lists": (_I, [_VP, C.POINTER(C.c_uint64), C.POINTER(_U32), C.POINTER(_U32), C.POINTER(_U32)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libgcre_b200.so (raises if it has not been built: run ``python -m geneticscre_b200.build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing - build the CUDA engine first (python geneticscre_b200/build.py); "
                               "there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class GcreError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"gcre status {status}: {message}")
        self.status = status


class GcreAssertion(GcreError):  # reference: std::logic_error("assertion")
    pass


class GcreOutOfRange(GcreError, IndexError):  # reference: std::out_of_range("assertion")
    pass


def check(status: int) -> None:
    if status == GCRE_OK:
        return
    msg = load().gcre_last_error().decode()
    if status == GCRE_ERR_ASSERT:
        raise GcreAssertion(status, msg)
    if status == GCRE_ERR_RANGE:
        raise GcreOutOfRange(status, msg)
    raise GcreError(status, msg)
