"""ctypes binding of libsrj_b200.so (the C ABI in include/srj_b200.h).

The library is the product: there is NO Python/CPU fallback.  If the shared object is missing
or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SRJ_B200_LIB") or os.path.join(_HERE, "libsrj_b200.so")  # env: development variants only

SRJ_OK, SRJ_EINVAL, SRJ_EUNSUPPORTED, SRJ_EOVERFLOW, SRJ_ECUDA, SRJ_ENOMEM = 0, -1, -2, -3, -4, -5
HASH_NONE, HASH_XXHASH64, HASH_MURMUR3_32, HASH_HIVE = 0, 1, 2, 3


class SrjColumn(C.Structure):
    pass


SrjColumn._fields_ = [("type_id", C.c_int32), ("scale", C.c_int32), ("size", C.c_int64), ("data", C.c_void_p),
                      ("null_mask", C.c_void_p), ("offsets", C.c_void_p), ("children", C.POINTER(SrjColumn)),
                      ("num_children", C.c_int32), ("reserved", C.c_int32)]


class SrjRowBatch(C.Structure):
    _fields_ = [("row_start", C.c_int64), ("row_count", C.c_int64), ("num_bytes", C.c_int64)]


class SrjLayout(C.Structure):
    _fields_ = [("num_columns", C.c_int32), ("num_string_columns", C.c_int32), ("validity_offset", C.c_int32),
                ("size_per_row", C.c_int32), ("fixed_row_size", C.c_int32), ("reserved", C.c_int32)]


class SrjFusedHash(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_keys", C.c_int32), ("key_columns", C.c_int32 * 16), ("seed", C.c_int64),
                ("out", C.c_void_p)]


# every symbol include/srj_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "srj_version": (C.c_char_p, []),
    "srj_last_error": (C.c_char_p, []),
    "srj_status_string": (C.c_char_p, [C.c_int]),
    "srj_compute_layout": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(SrjLayout), C.c_void_p, C.c_void_p]),
    "srj_plan_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "srj_plan_destroy": (None, [C.c_void_p]),
    "srj_plan_layout": (C.c_int, [C.c_void_p, C.POINTER(SrjLayout)]),
    "srj_to_rows_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "srj_to_rows_plan_batches": (C.c_int, [C.c_void_p, C.POINTER(SrjColumn), C.c_int64, C.c_void_p,
                                           C.POINTER(SrjRowBatch), C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "srj_convert_to_rows": (C.c_int, [C.c_void_p, C.POINTER(SrjColumn), C.c_int64, C.c_void_p,
                                      C.POINTER(SrjRowBatch), C.c_int32, C.POINTER(C.c_void_p),
                                      C.POINTER(C.c_void_p), C.c_void_p]),
    "srj_from_rows_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "srj_convert_from_rows_fixed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                              C.POINTER(SrjColumn), C.c_void_p, C.c_void_p,
                                              C.POINTER(SrjFusedHash), C.c_void_p, C.c_void_p]),
    "srj_convert_from_rows_strings": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                                C.POINTER(SrjColumn), C.c_void_p, C.c_void_p, C.c_void_p]),
    "srj_get_max_stack_depth": (C.c_int, []),
    "srj_xxhash64": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "srj_murmur_hash3_32": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_uint32, C.c_void_p,
                                      C.c_void_p]),
    "srj_hive_hash": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "srj_partition_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "srj_hash_partition": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "srj_partition_plan": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "srj_partition_columns": (C.c_int, [C.POINTER(SrjColumn), C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "srj_partition_strings": (C.c_int, [C.POINTER(SrjColumn), C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "srj_unsafe_row_layout": (C.c_int, [C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "srj_unsafe_row_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int64]),
    "srj_unsafe_row_sizes": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]),
    "srj_convert_to_unsafe_rows": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "srj_convert_from_unsafe_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(SrjColumn), C.c_int32, C.c_void_p, C.c_void_p,
                                               C.c_void_p]),
    "srj_convert_from_unsafe_rows_strings": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(SrjColumn), C.c_int32, C.c_void_p]),
    "srj_kudo_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "srj_kudo_split_sizes": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_int64),
                                       C.c_void_p, C.c_void_p]),
    "srj_kudo_split": (C.c_int, [C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "srj_kudo_assemble_sizes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int64),
                                          C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]),
    "srj_kudo_assemble": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SrjColumn), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "srj_kudo_nested_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "srj_kudo_assemble_nested_sizes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32,
                                                 C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]),
    "srj_kudo_assemble_nested": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SrjColumn), C.c_int32, C.c_void_p, C.c_void_p]),
    "srj_shard_rebase_offsets": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_void_p]),
    "srj_convert_from_rows_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(SrjColumn),
                                             C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "srj_convert_to_rows_host": (C.c_int, [C.c_void_p, C.POINTER(SrjColumn), C.c_int64, C.POINTER(SrjRowBatch), C.c_int32,
                                           C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p,
                                           C.c_void_p]),
}

HOST_ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int32, C.c_int64)     # srj_host_alloc_fn

_lib = None


def lib():
    """Load libsrj_b200.so (fails loudly when it has not been built: python spark-rapids-jni_b200/build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python spark-rapids-jni_b200/build.py` "
                              "(the CUDA library is the product; there is no fallback path)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(_lib, name)   # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
    return _lib


class CudfException(RuntimeError):
    """ai.rapids.cudf.CudfException (cudf::logic_error and friends, error.hpp:233-239)."""


class CudfColumnSizeOverflowException(CudfException):
    """std::overflow_error -> CudfColumnSizeOverflowException (error.hpp:181-230)."""


class CudaException(CudfException):
    """cudf::cuda_error -> ai.rapids.cudf.CudaException."""


def check(rc: int, what: str = ""):
    """Map a C-ABI status to the exception class the reference's JNI layer would throw."""
    if rc == SRJ_OK:
        return
    msg = lib().srj_last_error().decode("utf-8", "replace")
    if rc == SRJ_EOVERFLOW:
        raise CudfColumnSizeOverflowException(msg)
    if rc == SRJ_ENOMEM:
        raise MemoryError(msg)
    if rc == SRJ_ECUDA:
        raise CudaException(msg)
    raise CudfException(f"{what}: {msg}" if what else msg)
