"""ctypes binding of libb200_collective.so (the C ABI declared in include/b200_collective.h).

There is deliberately no CPU or library fallback: if the shared object is missing the
import fails loudly, and every entry point raises on a non-zero status.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_size_t, c_uint64, c_void_p
from pathlib import Path

LIB_NAME = "libb200_collective.so"
LIB_PATH = Path(__file__).resolve().parent / LIB_NAME
HANDLE_BYTES = 256
MAX_RANKS = 8

# status codes (b200_status_t)
OK = 0
ERR_INVALID = -1
ERR_CUDA = -2
ERR_SYSTEM = -3
ERR_UNSUPPORTED = -4
ERR_ABORTED = -5
ERR_TIMEOUT = -6
ERR_TOO_LARGE = -7

# dtypes (b200_dtype_t)
U8, I8, I32, U32, I64, U64, F16, BF16, F32, F64 = range(10)
# reduce ops (b200_op_t) -- same numbering as ray.util.collective.types.ReduceOp
SUM, PROD, MIN, MAX, AVG = range(5)
# tuning parameters (b200_param_t)
(PARAM_ONESHOT_MAX_BYTES, PARAM_NVLS_MIN_WORLD, PARAM_NVLS_CTAS, PARAM_LL_MAX_BYTES, PARAM_PIPE_MIN_BYTES,
 PARAM_PIPE_CHUNK_BYTES, PARAM_PIPE_COPY_CTAS, PARAM_PIPE_RED_CTAS, PARAM_PIPE_VARIANT,
 PARAM_P2P_BULK_MIN_CHUNK, PARAM_AG_PULL_MIN_BYTES) = range(11)
# algorithms (b200_algo_t)
ALGO_AUTO, ALGO_ONESHOT, ALGO_TWOSHOT, ALGO_NVLS, ALGO_LL, ALGO_PIPE = range(6)


class B200Config(ctypes.Structure):
    _fields_ = [
        ("staging_bytes", c_size_t),
        ("heap_bytes", c_size_t),
        ("inbox_bytes", c_size_t),
        ("enable_multicast", c_int),
        ("timeout_ms", c_int),
    ]


class B200Error(RuntimeError):
    """A libb200_collective call failed."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[b200 status {status}] {message}")
        self.status = status


class B200AbortedError(B200Error):
    """The communicator was aborted / destroyed (maps to ray.exceptions.RayChannelError)."""


class B200TimeoutError(B200Error):
    """A device-side wait hit the watchdog (a peer never arrived)."""


# Every exported symbol with (restype, argtypes).  tests/test_abi.py checks this table
# against include/b200_collective.h so the header, the binding and the .so cannot drift.
SIGNATURES = {
    "b200_comm_create": (c_int, [c_int, c_int, c_int, POINTER(B200Config), POINTER(c_void_p)]),
    "b200_comm_export_handle": (c_int, [c_void_p, c_void_p]),
    "b200_comm_connect": (c_int, [c_void_p, c_void_p]),
    "b200_comm_destroy": (c_int, [c_void_p]),
    "b200_comm_abort": (c_int, [c_void_p]),
    "b200_comm_status": (c_int, [c_void_p]),
    "b200_comm_rank": (c_int, [c_void_p]),
    "b200_comm_world_size": (c_int, [c_void_p]),
    "b200_comm_has_multicast": (c_int, [c_void_p]),
    "b200_symm_alloc": (c_int, [c_void_p, c_size_t, POINTER(c_void_p)]),
    "b200_symm_reset": (c_int, [c_void_p]),
    "b200_symm_contains": (c_int, [c_void_p, c_void_p, c_size_t]),
    "b200_pool_bind": (c_int, [c_void_p]),
    "b200_pool_alloc": (c_void_p, [c_size_t, c_int, c_void_p]),
    "b200_pool_free": (None, [c_void_p, c_size_t, c_int, c_void_p]),
    "b200_allreduce": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "b200_allgather": (c_int, [c_void_p, c_void_p, POINTER(c_void_p), c_size_t, c_int, c_void_p]),
    "b200_reducescatter": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "b200_broadcast": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "b200_reduce": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "b200_barrier": (c_int, [c_void_p, c_void_p]),
    "b200_send": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "b200_recv": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "b200_symm_base": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_size_t)]),
    "b200_get": (c_int, [c_void_p, c_void_p, c_int, c_size_t, c_size_t, c_void_p]),
    "b200_grad_allreduce": (c_int, [c_void_p, c_void_p, c_size_t, c_float, c_int, c_void_p]),
    "b200_allreduce_multi": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_size_t), c_int, c_int, c_int, c_void_p]),
    "b200_last_error": (c_char_p, []),
    "b200_version": (c_char_p, []),
    "b200_dtype_size": (c_size_t, [c_int]),
    "b200_comm_launch_count": (c_uint64, [c_void_p]),
    "b200_comm_set_blocks": (c_int, [c_void_p, c_int]),
    "b200_comm_set_param": (c_int, [c_void_p, c_int, ctypes.c_longlong]),
    "b200_selftest_pipe_geometry": (c_int, [c_size_t, c_size_t, c_int, c_int, c_int, ctypes.c_uint]),
    "b200_comm_trace_enable": (c_int, [c_void_p, ctypes.c_uint]),
    "b200_comm_trace_read": (c_int, [c_void_p, POINTER(ctypes.c_ulonglong), ctypes.c_uint, c_int]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared object (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("B200_COLLECTIVE_LIB", LIB_PATH))
    if not path.exists():
        raise ImportError(
            f"{path} not found: build it with `python -m ray_b200.build` "
            "(nvcc, sm_100a).  ray_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(str(path), mode=ctypes.RTLD_GLOBAL)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = ABI drift, fail loudly
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().b200_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int) -> None:
    if status == OK:
        return
    msg = last_error()
    if status == ERR_ABORTED:
        raise B200AbortedError(status, msg or "communicator aborted")
    if status == ERR_TIMEOUT:
        raise B200TimeoutError(status, msg or "device-side wait timed out")
    raise B200Error(status, msg or "unknown error")
