"""The C-ABI boundary: header, ctypes table and shared object must agree (CPU only,
no compute calls)."""
import ctypes
import os
import re
import subprocess

from ray_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200_collective.h")


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    # every prototype in the header starts with a return type and a b200_ name
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_what_the_binding_binds():
    declared = _declared_functions()
    assert declared, "no prototypes parsed from the header"
    assert sorted(_native.SIGNATURES) == declared


def _declared_enumerators(typedef):
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef enum \{([^}]*)\}\s*" + typedef + r";", text)
    assert body, f"enum {typedef} not found in the header"
    return {name: int(value) for name, value in re.findall(r"\b(B200_\w+)\s*=\s*(-?\d+)", body.group(1))}


def test_header_enums_match_the_binding_constants():
    """Parameter and algorithm numbers are part of the ABI: the binding's PARAM_* / ALGO_* must be
    exactly the header's enumerators, value for value."""
    for typedef, prefix, count in (("b200_param_t", "PARAM_", "B200_PARAM_COUNT"), ("b200_algo_t", "ALGO_", None)):
        declared = _declared_enumerators(typedef)
        assert declared, typedef
        if count:
            assert declared.pop(count) == len(declared), f"{count} is not the number of parameters"
            assert sorted(declared.values()) == list(range(len(declared))), f"{typedef} is not contiguous"
        bound = {f"B200_{k}": v for k, v in vars(_native).items() if k.startswith(prefix)}
        assert bound == declared, typedef


def test_library_exports_every_declared_symbol(native_lib):
    out = subprocess.run(["nm", "-D", "--defined-only", str(_native.LIB_PATH)], capture_output=True, text=True,
                         check=True).stdout
    exported = set(re.findall(r"\sT\s+(b200_[a-z0-9_]+)", out))
    missing = [n for n in _declared_functions() if n not in exported]
    assert not missing, f"not exported: {missing}"
    for name in _declared_functions():
        assert getattr(native_lib, name) is not None


def test_library_has_no_libcuda_or_torch_dependency(native_lib):
    out = subprocess.run(["ldd", str(_native.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    assert "libcuda.so" not in out and "libtorch" not in out and "libnccl" not in out, out


def test_no_nccl_symbols_referenced(native_lib):
    out = subprocess.run(["nm", "-D", str(_native.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    assert "nccl" not in out.lower()


def test_introspection_calls_work_without_a_gpu(native_lib):
    assert b"sm_100a" in native_lib.b200_version()
    sizes = {_native.U8: 1, _native.I8: 1, _native.F16: 2, _native.BF16: 2, _native.I32: 4, _native.U32: 4,
             _native.F32: 4, _native.I64: 8, _native.U64: 8, _native.F64: 8}
    for code, size in sizes.items():
        assert native_lib.b200_dtype_size(code) == size
    assert native_lib.b200_dtype_size(99) == 0


def test_invalid_arguments_fail_loudly_without_a_gpu(native_lib):
    h = ctypes.c_void_p()
    rc = native_lib.b200_comm_create(9, 0, 0, None, ctypes.byref(h))
    assert rc == _native.ERR_INVALID and "max 8" in _native.last_error()
    rc = native_lib.b200_comm_create(2, 2, 0, None, ctypes.byref(h))
    assert rc == _native.ERR_INVALID
    # null communicator
    assert native_lib.b200_barrier(None, None) == _native.ERR_INVALID
    assert native_lib.b200_allreduce(None, None, None, 4, _native.F32, _native.SUM, 0, None) == _native.ERR_INVALID


def test_sass_contains_blackwell_multicast_and_sys_scope_flags(native_lib):
    sass = subprocess.run(["cuobjdump", "-sass", str(_native.LIB_PATH)], capture_output=True, text=True)
    if sass.returncode != 0:
        import pytest

        pytest.skip("cuobjdump unavailable")
    text = sass.stdout
    assert "sm_100a" in text
    assert "LDGMC" in text, "multimem.ld_reduce missing from SASS"
    # north_star: "TMA bulk staging into shared memory": cp.async.bulk -> UBLKCP, mbarrier -> SYNCS
    assert "UBLKCP" in text and "SYNCS" in text, "bulk-copy engine (cp.async.bulk + mbarrier) missing from SASS"
    for kernel in ("p2p_bulk_kernel", "allreduce_pull_kernel", "allreduce_pipe_kernel", "allgather_pull_kernel", "get_bulk_kernel"):
        assert kernel in text, kernel
    assert re.search(r"ST\w*\.E\.\w*STRONG\.SYS|STG\.E\.STRONG\.SYS", text), "system-scope flag stores missing"
