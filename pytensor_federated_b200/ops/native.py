"""ctypes binding of ``libb200fed.so`` (the sm_100a kernels + host runtime).

The library is built in-tree by :mod:`pytensor_federated_b200.build`.  On a machine with a
GPU a missing/unloadable library is a hard error — there is no silent PyTorch fallback for
the fused path (the eager implementations in :mod:`pytensor_federated_b200.models` exist as
numerics references and as the CPU/gloo plumbing path only).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

_PKG = Path(__file__).resolve().parent.parent
LIB_PATH = _PKG / "libb200fed.so"

_lib: Optional[C.CDLL] = None

c_void_pp = C.POINTER(C.c_void_p)
c_ll_p = C.POINTER(C.c_longlong)
c_int_p = C.POINTER(C.c_int)
c_double_p = C.POINTER(C.c_double)
c_float_p = C.POINTER(C.c_float)


class NativeError(RuntimeError):
    pass


def _declare(lib: C.CDLL) -> None:
    def sig(name, restype, *argtypes):
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = list(argtypes)

    sig("b200_last_error", C.c_char_p)
    sig("b200_device_count", C.c_int)
    sig("b200_malloc", C.c_int, C.c_int, C.c_size_t, c_void_pp)
    sig("b200_free", C.c_int, C.c_int, C.c_void_p)
    sig("b200_ipc_get_handle", C.c_int, C.c_void_p, C.c_char_p)
    sig("b200_ipc_open_handle", C.c_int, C.c_int, C.c_char_p, c_void_pp)
    sig("b200_ipc_close_handle", C.c_int, C.c_void_p)
    sig("b200_enable_peer_access", C.c_int, C.c_int, C.c_int)
    sig("b200_comm_block_bytes", C.c_size_t, C.c_int, C.c_int, C.c_int)
    sig("b200_engine_create", C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int)
    sig("b200_engine_max_blocks", C.c_int, C.c_void_p)
    sig("b200_engine_sm_count", C.c_int, C.c_void_p)
    sig("b200_engine_alloc_comm", C.c_int, C.c_void_p, c_void_pp)
    sig("b200_engine_bind_comm", C.c_int, C.c_void_p, C.c_void_p, c_void_pp, C.c_void_p)
    sig("b200_engine_reset", C.c_int, C.c_void_p)
    sig("b200_engine_set_timeout", None, C.c_void_p, C.c_double)
    sig("b200_engine_set_grid", None, C.c_void_p, C.c_int)
    sig("b200_engine_set_idle_timeout", None, C.c_void_p, C.c_double)
    sig("b200_engine_set_speculative", C.c_int, C.c_void_p, C.c_double)
    sig("b200_engine_grid", C.c_int, C.c_void_p)
    sig("b200_engine_launches", C.c_ulonglong, C.c_void_p)
    sig("b200_engine_epoch", C.c_ulonglong, C.c_void_p)
    sig("b200_engine_stream", C.c_void_p, C.c_void_p)
    sig("b200_engine_host_theta", C.c_void_p, C.c_void_p)
    sig("b200_engine_host_result", C.c_void_p, C.c_void_p)
    sig(
        "b200_engine_set_linreg", C.c_int, C.c_void_p, C.c_int, c_void_pp, c_void_pp, c_ll_p,
        c_double_p, c_int_p, C.c_int,
    )
    sig(
        "b200_engine_set_glm", C.c_int, C.c_void_p, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_ll_p,
        c_int_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_int_p, C.c_int, C.c_int,
    )
    sig(
        "b200_engine_set_ode", C.c_int, C.c_void_p, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_int_p,
        c_int_p, c_float_p, c_int_p, c_int_p, c_int_p,
    )
    sig("b200_engine_set_custom_launcher", None, C.c_void_p, C.c_void_p)
    sig("b200_engine_set_ode_launcher", None, C.c_void_p, C.c_void_p)
    sig("b200_engine_launch", C.c_int, C.c_void_p)
    sig("b200_engine_set_device_theta", C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int)
    sig("b200_engine_wait", C.c_int, C.c_void_p, C.c_ulonglong, C.c_void_p, C.c_double)
    sig("b200_engine_eval", C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double)
    sig("b200_engine_serve", C.c_longlong, C.c_void_p, C.c_int, C.c_longlong)
    sig("b200_engine_stop_serving", None, C.c_void_p)
    sig("b200_engine_stop_peers", C.c_int, C.c_void_p)
    sig("b200_engine_sync", C.c_int, C.c_void_p)
    sig("b200_engine_trace", C.c_int, C.c_void_p, C.c_ulonglong, C.POINTER(C.c_ulonglong))
    sig("b200_glm_tc_chunk_table", C.c_int, c_ll_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_int_p, C.c_int)
    sig("b200_engine_enable_cta_trace", None, C.c_void_p, C.c_int)
    sig("b200_engine_cta_trace", C.c_int, C.c_void_p, C.POINTER(C.c_ulonglong), C.c_int)
    sig("b200_engine_destroy", None, C.c_void_p)


def load(build_if_missing: bool = True) -> C.CDLL:
    """Loads (building first when necessary and possible) the native library."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists() and build_if_missing:
        from .. import build as _build

        _build.build()
    if not LIB_PATH.exists():
        raise NativeError(f"{LIB_PATH} is missing; run `python -m pytensor_federated_b200.build`")
    # The library's RUNPATH points at the libcudart.so.12 of the CUDA runtime wheel (build.py), so it loads
    # on its own; gRPC-only processes (codec users) must not pay a multi-second `import torch` for it.
    # If that fails (relocated environment) torch is imported first: it brings the same libcudart along.
    try:
        lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_NOW | os.RTLD_LOCAL)
    except OSError:
        try:
            import torch  # noqa: F401

            lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_NOW | os.RTLD_LOCAL)
        except (OSError, ImportError) as ex:
            raise NativeError(f"could not load {LIB_PATH}: {ex}") from ex
    _declare(lib)
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise NativeError(f"{what or 'native call'} failed (rc={rc}): {last_error()}")


def available() -> bool:
    """True when the library loads and at least one CUDA device is visible."""
    try:
        return load(build_if_missing=False).b200_device_count() > 0
    except NativeError:
        return False


def void_p_array(values) -> "C.Array":
    arr = (C.c_void_p * len(values))()
    for i, v in enumerate(values):
        arr[i] = C.c_void_p(int(v) if v else None)
    return arr
