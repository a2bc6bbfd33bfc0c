"""ctypes binding of the C-ABI library (include/autogptq_b200.h).

The product has no CPU fallback: if the library is missing this module raises, and every compute
entry point fails when no CUDA device is present.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_int, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_C", "libautogptq_b200.so")

ABI_VERSION = 4
F16, BF16 = 0, 1
CHAIN_MAX_M = 2
CHAIN_X_PLAIN, CHAIN_X_SILU_MUL, CHAIN_X_SUM_PARTS = 0, 1, 2
CHAIN_DEBUG_NO_DEPS, CHAIN_DEBUG_NO_MATH = 1, 2
PEER_HANDLE_BYTES = 64
KERNEL_AUTO, KERNEL_GEMV, KERNEL_GEMM, KERNEL_SKINNY, KERNEL_IMMA = 0, 1, 2, 3, 6
GEMV_MAX_M = 4
SKINNY_MAX_M = 8
IMMA_MAX_M = 8

_lib = None


class B200KernelError(RuntimeError):
    """Raised when a C-ABI call returns a non-zero status (mirrors the reference's TORCH_CHECK -> RuntimeError)."""


def _declare(lib):
    P, I, S = c_void_p, c_int, c_size_t
    fwd = [P, P, P, P, P, P, P, P, I, I, I, I, I, P, S, P]
    sigs = {
        "agb200_abi_version": (I, []),
        "agb200_last_error": (c_char_p, []),
        "agb200_build_info": (c_char_p, []),
        "agb200_device_count": (I, []),
        "agb200_w4a16_forward": (I, fwd),
        "agb200_w4a16_forward_ex": (I, fwd + [I, I, I, I]),
        "agb200_w4a16_workspace_bytes": (S, [I, I, I]),
        "agb200_w4a16_forward_group": (I, [P, I, P, P, P, P, P, P, P, P, I, I, I, I, P, S, P]),
        "agb200_w4_prefetch_hint": (I, [I, P, P]),
        "agb200_w4a16_forward_host": (I, fwd),
        "agb200_w4a16_host_staging_bytes": (S, [I, I, I]),
        "agb200_w4_make_sequential": (I, [P, P, P, I, I, P]),
        "agb200_w4_prepare_tc": (I, [P, P, I, I, P]),
        "agb200_w4_dequantize": (I, [P, P, P, P, P, I, I, I, I, P]),
        "agb200_permute_columns": (I, [P, P, P, I, I, I, P]),
        "agb200_chain_plan_bytes": (S, [P, I, I]),
        "agb200_chain_parts_bytes": (S, [I, I, I]),
        "agb200_chain_create": (I, [P, I, I, I, P, S, P]),
        "agb200_chain_forward": (I, [P, I, P]),
        "agb200_chain_destroy": (I, [P]),
        "agb200_chain_info": (I, [P, P, P, P]),
        "agb200_chain_profile": (I, [P, P, I]),
        "agb200_peer_alloc": (I, [S, P]),
        "agb200_chain_diag": (I, [P]),
        "agb200_peer_free": (I, [P]),
        "agb200_peer_export": (I, [P, P]),
        "agb200_peer_open": (I, [P, P]),
        "agb200_peer_close": (I, [P]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return sigs


def load():
    """Load (once) and return the ctypes library; raises ImportError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. Build it with `python -m autogptq_b200.build` (needs nvcc). "
                "autogptq_b200 has no CPU / PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        _declare(lib)
        if lib.agb200_abi_version() != ABI_VERSION:
            raise ImportError(f"ABI version mismatch: library reports {lib.agb200_abi_version()}, binding expects {ABI_VERSION}")
        _lib = lib
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().agb200_last_error().decode(errors="replace")
        raise B200KernelError(f"{what or 'autogptq_b200'} failed (code {rc}): {msg}")


def declared_symbols():
    """Names bound above (used by the tests to cross-check against the header)."""
    class _Dummy:
        def __getattr__(self, k):
            class F:  # noqa: D401
                restype = None
                argtypes = None
            return F()
    return sorted(_declare(_Dummy()).keys())
