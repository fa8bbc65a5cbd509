"""ctypes binding of the C ABI declared in include/vlg.h.

The product path fails loudly when the CUDA library is missing: there is no CPU and no
PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
from ctypes import c_char_p, c_double, c_int, c_int64, c_size_t, c_uint64, c_void_p
from pathlib import Path

import os

LIB_PATH = Path(os.environ.get("VLG_B200_LIB", Path(__file__).resolve().parent / "libvlg_b200.so"))

_lib = None

# name -> (restype, argtypes); mirrors include/vlg.h one to one
SIGNATURES = {
    "vlg_error_string": (c_char_p, [c_int]),
    "vlg_last_cuda_error": (c_char_p, []),
    "vlg_abi_version": (c_int, []),
    "vlg_packed_decoders_bytes": (c_size_t, [c_int, c_int, c_int]),
    "vlg_pack_decoders": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p, c_void_p]),
    "vlg_workspace_bytes": (c_size_t, [c_int] * 6),
    "vlg_workspace_status": (c_int, [c_void_p, c_void_p, c_void_p]),
    "vlg_workspace_counters": (c_int, [c_void_p, c_void_p, c_void_p]),
    "vlg_optimize_steps": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,  # packed K X ..step0
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,         # a b omega m v
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_uint64, c_int64,  # basis t draws dec_base seed id0
                                   c_double, c_double, c_double, c_double, c_double,          # lr b1 b2 eps pen
                                   c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "vlg_curve_energy": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_uint64, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                 c_size_t, c_void_p]),
    "vlg_curve_energy_grad": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_uint64, c_int64, c_int,                      # seed id0 step
                                      c_void_p, c_void_p, c_void_p, c_void_p,         # energy grad_omega grad_a grad_b
                                      c_int, c_void_p, c_size_t, c_void_p]),
    "vlg_ensemble_std_norm": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vlg_spline_points": (c_int, [c_int, c_int, c_int] + [c_void_p] * 7),
    "vlg_spline_points_backward": (c_int, [c_int, c_int, c_int] + [c_void_p] * 7),
    "vlg_fit_splines": (c_int, [c_int, c_int, c_int] + [c_void_p] * 6),
}


# test hooks declared in include/vlg_selftest.h; they live in libvlg_b200_selftest.so (tests only)
SELFTEST_LIB_PATH = Path(__file__).resolve().parent / "libvlg_b200_selftest.so"
SELFTEST_SIGNATURES = {
    "vlg_selftest_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "vlg_selftest_umma_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
}


class VlgError(RuntimeError):
    pass


def load():
    """Load libvlg_b200.so (built in-tree by vlg_b200.build.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VlgError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "vlg_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.vlg_abi_version() != 2:
        raise VlgError("libvlg_b200.so ABI version mismatch")
    _lib = lib
    return lib


_selftest = None


def load_selftest():
    """Load the test-only library (built by vlg_b200.build.build_selftest)."""
    global _selftest
    if _selftest is None:
        if not SELFTEST_LIB_PATH.exists():
            raise VlgError(f"{SELFTEST_LIB_PATH} is missing: vlg_b200.build.build_selftest()")
        lib = ctypes.CDLL(str(SELFTEST_LIB_PATH))
        for name, (res, args) in SELFTEST_SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _selftest = lib
    return _selftest


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    lib = load()
    msg = lib.vlg_error_string(rc).decode()
    if rc == -3:
        msg += ": " + lib.vlg_last_cuda_error().decode()
    raise VlgError(f"{what} failed ({rc}): {msg}")
