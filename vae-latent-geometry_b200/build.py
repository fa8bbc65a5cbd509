"""In-tree build of libvlg_b200.so (nvcc, sm_100a only).  No JIT cache, no other arch."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libvlg_b200.so"
SOURCES = ["vlg_api.cu", "vlg_simt.cu", "vlg_pack.cu", "vlg_tc.cu", "vlg_decode.cu"]
# test-only kernels (tcgen05 building-block selftests, include/vlg_selftest.h): a separate library,
# never loaded by the product path
SELFTEST_LIB_PATH = PKG_DIR / "libvlg_b200_selftest.so"
SELFTEST_SOURCES = ["vlg_umma_test.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: cannot build libvlg_b200.so")


def needs_build(lib: Path = LIB_PATH) -> bool:
    if not lib.exists():
        return True
    newest = max(p.stat().st_mtime for p in list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) +
                 list(CSRC.glob("*.h")) + list((PKG_DIR.parent / "include").glob("*.h")))
    return newest > lib.stat().st_mtime


def _compile(lib: Path, sources, verbose: bool, extra=()) -> Path:
    srcs = [str(CSRC / s) for s in sources]
    cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-o", str(lib), *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return lib


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile the product CUDA sources for sm_100a into libvlg_b200.so."""
    if not force and not needs_build():
        return LIB_PATH
    return _compile(LIB_PATH, SOURCES, verbose)


def build_selftest(force: bool = False, verbose: bool = False) -> Path:
    """The tcgen05 building-block selftests (tests only) as their own library."""
    if not force and not needs_build(SELFTEST_LIB_PATH):
        return SELFTEST_LIB_PATH
    return _compile(SELFTEST_LIB_PATH, SELFTEST_SOURCES, verbose)
