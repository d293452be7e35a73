"""Builds the test-only native code of the kernel-level tests into build/probe/ and loads it with ctypes.

* build_probe(name): tests/kernels/<name>.cu, compiled with the library's own nvcc flags (__graft_entry__.NVCC_FLAGS,
  -fmad=false included: the bit-exact comparisons depend on it) into lib<name>.so.
* build_c(name): tests/kernels/<name>.c, compiled with gcc -O2 -std=c11 -ffp-contract=off (no GPU needed).

Both rebuild only when a source is newer than the library.  Also the small helpers the kernel tests share.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = os.path.join(ROOT, "tests", "kernels")
CSRC = os.path.join(ROOT, "pareben_b200", "csrc")
OUT_DIR = os.path.join(ROOT, "build", "probe")


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def build_probe(name):
    import __graft_entry__ as ge
    src = os.path.join(KERNELS, name + ".cu")
    lib = os.path.join(OUT_DIR, f"lib{name}.so")
    sources = ([src, os.path.join(ROOT, "__graft_entry__.py")] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
               + [os.path.join(KERNELS, f) for f in os.listdir(KERNELS) if f.endswith(".cuh")])
    if not _newer(lib, sources):
        os.makedirs(OUT_DIR, exist_ok=True)
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.run([nvcc, *ge.NVCC_FLAGS, "--shared", "-o", lib, src], check=True, cwd=OUT_DIR)
    return ctypes.CDLL(lib)


def build_c(name):
    src = os.path.join(KERNELS, name + ".c")
    lib = os.path.join(OUT_DIR, f"lib{name}.so")
    if not _newer(lib, [src]):
        os.makedirs(OUT_DIR, exist_ok=True)
        subprocess.run(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-o", lib, src, "-lm"],
                       check=True, cwd=OUT_DIR)
    return ctypes.CDLL(lib)


D = ctypes.POINTER(ctypes.c_double)
I = ctypes.POINTER(ctypes.c_int)


def dp(a):
    """float64 array -> double* (None -> NULL).  The array must be C-contiguous float64."""
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data_as(D)


def ip(a):
    if a is None:
        return None
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(I)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def bits_equal(a, b):
    """Bitwise equal (so +0 and -0 differ); any NaN equals any NaN (payloads are not part of the result)."""
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    if a.shape != b.shape:
        return False
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64), b[~nan].view(np.int64))
