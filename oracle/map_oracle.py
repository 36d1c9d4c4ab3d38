"""ctypes wrapper of the MAP-only screening oracle (map_oracle.c, compiled together with mdg_oracle.c).

TEST INFRASTRUCTURE ONLY, like oracle.py: imported by tests/, never by the product package `metadamage_b200`.
The library is built on first use with the flags of oracle/Makefile, next to its source, or in the temporary
directory when the tree is read-only.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from metadamage_b200._abi import MAP_RESULT_DTYPE, ptr

from .oracle import default_config  # noqa: F401  (the same mdg_fit_config defaults)

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = [os.path.join(_HERE, "map_oracle.c"), os.path.join(_HERE, "mdg_oracle.c"), os.path.join(_HERE, "..", "include", "mdg.h")]
_CFLAGS = ["-O2", "-fPIC", "-fopenmp", "-Wall", "-Wno-unused-function", "-Wno-misleading-indentation",
           "-Wno-maybe-uninitialized", "-ffp-contract=off", "-shared"]
_NAME = "libmdg_map_oracle.so"
_lib = None


def _fresh(path):
    return os.path.exists(path) and os.path.getmtime(path) >= max(os.path.getmtime(s) for s in _SOURCES)


def build(force=False):
    """Compile map_oracle.c with gcc (next to it, or in the temporary directory if oracle/ is read-only)."""
    for d in (_HERE, tempfile.gettempdir()):
        path = os.path.join(d, _NAME)
        if not force and _fresh(path):
            return path
        if os.access(d, os.W_OK):
            subprocess.run(["gcc", *_CFLAGS, "-o", path, os.path.join(_HERE, "map_oracle.c"), "-lm"], check=True)
            return path
    raise RuntimeError("no writable directory for the MAP oracle library")


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def map_batch(tax_id, k, N, cfg=None, mism12=None, noise3=None, n_threads=0):
    """Restatement of mdg_map_batch; returns a MAP_RESULT_DTYPE array."""
    cfg = cfg or default_config()
    tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
    k = np.ascontiguousarray(k, dtype=np.uint32)
    N = np.ascontiguousarray(N, dtype=np.uint32)
    n_tax, R = k.shape
    res = np.zeros(n_tax, dtype=MAP_RESULT_DTYPE)
    if mism12 is not None:
        mism12 = np.ascontiguousarray(mism12, dtype=np.uint32)
    if noise3 is not None:
        noise3 = np.ascontiguousarray(noise3, dtype=np.float64)
    rc = lib().orc_map_batch(C.c_int64(n_tax), C.c_int(R // 2), ptr(tax_id), ptr(k), ptr(N), ptr(mism12), ptr(noise3),
                             C.byref(cfg), ptr(res), C.c_int(n_threads))
    if rc != 0:
        raise RuntimeError(f"orc_map_batch failed with {rc}")
    return res


def lr_tail(lam):
    """(P, z) of the likelihood-ratio statistic as mdg_map_result computes them."""
    lam = np.ascontiguousarray(np.atleast_1d(lam), dtype=np.float64)
    P, z = np.zeros_like(lam), np.zeros_like(lam)
    lib().orc_test_lr_tail(C.c_int64(len(lam)), ptr(lam), ptr(P), ptr(z))
    return P, z
