"""ctypes wrapper of the profile-interval oracle (tests/map_profile_oracle.c, compiled as one unit with
oracle/map_oracle.c and oracle/mdg_oracle.c). Test infrastructure only. The library is built on first use with the
flags of the MAP oracle, next to its source, or in the temporary directory when the tree is read-only."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from metadamage_b200._abi import MAP_INTERVAL_DTYPE, MAP_RESULT_DTYPE, ptr
from oracle import map_oracle
from oracle.oracle import default_config

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "map_profile_oracle.c")
_SOURCES = [_SRC, *map_oracle._SOURCES]
_NAME = "libmdg_map_profile_oracle.so"
_lib = None


def build(force=False):
    for d in (_HERE, tempfile.gettempdir()):
        path = os.path.join(d, _NAME)
        if not force and os.path.exists(path) and os.path.getmtime(path) >= max(os.path.getmtime(s) for s in _SOURCES):
            return path
        if os.access(d, os.W_OK):
            subprocess.run(["gcc", *map_oracle._CFLAGS, "-o", path, _SRC, "-lm"], check=True)
            return path
    raise RuntimeError("no writable directory for the profile oracle library")


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_map_profile.argtypes = [C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                         C.c_void_p, C.c_int]
    return _lib


def map_profile(k, N, map_rows, cfg=None, level=0.68, n_threads=0):
    """Restatement of mdg_map_profile; returns a MAP_INTERVAL_DTYPE array."""
    cfg = cfg or default_config()
    k = np.ascontiguousarray(k, dtype=np.uint32)
    N = np.ascontiguousarray(N, dtype=np.uint32)
    map_rows = np.ascontiguousarray(map_rows, dtype=MAP_RESULT_DTYPE)
    n_tax, R = k.shape
    out = np.zeros(n_tax, MAP_INTERVAL_DTYPE)
    rc = lib().orc_map_profile(n_tax, R // 2, ptr(k), ptr(N), C.addressof(cfg), ptr(map_rows), float(level), ptr(out),
                               n_threads)
    if rc != 0:
        raise ValueError(f"orc_map_profile failed with {rc}")
    return out

