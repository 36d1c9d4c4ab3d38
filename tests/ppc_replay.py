"""ctypes wrapper of the posterior-predictive replay (tests/ppc_replay.c, compiled as one unit with
oracle/mdg_oracle.c), and a numpy restatement of the order statistics K6 takes of the draws. Test infrastructure only.
The library is built on first use with the flags of the MAP oracle, next to its source, or in the temporary directory
when the tree is read-only."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from metadamage_b200._abi import FIT_FAILED, ptr
from oracle import map_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ppc_replay.c")
_SOURCES = [_SRC, *map_oracle._SOURCES[1:]]  # mdg_oracle.c and mdg.h
_NAME = "libmdg_ppc_replay.so"
_lib = None


def build(force=False):
    for d in (_HERE, tempfile.gettempdir()):
        path = os.path.join(d, _NAME)
        if not force and os.path.exists(path) and os.path.getmtime(path) >= max(os.path.getmtime(s) for s in _SOURCES):
            return path
        if os.access(d, os.W_OK):
            subprocess.run(["gcc", *map_oracle._CFLAGS, "-o", path, _SRC, "-lm"], check=True)
            return path
    raise RuntimeError("no writable directory for the predictive replay library")


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_ppc_replay.argtypes = [C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.POINTER(C.c_int64), C.c_int]
    return _lib


def items_per_tax(P, cfg):
    return 2 * P + (2 if cfg.do_fwd_rev else 0)


def draws(tax_id, N, samples, status, cfg, n_threads=0):
    """The kernel's integer draws y [n_tax][items_per_tax][S] (uint32) from the constrained draws `samples`
    [n_tax][6][S][4] that fit_batch(want_samples=True) returned. Items of failed TaxIDs and of N = 0 are 0."""
    tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
    N = np.ascontiguousarray(N, dtype=np.uint32)
    status = np.ascontiguousarray(status, dtype=np.uint32)
    samples = np.ascontiguousarray(samples, dtype=np.float64)
    n_tax, R = N.shape
    S = cfg.num_samples
    assert samples.shape == (n_tax, 6, S, 4) and len(tax_id) == n_tax == len(status)
    y = np.zeros((n_tax, items_per_tax(R // 2, cfg), S), np.uint32)
    bad = C.c_int64(-1)
    if lib().orc_ppc_replay(n_tax, R // 2, ptr(tax_id), ptr(N), C.byref(cfg), ptr(status), ptr(samples), ptr(y),
                            C.byref(bad), n_threads) != 0:
        t, rest = divmod(bad.value, y.shape[1] * S)
        raise ValueError(f"TaxID {tax_id[t]} (row {t}), item {rest // S}, draw {rest % S}: q outside (0, 1) or a "
                         "non-finite Beta parameter in a fit not marked failed")
    return y


def median_hpdi(frac, prob):
    """np.median and numpyro 0.4.1's diagnostics.hpdi(frac, prob) over the last axis, with K6's clamp of the window
    length L = int(prob * S) to S - 1 (hpdi itself has no window at prob = 1)."""
    S = frac.shape[-1]
    s = np.sort(frac, axis=-1)
    L = min(int(prob * S), S - 1)
    i = np.argmin(s[..., L:] - s[..., :S - L], axis=-1)[..., None]
    return (np.median(frac, axis=-1), np.take_along_axis(s, i, -1)[..., 0], np.take_along_axis(s, i + L, -1)[..., 0])


def predictive(tax_id, N, samples, status, cfg, n_threads=0):
    """What K6 and the assembly make of the replayed draws: `median`, `hpdi_lo`, `hpdi_hi` [n_tax][2P] float32 and
    the FP64 D_max columns of mdg_fit_result; NaN where N = 0 and for failed TaxIDs, and D_max_forward /
    D_max_reverse NaN without do_fwd_rev. Also returns the draws under "y"."""
    N = np.ascontiguousarray(N, dtype=np.uint32)
    status = np.asarray(status)
    n_tax, R = N.shape
    P = R // 2
    y = draws(tax_id, N, samples, status, cfg, n_threads)
    dense = np.r_[np.arange(R), [0, 0 if cfg.reference_quirks else P]][:y.shape[1]]
    Nj = N[:, dense].astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        frac = y / Nj[..., None]
    frac[Nj == 0] = np.nan
    frac[(status & FIT_FAILED) != 0] = np.nan
    med, lo, hi = median_hpdi(frac, cfg.hpdi_prob)
    nan = np.full(n_tax, np.nan)
    out = dict(y=y, median=med[:, :R].astype(np.float32), hpdi_lo=lo[:, :R].astype(np.float32),
               hpdi_hi=hi[:, :R].astype(np.float32), D_max=med[:, 0], D_max_lower_hpdi=lo[:, 0],
               D_max_upper_hpdi=hi[:, 0], D_max_forward=med[:, R] if cfg.do_fwd_rev else nan,
               D_max_reverse=med[:, R + 1] if cfg.do_fwd_rev else nan)
    return out


PREDICTIVE_COLUMNS = ("D_max", "D_max_lower_hpdi", "D_max_upper_hpdi", "D_max_forward", "D_max_reverse")


def same_bits(a, b):
    """Bit-identical floats, except that any NaN matches any NaN (the NaN payloads are not part of the output)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    u = np.uint32 if a.dtype == np.float32 else np.uint64
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(u), b[~nb].view(u))


def mismatches(got, want):
    """Names of the outputs where fit_batch's `got` (result rows + median/hpdi arrays) and the replay `want`
    differ."""
    bad = [key for key in ("median", "hpdi_lo", "hpdi_hi") if not same_bits(got[key], want[key])]
    return bad + [key for key in PREDICTIVE_COLUMNS if not same_bits(np.ascontiguousarray(got["result"][key]), want[key])]
