"""Host-side driver of the B200 hot path: one `Context` per GPU wrapping the C-ABI calls
`mdg_counts_reduce` (K1) and `mdg_fit_batch` (K3-K7) for numpy (host) or torch-CUDA (device)
buffers. PyTorch is used for device memory and streams only."""
import ctypes as C

import numpy as np

from . import _lib
from ._abi import FIT_RESULT_DTYPE, MAP_RESULT_DTYPE, MDG_DEVICE, MDG_HOST, NUM_RUNS, Timings, ptr

BASES = "ACGT"
OFFDIAG_COLUMNS = [r + o for r in BASES for o in BASES if r != o]  # AC,AG,AT,CA,CG,CT,GA,GC,GT,TA,TC,TG


def _base_index(sub):
    if len(sub) != 2 or sub[0] not in BASES or sub[1] not in BASES:
        raise ValueError(f"substitution bases must be two of ACGT, got {sub!r}")
    return BASES.index(sub[0]), BASES.index(sub[1])


def _dptr(t, rows_ok=False):
    """device pointer of a contiguous torch CUDA tensor (None -> NULL); `rows_ok`: a 2-D tensor whose rows are
    contiguous (a column range of a wider buffer; the row stride is passed separately) is accepted too"""
    if t is None:
        return None
    if not t.is_cuda or not (t.is_contiguous() or (rows_ok and t.dim() == 2 and t.stride(1) == 1)):
        raise ValueError("device buffers must be contiguous CUDA tensors")
    return C.c_void_p(t.data_ptr())


def _text_arg(text):
    """bytes-like or a contiguous uint8 ndarray (e.g. counts.read_file_bytes' pinned buffer) -> (ctypes argument, length,
    keep-alive object)"""
    if isinstance(text, np.ndarray):
        if text.dtype != np.uint8 or not text.flags["C_CONTIGUOUS"]:
            raise TypeError("text array must be contiguous uint8")
        return C.cast(text.ctypes.data, C.c_char_p), int(text.size), text
    if not isinstance(text, (bytes, bytearray, memoryview)):
        raise TypeError("text must be bytes or a uint8 array")
    b = bytes(text)
    return b, len(b), b


class Context:
    """One GPU, one stream. Not thread-safe; use one Context per host thread / process."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        handle = C.c_void_p()
        _lib.check(self._lib.mdg_ctx_create(int(device), C.byref(handle)))
        self._h = handle
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.mdg_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_handle):
        _lib.check(self._lib.mdg_ctx_set_stream(self._h, C.c_void_p(cuda_stream_handle or 0)))

    def synchronize(self):
        _lib.check(self._lib.mdg_ctx_synchronize(self._h))

    @staticmethod
    def _timings_dict(t):
        return {
            "counts_ms": t.counts_ms, "map_ms": t.map_ms, "nuts_ms": t.nuts_ms, "ppc_ms": t.ppc_ms,
            "assemble_ms": t.assemble_ms, "total_ms": t.total_ms, "n_launches": int(t.n_launches),
            "leapfrogs": [int(v) for v in t.leapfrogs], "nuts_union_ms": t.nuts_union_ms,
            "nuts_begin_ms": t.nuts_begin_ms, "nuts_end_ms": t.nuts_end_ms,
        }

    def timings(self):
        t = Timings()
        _lib.check(self._lib.mdg_ctx_get_timings(self._h, C.byref(t)))
        return self._timings_dict(t)

    def fp64_peak_tflops(self):
        out = C.c_double(0)
        _lib.check(self._lib.mdg_measure_fp64_peak(self._h, C.byref(out)))
        return out.value

    # ------------------------------------------------------------------ K0
    def tsv_parse(self, text, want_spans=False):
        """Tokenise a mismatch-matrix file (bytes) on the GPU -> SoA numpy columns (counts.py:229-235)."""
        arg, n_bytes, _keep = _text_arg(text)
        cap = (int(np.count_nonzero(text == 10)) if isinstance(text, np.ndarray) else _keep.count(b"\n")) + 1
        out = dict(tax_id=np.empty(cap, np.int64), n_alignments=np.empty(cap, np.uint32), is_reverse=np.empty(cap, np.uint8),
                   pos0=np.empty(cap, np.uint8), counts16=np.empty((16, cap), np.uint32),
                   name_span=np.empty((cap, 2), np.int64) if want_spans else None,
                   rank_span=np.empty((cap, 2), np.int64) if want_spans else None)
        n_rows, n_cols = C.c_int64(0), C.c_int32(0)
        _lib.check(self._lib.mdg_tsv_parse(self._h, MDG_HOST, arg, n_bytes, cap, ptr(out["tax_id"]), ptr(out["n_alignments"]),
                                           ptr(out["is_reverse"]), ptr(out["pos0"]), ptr(out["counts16"]), cap,
                                           ptr(out["name_span"]), ptr(out["rank_span"]), C.byref(n_rows), C.byref(n_cols)))
        n = n_rows.value
        res = {k: (v[:n] if v is not None and k != "counts16" else v) for k, v in out.items()}
        res["counts16"] = np.ascontiguousarray(out["counts16"][:, :n])
        res["n_rows"], res["n_cols"] = n, n_cols.value
        return res

    def tsv_parse_device(self, text, want_spans=False):
        """K0 with the parsed columns left on the GPU (torch CUDA tensors), ready for `counts_reduce_device`:
        nothing but the text crosses PCIe. Returns (cols, n_rows, n_cols); `cols` also carries `name_span` /
        `rank_span` ([rows][2] int64, 22-column layout) when asked for."""
        import torch

        arg, n_bytes, _keep = _text_arg(text)
        # room for the rows without counting the newlines on the host (70 ms per 100 MB): a data line is at least
        # 39 bytes long (20 fields, 19 tabs, newline, an empty strand field at worst; 22-column lines are longer still)
        cap = n_bytes // 38 + 2
        dev = torch.device("cuda", self.device)
        cols = dict(tax_id=torch.empty(cap, dtype=torch.int64, device=dev), n_alignments=torch.empty(cap, dtype=torch.int32, device=dev),
                    is_reverse=torch.empty(cap, dtype=torch.uint8, device=dev), pos0=torch.empty(cap, dtype=torch.uint8, device=dev),
                    counts16=torch.empty((16, cap), dtype=torch.int32, device=dev))
        if want_spans:
            cols["name_span"] = torch.empty((cap, 2), dtype=torch.int64, device=dev)
            cols["rank_span"] = torch.empty((cap, 2), dtype=torch.int64, device=dev)
        n_rows, n_cols = C.c_int64(0), C.c_int32(0)
        _lib.check(self._lib.mdg_tsv_parse(self._h, MDG_DEVICE, arg, n_bytes, cap, _dptr(cols["tax_id"]), _dptr(cols["n_alignments"]),
                                           _dptr(cols["is_reverse"]), _dptr(cols["pos0"]), _dptr(cols["counts16"]), cap,
                                           _dptr(cols.get("name_span")), _dptr(cols.get("rank_span")), C.byref(n_rows), C.byref(n_cols)))
        n = n_rows.value
        out = {key: (val[:n] if key != "counts16" else val[:, :n]) for key, val in cols.items()}
        return out, n, n_cols.value

    # ------------------------------------------------------------------ K1
    def counts_reduce(self, tax_id, n_alignments, is_reverse, pos0, counts16, fwd="CT", rev="GA",
                      max_position=15, min_alignments=10, min_y_sum=10, want_noise=False, want_rows=True, out=None):
        """counts.py:237-256 on host SoA columns (numpy). Returns a dict of numpy arrays.
        `out` (optional): a dict from an earlier call with the same shapes (or caller-allocated, e.g.
        pinned, arrays under the same keys); its buffers are reused instead of allocating new ones."""
        n = len(tax_id)
        P = int(max_position)
        tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
        n_alignments = np.ascontiguousarray(n_alignments, dtype=np.uint32)
        is_reverse = np.ascontiguousarray(is_reverse, dtype=np.uint8)
        pos0 = np.ascontiguousarray(pos0, dtype=np.uint8)
        counts16 = np.ascontiguousarray(counts16, dtype=np.uint32)
        if counts16.shape != (16, n):
            raise ValueError("counts16 must be [16][n_rows] (ref-major ACGT x ACGT)")
        fr, fo = _base_index(fwd)
        rr, ro = _base_index(rev)
        # room for every run of equal tax_id (an upper bound of the kept TaxIDs)
        m_cap = int(np.count_nonzero(tax_id[1:] != tax_id[:-1])) + 1 if n else 0
        reuse = out if out is not None else {}

        def buf(key, shape, dtype):
            a = reuse.get("_buf_" + key, reuse.get(key))
            shape = shape if isinstance(shape, tuple) else (shape,)
            if a is not None and a.dtype == np.dtype(dtype) and a.shape[1:] == shape[1:] and a.shape[0] >= shape[0] and a.flags["C_CONTIGUOUS"]:
                return a
            return np.empty(shape, dtype)

        out = {}
        if want_rows:
            out.update(
                n_fwd_ref=buf("n_fwd_ref", n, np.uint32), n_rev_ref=buf("n_rev_ref", n, np.uint32),
                f_fwd=buf("f_fwd", n, np.float32), f_rev=buf("f_rev", n, np.float32),
                z=buf("z", n, np.int8), y_sum_total=buf("y_sum_total", n, np.uint64), keep=buf("keep", n, np.uint8),
            )
        out.update(
            tax_id=buf("tax_id", m_cap, np.int64), n_alignments=buf("n_alignments", m_cap, np.uint32), first_row=buf("first_row", m_cap, np.int64),
            k=buf("k", (m_cap, 2 * P), np.uint32), N=buf("N", (m_cap, 2 * P), np.uint32),
            noise=buf("noise", (m_cap, 3), np.float64) if want_noise else None,
        )
        full = {"_buf_" + key: val for key, val in out.items() if val is not None}  # full-capacity buffers, for the next call
        n_tax = C.c_int64(0)
        g = out.get
        _lib.check(self._lib.mdg_counts_reduce(
            self._h, MDG_HOST, n, ptr(tax_id), ptr(n_alignments), ptr(is_reverse), ptr(pos0), ptr(counts16), n,
            fr, fo, rr, ro, P, int(min_alignments), int(min_y_sum),
            ptr(g("n_fwd_ref")), ptr(g("n_rev_ref")), ptr(g("f_fwd")), ptr(g("f_rev")), ptr(g("z")),
            ptr(g("y_sum_total")), ptr(g("keep")), ptr(out["tax_id"]), ptr(out["n_alignments"]),
            ptr(out["first_row"]), ptr(out["k"]), ptr(out["N"]), ptr(out["noise"]), m_cap, C.byref(n_tax)))
        m = n_tax.value
        for key in ("tax_id", "n_alignments", "first_row", "k", "N", "noise"):
            if out[key] is not None:
                out[key] = out[key][:m]
        if want_rows:
            for key in ("n_fwd_ref", "n_rev_ref", "f_fwd", "f_rev", "z", "y_sum_total", "keep"):
                out[key] = out[key][:n]
        out["n_tax"] = m
        if reuse:
            out.update(full)
        return out

    def counts_reduce_device(self, cols, outs, fwd="CT", rev="GA", max_position=15, min_alignments=10,
                             min_y_sum=10):
        """K1 on torch CUDA tensors. cols: tax_id(i64) n_alignments(i32 bits of u32) is_reverse(u8)
        pos0(u8) counts16([16][n] i32). outs: dict of preallocated CUDA tensors (missing -> skipped).
        Returns the number of kept TaxIDs (forces a stream sync)."""
        n = cols["tax_id"].numel()
        fr, fo = _base_index(fwd)
        rr, ro = _base_index(rev)
        n_tax = C.c_int64(0)
        g = lambda k: _dptr(outs.get(k))  # noqa: E731
        _lib.check(self._lib.mdg_counts_reduce(
            self._h, MDG_DEVICE, n, _dptr(cols["tax_id"]), _dptr(cols["n_alignments"]), _dptr(cols["is_reverse"]),
            _dptr(cols["pos0"]), _dptr(cols["counts16"], rows_ok=True), cols["counts16"].stride(0),
            fr, fo, rr, ro, int(max_position), int(min_alignments), int(min_y_sum),
            g("n_fwd_ref"), g("n_rev_ref"), g("f_fwd"), g("f_rev"), g("z"), g("y_sum_total"), g("keep"),
            g("tax_id"), g("n_alignments"), g("first_row"), g("k"), g("N"), g("noise"), int(outs["k"].shape[0]), C.byref(n_tax)))
        return n_tax.value

    # ------------------------------------------------------------------ K1d (C8)
    def counts_order(self, tax_id_row, z_row, keep_row, first_row, tax_order):
        """Row permutation of counts.py:167-172 on host arrays: source row of every output row (kept rows only)."""
        tax_id_row = np.ascontiguousarray(tax_id_row, dtype=np.int64)
        z_row = np.ascontiguousarray(z_row, dtype=np.int8)
        keep_row = None if keep_row is None else np.ascontiguousarray(keep_row, dtype=np.uint8)
        first_row = np.ascontiguousarray(first_row, dtype=np.int64)
        tax_order = np.ascontiguousarray(tax_order, dtype=np.int64)
        cap = len(tax_id_row) if keep_row is None else int(np.count_nonzero(keep_row))
        perm = np.empty(cap, np.int64)
        n_out = C.c_int64(0)
        _lib.check(self._lib.mdg_counts_order(self._h, MDG_HOST, len(tax_id_row), ptr(tax_id_row), ptr(z_row), ptr(keep_row), len(first_row),
                                              ptr(first_row), ptr(tax_order), ptr(perm), cap, C.byref(n_out)))
        return perm[: n_out.value]

    def counts_order_device(self, cols, outs, n_tax, tax_order, out_perm):
        """K1d on torch CUDA tensors (`cols` / `outs` of counts_reduce_device; tax_order, out_perm: int64 CUDA tensors).
        Returns the number of kept rows written to out_perm."""
        n_out = C.c_int64(0)
        _lib.check(self._lib.mdg_counts_order(self._h, MDG_DEVICE, cols["tax_id"].numel(), _dptr(cols["tax_id"]), _dptr(outs["z"]),
                                              _dptr(outs.get("keep")), int(n_tax), _dptr(outs["first_row"]), _dptr(tax_order),
                                              _dptr(out_perm), out_perm.numel(), C.byref(n_out)))
        return n_out.value

    # ------------------------------------------------------------------ K8 (N3)
    def select_top(self, tax_id_row, n_alignments_row, keep_row, tax_id, first_row, n_top, want_weight=False):
        """fits.extract_top_max_fits (fits.py:736-744) on the arrays counts_reduce returns: positions (in the
        per-TaxID arrays, ascending = df_counts order) of the n_top TaxIDs with the largest sum of
        N_alignments over their kept rows; ties at the cut go to the smaller tax id."""
        tax_id_row = np.ascontiguousarray(tax_id_row, dtype=np.int64)
        n_alignments_row = np.ascontiguousarray(n_alignments_row, dtype=np.uint32)
        keep_row = None if keep_row is None else np.ascontiguousarray(keep_row, dtype=np.uint8)
        tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
        first_row = np.ascontiguousarray(first_row, dtype=np.int64)
        n_tax = len(tax_id)
        index = np.empty(max(0, min(int(n_top), n_tax)), np.int64)
        weight = np.empty(n_tax, np.uint64) if want_weight else None
        n_out = C.c_int64(0)
        _lib.check(self._lib.mdg_select_top(self._h, MDG_HOST, len(tax_id_row), ptr(tax_id_row), ptr(n_alignments_row), ptr(keep_row),
                                            n_tax, ptr(tax_id), ptr(first_row), int(n_top), ptr(weight), ptr(index), C.byref(n_out)))
        index = index[:n_out.value]
        return (index, weight) if want_weight else index

    def select_top_device(self, cols, outs, n_tax, n_top, out_index, out_weight=None):
        """K8 on torch CUDA tensors: `cols` / `outs` as given to / filled by counts_reduce_device;
        out_index: int64 CUDA tensor with room for min(n_top, n_tax) entries. Returns how many were selected."""
        n_out = C.c_int64(0)
        _lib.check(self._lib.mdg_select_top(self._h, MDG_DEVICE, cols["tax_id"].numel(), _dptr(cols["tax_id"]), _dptr(cols["n_alignments"]),
                                            _dptr(outs.get("keep")), int(n_tax), _dptr(outs["tax_id"]), _dptr(outs["first_row"]), int(n_top),
                                            _dptr(out_weight), _dptr(out_index), C.byref(n_out)))
        return n_out.value

    # ------------------------------------------------------------------ K3-K7
    def fit_batch(self, tax_id, k, N, cfg=None, mism12=None, noise3=None, want_samples=False,
                  want_trace=False, want_waic=False):
        """fits.py:428-469 for a dense batch of TaxIDs on host numpy arrays."""
        cfg = cfg or _lib.default_config()
        tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
        k = np.ascontiguousarray(k, dtype=np.uint32)
        N = np.ascontiguousarray(N, dtype=np.uint32)
        if k.ndim != 2 or k.shape != N.shape or k.shape[0] != len(tax_id) or k.shape[1] % 2:
            raise ValueError("k and N must be [n_tax][2*max_position]")
        n_tax, R = k.shape
        S, W = cfg.num_samples, cfg.num_warmup
        res = np.zeros(n_tax, dtype=FIT_RESULT_DTYPE)
        med = np.empty((n_tax, R), np.float32)
        lo = np.empty((n_tax, R), np.float32)
        hi = np.empty((n_tax, R), np.float32)
        samples = np.empty((n_tax, NUM_RUNS, S, 4)) if want_samples else None
        trace = np.empty((n_tax, NUM_RUNS, W + S, 4)) if want_trace else None
        waic = np.empty((n_tax, NUM_RUNS, 2, R)) if want_waic else None
        if mism12 is not None:
            mism12 = np.ascontiguousarray(mism12, dtype=np.uint32)
            if mism12.shape != (n_tax, R, 12):
                raise ValueError("mism12 must be [n_tax][2*max_position][12]")
        if noise3 is not None:
            noise3 = np.ascontiguousarray(noise3, dtype=np.float64)
        _lib.check(self._lib.mdg_fit_batch(
            self._h, MDG_HOST, n_tax, R // 2, ptr(tax_id), ptr(k), ptr(N), ptr(mism12), ptr(noise3), C.byref(cfg),
            ptr(res), ptr(med), ptr(lo), ptr(hi), ptr(samples), ptr(trace), ptr(waic)))
        return dict(result=res, median=med, hpdi_lo=lo, hpdi_hi=hi, samples=samples, trace=trace, waic=waic)

    def fit_batch_device(self, tax_id, k, N, out, cfg=None, median=None, hpdi_lo=None, hpdi_hi=None,
                         mism12=None, noise3=None):
        """K3-K7 on torch CUDA tensors; `out` is a uint8 CUDA tensor of n_tax*sizeof(mdg_fit_result)."""
        self.fit_wait(self.fit_submit_device(tax_id, k, N, out, cfg, median, hpdi_lo, hpdi_hi, mism12, noise3))

    # ------------------------------------------------------------------ asynchronous fits (mdg_fit_batch_submit / _wait)
    def fit_submit_device(self, tax_id, k, N, out, cfg=None, median=None, hpdi_lo=None, hpdi_hi=None,
                          mism12=None, noise3=None):
        """Enqueue K3-K7 on torch CUDA tensors and return a ticket; nothing waits for the GPU. The tensors must
        stay alive and untouched until `fit_wait(ticket)`. At most two batches per Context are in flight."""
        cfg = cfg or _lib.default_config()
        n_tax, R = k.shape
        if out.numel() * out.element_size() < n_tax * FIT_RESULT_DTYPE.itemsize:
            raise ValueError("out buffer too small")
        ticket = C.c_int64(0)
        _lib.check(self._lib.mdg_fit_batch_submit(
            self._h, MDG_DEVICE, n_tax, R // 2, _dptr(tax_id), _dptr(k), _dptr(N), _dptr(mism12), _dptr(noise3),
            C.byref(cfg), _dptr(out), _dptr(median), _dptr(hpdi_lo), _dptr(hpdi_hi), None, None, None, C.byref(ticket)))
        keep = (tax_id, k, N, out, median, hpdi_lo, hpdi_hi, mism12, noise3)
        return {"id": ticket.value, "keep": keep}

    def fit_submit(self, tax_id, k, N, cfg=None, noise3=None, out=None):
        """Enqueue K3-K7 on host numpy arrays (pinned ones make the copies asynchronous) and return a ticket.
        `out` (optional): dict with preallocated `result` / `median` / `hpdi_lo` / `hpdi_hi` arrays (e.g. pinned)."""
        cfg = cfg or _lib.default_config()
        tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
        k = np.ascontiguousarray(k, dtype=np.uint32)
        N = np.ascontiguousarray(N, dtype=np.uint32)
        if k.ndim != 2 or k.shape != N.shape or k.shape[0] != len(tax_id) or k.shape[1] % 2:
            raise ValueError("k and N must be [n_tax][2*max_position]")
        n_tax, R = k.shape
        out = out or {}

        def buf(key, shape, dtype):
            a = out.get(key)
            if a is not None and a.dtype == dtype and a.flags["C_CONTIGUOUS"] and a.shape[0] >= shape[0] and a.shape[1:] == shape[1:]:
                return a[: shape[0]]
            return np.zeros(shape, dtype) if key == "result" else np.empty(shape, dtype)

        res = buf("result", (n_tax,), FIT_RESULT_DTYPE)
        med, lo, hi = (buf(key, (n_tax, R), np.float32) for key in ("median", "hpdi_lo", "hpdi_hi"))
        if noise3 is not None:
            noise3 = np.ascontiguousarray(noise3, dtype=np.float64)
        ticket = C.c_int64(0)
        _lib.check(self._lib.mdg_fit_batch_submit(
            self._h, MDG_HOST, n_tax, R // 2, ptr(tax_id), ptr(k), ptr(N), None, ptr(noise3), C.byref(cfg),
            ptr(res), ptr(med), ptr(lo), ptr(hi), None, None, None, C.byref(ticket)))
        return {"id": ticket.value, "keep": (tax_id, k, N, noise3, cfg),
                "result": dict(result=res, median=med, hpdi_lo=lo, hpdi_hi=hi)}

    def fit_wait(self, ticket):
        """Block until the batch of `ticket` is complete; returns its result dict (host submits) with the
        batch's device timings under "timings"."""
        t = Timings()
        _lib.check(self._lib.mdg_fit_batch_wait(self._h, C.c_int64(ticket["id"]), C.byref(t)))
        ticket["keep"] = None
        res = ticket.get("result") or {}
        res["timings"] = self._timings_dict(t)
        return res

    # ------------------------------------------------------------------ K3m MAP-only screening
    def map_batch(self, tax_id, k, N, cfg=None, mism12=None, noise3=None):
        """mdg_map_batch on host numpy arrays: six MAP fits per TaxID with Laplace uncertainties and the
        likelihood-ratio statistic, no NUTS. Returns a MAP_RESULT_DTYPE array."""
        cfg = cfg or _lib.default_config()
        tax_id = np.ascontiguousarray(tax_id, dtype=np.int64)
        k = np.ascontiguousarray(k, dtype=np.uint32)
        N = np.ascontiguousarray(N, dtype=np.uint32)
        if k.ndim != 2 or k.shape != N.shape or k.shape[0] != len(tax_id) or k.shape[1] % 2:
            raise ValueError("k and N must be [n_tax][2*max_position]")
        n_tax, R = k.shape
        if mism12 is not None:
            mism12 = np.ascontiguousarray(mism12, dtype=np.uint32)
            if mism12.shape != (n_tax, R, 12):
                raise ValueError("mism12 must be [n_tax][2*max_position][12]")
        if noise3 is not None:
            noise3 = np.ascontiguousarray(noise3, dtype=np.float64)
        res = np.zeros(n_tax, dtype=MAP_RESULT_DTYPE)
        _lib.check(self._lib.mdg_map_batch(self._h, MDG_HOST, n_tax, R // 2, ptr(tax_id), ptr(k), ptr(N), ptr(mism12),
                                           ptr(noise3), C.byref(cfg), ptr(res)))
        return res

    def map_batch_device(self, tax_id, k, N, out, cfg=None, mism12=None, noise3=None):
        """mdg_map_batch on torch CUDA tensors (k, N: [n_tax][2P] int32 bits of uint32); `out` is a uint8 CUDA tensor
        of at least n_tax * MAP_RESULT_DTYPE.itemsize bytes. Synchronous."""
        cfg = cfg or _lib.default_config()
        n_tax, R = k.shape
        if out.numel() * out.element_size() < n_tax * MAP_RESULT_DTYPE.itemsize:
            raise ValueError("out buffer too small")
        _lib.check(self._lib.mdg_map_batch(self._h, MDG_DEVICE, n_tax, R // 2, _dptr(tax_id), _dptr(k), _dptr(N), _dptr(mism12),
                                           _dptr(noise3), C.byref(cfg), _dptr(out)))

    # ------------------------------------------------------------------ test hooks
    def lgamma_digamma(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        lg = np.empty_like(x)
        dg = np.empty_like(x)
        _lib.check(self._lib.mdg_test_lgamma_digamma(self._h, x.size, ptr(x), ptr(lg), ptr(dg)))
        return lg, dg

    def exp_log(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        ex = np.empty_like(x)
        lg = np.empty_like(x)
        _lib.check(self._lib.mdg_test_exp_log(self._h, x.size, ptr(x), ptr(ex), ptr(lg)))
        return ex, lg

    def philox(self, key2, ctr4):
        key2 = np.ascontiguousarray(key2, dtype=np.uint32).reshape(-1, 2)
        ctr4 = np.ascontiguousarray(ctr4, dtype=np.uint32).reshape(-1, 4)
        out = np.empty_like(ctr4)
        _lib.check(self._lib.mdg_test_philox(self._h, len(ctr4), ptr(key2), ptr(ctr4), ptr(out)))
        return out

    def logp_grad(self, k, N, u, cfg=None, model=0, lane_mask=0, with_jacobian=True):
        cfg = cfg or _lib.default_config()
        k = np.ascontiguousarray(k, dtype=np.uint32).ravel()
        N = np.ascontiguousarray(N, dtype=np.uint32).ravel()
        P = len(k) // 2
        u = np.ascontiguousarray(np.atleast_2d(u), dtype=np.float64)
        if u.shape[1] != 4:
            u = np.ascontiguousarray(np.pad(u, ((0, 0), (0, 4 - u.shape[1]))))
        ne = u.shape[0]
        logp = np.empty(ne)
        grad = np.empty((ne, 4))
        ll = np.empty((ne, 2 * P))
        _lib.check(self._lib.mdg_test_logp_grad(self._h, P, ptr(k), ptr(N), C.byref(cfg), model, lane_mask,
                                                int(with_jacobian), ne, ptr(u), ptr(logp), ptr(grad), ptr(ll)))
        return logp, grad, ll
