"""-m gpu: every C-ABI entry point gives the same bytes whether its buffers are on the host (MDG_HOST: staged through
the context's arena) or on the device (MDG_DEVICE: used in place), also with each optional output left NULL; and
every entry point leaves the caller's current device as it found it."""
import ctypes as C

import numpy as np
import pytest

from metadamage_b200 import _lib, synthetic as syn
from metadamage_b200._abi import FIT_RESULT_DTYPE, MAP_RESULT_DTYPE, MDG_DEVICE, MDG_HOST, NUM_RUNS, ptr

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

P = 15
R = 2 * P
ROW_OUTS = [("n_fwd_ref", np.uint32), ("n_rev_ref", np.uint32), ("f_fwd", np.float32), ("f_rev", np.float32), ("z", np.int8),
            ("y_sum_total", np.uint64), ("keep", np.uint8)]
TAX_OUTS = [("tax_id", np.int64, ()), ("n_alignments", np.uint32, ()), ("first_row", np.int64, ()), ("k", np.uint32, (R,)),
            ("N", np.uint32, (R,)), ("noise", np.float64, (3,))]


def lib():
    return _lib.load()


def on_device(a):
    """numpy array -> CUDA tensor holding the same bytes"""
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda()


def dptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def to_host(t, like):
    return t.cpu().numpy().view(like.dtype).reshape(like.shape)


def call(mem, fn, *args):
    """args: numpy arrays (inputs or outputs) or scalars; MDG_DEVICE runs on device copies of the arrays. Returns the
    arrays as the call left them (host numpy in both cases)."""
    arrays = [a if isinstance(a, np.ndarray) else None for a in args]
    if mem == MDG_HOST:
        cargs = [ptr(a) if isinstance(a, np.ndarray) else a for a in args]
        _lib.check(fn(*cargs))
        return arrays
    dev = [on_device(a) if a is not None else None for a in arrays]
    cargs = [dptr(d) if isinstance(a, np.ndarray) else a for a, d in zip(args, dev)]
    _lib.check(fn(*cargs))
    torch.cuda.synchronize()
    return [to_host(d, a) if a is not None else None for a, d in zip(arrays, dev)]


def assert_same_bytes(host, device):
    for i, (h, d) in enumerate(zip(host, device)):
        if h is not None:
            assert h.tobytes() == d.tobytes(), f"argument {i}"


@pytest.fixture(scope="module")
def gen():
    return syn.make_mismatch_matrix(700, max_position=P, seed=41)


@pytest.fixture(scope="module")
def reduced(ctx, gen):
    return ctx.counts_reduce(gen["tax_id"], gen["n_alignments"], gen["is_reverse"], gen["pos0"], gen["counts16"], max_position=P,
                             want_noise=True)


@pytest.mark.parametrize("spans", [False, True])
def test_tsv_parse_host_vs_device(ctx, gen, tmp_path, spans):
    text = open(syn.write_tsv(gen, str(tmp_path / "m.txt")), "rb").read()
    cap = text.count(b"\n") + 1
    outs = [np.zeros(cap, np.int64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint8), np.zeros(cap, np.uint8),
            np.zeros((16, cap), np.uint32)]
    span = [np.zeros((cap, 2), np.int64) if spans else None for _ in range(2)]
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        n_rows, n_cols = C.c_int64(0), C.c_int32(0)
        args = [ctx._h, mem, text, len(text), cap, *[o.copy() for o in outs], cap, *[s.copy() if s is not None else None for s in span],
                C.byref(n_rows), C.byref(n_cols)]
        got = call(mem, lib().mdg_tsv_parse, *args)
        res[mem] = (got, n_rows.value, n_cols.value)
    assert res[MDG_HOST][1:] == res[MDG_DEVICE][1:] == (len(gen["tax_id"]), 22)
    assert_same_bytes(res[MDG_HOST][0], res[MDG_DEVICE][0])


@pytest.mark.parametrize("missing", [None] + [name for name, _ in ROW_OUTS] + [name for name, *_ in TAX_OUTS] + ["first_row only"])
def test_counts_reduce_host_vs_device(ctx, gen, missing):
    """`first_row only`: no out_first_row but out_noise, which needs the first rows in scratch."""
    n = len(gen["tax_id"])
    cap = int(np.count_nonzero(gen["tax_id"][1:] != gen["tax_id"][:-1])) + 1
    ins = [np.ascontiguousarray(gen[key], dtype=dt) for key, dt in
           (("tax_id", np.int64), ("n_alignments", np.uint32), ("is_reverse", np.uint8), ("pos0", np.uint8), ("counts16", np.uint32))]
    rows = [np.zeros(n, dt) for _, dt in ROW_OUTS]
    taxs = [np.zeros((cap, *shape), dt) for _, dt, shape in TAX_OUTS]
    names = [name for name, _ in ROW_OUTS] + [name for name, *_ in TAX_OUTS]
    outs = [None if name == missing or (missing == "first_row only" and name == "first_row") else a for name, a in zip(names, rows + taxs)]
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        n_tax = C.c_int64(0)
        args = [ctx._h, mem, n, *[a.copy() for a in ins], n, 1, 3, 2, 0, P, 10, 10,
                *[a.copy() if a is not None else None for a in outs], cap, C.byref(n_tax)]
        res[mem] = (call(mem, lib().mdg_counts_reduce, *args), n_tax.value)
    assert res[MDG_HOST][1] == res[MDG_DEVICE][1] > 0
    assert_same_bytes(*(res[mem][0] for mem in (MDG_HOST, MDG_DEVICE)))


@pytest.mark.parametrize("with_keep", [False, True])
def test_counts_order_host_vs_device(ctx, gen, reduced, with_keep):
    n = len(gen["tax_id"])
    m = reduced["n_tax"]
    keep = np.ascontiguousarray(reduced["keep"]) if with_keep else None
    cap = int(np.count_nonzero(keep)) if with_keep else n
    order = np.random.default_rng(3).permutation(m).astype(np.int64)
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        n_out = C.c_int64(0)
        args = [ctx._h, mem, n, gen["tax_id"].astype(np.int64), np.ascontiguousarray(reduced["z"]), keep, m,
                np.ascontiguousarray(reduced["first_row"]), order, np.zeros(cap, np.int64), cap, C.byref(n_out)]
        res[mem] = (call(mem, lib().mdg_counts_order, *args), n_out.value)
    assert res[MDG_HOST][1] == res[MDG_DEVICE][1] > 0
    assert_same_bytes(res[MDG_HOST][0], res[MDG_DEVICE][0])


@pytest.mark.parametrize("n_top,with_weight,with_keep", [(10, True, True), (10, False, False), (10**6, True, False), (0, True, True)])
def test_select_top_host_vs_device(ctx, gen, reduced, n_top, with_weight, with_keep):
    n = len(gen["tax_id"])
    m = reduced["n_tax"]
    take = min(n_top, m)
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        n_out = C.c_int64(0)
        args = [ctx._h, mem, n, gen["tax_id"].astype(np.int64), gen["n_alignments"].astype(np.uint32),
                np.ascontiguousarray(reduced["keep"]) if with_keep else None, m, np.ascontiguousarray(reduced["tax_id"]),
                np.ascontiguousarray(reduced["first_row"]), n_top, np.zeros(m, np.uint64) if with_weight else None,
                np.zeros(max(take, 1), np.int64), C.byref(n_out)]
        res[mem] = (call(mem, lib().mdg_select_top, *args), n_out.value)
    assert res[MDG_HOST][1] == res[MDG_DEVICE][1] == take
    assert_same_bytes(res[MDG_HOST][0], res[MDG_DEVICE][0])


@pytest.fixture(scope="module")
def fit_inputs():
    tax_id, k, N, _ = syn.dense_fit_batch(9, max_position=P, seed=43)
    rng = np.random.default_rng(5)
    mism12 = rng.integers(0, 50, (len(tax_id), R, 12), dtype=np.uint32)
    noise3 = rng.random((len(tax_id), 3))
    return tax_id.astype(np.int64), k.astype(np.uint32), N.astype(np.uint32), mism12, noise3


@pytest.mark.parametrize("case", ["all", "no_median_hpdi", "no_draws", "no_mism12_noise"])
def test_fit_batch_host_vs_device(ctx, fit_inputs, monkeypatch, case):
    """MDG_FIT_CHUNK=4: three chunks, so the per-chunk copies back start at rows 0, 4 and 8."""
    monkeypatch.setenv("MDG_FIT_CHUNK", "4")
    tax_id, k, N, mism12, noise3 = fit_inputs
    if case == "no_mism12_noise":
        mism12 = noise3 = None
    n = len(tax_id)
    cfg = _lib.default_config(num_warmup=40, num_samples=30, seed=7)
    S, W = cfg.num_samples, cfg.num_warmup
    stats = [np.zeros((n, R), np.float32) if case != "no_median_hpdi" else None for _ in range(3)]
    draws = [np.zeros((n, NUM_RUNS, S, 4)), np.zeros((n, NUM_RUNS, W + S, 4)), np.zeros((n, NUM_RUNS, 2, R))]
    if case == "no_draws":
        draws = [None] * 3
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        args = [ctx._h, mem, n, P, tax_id, k, N, mism12, noise3, C.byref(cfg), np.zeros(n, FIT_RESULT_DTYPE),
                *[a.copy() if a is not None else None for a in stats + draws]]
        res[mem] = call(mem, lib().mdg_fit_batch, *args)
    assert_same_bytes(res[MDG_HOST], res[MDG_DEVICE])


@pytest.mark.parametrize("with_extras", [False, True])
def test_map_batch_host_vs_device(ctx, fit_inputs, with_extras):
    tax_id, k, N, mism12, noise3 = fit_inputs
    if not with_extras:
        mism12 = noise3 = None
    cfg = _lib.default_config()
    res = {}
    for mem in (MDG_HOST, MDG_DEVICE):
        args = [ctx._h, mem, len(tax_id), P, tax_id, k, N, mism12, noise3, C.byref(cfg), np.zeros(len(tax_id), MAP_RESULT_DTYPE)]
        res[mem] = call(mem, lib().mdg_map_batch, *args)
    assert_same_bytes(res[MDG_HOST], res[MDG_DEVICE])


def test_entry_points_restore_the_current_device(gen, reduced, fit_inputs):
    """Every entry point, called on a context of GPU 1 by a thread whose current device is 0, leaves it at 0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from metadamage_b200.backend import Context

    torch.cuda.set_device(0)
    tax_id, k, N, _, _ = fit_inputs
    cfg = _lib.default_config(num_warmup=20, num_samples=20)
    m = reduced["n_tax"]
    with Context(1) as c1:
        calls = {
            "tsv_parse": lambda: c1.tsv_parse(b"1\t10\t5'\t0" + b"\t1" * 16 + b"\n"),
            "counts_reduce": lambda: c1.counts_reduce(gen["tax_id"], gen["n_alignments"], gen["is_reverse"], gen["pos0"],
                                                      gen["counts16"], max_position=P),
            "counts_order": lambda: c1.counts_order(gen["tax_id"], reduced["z"], reduced["keep"], reduced["first_row"],
                                                    np.arange(m, dtype=np.int64)),
            "select_top": lambda: c1.select_top(gen["tax_id"], gen["n_alignments"], reduced["keep"], reduced["tax_id"],
                                                reduced["first_row"], 5),
            "fit_batch": lambda: c1.fit_batch(tax_id, k, N, cfg),
            "fit_submit_wait": lambda: c1.fit_wait(c1.fit_submit(tax_id, k, N, cfg)),
            "map_batch": lambda: c1.map_batch(tax_id, k, N, cfg),
            "synchronize": c1.synchronize,
        }
        for name, fn in calls.items():
            fn()
            assert torch.cuda.current_device() == 0, name
