"""-m gpu: the CUDA counts kernel (K1), called through the C-ABI, vs the oracle and the
reference-generated goldens. Bit-exact on every integer / byte / float32 column."""
import numpy as np
import pytest

from test_oracle_counts import CASES, check_against_golden, run_case
from metadamage_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

ROW_KEYS = ("n_fwd_ref", "n_rev_ref", "z", "y_sum_total", "keep")
TAX_KEYS = ("tax_id", "n_alignments", "first_row", "k", "N")


def assert_same(r, o, noise=True):
    assert r["n_tax"] == o["n_tax"]
    for key in ROW_KEYS + TAX_KEYS:
        assert np.array_equal(r[key], o[key]), key
    for key in ("f_fwd", "f_rev"):
        assert np.array_equal(r[key].view(np.uint32), o[key].view(np.uint32)), key
    if noise and r.get("noise") is not None:
        np.testing.assert_allclose(r["noise"], o["noise"], rtol=1e-11, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("name", list(CASES))
def test_counts_match_reference_goldens(ctx, sample_inputs, counts_golden, name):
    r, s = run_case(ctx.counts_reduce, sample_inputs, name)
    check_against_golden(r, s, counts_golden, name, CASES[name][1], CASES[name][2])


@pytest.mark.parametrize("name", list(CASES))
def test_counts_match_oracle_on_samples(ctx, oracle, sample_inputs, name):
    src, fwd, rev, min_al, min_y = CASES[name]
    s = sample_inputs[src]
    kw = dict(fwd=fwd, rev=rev, max_position=15, min_alignments=min_al, min_y_sum=min_y)
    r = ctx.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"], want_noise=True, **kw)
    o = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"], **kw)
    assert_same(r, o)


def test_counts_output_buffers_can_be_reused(ctx, oracle):
    """Context.counts_reduce(out=...) writes into the arrays of an earlier result (or caller-allocated,
    e.g. pinned, ones) instead of allocating: same values, same memory."""
    g = syn.make_mismatch_matrix(800, seed=12)
    args = (g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"])
    first = ctx.counts_reduce(*args, want_noise=True)
    snapshot = {key: np.array(val, copy=True) for key, val in first.items() if isinstance(val, np.ndarray)}
    second = ctx.counts_reduce(*args, want_noise=True, out=first)
    third = ctx.counts_reduce(*args, want_noise=True, out=second)
    for key, val in snapshot.items():
        assert np.array_equal(third[key], val, equal_nan=True), key
    assert np.shares_memory(third["n_fwd_ref"], first["n_fwd_ref"]) and np.shares_memory(third["k"], second["k"])
    assert_same({k_: v for k_, v in third.items() if not k_.startswith("_buf_")}, oracle.counts_reduce(*args))
    # buffers of the wrong shape are simply not used
    other = ctx.counts_reduce(*args, max_position=7, out=third)
    assert other["k"].shape[1] == 14 and not np.shares_memory(other["k"], third["k"])


@pytest.mark.parametrize("P,seed,fwd,rev", [(15, 1, "CT", "GA"), (25, 2, "GA", "CT"), (7, 3, "CT", "GA"), (40, 4, "AG", "TC")])
def test_counts_match_oracle_on_synthetic(ctx, oracle, P, seed, fwd, rev):
    g = syn.make_mismatch_matrix(3000, max_position=P, seed=seed, fwd=fwd, rev=rev)
    kw = dict(fwd=fwd, rev=rev, max_position=P, min_alignments=10, min_y_sum=10)
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], want_noise=True, **kw)
    o = oracle.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"], **kw)
    assert_same(r, o)
    assert np.array_equal(r["tax_id"], g["tax_ids"][g["passes"]])


def ragged_input(rng, n_tax, max_rows, P):
    """TaxIDs with 1..max_rows rows, random strands/positions (duplicates, gaps, |z| > P included)."""
    lens = rng.integers(1, max_rows + 1, n_tax)
    tax = np.repeat(rng.permutation(n_tax).astype(np.int64) * 7 + 3, lens)
    n = len(tax)
    nal = np.repeat(rng.integers(1, 200, n_tax).astype(np.uint32), lens)
    rev = rng.integers(0, 2, n).astype(np.uint8)
    pos = rng.integers(0, P + 6, n).astype(np.uint8)
    c16 = rng.integers(0, 50, (16, n)).astype(np.uint32)
    c16[:, rng.random(n) < 0.05] = 0  # all-zero rows: N = 0 -> f = 0
    return tax, nal, rev, pos, c16


@pytest.mark.parametrize("max_rows,n_tax", [(1, 5000), (9, 4000), (70, 2000), (400, 300), (1500, 40)])
def test_counts_ragged_segments(ctx, oracle, max_rows, n_tax):
    """Segment lengths from 1 to 1500 rows: a TaxID that runs past its warp's 128 rows is read on, 32 rows at a
    time, up to MDG_MAX_SEGMENT_ROWS."""
    rng = np.random.default_rng(max_rows)
    tax, nal, rev, pos, c16 = ragged_input(rng, n_tax, max_rows, 15)
    kw = dict(max_position=15, min_alignments=20, min_y_sum=5)
    r = ctx.counts_reduce(tax, nal, rev, pos, c16, want_noise=True, **kw)
    o = oracle.counts_reduce(tax, nal, rev, pos, c16, **kw)
    assert_same(r, o)


def test_counts_empty_and_tiny(ctx, oracle):
    e = np.zeros(0)
    r = ctx.counts_reduce(e, e, e, e, np.zeros((16, 0)))
    assert r["n_tax"] == 0 and r["k"].shape == (0, 30)
    rng = np.random.default_rng(9)
    for n in (1, 2, 15, 16, 17, 1023, 1024, 1025, 1151, 1153):
        tax, nal, rev, pos, c16 = ragged_input(rng, max(1, n // 10), 12, 15)
        tax, nal, rev, pos, c16 = tax[:n], nal[:n], rev[:n], pos[:n], np.ascontiguousarray(c16[:, :n])
        r = ctx.counts_reduce(tax, nal, rev, pos, c16, min_alignments=1, min_y_sum=0, want_noise=True)
        o = oracle.counts_reduce(tax, nal, rev, pos, c16, min_alignments=1, min_y_sum=0)
        assert_same(r, o)


def test_counts_segment_too_long_is_an_error(ctx):
    from metadamage_b200._lib import MdgError

    n = 6000
    tax = np.zeros(n, np.int64)
    with pytest.raises(MdgError, match="rows"):
        ctx.counts_reduce(tax, np.full(n, 50, np.uint32), np.zeros(n, np.uint8), np.zeros(n, np.uint8), np.ones((16, n), np.uint32))


def test_counts_uint32_overflow_is_an_error(ctx):
    from metadamage_b200._lib import MdgError

    c16 = np.full((16, 4), 2 ** 31, np.uint32)
    with pytest.raises(MdgError, match="uint32"):
        ctx.counts_reduce(np.zeros(4, np.int64), np.full(4, 50, np.uint32), np.zeros(4, np.uint8), np.arange(4, dtype=np.uint8), c16)


def test_counts_full_size_properties(ctx):
    """BASELINE config 5: 10M rows. Size-independent properties instead of an oracle run:
    conservation of k and N, y_sum_total broadcast, idempotence, and exact agreement with the
    generator's own dense k/N."""
    g = syn.make_mismatch_matrix(333_334, max_position=15, seed=syn.SEEDS["cfg5"])
    n = len(g["tax_id"])
    assert n >= 10_000_000
    r = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"])
    sel = g["passes"]
    assert r["n_tax"] == int(sel.sum())
    assert np.array_equal(r["tax_id"], g["tax_ids"][sel])
    assert np.array_equal(r["k"], g["k"][sel]) and np.array_equal(r["N"], g["N"][sel])
    keep = r["keep"].astype(bool)
    assert keep.sum() == 30 * r["n_tax"]
    # y_sum_total of a kept row equals the dense row sum of its TaxID
    ysum = r["k"].sum(axis=1, dtype=np.uint64)
    assert np.array_equal(r["y_sum_total"][keep].reshape(-1, 30)[:, 0], ysum)
    assert np.array_equal(np.abs(r["z"].astype(int)), g["pos0"].astype(int) + 1)
    # checksum of checksums: total N over kept rows (picked by strand) == total dense N
    n_pick = np.where(g["is_reverse"] == 1, r["n_rev_ref"], r["n_fwd_ref"]).astype(np.uint64)
    assert int(n_pick[keep].sum()) == int(r["N"].sum(dtype=np.uint64))
    r2 = ctx.counts_reduce(g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], g["counts16"])
    for key in ROW_KEYS + TAX_KEYS + ("f_fwd", "f_rev"):
        assert r[key].tobytes() == r2[key].tobytes()


def test_counts_full_size_bit_exact_vs_oracle(ctx, oracle):
    """BASELINE config 5 at full size (10M rows, 333 334 TaxIDs): EVERY output of K1 — the per-row
    columns n_fwd_ref, n_rev_ref, f_fwd, f_rev (float32 bit patterns), z, y_sum_total, keep and the
    per-TaxID tax_id, n_alignments, first_row, dense k/N, noise — against the oracle's restatement of
    counts.py:237-256 on the same rows, including N = 0 rows (0/0 -> 0) and the failing TaxIDs."""
    g = syn.make_mismatch_matrix(333_334, max_position=15, seed=syn.SEEDS["cfg5"])
    # force some all-zero reference rows (N = 0 -> f = 0, counts.py:254) and k = 0 rows into the stress input
    rng = np.random.default_rng(5)
    c16 = g["counts16"].copy()
    n = c16.shape[1]
    c16[:, rng.integers(0, n, 50_000)] = 0
    c16[7, rng.integers(0, n, 200_000)] = 0   # CT
    c16[8, rng.integers(0, n, 200_000)] = 0   # GA
    args = (g["tax_id"], g["n_alignments"], g["is_reverse"], g["pos0"], c16)
    r = ctx.counts_reduce(*args, want_noise=True)
    o = oracle.counts_reduce(*args)
    assert n >= 10_000_000 and o["n_tax"] > 50_000
    assert (o["n_fwd_ref"] == 0).sum() > 1000 and (o["keep"] == 0).sum() > 1_000_000
    assert_same(r, o)
