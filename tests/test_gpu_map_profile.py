"""-m gpu: profile intervals of D_max (mdg_map_profile, K3p) against the oracle, host / device buffers and partitions,
a million TaxIDs in one call, and `metadamage fit --map-only --profile-interval` end to end."""
import numpy as np
import pytest
from typer.testing import CliRunner

from metadamage_b200 import _lib, synthetic as syn
from metadamage_b200._abi import FIT_FAILED, MAP_INTERVAL_DTYPE, MAP_RESULT_DTYPE, PROFILE_AT_BOUND, PROFILE_FAILED
from test_gpu_map import map_matches_oracle_batch
from test_host import write_tsv

pytestmark = pytest.mark.gpu

UNUSABLE = PROFILE_FAILED | FIT_FAILED


@pytest.fixture(scope="module")
def prof():
    import map_profile_oracle as P

    P.build()
    return P


@pytest.mark.parametrize("P", [15, 25, 40])
@pytest.mark.parametrize("fwd_rev", [0, 1])
def test_profile_matches_oracle(ctx, oracle, sample_inputs, prof, P, fwd_rev):
    """Both sides profile the same CUDA MAP rows. An end is a root of h(D) = 2 (logp^ - pl(D)) - t found to |h| <= 1e-7
    or a bracket of 1e-9. The two inner fits reach pl(D) to within their acceptance slack (1e-14 of sum lgamma(N + 1):
    up to a few 1e-7 at the sample file's coverage; logp within 1e-6 is asserted below), so h differs by up to ~2e-6
    between them; with |dh/dD| ~ 4 sqrt(t) / width near a root the ends then agree to ~1e-6 of the interval width plus
    the bracket. The bound is 1e-5 of the width plus 2e-9."""
    tid, k, N = map_matches_oracle_batch(oracle, sample_inputs, n=64, P=P, seed=5 + P)
    cfg = _lib.default_config(do_fwd_rev=fwd_rev)
    rows = ctx.map_batch(tid, k, N, cfg)
    got = ctx.map_profile(k, N, rows, cfg)
    exp = prof.map_profile(k, N, rows, oracle.default_config(do_fwd_rev=fwd_rev))
    assert np.array_equal(got["tax_id"], tid) and np.array_equal(got["threshold"], exp["threshold"])
    n_prof = 3 if fwd_rev else 1
    for i in range(n_prof):
        g, e = got["end"][:, i], exp["end"][:, i]
        clean = ((g["flags"] | e["flags"]) & UNUSABLE) == 0
        assert clean.mean() >= 0.95, (i, clean.mean())
        assert np.array_equal(g["flags"][clean], e["flags"][clean]), i
        assert np.array_equal(g["flags"] & FIT_FAILED, e["flags"] & FIT_FAILED), i
        width = np.abs(e["D"][:, 1] - e["D"][:, 0])[:, None] * np.ones(2)
        dD = np.abs(g["D"] - e["D"])[clean]
        assert (dD <= 1e-5 * width[clean] + 2e-9).all(), (i, tid[clean.any(axis=1)], np.max(dD / width[clean]))
        assert (np.abs(g["logp"] - e["logp"])[clean] < 1e-6).all(), i
    if not fwd_rev:
        assert np.all(np.isnan(got["end"]["D"][:, 1:])) and np.all(got["end"]["n_eval"][:, 1:] == 0)


def test_host_device_partitions_and_timings(ctx):
    import torch

    tid, k, N, _ = syn.dense_fit_batch(300, seed=21)
    cfg = _lib.default_config()
    rows = ctx.map_batch(tid, k, N, cfg)
    host = ctx.map_profile(k, N, rows, cfg)
    t = ctx.timings()
    assert t["map_ms"] > 0 and t["total_ms"] > 0 and t["n_launches"] == 2
    assert t["nuts_ms"] == 0 and t["ppc_ms"] == 0 and t["assemble_ms"] == 0 and t["counts_ms"] == 0
    assert t["leapfrogs"] == [int(host["end"][:, r // 2]["n_eval"].sum()) if r % 2 == 0 else 0 for r in range(6)]
    dev = torch.device("cuda", 0)
    out = torch.zeros(len(tid) * MAP_INTERVAL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    d_rows = torch.from_numpy(rows.view(np.uint8)).to(dev)
    ctx.map_profile_device(torch.from_numpy(k.view(np.int32)).to(dev), torch.from_numpy(N.view(np.int32)).to(dev), d_rows, out, cfg)
    assert out.cpu().numpy().tobytes() == host.tobytes()
    split = np.concatenate([ctx.map_profile(k[:117], N[:117], rows[:117], cfg), ctx.map_profile(k[117:], N[117:], rows[117:], cfg)])
    assert split.tobytes() == host.tobytes()
    empty = ctx.map_profile(k[:0], N[:0], rows[:0], cfg)
    assert len(empty) == 0 and ctx.timings()["leapfrogs"] == [0] * 6
    for level in (0.0, 1.0, float("nan")):
        with pytest.raises(_lib.MdgError):
            ctx.map_profile(k, N, rows, cfg, level=level)


def test_one_million_taxids_in_one_call(ctx):
    tid, k, N = syn.dense_fit_batch_shares(1_000_000, 8)
    rows = ctx.map_batch(tid, k, N)
    iv = ctx.map_profile(k, N, rows)
    assert np.array_equal(iv["tax_id"], tid)
    ends = iv["end"][:, 0]
    usable = (iv["status"] & UNUSABLE) == 0
    assert usable.mean() > 0.99, usable.mean()
    at_bound = (ends["flags"] & PROFILE_AT_BOUND) != 0
    assert np.all(np.isfinite(ends["D"][usable]) | at_bound[usable])
    assert np.all(ends["D"][usable, 0] <= rows["D_max"][usable]) and np.all(rows["D_max"][usable] <= ends["D"][usable, 1])
    sl = slice(999_000, None)
    assert ctx.map_profile(k[sl], N[sl], rows[sl]).tobytes() == iv[sl].tobytes()


def run_cli(args):
    from metadamage.cli import cli_app

    result = CliRunner().invoke(cli_app, ["fit", *map(str, args)])
    assert result.exit_code == 0, result.output
    return result


def test_cli_profile_interval_end_to_end(tmp_path, sample_inputs, monkeypatch):
    from metadamage_b200 import fits, io

    path = tmp_path / "data_ancient.txt"
    write_tsv(path, sample_inputs["ancient"], True)
    plain_dir, iv_dir = tmp_path / "plain", tmp_path / "iv"
    run_cli([path, "--map-only", "--out-dir", plain_dir])
    run_cli([path, "--map-only", "--profile-interval", "--out-dir", iv_dir])
    plain = io.Parquet(plain_dir / "map_results" / "data_ancient.parquet").load()
    df = io.Parquet(iv_dir / "map_results" / "data_ancient.parquet").load()
    assert list(df.columns) == fits.MAP_RESULT_COLUMNS + fits.MAP_INTERVAL_COLUMNS
    assert df[fits.MAP_RESULT_COLUMNS].equals(plain)
    assert io.Parquet(iv_dir / "map_results" / "data_ancient.parquet").load_metadata()["profile_interval"] == 0.68
    # the strongly damaged ancient TaxIDs: an interval away from 0 around the mode
    assert df["interval_valid"].all() and (df["D_max_lower"] > 0).all()
    assert ((df["D_max_lower"] < df["D_max"]) & (df["D_max"] < df["D_max_upper"])).all()
    # cache: an interval run reuses an interval table, a plain run recomputes, --forced recomputes
    calls = []
    real = fits.compute_map_fits
    monkeypatch.setattr(fits, "compute_map_fits", lambda *a, **kw: calls.append(kw.get("profile_interval")) or real(*a, **kw))
    run_cli([path, "--map-only", "--profile-interval", "--out-dir", iv_dir])
    assert calls == []
    run_cli([path, "--map-only", "--out-dir", iv_dir])
    assert calls == [False]
    assert io.Parquet(iv_dir / "map_results" / "data_ancient.parquet").load().equals(plain)
    run_cli([path, "--map-only", "--out-dir", plain_dir])
    assert calls == [False]
    run_cli([path, "--map-only", "--profile-interval", "--out-dir", iv_dir, "--forced"])
    assert calls == [False, True]


def test_cli_profile_interval_two_gpus_equal_one(tmp_path):
    from metadamage_b200 import io

    if _lib.load().mdg_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    g = syn.make_mismatch_matrix(0, n_fit=300, seed=11)
    path = tmp_path / "synth.txt"
    syn.write_tsv(g, str(path))
    run_cli([path, "--map-only", "--profile-interval", "--out-dir", tmp_path / "o1"])
    run_cli([path, "--map-only", "--profile-interval", "--out-dir", tmp_path / "o2", "--gpus", 2])
    a = io.Parquet(tmp_path / "o1" / "map_results" / "synth.parquet").load()
    b = io.Parquet(tmp_path / "o2" / "map_results" / "synth.parquet").load()
    assert a.equals(b)
