"""-m gpu: the MAP-only screening path (mdg_map_batch, K3m) against mdg_fit_batch's MAP fields and the oracle, its
partition invariance, edge cases, and `metadamage fit --map-only` end to end."""
import numpy as np
import pytest
from scipy import special
from typer.testing import CliRunner

from metadamage_b200 import _lib, synthetic as syn
from metadamage_b200._abi import FIT_FAILED, MAP_RESULT_DTYPE
from test_gpu_fits import small_batch
from test_host import make_cfg, write_tsv

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def map_oracle(oracle):
    from oracle import map_oracle as M

    M.build()
    return M


def map_matches_oracle_batch(oracle, sample_inputs, n=96, P=15, seed=5):
    """test_map_matches_oracle's batch: synthetic TaxIDs plus the six high-coverage sample TaxIDs (P = 15)"""
    tid, k, N = small_batch(n, P=P, seed=seed)
    if P == 15:
        for name in ("ancient", "control"):
            s = sample_inputs[name]
            r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
            tid = np.r_[tid, r["tax_id"] + 10 ** 6]
            k = np.vstack([k, r["k"]])
            N = np.vstack([N, r["N"]])
    return tid, k, N


def test_all_position_fits_bit_identical_to_fit_batch(ctx, oracle, sample_inputs):
    tid, k, N = map_matches_oracle_batch(oracle, sample_inputs)
    cfg = _lib.default_config(num_warmup=4, num_samples=4, do_fwd_rev=0)
    fit = ctx.fit_batch(tid, k, N, cfg)["result"]
    res = ctx.map_batch(tid, k, N, _lib.default_config())
    r = res["run"]
    for a, b in (("q", "map_q"), ("A", "map_A"), ("c", "map_c"), ("phi", "map_phi"), ("logp", "map_logp")):
        assert r[:, 0][a].tobytes() == fit[b].tobytes(), a
    for a, b in (("q", "map_null_q"), ("phi", "map_null_phi"), ("logp", "map_null_logp")):
        assert r[:, 1][a].tobytes() == fit[b].tobytes(), a
    assert np.array_equal(r[:, 0]["iters"], fit["map_iters"])
    assert res["D_max"].tobytes() == fit["map_D_max"].tobytes()


def close(a, b, rtol, atol=0.0):
    return np.abs(a - b) <= rtol * np.abs(b) + atol


@pytest.mark.parametrize("P", [15, 25, 40])
@pytest.mark.parametrize("fwd_rev", [0, 1])
def test_map_batch_matches_oracle(ctx, oracle, sample_inputs, P, fwd_rev, map_oracle):
    tid, k, N = map_matches_oracle_batch(oracle, sample_inputs, n=64, P=P, seed=5 + P)
    got = ctx.map_batch(tid, k, N, _lib.default_config(do_fwd_rev=fwd_rev))
    exp = map_oracle.map_batch(tid, k, N, oracle.default_config(do_fwd_rev=fwd_rev))
    for f in ("tax_id", "N_z1_forward", "N_z1_reverse", "N_sum_forward", "N_sum_reverse", "N_sum_total", "y_sum_forward",
              "y_sum_reverse", "y_sum_total"):
        assert np.array_equal(got[f], exp[f]), f
    n_runs = 6 if fwd_rev else 2
    for run in range(n_runs):
        g, e = got["run"][:, run], exp["run"][:, run]
        conv = ((g["flags"] | e["flags"]) & 0x2) == 0
        assert conv.mean() >= 0.95, (run, conv.mean())
        assert np.array_equal(g["flags"][conv], e["flags"][conv]), run
        names = ("q", "A", "c", "phi") if run % 2 == 0 else ("q", "phi")
        for f in names:
            assert close(g[f][conv], e[f][conv], 1e-5, 1e-9).all(), (run, f)
        cov = conv & ((e["flags"] & 0x10) == 0)
        stds = ("q_std", "A_std", "c_std", "phi_std") if run % 2 == 0 else ("q_std", "phi_std")
        for f in stds:
            assert close(g[f][cov], e[f][cov], 1e-4, 1e-9).all(), (run, f)
        for f in ("logp", "loglik"):
            assert np.max(np.abs(g[f][conv] - e[f][conv])) < 1e-6, (run, f)
    both = ((got["status"] | exp["status"]) & 0x2) == 0
    assert np.array_equal(got["status"][both], exp["status"][both])
    ok = both & ((exp["status"] & 0x10) == 0)
    # rho_Ac = cov_Ac / (A_std c_std). An off-diagonal entry of H^-1 carries an error of the size of the diagonal ones
    # times their relative error (it passes through zero by cancellation), so rho's error is absolute on the [-1, 1]
    # scale: the stds' 1e-4 relative bound becomes 1e-4 relative plus 1e-4 absolute here
    d_rho = np.abs(got["rho_Ac"][ok] - exp["rho_Ac"][ok])
    worst = int(np.argmax(d_rho))
    assert close(got["rho_Ac"][ok], exp["rho_Ac"][ok], 1e-4, 1e-4).all(), (d_rho.max(), got["rho_Ac"][ok][worst], exp["rho_Ac"][ok][worst])
    assert close(got["D_max_std"][ok], exp["D_max_std"][ok], 1e-4, 1e-9).all()
    lam_g, lam_e = got["lambda_LR"][both], exp["lambda_LR"][both]
    assert (np.abs(lam_g - lam_e) <= 2e-6 * (1 + np.abs(lam_e))).all()
    # the tail statistics of the CUDA rows are scipy's of their own lambda
    lam = np.maximum(got["lambda_LR"][both], 0.0)
    np.testing.assert_allclose(got["lambda_LR_P"][both], np.exp(-lam / 2), rtol=1e-12)
    np.testing.assert_allclose(got["lambda_LR_z"][both], -special.ndtri_exp(-lam / 2), rtol=1e-10)
    if fwd_rev:
        for side, pmd, null in (("forward", 2, 3), ("reverse", 4, 5)):
            rr = got["run"]
            assert got[side + "_D_max"].tobytes() == (rr[:, pmd]["A"] + rr[:, pmd]["c"]).tobytes()
            assert got[side + "_lambda_LR"].tobytes() == (2.0 * (rr[:, pmd]["loglik"] - rr[:, null]["loglik"])).tobytes()
    else:
        assert np.all(np.isnan(got["forward_D_max"])) and np.all(got["run"][:, 2:]["n_eval"] == 0)


def test_host_device_and_partitions_bit_identical(ctx):
    import torch

    tid, k, N = small_batch(300, seed=21)
    cfg = _lib.default_config()
    noise3 = np.random.default_rng(0).random((len(tid), 3))
    host = ctx.map_batch(tid, k, N, cfg, noise3=noise3)
    t = ctx.timings()
    assert t["map_ms"] > 0 and t["assemble_ms"] > 0 and t["total_ms"] > 0 and t["n_launches"] == 2
    assert t["nuts_ms"] == 0 and t["ppc_ms"] == 0
    assert t["leapfrogs"] == [int(host["run"][:, r]["n_eval"].sum()) for r in range(6)]
    np.testing.assert_array_equal(host["normalized_noise_reverse"], noise3[:, 2])
    dev = torch.device("cuda", 0)
    out = torch.zeros(len(tid) * MAP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    ctx.map_batch_device(torch.from_numpy(tid).to(dev), torch.from_numpy(k.view(np.int32)).to(dev),
                         torch.from_numpy(N.view(np.int32)).to(dev), out, cfg, noise3=torch.from_numpy(noise3).to(dev))
    assert out.cpu().numpy().tobytes() == host.tobytes()
    split = np.concatenate([ctx.map_batch(tid[:117], k[:117], N[:117], cfg, noise3=noise3[:117]),
                            ctx.map_batch(tid[117:], k[117:], N[117:], cfg, noise3=noise3[117:])])
    assert split.tobytes() == host.tobytes()


def test_noise_from_mism12_equals_fit_batch(ctx):
    tid, k, N, g = syn.dense_fit_batch(40, seed=31)
    first = np.flatnonzero(np.r_[True, g["tax_id"][1:] != g["tax_id"][:-1]])
    m12 = syn.mism12_from_counts16(g["counts16"], first[g["passes"]], 15)
    cfg = _lib.default_config(num_warmup=4, num_samples=4, do_fwd_rev=0)
    fit = ctx.fit_batch(tid, k, N, cfg, mism12=m12)["result"]
    res = ctx.map_batch(tid, k, N, cfg, mism12=m12)
    for f in ("normalized_noise", "normalized_noise_forward", "normalized_noise_reverse", "N_sum_total", "y_sum_reverse"):
        assert res[f].tobytes() == fit[f].tobytes(), f


def test_one_million_taxids_in_one_call(ctx):
    tid, k, N = syn.dense_fit_batch_shares(1_000_000, 8)
    assert len(tid) == 1_000_000
    res = ctx.map_batch(tid, k, N)
    assert np.array_equal(res["tax_id"], tid)
    assert (res["status"] & FIT_FAILED).sum() == 0
    assert np.isfinite(res["D_max"]).all()
    # the last rows equal a call on those TaxIDs alone
    sl = slice(999_000, None)
    assert ctx.map_batch(tid[sl], k[sl], N[sl]).tobytes() == res[sl].tobytes()


def test_edge_cases(ctx, oracle, map_oracle):
    for P in (15, 40):
        empty = ctx.map_batch(np.zeros(0, np.int64), np.zeros((0, 2 * P), np.uint32), np.zeros((0, 2 * P), np.uint32))
        assert len(empty) == 0 and ctx.timings()["leapfrogs"] == [0] * 6
        z = np.zeros((2, 2 * P), np.uint32)
        tid = np.array([7, 8], np.int64)
        got = ctx.map_batch(tid, z, z)
        exp = map_oracle.map_batch(tid, z, z)
        assert np.array_equal(got["status"], exp["status"]) and np.array_equal(got["run"]["flags"], exp["run"]["flags"])
        assert np.isfinite(got["run"][:, 0]["q"]).all() and (got["N_sum_total"] == 0).all()


def run_cli(args):
    from metadamage.cli import cli_app

    result = CliRunner().invoke(cli_app, ["fit", *map(str, args)])
    assert result.exit_code == 0, result.output
    return result


def test_cli_map_only_end_to_end(tmp_path, sample_inputs, monkeypatch):
    from metadamage_b200 import counts, fits, io

    path = tmp_path / "data_ancient.txt"
    write_tsv(path, sample_inputs["ancient"], True)
    out = tmp_path / "out"
    run_cli([path, "--map-only", "--out-dir", out])
    assert sorted(p.name for p in out.iterdir()) == ["counts", "map_results"]
    df = io.Parquet(out / "map_results" / "data_ancient.parquet").load()
    assert list(df.columns) == fits.MAP_RESULT_COLUMNS and len(df) == 3
    cfg = make_cfg(out)
    cfg.add_filename(path)
    df_counts = counts.load_counts(cfg)
    want = fits.compute_map_fits(df_counts, cfg)
    pd_equal = df.drop(columns=["shortname"]).reset_index(drop=True).equals(want.drop(columns=["shortname"]).reset_index(drop=True))
    assert pd_equal
    assert (df["lambda_LR"] > 150).all() and df["valid"].all()
    # cached second run; --forced recomputes
    calls = []
    real = fits.compute_map_fits
    monkeypatch.setattr(fits, "compute_map_fits", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    run_cli([path, "--map-only", "--out-dir", out])
    assert calls == []
    run_cli([path, "--map-only", "--out-dir", out, "--forced"])
    assert calls == [1]
    # --max-fits applies
    run_cli([path, "--map-only", "--out-dir", tmp_path / "top", "--max-fits", 2])
    assert len(io.Parquet(tmp_path / "top" / "map_results" / "data_ancient.parquet").load()) == 2


def test_cli_map_only_two_gpus_equal_one(tmp_path):
    from metadamage_b200 import io

    if _lib.load().mdg_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    g = syn.make_mismatch_matrix(0, n_fit=300, seed=11)
    path = tmp_path / "synth.txt"
    syn.write_tsv(g, str(path))
    run_cli([path, "--map-only", "--out-dir", tmp_path / "o1"])
    run_cli([path, "--map-only", "--out-dir", tmp_path / "o2", "--gpus", 2])
    a = io.Parquet(tmp_path / "o1" / "map_results" / "synth.parquet").load()
    b = io.Parquet(tmp_path / "o2" / "map_results" / "synth.parquet").load()
    assert a.equals(b)
