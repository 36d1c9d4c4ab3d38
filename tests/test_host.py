"""Host-side logic (no GPU): CLI behaviour mirroring the reference's own tests
(tests/test_metadamage.py:17-69), TSV layouts, row ordering, schemas, caching metadata."""
import json
import os
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
from typer.testing import CliRunner

from metadamage.cli import cli_app
from metadamage.utils import extract_name
from metadamage_b200 import counts, fits, io, utils
from metadamage_b200._abi import FIT_RESULT_DTYPE


# ---- the reference's five tests, verbatim in behaviour ----
def test_extracting_name_from_string():
    assert extract_name("./data/input/data_ancient.txt") == "data_ancient"


def test_extracting_name_from_path():
    assert extract_name(Path("./data/input/data_ancient.txt")) == "data_ancient"


def test_cli_fit_bad_file():
    result = CliRunner().invoke(cli_app, ["fit", "file_which_does_not_exist.txt"])
    assert result.exit_code == 1
    assert isinstance(result.exception, Exception)


def test_cli_fit_bad_files():
    result = CliRunner().invoke(cli_app, ["fit", "file_which_does_not_exist.txt", "another_file_which_does_not_exist.txt"])
    assert result.exit_code == 1
    assert isinstance(result.exception, Exception)


def test_cli_fit_version():
    result = CliRunner().invoke(cli_app, ["--version"])
    assert result.exit_code == 0
    assert "version" in result.stdout


# ---- options ----
def test_cli_fit_options_present():
    """The reference's options (cli.py:97-126, README.md:112-135) plus --max-position, same defaults."""
    import typer

    fit = typer.main.get_command(cli_app).commands["fit"]
    opts = {o: p for p in fit.params for o in p.opts}
    for opt in ("--max-position", "--min-alignments", "--min-y-sum", "--substitution-bases-forward",
                "--substitution-bases-reverse", "--max-fits", "--max-cores", "--forced", "--out-dir"):
        assert opt in opts
    assert opts["--max-position"].default == 15 and opts["--min-alignments"].default == 10
    assert opts["--min-y-sum"].default == 10 and opts["--max-cores"].default == 1 and opts["--max-fits"].default is None
    assert opts["--substitution-bases-forward"].default.value == "CT" and opts["--substitution-bases-reverse"].default.value == "GA"


def make_cfg(tmp_path, **kw):
    base = dict(out_dir=tmp_path, max_fits=None, max_cores=1, min_alignments=10, min_y_sum=10,
                substitution_bases_forward="CT", substitution_bases_reverse="GA", forced=False, version="0.0.0")
    base.update(kw)
    return utils.Config(**base)


def test_config_semantics(tmp_path):
    cfg = make_cfg(tmp_path, max_cores=-1)
    assert cfg.N_cores == utils._available_cores() - 1
    cfg = make_cfg(tmp_path, max_cores=10 ** 6)
    assert cfg.N_cores == utils._available_cores() - 1
    cfg.add_filename("x/y/KapK-12-1.sorted.txt")
    assert cfg.shortname == "KapK-12-1"
    assert cfg.filename_counts == tmp_path / "counts" / "KapK-12-1.parquet"
    assert cfg.filename_fit_results == tmp_path / "fit_results" / "KapK-12-1.parquet"
    d = cfg.to_dict()
    assert d["max_position"] == 15 and isinstance(d["out_dir"], str)
    json.dumps(d)
    with pytest.raises(ValueError):
        make_cfg(tmp_path, max_position=0)


def write_tsv(path, sample, legacy):
    s = sample
    cols = {"tax_id": s["tax_id"], "N_alignments": s["n_alignments"],
            "strand": np.where(s["is_reverse"] == 1, "3'", "5'"), "position": s["pos0"]}
    df = pd.DataFrame(cols)
    for i, name in enumerate(counts.REF_OBS_BASES):
        df[name] = s["counts16"][i]
    if legacy:
        df.columns = ["#taxid", "Nalignments", "Direction", "Pos"] + counts.REF_OBS_BASES
        df.to_csv(path, sep="\t", index=False)
    else:
        df.insert(1, "tax_name", "Homo sapiens")
        df.insert(2, "tax_rank", "species")
        df.to_csv(path, sep="\t", index=False, header=False)


@pytest.mark.parametrize("legacy", [True, False])
def test_read_mismatch_table_both_layouts(tmp_path, sample_inputs, legacy):
    path = tmp_path / "data.txt"
    write_tsv(path, sample_inputs["ancient"], legacy)
    df = counts.read_mismatch_table(path)
    assert list(df.columns) == counts.COLUMNS and len(df) == 90
    cols = counts.soa_columns(df)
    for key in ("tax_id", "n_alignments", "is_reverse", "pos0", "counts16"):
        assert np.array_equal(cols[key], sample_inputs["ancient"][key])


def test_rows_are_regrouped_when_interleaved(sample_inputs):
    s = sample_inputs["control"]
    df = pd.DataFrame({"tax_id": s["tax_id"], "x": np.arange(90)})
    perm = np.r_[np.arange(0, 90, 2), np.arange(1, 90, 2)]  # every TaxID split in two runs
    out = counts.group_rows_by_tax_id(df.iloc[perm].reset_index(drop=True))
    heads = np.flatnonzero(np.r_[True, out.tax_id.values[1:] != out.tax_id.values[:-1]])
    assert len(heads) == 3
    same = counts.group_rows_by_tax_id(df)
    assert same is df


def test_reference_row_order_matches_reference(counts_golden, sample_inputs):
    """counts.py:167-172 on the golden rows: shuffling them and re-ordering restores the reference order."""
    g = counts_golden
    n_al, tax, z = g["control_CT_GA__N_alignments"], g["control_CT_GA__tax_id"], g["control_CT_GA__position"]
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(z))
    order = counts.reference_row_order(n_al[perm], tax[perm], z[perm])
    assert np.array_equal(z[perm][order], z) and np.array_equal(tax[perm][order], tax)
    assert list(z[:30]) == list(range(1, 16)) + list(range(-1, -16, -1))


def test_downcast_dataframe_dtypes():
    df = pd.DataFrame({"tax_id": [1, 2], "position": [1, -1], "N": [5, 2 ** 31], "f": [0.5, 0.25], "name": ["a", "b"]})
    out = utils.downcast_dataframe(df, ["tax_id", "name", "missing"])
    assert str(out.dtypes["tax_id"]) == "category" and str(out.dtypes["name"]) == "category"
    assert out.dtypes["position"] == np.int8 and out.dtypes["N"] == np.uint32 and out.dtypes["f"] == np.float32
    with pytest.raises(AssertionError):
        utils.downcast_dataframe(pd.DataFrame({"N": [2 ** 33]}), [])


def test_metadata_is_similar():
    a = dict(min_alignments=10, shortname="x", extra=1)
    assert utils.metadata_is_similar(a, dict(a))
    assert not utils.metadata_is_similar(a, dict(a, more=2))
    assert utils.metadata_is_similar(a, dict(a, extra=2), include=["min_alignments", "shortname"])
    assert not utils.metadata_is_similar(a, dict(a, shortname="y"), include=["min_alignments", "shortname"])


def test_parquet_roundtrip_with_metadata(tmp_path):
    df = utils.downcast_dataframe(pd.DataFrame({"tax_id": [3, 3, 5], "position": [1, -1, 1], "f": [0.1, 0.2, 0.3]}), ["tax_id"])
    pq = io.Parquet(tmp_path / "sub" / "x.parquet")
    assert not pq.exists()
    pq.save(df, metadata={"shortname": "x", "min_y_sum": 10})
    assert pq.exists() and not pq.exists(forced=True)
    assert pq.load_metadata() == {"shortname": "x", "min_y_sum": 10}
    back = pq.load()
    assert str(back.dtypes["tax_id"]) == "category" and back["position"].dtype == np.int8
    assert len(io.Parquet(tmp_path / "sub").load(shortname="x", tax_id=3)) == 2


def fake_df_counts(sample, cfg):
    """df_counts as compute_counts would build it, from plain numpy (no GPU)."""
    s = sample
    df = pd.DataFrame({"tax_id": s["tax_id"], "tax_name": "n", "tax_rank": "r", "N_alignments": s["n_alignments"],
                       "strand": np.where(s["is_reverse"] == 1, "3'", "5'"),
                       "position": np.where(s["is_reverse"] == 1, -(s["pos0"].astype(int) + 1), s["pos0"].astype(int) + 1)})
    for i, name in enumerate(counts.REF_OBS_BASES):
        df[name] = s["counts16"][i]
    df["C"] = s["counts16"][4:8].sum(0)
    df["G"] = s["counts16"][8:12].sum(0)
    return df


def dense_by_oracle(s, oracle):
    """What counts.dense_from_df_counts returns (it needs the GPU: K1 on the frame's columns), built from the oracle."""
    r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
    n = r["n_tax"]
    return dict(tax_id=r["tax_id"], tax_name=np.array([""] * n, dtype=object), tax_rank=np.array([""] * n, dtype=object),
                N_alignments=r["n_alignments"], k=r["k"], N=r["N"], noise=r["noise"], mism12=None, first_row=r["first_row"],
                max_position=15, fwd="CT", rev="GA")


@pytest.mark.gpu
def test_dense_from_df_counts(tmp_path, sample_inputs, oracle):
    """K1 on a df_counts frame's own columns (the parquet-cache path of compute_fits) == the oracle's dense k/N/noise."""
    cfg = make_cfg(tmp_path)
    s = sample_inputs["ancient"]
    dense = counts.dense_from_df_counts(fake_df_counts(s, cfg), cfg)
    r = oracle.counts_reduce(s["tax_id"], s["n_alignments"], s["is_reverse"], s["pos0"], s["counts16"])
    assert np.array_equal(dense["k"], r["k"]) and np.array_equal(dense["N"], r["N"])
    assert list(dense["tax_id"]) == [0, 1, 2] and dense["mism12"] is None
    np.testing.assert_allclose(dense["noise"], r["noise"], rtol=1e-11)


def test_fit_dataframes_have_reference_schema(tmp_path, sample_inputs, oracle):
    cfg = make_cfg(tmp_path)
    cfg.add_filename("data_ancient.txt")
    dense = dense_by_oracle(sample_inputs["ancient"], oracle)
    res = np.zeros(3, dtype=FIT_RESULT_DTYPE)
    res["tax_id"] = dense["tax_id"]
    res["D_max"] = [0.4, 0.41, 0.42]
    res["status"] = [0, 1, 0]  # the middle fit failed -> dropped like a timed-out fit
    res["N_sum_total"] = dense["N"].sum(1)
    df, ok = fits.make_df_fit_results(res, dense, cfg)
    assert list(df.columns) == fits.FIT_RESULT_COLUMNS + ["shortname"]
    assert list(df["tax_id"]) == [0, 2]
    for col in ("tax_id", "tax_name", "tax_rank", "shortname"):
        assert str(df.dtypes[col]) == "category"
    assert df.dtypes["D_max"] == np.float32 and df.dtypes["N_sum_total"] == np.uint32 and df.dtypes["N_alignments"] == np.uint32
    out = dict(median=np.zeros((3, 30), np.float32), hpdi_lo=np.zeros((3, 30), np.float32), hpdi_hi=np.ones((3, 30), np.float32))
    dfp = fits.make_df_fit_predictions(out, dense, ok, cfg)
    assert list(dfp.columns) == ["tax_id", "position", "median", "hdpi_lower", "hdpi_upper", "shortname"]
    assert len(dfp) == 60 and dfp["position"].dtype == np.int8
    assert list(dfp["position"][:30]) == list(range(1, 16)) + list(range(-1, -16, -1))


def test_top_max_fits_selection():
    df = pd.DataFrame({"tax_id": np.repeat([1, 2, 3, 4], 2), "N_alignments": np.repeat([5, 50, 20, 7], 2)})
    assert sorted(pd.unique(fits.get_top_max_fits(df, 2)["tax_id"])) == [2, 3]
    assert len(fits.get_top_max_fits(df, None)) == 8 and len(fits.get_top_max_fits(df, 0)) == 8


def test_main_raises_when_all_files_are_bad(tmp_path):
    from metadamage_b200.main import main

    empty = tmp_path / "empty.txt"
    empty.write_text("")
    with pytest.raises(Exception, match="All files were bad"):
        main([empty], make_cfg(tmp_path))


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the CPU arm of the measurement contract): exactly one line on stdout, valid
    JSON, with the keys the driver reads; the oracle port is the timed thing, no GPU involved."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "taxid_damage_fits_per_sec" and d["unit"] == "fits/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data"):
        assert key in d, key
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["steps"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_split_text_at_taxid_boundaries():
    """The multi-GPU counts stage cuts the file where a new TaxID starts (no TaxID spans two pieces)."""
    lines = []
    for t in range(300):
        for r in range(1 + (t * 7) % 40):
            lines.append(f"{t * 3 + 1}\tname\trank\t{10 + t}\t5'\t{r}" + "\t1" * 16)
    text = ("\n".join(lines) + "\n").encode() * 1
    text = text * 1
    for n_parts in (1, 2, 3, 8):
        spans = counts.split_text_at_taxid_boundaries(text * 4 if False else text, n_parts)
        assert spans[0][0] == 0 and spans[-1][1] == len(text)
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        seen = []
        for a, b in spans:
            assert a == 0 or text[a - 1:a] == b"\n"
            ids = [ln.split(b"\t")[0] for ln in text[a:b].splitlines()]
            runs = [ids[i] for i in range(len(ids)) if i == 0 or ids[i] != ids[i - 1]]
            seen.append(set(runs))
        for i in range(len(seen)):
            for j in range(i + 1, len(seen)):
                assert not (seen[i] & seen[j])
    big = text * 3  # large enough to be cut
    assert len(counts.split_text_at_taxid_boundaries(big, 4)) >= 2


def test_decode_spans_and_pinned_file_reader(tmp_path):
    """The counts seam cuts tax_name / tax_rank out of the file bytes through (offset, length) spans: one vectorised
    gather for ASCII, string by string for anything else; the file text lands in a reusable staging buffer."""
    text = "1\tHomo sapiens\tspecies\n2\tÆgir é\tgenus\n3\t\tno rank\n".encode("utf-8")
    spans, pos = [], 0
    for line in text.split(b"\n")[:-1]:
        f = line.split(b"\t")
        o1 = pos + len(f[0]) + 1
        o2 = o1 + len(f[1]) + 1
        spans.append(((o1, len(f[1])), (o2, len(f[2]))))
        pos += len(line) + 1
    names = counts._decode_spans(text, np.array([s[0] for s in spans]))
    ranks = counts._decode_spans(np.frombuffer(text, np.uint8), np.array([s[1] for s in spans]))
    assert names == ["Homo sapiens", "Ægir é", ""] and ranks == ["species", "genus", "no rank"]
    assert counts._decode_spans(text, np.zeros((0, 2), np.int64)) == []
    assert counts._decode_spans(b"abc def", np.array([[0, 3], [4, 3]])) == ["abc", "def"]  # the ASCII fast path
    path = tmp_path / "table.txt"
    path.write_bytes(text * 1000)
    first = counts.read_file_bytes(str(path))
    assert first.dtype == np.uint8 and first.tobytes() == text * 1000
    path.write_bytes(text)
    again = counts.read_file_bytes(str(path))  # a shorter file in the same buffer
    assert again.tobytes() == text
    # the TaxID-boundary split takes the byte array as well as bytes
    big = b"".join(f"{t}\tn\tr\t10\t5'\t1".encode() + b"\t1" * 16 + b"\n" for t in range(3000) for _ in range(3))
    assert counts.split_text_at_taxid_boundaries(big, 3) == counts.split_text_at_taxid_boundaries(np.frombuffer(big, np.uint8), 3)


def test_bench_workloads_follow_baseline_configs():
    """N = 1 is BASELINE config 2 (10 000 fitted TaxIDs, seed 20240001); N > 1 steps over config 3's per-GPU share
    (seed 20240002, 125 000 TaxIDs per GPU = 1M over 8 GPUs), the same description for both arms."""
    import argparse
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench

    one = bench.workload_config(argparse.Namespace(max_position=15, taxa_per_gpu=10_000, inflight=1), 1)
    assert "cfg2" in one["workload"] and "20240001" in one["workload"] and one["taxa_per_gpu"] == 10_000
    eight = bench.workload_config(argparse.Namespace(max_position=15, taxa_per_gpu=125_000, inflight=1), 8)
    assert "cfg3" in eight["workload"] and "20240002" in eight["workload"] and "over 8 GPUs" in eight["workload"]
    assert eight["taxa_per_gpu"] * 8 == 1_000_000 and "model" not in eight
    src = open(os.path.join(root, "bench.py")).read()
    assert src.count("125_000") >= 2  # the default of both arms


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """bench.py --dump-outputs: every array lands as <name>.npy holding finite numbers only (NaN / inf marked in a
    companion file); a group beyond the byte budget is cut to the same seeded rows in each of its arrays, and the
    files stay within the budget."""
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    noise = np.linspace(0, 1, 300).reshape(100, 3)
    noise[[3, 7], 1] = np.nan
    noise[9] = [np.inf, -np.inf, np.nan]
    taxa = {"fit_D_max": np.linspace(0, 1, 100), "fit_median": np.ones((100, 30), np.float32), "counts_noise": noise}
    rows = {"counts_f_fwd": np.arange(50_000, dtype=np.float32), "counts_z": np.arange(50_000, dtype=np.float64) % 31}
    budget = 200_000
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), [taxa, rows], budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["counts_f_fwd.npy", "counts_noise.npy", "counts_noise_nonfinite.npy", "counts_z.npy", "fit_D_max.npy", "fit_median.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget
    for f in files:
        a = np.load(tmp_path / "a" / f)
        assert a.dtype in (np.float32, np.float64) and np.all(np.isfinite(a)), f
        assert np.array_equal(a, np.load(tmp_path / "b" / f))
    assert np.array_equal(np.load(tmp_path / "a" / "fit_median.npy"), taxa["fit_median"])  # the first group fits whole
    # NaN / inf entries are written as 0 and marked: 1 NaN, 2 +inf, 3 -inf
    code = np.load(tmp_path / "a" / "counts_noise_nonfinite.npy")
    want = np.zeros((100, 3), np.float32)
    want[[3, 7], 1] = 1
    want[9] = [2, 3, 1]
    assert np.array_equal(code, want)
    ok = want == 0
    assert np.array_equal(np.load(tmp_path / "a" / "counts_noise.npy")[ok], noise[ok])
    assert np.all(np.load(tmp_path / "a" / "counts_noise.npy")[~ok] == 0)
    f_fwd, z = np.load(tmp_path / "a" / "counts_f_fwd.npy"), np.load(tmp_path / "a" / "counts_z.npy")
    assert 0 < len(f_fwd) < 50_000 and np.all(np.diff(f_fwd) > 0)
    assert np.array_equal(z, f_fwd.astype(np.int64) % 31)  # the same rows in both arrays
