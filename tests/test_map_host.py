"""Host side of the MAP-only screening mode (no GPU): struct layout against the header, the table built from a
result array, and the `--map-only` switch of the CLI and the per-file loop."""
import logging
import os
import subprocess

import numpy as np
import pandas as pd
from typer.testing import CliRunner

from conftest import ROOT
from metadamage.cli import cli_app
from metadamage_b200 import fits
from metadamage_b200._abi import FIT_COV_INVALID, FIT_FAILED, FIT_MAP_NOT_CONVERGED, MAP_RESULT_DTYPE, MAP_RUN_DTYPE
from test_host import make_cfg


def test_map_struct_layouts_match_header(tmp_path):
    fields = ["loglik", "flags"]
    rfields = ["D_max", "lambda_LR_z", "normalized_noise", "N_z1_forward", "y_sum_total", "run"]
    src = tmp_path / "sz.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "mdg.h"\nint main(){printf("%zu %zu'
        + " %zu" * (len(fields) + len(rfields)) + '\\n",sizeof(mdg_map_run),sizeof(mdg_map_result)'
        + "".join(f",offsetof(mdg_map_run,{f})" for f in fields)
        + "".join(f",offsetof(mdg_map_result,{f})" for f in rfields) + ");return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    sizes = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [MAP_RUN_DTYPE.itemsize, MAP_RESULT_DTYPE.itemsize] + [MAP_RUN_DTYPE.fields[f][1] for f in fields] + \
        [MAP_RESULT_DTYPE.fields[f][1] for f in rfields]
    assert MAP_RUN_DTYPE.itemsize == 104 and MAP_RESULT_DTYPE.itemsize == 832


def hand_built(n=4):
    res = np.zeros(n, MAP_RESULT_DTYPE)
    res["tax_id"] = np.arange(n) + 100
    res["D_max"] = np.linspace(0.1, 0.4, n)
    res["lambda_LR"] = np.arange(n) * 10.0
    res["N_sum_total"] = 1000 + np.arange(n)
    res["run"]["q"] = np.arange(n)[:, None] * 0.01 + np.arange(6)[None, :] * 0.1
    res["run"]["loglik"] = -5.0
    res["status"] = [0, FIT_FAILED, FIT_MAP_NOT_CONVERGED | FIT_COV_INVALID, FIT_COV_INVALID][:n]
    dense = dict(tax_id=res["tax_id"].copy(), tax_name=np.array(["a", "b", "c", "d"][:n], object),
                 tax_rank=np.array(["species"] * n, object), N_alignments=np.arange(n, dtype=np.uint32) + 50)
    return res, dense


def test_make_df_map_results_columns_dtypes_and_drops(tmp_path, caplog):
    res, dense = hand_built()
    cfg = make_cfg(tmp_path)
    cfg.add_filename("x/sample.txt")
    with caplog.at_level(logging.WARNING):
        df = fits.make_df_map_results(res, dense, cfg)
    assert "no valid fit for tax_id 101" in caplog.text
    assert list(df.columns) == fits.MAP_RESULT_COLUMNS
    assert fits.MAP_RESULT_COLUMNS[:4] == ["tax_id", "tax_name", "tax_rank", "N_alignments"]
    assert fits.MAP_RESULT_COLUMNS[-2:] == ["valid", "shortname"]
    assert list(df["tax_id"]) == [100, 102, 103]
    assert df["valid"].tolist() == [True, False, False] and df["valid"].dtype == bool
    for col in ("tax_id", "tax_name", "tax_rank", "shortname"):
        assert isinstance(df[col].dtype, pd.CategoricalDtype), col
    for col in ("N_alignments", "N_z1_forward", "N_sum_total", "y_sum_total"):
        assert df[col].dtype == np.uint32, col
    for col in ("D_max", "q", "null_q", "lambda_LR", "lambda_LR_z", "forward_D_max", "normalized_noise"):
        assert df[col].dtype == np.float32, col
    np.testing.assert_allclose(df["q"], res["run"][[0, 2, 3], 0]["q"].astype(np.float32))
    np.testing.assert_allclose(df["null_q"], res["run"][[0, 2, 3], 1]["q"].astype(np.float32))
    assert df["N_sum_total"].tolist() == [1000, 1002, 1003] and df["N_alignments"].tolist() == [50, 52, 53]
    assert df["shortname"].tolist() == ["sample"] * 3


def test_make_df_map_results_empty(tmp_path):
    cfg = make_cfg(tmp_path)
    cfg.add_filename("x/sample.txt")
    dense = dict(tax_id=np.zeros(0, np.int64), tax_name=np.zeros(0, object), tax_rank=np.zeros(0, object),
                 N_alignments=np.zeros(0, np.uint32))
    df = fits.make_df_map_results(np.zeros(0, MAP_RESULT_DTYPE), dense, cfg)
    assert len(df) == 0 and list(df.columns) == fits.MAP_RESULT_COLUMNS


def test_cli_lists_map_only():
    result = CliRunner().invoke(cli_app, ["fit", "--help"])
    assert result.exit_code == 0 and "--map-only" in result.stdout


def test_map_results_path_and_metadata_unchanged(tmp_path):
    cfg = make_cfg(tmp_path)
    cfg.add_filename("x/y/KapK-12-1.sorted.txt")
    assert cfg.filename_map_results == tmp_path / "map_results" / "KapK-12-1.parquet"
    assert not any("map" in key for key in cfg.to_dict())  # the switch is an argument, not configuration


def test_main_map_only_calls_get_map_fits(tmp_path, monkeypatch):
    from metadamage_b200 import counts, main as main_mod

    calls = []
    path = tmp_path / "data.txt"
    path.write_text("x\n")
    monkeypatch.setattr(counts, "load_counts", lambda cfg: pd.DataFrame({"tax_id": [1]}))
    monkeypatch.setattr(fits, "get_map_fits", lambda df, cfg: calls.append("map"))
    monkeypatch.setattr(fits, "get_fits", lambda df, cfg: calls.append("fits"))
    cfg = make_cfg(tmp_path / "out")
    main_mod.main([path], cfg, map_only=True)
    assert calls == ["map"]
    main_mod.main([path], cfg)
    assert calls == ["map", "fits"]


def test_cli_map_only_reaches_main(tmp_path, monkeypatch):
    from metadamage_b200 import main as main_mod

    seen = {}
    monkeypatch.setattr(main_mod, "main", lambda filenames, cfg, map_only=False: seen.update(map_only=map_only))
    path = tmp_path / "data.txt"
    path.write_text("x\n")
    assert CliRunner().invoke(cli_app, ["fit", str(path), "--map-only", "--out-dir", str(tmp_path)]).exit_code == 0
    assert seen == {"map_only": True}
    assert CliRunner().invoke(cli_app, ["fit", str(path), "--out-dir", str(tmp_path)]).exit_code == 0
    assert seen == {"map_only": False}


def test_public_names_reexported():
    import metadamage.fits as mf

    for name in ("MAP_RESULT_COLUMNS", "map_dense", "make_df_map_results", "compute_map_fits", "get_map_fits"):
        assert getattr(mf, name) is getattr(fits, name)
