"""Host side of the profile intervals of the MAP-only mode (no GPU): struct layouts against the header, the columns
the table builder appends, the `--profile-interval` switch and the cache key it adds."""
import os
import subprocess

import numpy as np
import pandas as pd
from typer.testing import CliRunner

from conftest import ROOT
from metadamage.cli import cli_app
from metadamage_b200 import fits, io
from metadamage_b200._abi import (FIT_FAILED, MAP_INTERVAL_DTYPE, PROFILE_AT_BOUND, PROFILE_END_DTYPE, PROFILE_FAILED)
from test_host import make_cfg
from test_map_host import hand_built


def test_profile_struct_layouts_match_header(tmp_path):
    efields = ["D", "logp", "n_eval", "flags"]
    ifields = ["status", "level", "threshold", "end"]
    src = tmp_path / "sz.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "mdg.h"\nint main(){printf("%zu %zu'
        + " %zu" * (len(efields) + len(ifields)) + '\\n",sizeof(mdg_profile_end),sizeof(mdg_map_interval)'
        + "".join(f",offsetof(mdg_profile_end,{f})" for f in efields)
        + "".join(f",offsetof(mdg_map_interval,{f})" for f in ifields) + ");return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    sizes = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [PROFILE_END_DTYPE.itemsize, MAP_INTERVAL_DTYPE.itemsize] + \
        [PROFILE_END_DTYPE.fields[f][1] for f in efields] + [MAP_INTERVAL_DTYPE.fields[f][1] for f in ifields]
    assert PROFILE_END_DTYPE.itemsize == 56 and MAP_INTERVAL_DTYPE.itemsize == 368


def test_make_df_map_results_interval_columns(tmp_path):
    res, dense = hand_built()
    iv = np.zeros(len(res), MAP_INTERVAL_DTYPE)
    iv["end"]["D"] = np.arange(len(res))[:, None, None] * 0.1 + np.arange(3)[None, :, None] * 0.01 + np.array([0.0, 0.5])
    iv["status"] = [0, FIT_FAILED, PROFILE_AT_BOUND, PROFILE_FAILED]
    cfg = make_cfg(tmp_path)
    cfg.add_filename("x/sample.txt")
    plain = fits.make_df_map_results(res, dense, cfg)
    df = fits.make_df_map_results(res, dense, cfg, iv)
    assert list(df.columns) == fits.MAP_RESULT_COLUMNS + fits.MAP_INTERVAL_COLUMNS
    assert df[fits.MAP_RESULT_COLUMNS].equals(plain)
    for col in fits.MAP_INTERVAL_COLUMNS[:-1]:
        assert df[col].dtype == np.float32, col
    assert df["interval_valid"].dtype == bool and df["interval_valid"].tolist() == [True, True, False]
    rows = [0, 2, 3]  # row 1 has no valid fit and is dropped
    np.testing.assert_array_equal(df["D_max_lower"], iv["end"][rows, 0, 0]["D"].astype(np.float32))
    np.testing.assert_array_equal(df["forward_D_max_upper"], iv["end"][rows, 1, 1]["D"].astype(np.float32))
    np.testing.assert_array_equal(df["reverse_D_max_lower"], iv["end"][rows, 2, 0]["D"].astype(np.float32))


def test_cli_lists_profile_interval_and_needs_map_only(tmp_path):
    result = CliRunner().invoke(cli_app, ["fit", "--help"])
    assert result.exit_code == 0 and "--profile-interval" in result.stdout
    path = tmp_path / "data.txt"
    path.write_text("x\n")
    result = CliRunner().invoke(cli_app, ["fit", str(path), "--profile-interval", "--out-dir", str(tmp_path)])
    assert result.exit_code == 2


def test_cli_profile_interval_reaches_main_only_when_set(tmp_path, monkeypatch):
    from metadamage_b200 import main as main_mod

    seen = []
    monkeypatch.setattr(main_mod, "main", lambda filenames, cfg, **kw: seen.append(kw))
    path = tmp_path / "data.txt"
    path.write_text("x\n")
    assert CliRunner().invoke(cli_app, ["fit", str(path), "--map-only", "--profile-interval", "--out-dir", str(tmp_path)]).exit_code == 0
    assert CliRunner().invoke(cli_app, ["fit", str(path), "--map-only", "--out-dir", str(tmp_path)]).exit_code == 0
    assert seen == [{"map_only": True, "profile_interval": True}, {"map_only": True}]


def test_main_passes_profile_interval_only_when_set(tmp_path, monkeypatch):
    from metadamage_b200 import counts, main as main_mod

    calls = []
    path = tmp_path / "data.txt"
    path.write_text("x\n")
    monkeypatch.setattr(counts, "load_counts", lambda cfg: pd.DataFrame({"tax_id": [1]}))
    monkeypatch.setattr(fits, "get_map_fits", lambda df, cfg, **kw: calls.append(kw))
    cfg = make_cfg(tmp_path / "out")
    main_mod.main([path], cfg, map_only=True, profile_interval=True)
    main_mod.main([path], cfg, map_only=True)
    assert calls == [{"profile_interval": True}, {}]


def test_cache_key_only_with_intervals(tmp_path, monkeypatch):
    """The metadata of map_results carries "profile_interval" only for a table with intervals; a cached table is
    reused only when that key matches, and --forced recomputes."""
    computed = []

    def fake(df_counts, cfg, n_fits=None, profile_interval=False):
        computed.append(profile_interval)
        return pd.DataFrame({"x": [1.0]})

    monkeypatch.setattr(fits, "compute_map_fits", fake)
    cfg = make_cfg(tmp_path)
    cfg.add_filename("x/sample.txt")
    fits.get_map_fits(None, cfg)
    assert "profile_interval" not in io.Parquet(cfg.filename_map_results).load_metadata()
    assert io.Parquet(cfg.filename_map_results).load_metadata() == cfg.to_dict()
    fits.get_map_fits(None, cfg)  # cached
    fits.get_map_fits(None, cfg, profile_interval=True)  # key differs: recompute
    assert io.Parquet(cfg.filename_map_results).load_metadata()["profile_interval"] == 0.68
    fits.get_map_fits(None, cfg, profile_interval=True)  # cached
    fits.get_map_fits(None, cfg)  # plain run after an interval run: recompute
    assert computed == [False, True, False]
    forced = make_cfg(tmp_path, forced=True)
    forced.add_filename("x/sample.txt")
    fits.get_map_fits(None, forced)
    assert computed == [False, True, False, False]
