"""Generate the golden fixtures under tests/golden/ by running the REFERENCE's own functions.

Run with a checkout of the reference project (no GPU needed):

    python tests/golden/make_golden.py /path/to/reference

The reference imports numpyro / jax / dask / ... at module level; none of them is installable
offline, so they are replaced by inert stub modules here. Only reference functions that are
pure pandas / numpy are then executed:

  counts.py : add_reference_counts, add_error_rates, make_position_1_indexed,
              make_reverse_position_negative, replace_nans_with_zeroes, compute_y_sum_total,
              filter_cut_based_on_cfg, sort_by_alignments            (counts.py:86-209)
              (the dask groupby/merge of add_y_sum_counts, counts.py:192-204, is replaced by the
              equivalent pandas groupby/merge; everything else is the reference's code)
  fits.py   : get_lppd_and_waic (with compute_log_likelihood monkey-patched to return a fixed
              matrix), compute_n_sigma, compute_assymmetry_combined_vs_forwardreverse,
              add_noise_estimates, group_to_numpyro_data              (fits.py:147-227, 359-419)

              extract_top_max_fits / get_top_max_fits                  (fits.py:736-751)

  dashboard/fit_results.py : FitResults' pandas half (derived columns, ranges, marker sizes, filter,
              single-TaxID fetches; lines 74-239), loaded stand-alone without Dash / Plotly

Outputs: counts_golden.npz, fits_golden.npz, topn_golden.npz, lookups_golden.npz (small; committed).
"""
import importlib
import os
import sys
import tempfile
import types
import warnings

import numpy as np
import pandas as pd

REF = None  # the reference checkout, from the command line
HERE = os.path.dirname(os.path.abspath(__file__))


class _Anything:
    """Inert stand-in: callable, attribute-able, usable as decorator / base class."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        if len(a) == 1 and callable(a[0]) and not k:
            return a[0]  # decorator use
        return _Anything()

    def __getattr__(self, name):
        return _Anything()


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    mod.__getattr__ = lambda attr: _Anything()  # type: ignore[attr-defined]
    sys.modules[name] = mod
    return mod


def install_stubs():
    for name in [
        "dask", "dask.dataframe", "dask.diagnostics", "dask.distributed", "jax", "jax.numpy", "jax.random",
        "numpyro", "numpyro.distributions", "numpyro.infer", "timeout_decorator", "matplotlib",
        "matplotlib.pyplot", "PyPDF2", "dill", "toml", "plotly", "dash",
    ]:
        _stub(name)
    sys.modules["jax"].jit = lambda f=None, **k: f if f is not None else (lambda g: g)
    sys.modules["timeout_decorator"].TimeoutError = type("TimeoutError", (Exception,), {})
    sys.modules["numpyro"].enable_x64 = lambda *a, **k: None

    class _Base:
        def __init__(self, *a, **k):
            pass

    _stub("click_help_colors", HelpColorsCommand=_Base, HelpColorsGroup=_Base)


def load_reference():
    install_stubs()
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(tempfile.gettempdir())  # the reference's logger writes ./logs/
    try:
        counts = importlib.import_module("metadamage.counts")
        fits = importlib.import_module("metadamage.fits")
        utils = importlib.import_module("metadamage.utils")
    finally:
        os.chdir(cwd)
    # scipy / numpy probe sys.modules for jax and dask; the reference modules already hold
    # their own references to the stubs, so drop them again
    for name in [m for m in sys.modules if m.split(".")[0] in ("jax", "dask")]:
        del sys.modules[name]
    return counts, fits, utils


class Cfg:
    def __init__(self, fwd="CT", rev="GA", min_alignments=10, min_y_sum=10):
        self.substitution_bases_forward = fwd
        self.substitution_bases_reverse = rev
        self.min_alignments = min_alignments
        self.min_y_sum = min_y_sum
        self.shortname = "golden"


def read_sample(path, counts):
    """20-column legacy layout with header -> the reference's 22 columns (counts.py:37-45)."""
    df = pd.read_csv(path, sep="\t")
    df.columns = ["tax_id", "N_alignments", "strand", "position"] + list(df.columns[4:])
    df.insert(1, "tax_name", "name")
    df.insert(2, "tax_rank", "rank")
    assert list(df.columns) == counts.columns
    return df


def reference_counts(df, cfg, counts):
    """counts.py:229-264 with pandas in place of dask."""
    fwd, rev = cfg.substitution_bases_forward, cfg.substitution_bases_reverse
    df = (
        df.copy()
        .pipe(counts.add_reference_counts, ref=fwd[0])
        .pipe(counts.add_reference_counts, ref=rev[0])
        .pipe(counts.add_error_rates, ref=fwd[0], obs=fwd[1])
        .pipe(counts.add_error_rates, ref=rev[0], obs=rev[1])
        .pipe(counts.make_position_1_indexed)
        .pipe(counts.make_reverse_position_negative)
        .pipe(counts.replace_nans_with_zeroes)
    )
    ds = (
        df.groupby("tax_id")[list(df.columns)]
        .apply(counts.compute_y_sum_total, cfg)
        .rename("y_sum_total")
        .reset_index()
    )
    df = pd.merge(df, ds, on=["tax_id"])
    df = (
        df.pipe(counts.filter_cut_based_on_cfg, cfg)
        .reset_index(drop=True)
        .pipe(counts.sort_by_alignments)
        .reset_index(drop=True)
    )
    return df


def make_counts_golden(counts):
    out = {}
    cases = {
        "ancient_CT_GA": ("data_ancient.txt", Cfg()),
        "control_CT_GA": ("data_control.txt", Cfg()),
        "ancient_GA_CT": ("data_ancient.txt", Cfg(fwd="GA", rev="CT")),
        "control_cut": ("data_control.txt", Cfg(min_alignments=200000, min_y_sum=7000)),
        "ancient_same_ref": ("data_ancient.txt", Cfg(fwd="CT", rev="CA")),
    }
    for name, (fname, cfg) in cases.items():
        df_in = read_sample(os.path.join(REF, "data", "input", fname), counts)
        df = reference_counts(df_in, cfg, counts)
        fwd, rev = cfg.substitution_bases_forward, cfg.substitution_bases_reverse
        out[f"{name}__columns"] = np.array(list(df.columns))
        out[f"{name}__cfg"] = np.array([fwd, rev, str(cfg.min_alignments), str(cfg.min_y_sum)])
        out[f"{name}__tax_id"] = df["tax_id"].to_numpy(np.int64)
        out[f"{name}__N_alignments"] = df["N_alignments"].to_numpy(np.int64)
        out[f"{name}__position"] = df["position"].to_numpy(np.int64)
        out[f"{name}__n_fwd_ref"] = df[fwd[0]].to_numpy(np.int64)
        out[f"{name}__n_rev_ref"] = df[rev[0]].to_numpy(np.int64)
        out[f"{name}__f_fwd"] = df[f"f_{fwd}"].to_numpy(np.float64)
        out[f"{name}__f_rev"] = df[f"f_{rev}"].to_numpy(np.float64)
        out[f"{name}__y_sum_total"] = df["y_sum_total"].to_numpy(np.int64)
        out[f"{name}__k_fwd"] = df[fwd].to_numpy(np.int64)
        out[f"{name}__k_rev"] = df[rev].to_numpy(np.int64)
    np.savez_compressed(os.path.join(HERE, "counts_golden.npz"), **out)
    return out


def make_fits_golden(counts, fits):
    from scipy import stats

    rng = np.random.default_rng(12345)
    out = {}
    df_in = read_sample(os.path.join(REF, "data", "input", "data_control.txt"), counts)
    cfg = Cfg()
    df = reference_counts(df_in, cfg, counts)
    group = df[df.tax_id == 1]
    data = fits.group_to_numpyro_data(group, cfg)
    out["data_z"], out["data_y"], out["data_N"] = data["z"], data["y"], data["N"]

    # a fixed "posterior": 200 draws around the MAP of control tax 1
    S = 200
    q = np.clip(rng.normal(0.34, 0.1, S), 0.05, 0.9)
    A = np.clip(rng.normal(0.007, 0.002, S), 1e-4, 0.5)
    c = np.clip(rng.normal(0.0085, 0.001, S), 1e-4, 0.5)
    phi = 2 + rng.gamma(4.0, 15.0, S)
    out["theta_pmd"] = np.stack([q, A, c, phi], 1)
    z = np.abs(data["z"])
    Dz = A[:, None] * (1 - q[:, None]) ** (z[None, :] - 1) + c[:, None]
    lp_pmd = stats.betabinom.logpmf(data["y"][None, :], data["N"][None, :], Dz * phi[:, None], (1 - Dz) * phi[:, None])
    qn = np.clip(rng.normal(0.0095, 0.001, S), 1e-4, 0.5)
    phin = 2 + rng.gamma(4.0, 12.0, S)
    out["theta_null"] = np.stack([qn, phin], 1)
    lp_null = stats.betabinom.logpmf(data["y"][None, :], data["N"][None, :], qn[:, None] * phin[:, None],
                                     (1 - qn[:, None]) * phin[:, None])
    out["logprob_pmd"], out["logprob_null"] = lp_pmd, lp_null

    # fits.get_lppd_and_waic with the log-likelihood matrix injected (fits.py:147-172)
    def waic_of(mat):
        fits.compute_log_likelihood = lambda mcmc, data_: mat
        return fits.get_lppd_and_waic(None, None)

    d_pmd, d_null = waic_of(lp_pmd), waic_of(lp_null)
    for key in ("lppd_i", "pWAIC_i", "waic_i"):
        out[f"pmd_{key}"], out[f"null_{key}"] = d_pmd[key], d_null[key]
    out["pmd_waic"], out["null_waic"] = d_pmd["waic"], d_null["waic"]
    out["n_sigma"] = fits.compute_n_sigma(d_pmd, d_null)  # fits.py:194-201
    d_f, d_r = waic_of(lp_pmd[:, :15] * 0.97), waic_of(lp_pmd[:, 15:] * 1.02)
    out["fwd_waic_i"], out["rev_waic_i"] = d_f["waic_i"], d_r["waic_i"]
    out["asymmetry"] = fits.compute_assymmetry_combined_vs_forwardreverse(d_pmd, d_f, d_r)  # fits.py:204-227

    # noise estimates on every TaxID of both sample files (fits.py:359-376)
    off = [a + b for a in "ACGT" for b in "ACGT" if a != b]
    noise_in, noise_out = [], []
    for fname in ("data_ancient.txt", "data_control.txt"):
        dfc = reference_counts(read_sample(os.path.join(REF, "data", "input", fname), counts), cfg, counts)
        for _, grp in dfc.groupby("tax_id", sort=False):
            fr = {}
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                fits.add_noise_estimates(grp, fr)
            noise_in.append(grp[off].to_numpy(np.int64))
            noise_out.append([fr["normalized_noise"], fr["normalized_noise_forward"], fr["normalized_noise_reverse"]])
    out["noise_mism12"] = np.stack(noise_in)
    out["noise_expected"] = np.array(noise_out)

    # median / hpdi restatement target: numpyro.diagnostics.hpdi is not importable; pin np.median only
    x = rng.integers(0, 50, (1000, 4)) / 49.0
    out["median_in"], out["median_out"] = x, np.median(x, axis=0)
    np.savez_compressed(os.path.join(HERE, "fits_golden.npz"), **out)
    return out


def make_topn_golden(fits):
    """fits.extract_top_max_fits / get_top_max_fits (fits.py:736-751) on df_counts-like frames with many
    ties in the per-TaxID sums: the selected TaxIDs in df_counts order."""
    rng = np.random.default_rng(20240018)
    out = {}
    for case, (n_tax, levels) in enumerate([(200, 12), (64, 3), (1000, 40)]):
        tax = rng.permutation(rng.choice(10 ** 6, n_tax, replace=False)).astype(np.int64)
        nal = rng.choice(np.sort(rng.integers(10, 5000, levels)), n_tax).astype(np.uint32)
        rows = rng.choice([30, 30, 30, 28, 16, 2], n_tax)
        order = np.lexsort((-tax, -nal.astype(np.int64)))  # counts.sort_by_alignments: N_alignments desc, tax_id desc
        tax, nal, rows = tax[order], nal[order], rows[order]
        tax_row = np.repeat(tax, rows)
        nal_row = np.repeat(nal, rows)
        df = pd.DataFrame({"tax_id": pd.Series(tax_row).astype("category"), "N_alignments": nal_row.astype(np.uint32),
                           "position": np.concatenate([np.arange(r) for r in rows]).astype(np.int8)})
        out[f"case{case}_tax_id_row"] = tax_row
        out[f"case{case}_n_alignments_row"] = nal_row
        for n_top in (1, 5, 17, n_tax // 2, n_tax - 1, n_tax, n_tax + 7):
            top = fits.get_top_max_fits(df, n_top)
            out[f"case{case}_top{n_top}"] = pd.unique(top["tax_id"]).astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "topn_golden.npz"), **out)
    return out


def load_reference_fit_results():
    """dashboard/fit_results.py as a stand-alone module: the dashboard package itself needs Dash, Plotly,
    ete3, ...; only FitResults' pandas half is executed, with dashboard.utils loaded from its file."""
    import importlib.util

    class Ctx(_Anything):
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    for name in ["about_time", "dill", "plotly.express", "plotly.graph_objects", "plotly.io", "PIL"]:
        _stub(name)
    sys.modules["about_time"].about_time = lambda *a, **k: Ctx()
    d3 = ["#1F77B4", "#FF7F0E", "#2CA02C", "#D62728", "#9467BD", "#8C564B", "#E377C2", "#7F7F7F", "#BCBD22", "#17BECF"]
    sys.modules["plotly.express"].colors = types.SimpleNamespace(qualitative=types.SimpleNamespace(D3=d3))  # _set_cmap
    sys.modules["plotly"].express = sys.modules["plotly.express"]  # `import plotly.express as px` goes through the parent
    import joblib

    class _NoMemory:  # joblib.Memory would write ./memoization
        def __init__(self, *a, **k):
            pass

        def cache(self, f):
            return f

    real_memory, joblib.Memory = joblib.Memory, _NoMemory

    def from_file(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    dash_pkg = types.ModuleType("metadamage.dashboard")
    dash_pkg.__path__ = []
    sys.modules["metadamage.dashboard"] = dash_pkg
    importlib.import_module("metadamage").dashboard = dash_pkg
    dash_pkg.utils = from_file("metadamage.dashboard.utils", os.path.join(REF, "metadamage", "dashboard", "utils.py"))
    mod = from_file("metadamage.dashboard.fit_results", os.path.join(REF, "metadamage", "dashboard", "fit_results.py"))
    joblib.Memory = real_memory
    return mod


def make_lookups_golden(fit_results_mod):
    """The reference's FitResults (dashboard/fit_results.py:74-239) on result files written with the
    reference's column schema: derived columns, ranges, marker sizes, filters, single-TaxID fetches."""
    import shutil
    import tempfile

    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from metadamage_b200 import fits as our_fits, io as our_io  # the writers under test
    rng = np.random.default_rng(20240019)
    folder = tempfile.mkdtemp(prefix="mdg_lookups_")
    out = {}
    try:
        frames, preds = [], []
        for shortname, n in (("sampleA", 40), ("sampleB", 25)):
            tax = rng.choice(10 ** 5, n, replace=False).astype(np.int64)
            df = pd.DataFrame({c: rng.normal(1.0, 1.0, n).astype(np.float32) for c in our_fits.FIT_RESULT_COLUMNS})
            df["tax_id"] = tax
            df["tax_name"] = [f"name{t % 7}" for t in tax]
            df["tax_rank"] = [("species", "genus", "family")[t % 3] for t in tax]
            for c in ("N_alignments", "N_z1_forward", "N_z1_reverse", "N_sum_forward", "N_sum_reverse", "N_sum_total",
                      "y_sum_forward", "y_sum_reverse", "y_sum_total"):
                df[c] = rng.integers(0 if c == "N_sum_total" else 1, 10 ** 6, n).astype(np.uint32)
            df.loc[0, "N_sum_total"] = 0  # log10 -> -inf, must be ignored by the ranges
            df.loc[1, "n_sigma"] = np.nan
            df["shortname"] = shortname
            for c in ("tax_id", "tax_name", "tax_rank", "shortname"):
                df[c] = df[c].astype("category")
            our_io.Parquet(os.path.join(folder, "fit_results", f"{shortname}.parquet")).save(df, metadata={"shortname": shortname})
            pr = pd.DataFrame({"tax_id": np.repeat(tax, 30), "position": np.tile(np.r_[1:16, -1:-16:-1], n).astype(np.int8),
                               "median": rng.random(30 * n).astype(np.float32), "hdpi_lower": rng.random(30 * n).astype(np.float32),
                               "hdpi_upper": rng.random(30 * n).astype(np.float32)})
            pr["shortname"] = shortname
            for c in ("tax_id", "shortname"):
                pr[c] = pr[c].astype("category")
            our_io.Parquet(os.path.join(folder, "fit_predictions", f"{shortname}.parquet")).save(pr, metadata={"shortname": shortname})
            cn = pd.DataFrame({"tax_id": np.repeat(tax, 30), "position": np.tile(np.r_[1:16, -1:-16:-1], n).astype(np.int8),
                               "N_alignments": np.repeat(df["N_alignments"].to_numpy(), 30)})
            cn["tax_id"] = cn["tax_id"].astype("category")
            our_io.Parquet(os.path.join(folder, "counts", f"{shortname}.parquet")).save(cn, metadata={"shortname": shortname})
            frames.append(df)
        cwd = os.getcwd()
        os.chdir(tempfile.gettempdir())
        try:
            fr = fit_results_mod.FitResults(folder)
        finally:
            os.chdir(cwd)
        d = fr.df_fit_results
        out["folder_tables"] = np.array(["fit_results", "fit_predictions", "counts"])
        for c in ("N_alignments_log10", "N_alignments_sqrt", "N_sum_total_log10", "size"):
            out[f"col_{c}"] = d[c].to_numpy(np.float64).copy()
        out["tax_id_order"] = d["tax_id"].to_numpy(np.int64)
        out["range_keys"] = np.array(sorted(fr.ranges))
        out["range_values"] = np.array([fr.ranges[k] for k in sorted(fr.ranges)], dtype=np.float64)
        out["max_of_size"] = np.float64(fr.max_of_size)
        for tr in ("identity", "log10", "constant"):
            fr.set_marker_size(tr, 12)
            out[f"size_{tr}"] = fr.df_fit_results["size"].to_numpy(np.float64).copy()  # (to_numpy is a view; the next call overwrites it)
            out[f"max_of_size_{tr}"] = np.float64(fr.max_of_size)
        fr.set_marker_size("sqrt")
        some = [int(t) for t in d["tax_id"].to_numpy()[[3, 9, 44]]]
        filters = [
            {"shortnames": ["sampleA"], "n_sigma": (0.0, 2.5)},
            {"shortname": "sampleB", "N_alignments": (2.0, 5.5), "D_max": (-1.0, 3.0)},
            {"tax_ids": some},
            {"tax_id": some[0], "y_sum_total": (-1.0, 7.0)},
            {"tax_ranks": ["species", "genus"], "tax_names": ["name1", "name2", "name3"], "q_mean": None},
            {"tax_rank": "'family'", "N_sum_total": (0.0, 6.0)},
        ]
        out["n_filters"] = np.int64(len(filters))
        import json
        out["filters_json"] = np.array(json.dumps(filters))
        for i, f in enumerate(filters):
            out[f"filter{i}_index"] = fr.filter(f).index.to_numpy(np.int64)
        out["single_pred_tax"] = np.int64(some[1])
        out["single_pred_median"] = fr.get_single_fit_prediction("sampleA", some[1])["median"].to_numpy(np.float64)
        out["single_count_rows"] = np.int64(len(fr.get_single_count_group("sampleA", some[1])))
        # the files themselves travel with the fixture (tiny)
        import io as _io
        import zipfile
        buf = _io.BytesIO()
        with zipfile.ZipFile(buf, "w", zipfile.ZIP_DEFLATED) as z:
            for root, _, files in os.walk(folder):
                for fn in files:
                    full = os.path.join(root, fn)
                    z.write(full, os.path.relpath(full, folder))
        out["files_zip"] = np.frombuffer(buf.getvalue(), dtype=np.uint8)
    finally:
        shutil.rmtree(folder, ignore_errors=True)
    np.savez_compressed(os.path.join(HERE, "lookups_golden.npz"), **out)
    return out


def main():
    global REF
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_golden.py /path/to/reference")
    REF = os.path.abspath(sys.argv[1])
    counts, fits, utils = load_reference()
    c = make_counts_golden(counts)
    f = make_fits_golden(counts, fits)
    t = make_topn_golden(fits)
    print("topn_golden.npz:", len(t), "arrays")
    lk = make_lookups_golden(load_reference_fit_results())
    print("lookups_golden.npz:", len(lk), "arrays")
    print("counts_golden.npz:", len(c), "arrays;", "fits_golden.npz:", len(f), "arrays")
    print("n_sigma", f["n_sigma"], "asymmetry", f["asymmetry"])
    print("noise", f["noise_expected"])


if __name__ == "__main__":
    main()
