"""Fits stage: df_counts -> (df_fit_results, df_fit_predictions), computed on the GPU(s).

Keeps the reference's seams `compute_fits(df_counts, cfg, mcmc_kwargs)` and
`get_fits(df_counts, cfg)` (fits.py:709-730, 754-807): same two DataFrames (columns, order,
dtypes; fits.py:242-293, 632-680), same parquet cache rules, same --max-fits selection
(fits.py:736-751). The per-TaxID Python/numpyro work (fits.py:428-469) and the
multiprocessing fan-out (fits.py:569-626) are replaced by `mdg_fit_batch` on each GPU's
contiguous share of the TaxID batch. The MAP fit (new) is written to fit_map/<shortname>.parquet
so that the two reference schemas stay unchanged.

`get_map_fits` / `compute_map_fits` are the MAP-only screening mode (`metadamage fit --map-only`): six MAP
fits per TaxID with Laplace uncertainties and a likelihood-ratio statistic through `mdg_map_batch`, no NUTS,
one table in map_results/<shortname>.parquet. With `profile_interval` (`--profile-interval`) the table also gets
profile intervals of D_max at level 0.68 through `mdg_map_profile` (MAP_INTERVAL_COLUMNS).
"""
import logging

import numpy as np
import pandas as pd

from . import _lib, io, utils
from ._abi import FIT_COV_INVALID, FIT_FAILED, FIT_MAP_NOT_CONVERGED, MAP_INTERVAL_DTYPE, MAP_RESULT_DTYPE, PROFILE_FAILED
from .counts import dense_from_df_counts, get_context
from .parallel import run_on_gpus

logger = logging.getLogger(__name__)

# column order of the reference's fit_result dict (fits.py:242-293, 317-356, 374-376)
FIT_RESULT_COLUMNS = [
    "tax_id", "tax_name", "tax_rank", "D_max", "n_sigma", "D_max_lower_hpdi", "D_max_upper_hpdi", "q_mean",
    "concentration_mean", "D_max_marginalized_mean", "N_alignments", "N_z1_forward", "N_z1_reverse",
    "N_sum_forward", "N_sum_reverse", "N_sum_total", "y_sum_forward", "y_sum_reverse", "y_sum_total",
    "n_sigma_forward", "D_max_forward", "q_mean_forward", "n_sigma_reverse", "D_max_reverse", "q_mean_reverse",
    "asymmetry", "normalized_noise", "normalized_noise_forward", "normalized_noise_reverse",
]
FIT_MAP_COLUMNS = ["map_A", "map_q", "map_c", "map_phi", "map_D_max", "map_logp", "map_null_q", "map_null_phi",
                   "map_null_logp"]

# the MAP-only table (map_results/<shortname>.parquet). D_max is A + c at the PMD mode, not the posterior predictive
# median of fit_results; lambda_LR_P / lambda_LR_z are a screening scale (the null model sits on the boundary A = 0 of
# the PMD model), not calibrated p-values.
MAP_RESULT_COLUMNS = [
    "tax_id", "tax_name", "tax_rank", "N_alignments", "N_z1_forward", "N_z1_reverse", "N_sum_forward", "N_sum_reverse",
    "N_sum_total", "y_sum_forward", "y_sum_reverse", "y_sum_total",
    "D_max", "D_max_std", "significance", "q", "q_std", "A", "A_std", "c", "c_std", "phi", "phi_std", "rho_Ac", "logp",
    "loglik",
    "null_q", "null_q_std", "null_phi", "null_phi_std", "null_logp", "null_loglik",
    "lambda_LR", "lambda_LR_P", "lambda_LR_z",
    "forward_D_max", "forward_D_max_std", "forward_lambda_LR", "reverse_D_max", "reverse_D_max_std", "reverse_lambda_LR",
    "normalized_noise", "normalized_noise_forward", "normalized_noise_reverse", "valid", "shortname",
]
# columns taken from one run's record: column -> (run kind, mdg_map_run field)
_MAP_RUN_COLUMNS = {
    **{name: (0, name) for name in ("q", "q_std", "A", "A_std", "c", "c_std", "phi", "phi_std", "logp", "loglik")},
    **{"null_" + name: (1, name) for name in ("q", "q_std", "phi", "phi_std", "logp", "loglik")},
}
# profile intervals of D_max appended to the MAP-only table with --profile-interval, at the level of fit_results' HPDI
# (fits.py:119). interval_valid: both all-position ends were found (an end at a bound included).
PROFILE_INTERVAL_LEVEL = 0.68
MAP_INTERVAL_COLUMNS = ["D_max_lower", "D_max_upper", "forward_D_max_lower", "forward_D_max_upper", "reverse_D_max_lower",
                        "reverse_D_max_upper", "interval_valid"]


def mcmc_kwargs_default():
    """fits.py:792-799."""
    return dict(progress_bar=False, num_warmup=500, num_samples=1000, num_chains=1, chain_method="sequential")


def fit_config_from(cfg, mcmc_kwargs=None):
    kw = dict(mcmc_kwargs_default(), **(mcmc_kwargs or {}))
    if kw.get("num_chains", 1) != 1:
        raise ValueError("only num_chains=1 is supported (as in the reference, fits.py:796)")
    return _lib.default_config(num_warmup=int(kw["num_warmup"]), num_samples=int(kw["num_samples"]),
                               seed=int(getattr(cfg, "seed", 0)))


def extract_top_max_fits(df_counts, max_fits):
    """fits.py:736-744: the TaxIDs with the largest sum of N_alignments over their rows."""
    top = df_counts.groupby("tax_id", observed=True)["N_alignments"].sum().nlargest(max_fits).index
    return df_counts[df_counts["tax_id"].isin(top)]


def get_top_max_fits(df_counts, n_fits):
    if n_fits is not None and n_fits > 0:
        return extract_top_max_fits(df_counts, n_fits)
    return df_counts


def fit_dense(dense, cfg, fit_cfg, n_gpus=1):
    """Run mdg_fit_batch over `n_gpus` contiguous shares of the dense batch; host-side concat."""
    n_tax = len(dense["tax_id"])
    R = dense["k"].shape[1]
    if n_tax == 0:
        from ._abi import FIT_RESULT_DTYPE

        e = np.zeros((0, R), np.float32)
        return dict(result=np.zeros(0, FIT_RESULT_DTYPE), median=e, hpdi_lo=e.copy(), hpdi_hi=e.copy())
    n_dev = max(1, min(int(n_gpus), _lib.load().mdg_device_count() or 1))

    def worker(rank, start, stop):
        sl = slice(start, stop)
        return get_context(rank).fit_batch(dense["tax_id"][sl], dense["k"][sl], dense["N"][sl], fit_cfg,
                                        mism12=dense["mism12"][sl] if dense.get("mism12") is not None else None,
                                        noise3=dense["noise"][sl] if dense.get("noise") is not None else None)

    parts = [p for p in run_on_gpus(n_tax, n_dev, worker) if p is not None]
    return {key: np.concatenate([p[key] for p in parts]) for key in ("result", "median", "hpdi_lo", "hpdi_hi")}


def map_dense(dense, cfg, fit_cfg, n_gpus=1, level=None):
    """Run mdg_map_batch over `n_gpus` contiguous shares of the dense batch (as fit_dense); host-side concat. With
    `level`, each GPU also profiles its share (mdg_map_profile) right after its MAP pass, and (rows, intervals) is
    returned."""
    n_tax = len(dense["tax_id"])
    if n_tax == 0:
        rows = np.zeros(0, MAP_RESULT_DTYPE)
        return rows if level is None else (rows, np.zeros(0, MAP_INTERVAL_DTYPE))
    n_dev = max(1, min(int(n_gpus), _lib.load().mdg_device_count() or 1))

    def worker(rank, start, stop):
        sl = slice(start, stop)
        ctx = get_context(rank)
        rows = ctx.map_batch(dense["tax_id"][sl], dense["k"][sl], dense["N"][sl], fit_cfg,
                             mism12=dense["mism12"][sl] if dense.get("mism12") is not None else None,
                             noise3=dense["noise"][sl] if dense.get("noise") is not None else None)
        if level is None:
            return rows
        return rows, ctx.map_profile(dense["k"][sl], dense["N"][sl], rows, fit_cfg, level)

    parts = [p for p in run_on_gpus(n_tax, n_dev, worker) if p is not None]
    if level is None:
        return np.concatenate(parts)
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def select_top_dense(df_counts, dense, n_fits, ctx=None):
    """`--max-fits` on the device (mdg_select_top, K8): fits.py:736-744 on the arrays instead of the pandas
    groupby / nlargest / isin (kept as `extract_top_max_fits`, the test oracle): the n_fits TaxIDs with the largest
    sum of N_alignments over their rows, ties to the smaller tax id, in df_counts order."""
    n_tax = len(dense["tax_id"])
    if n_fits is None or n_fits <= 0 or n_fits >= n_tax:
        return dense
    ctx = ctx or get_context(0)
    idx = ctx.select_top(df_counts["tax_id"].to_numpy(np.int64), df_counts["N_alignments"].to_numpy(np.uint32), None,
                         dense["tax_id"], dense["first_row"], int(n_fits))
    out = dict(dense)
    for key in ("tax_id", "tax_name", "tax_rank", "N_alignments", "k", "N", "noise", "mism12", "first_row"):
        if out.get(key) is not None:
            out[key] = out[key][idx]
    return out


def _category_of(values):
    """what Series.astype("category") builds (sorted distinct values + codes), from one np.unique"""
    values = np.asarray(values)
    uniq, inv = np.unique(values, return_inverse=True)
    return uniq, inv.astype(np.int32 if len(uniq) > 32767 else (np.int16 if len(uniq) > 127 else np.int8))


def _final_dtype(arr, col):
    """utils.downcast_dataframe's rule, applied while the column is built: integers -> uint32 (position -> int8,
    with its overflow check), floats -> float32"""
    arr = np.asarray(arr)
    if arr.dtype.kind in "iu":
        if len(arr) and arr.max() > np.iinfo("uint32").max:
            raise AssertionError("Dataframe contains too large values.")
        return arr.astype("int8" if col == "position" else "uint32", copy=False)
    if arr.dtype.kind == "f":
        return arr.astype("float32", copy=False)
    return arr


def make_df_fit_results(res, dense, cfg):
    """fits.py:668-680: one row per fitted TaxID in df_counts order; failed fits are dropped
    with a warning, like the reference's timed-out fits (fits.py:520-521, 603-606). Every column is built in its
    final dtype (what utils.downcast_dataframe(df, [tax_id, tax_name, tax_rank, shortname]) gives)."""
    ok = (res["status"] & FIT_FAILED) == 0
    for tax in dense["tax_id"][~ok]:
        logger.warning("Fit: no valid fit for tax_id %s. Skipping for now", tax)
    n = int(ok.sum())
    data = {}
    for col in FIT_RESULT_COLUMNS:
        if col in ("tax_id", "tax_name", "tax_rank"):
            vals = dense[col][ok]
            if col == "tax_id" and n:
                uniq, codes = _category_of(vals)
                data[col] = pd.Categorical.from_codes(codes, categories=uniq)
            else:
                data[col] = pd.Categorical(np.asarray(vals, dtype=np.int64 if col == "tax_id" else object))
        elif col == "N_alignments":
            data[col] = _final_dtype(dense[col][ok], col)
        else:
            data[col] = _final_dtype(res[col][ok], col)
    data["shortname"] = pd.Categorical.from_codes(np.zeros(n, np.int8), categories=[cfg.shortname])
    return pd.DataFrame(data, copy=False), ok


def make_df_fit_predictions(out, dense, ok, cfg):
    """fits.py:632-665: 2P rows per TaxID: tax_id, position, median, hdpi_lower, hdpi_upper (sic); final dtypes
    (category, int8, float32) built directly instead of through a 2P-times-longer object / float64 frame."""
    P = int(cfg.max_position)
    z = np.arange(P, dtype=np.int8) + 1
    position = np.concatenate([z, -z])
    n = int(ok.sum())
    uniq, codes = _category_of(dense["tax_id"][ok]) if n else (np.zeros(0, np.int64), np.zeros(0, np.int8))
    return pd.DataFrame({
        "tax_id": pd.Categorical.from_codes(np.repeat(codes, 2 * P), categories=uniq),
        "position": np.tile(position, n),
        "median": np.ascontiguousarray(out["median"][ok], dtype=np.float32).ravel(),
        "hdpi_lower": np.ascontiguousarray(out["hpdi_lo"][ok], dtype=np.float32).ravel(),
        "hdpi_upper": np.ascontiguousarray(out["hpdi_hi"][ok], dtype=np.float32).ravel(),
        "shortname": pd.Categorical.from_codes(np.zeros(n * 2 * P, np.int8), categories=[cfg.shortname]),
    }, copy=False)


def make_df_fit_map(res, dense, ok, cfg):
    n = int(ok.sum())
    uniq, codes = _category_of(dense["tax_id"][ok]) if n else (np.zeros(0, np.int64), np.zeros(0, np.int8))
    data = {"tax_id": pd.Categorical.from_codes(codes, categories=uniq), **{c: _final_dtype(res[c][ok], c) for c in FIT_MAP_COLUMNS}}
    data["shortname"] = pd.Categorical.from_codes(np.zeros(n, np.int8), categories=[cfg.shortname])
    return pd.DataFrame(data, copy=False)


def make_df_map_results(res, dense, cfg, intervals=None):
    """The MAP-only table: one row per TaxID in df_counts order, columns MAP_RESULT_COLUMNS in their final dtypes
    (as make_df_fit_results). TaxIDs whose all-position PMD or null fit had no finite starting point are dropped with
    the same warning. `valid`: both all-position fits converged and have a Laplace covariance. `intervals` (the
    MAP_INTERVAL_DTYPE rows of mdg_map_profile for the same TaxIDs) appends MAP_INTERVAL_COLUMNS."""
    ok = (res["status"] & FIT_FAILED) == 0
    for tax in dense["tax_id"][~ok]:
        logger.warning("Fit: no valid fit for tax_id %s. Skipping for now", tax)
    n = int(ok.sum())
    r = res[ok]
    data = {}
    for col in MAP_RESULT_COLUMNS:
        if col in ("tax_id", "tax_name", "tax_rank"):
            vals = dense[col][ok]
            if col == "tax_id" and n:
                uniq, codes = _category_of(vals)
                data[col] = pd.Categorical.from_codes(codes, categories=uniq)
            else:
                data[col] = pd.Categorical(np.asarray(vals, dtype=np.int64 if col == "tax_id" else object))
        elif col == "N_alignments":
            data[col] = _final_dtype(dense[col][ok], col)
        elif col in _MAP_RUN_COLUMNS:
            run, field = _MAP_RUN_COLUMNS[col]
            data[col] = _final_dtype(r["run"][:, run][field], col)
        elif col == "valid":
            data[col] = (r["status"] & (FIT_MAP_NOT_CONVERGED | FIT_COV_INVALID)) == 0
        elif col == "shortname":
            data[col] = pd.Categorical.from_codes(np.zeros(n, np.int8), categories=[cfg.shortname])
        else:
            data[col] = _final_dtype(r[col], col)
    if intervals is not None:
        ends = intervals[ok]["end"]
        for i, prefix in enumerate(("", "forward_", "reverse_")):
            data[prefix + "D_max_lower"] = _final_dtype(ends[:, i, 0]["D"], "D")
            data[prefix + "D_max_upper"] = _final_dtype(ends[:, i, 1]["D"], "D")
        data["interval_valid"] = (intervals[ok]["status"] & (PROFILE_FAILED | FIT_FAILED)) == 0
    return pd.DataFrame(data, copy=False)


def compute_map_fits(df_counts, cfg, n_fits=None, profile_interval=False):
    """MAP-only screening of every TaxID of df_counts (or of the top `n_fits`, as compute_fits): the table of
    make_df_map_results, with the profile intervals of D_max at PROFILE_INTERVAL_LEVEL if `profile_interval`."""
    dense = select_top_dense(df_counts, dense_from_df_counts(df_counts, cfg), n_fits)
    n_gpus = getattr(cfg, "gpus", 1)
    if not profile_interval:
        return make_df_map_results(map_dense(dense, cfg, fit_config_from(cfg), n_gpus=n_gpus), dense, cfg)
    res, intervals = map_dense(dense, cfg, fit_config_from(cfg), n_gpus=n_gpus, level=PROFILE_INTERVAL_LEVEL)
    return make_df_map_results(res, dense, cfg, intervals)


def compute_fits(df_counts, cfg, mcmc_kwargs=None, return_map=False, n_fits=None):
    """The GPU replacement of fits.compute_fits (fits.py:709-730). `n_fits`: fit only the top TaxIDs of
    fits.py:736-744 (what get_fits does by filtering the frame first), selected on the device."""
    dense = select_top_dense(df_counts, dense_from_df_counts(df_counts, cfg), n_fits)
    fit_cfg = fit_config_from(cfg, mcmc_kwargs)
    out = fit_dense(dense, cfg, fit_cfg, n_gpus=getattr(cfg, "gpus", 1))
    df_fit_results, ok = make_df_fit_results(out["result"], dense, cfg)
    df_fit_predictions = make_df_fit_predictions(out, dense, ok, cfg)
    if return_map:
        return df_fit_results, df_fit_predictions, make_df_fit_map(out["result"], dense, ok, cfg)
    return df_fit_results, df_fit_predictions


CACHE_KEYS = ["min_alignments", "min_y_sum", "substitution_bases_forward", "substitution_bases_reverse",
              "N_fits", "shortname", "filename", "max_position"]


def get_fits(df_counts, cfg):
    """fits.py:754-807: reuse both parquet files iff present, not --forced and metadata match."""
    pq_results = io.Parquet(cfg.filename_fit_results)
    pq_predictions = io.Parquet(cfg.filename_fit_predictions)
    if pq_results.exists(cfg.forced) and pq_predictions.exists(cfg.forced):
        meta = cfg.to_dict()
        if utils.metadata_is_similar(pq_results.load_metadata(), meta, include=CACHE_KEYS) and \
                utils.metadata_is_similar(pq_predictions.load_metadata(), meta, include=CACHE_KEYS):
            logger.info("Fit: Loading fits from parquet-file.")
            return pq_results.load(), pq_predictions.load()
    logger.info("Fit: Generating fits and saving to file.")
    df_fit_results, df_fit_predictions, df_fit_map = compute_fits(df_counts, cfg, mcmc_kwargs_default(), return_map=True,
                                                                  n_fits=cfg.N_fits)
    meta = cfg.to_dict()
    pq_results.save(df_fit_results, metadata=meta)
    pq_predictions.save(df_fit_predictions, metadata=meta)
    io.Parquet(cfg.filename_fit_map).save(df_fit_map, metadata=meta)
    return df_fit_results, df_fit_predictions


def get_map_fits(df_counts, cfg, profile_interval=False):
    """`metadamage fit --map-only [--profile-interval]`: the cache rules of get_fits on map_results/<shortname>.parquet.
    With intervals the metadata also records "profile_interval": PROFILE_INTERVAL_LEVEL, and a cached table is reused
    only if its own key matches (a missing key means a table without intervals)."""
    pq = io.Parquet(cfg.filename_map_results)
    meta = cfg.to_dict()
    if profile_interval:
        meta["profile_interval"] = PROFILE_INTERVAL_LEVEL
    if pq.exists(cfg.forced):
        if utils.metadata_is_similar(pq.load_metadata(), meta, include=CACHE_KEYS + ["profile_interval"]):
            logger.info("Fit: Loading MAP fits from parquet-file.")
            return pq.load()
    logger.info("Fit: Generating MAP fits and saving to file.")
    df_map_results = compute_map_fits(df_counts, cfg, n_fits=cfg.N_fits, profile_interval=profile_interval)
    pq.save(df_map_results, metadata=meta)
    return df_map_results
