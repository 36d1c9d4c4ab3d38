"""Per-file loop of `metadamage fit` (main.py:28-74): counts, then fits, for every valid file. With `map_only` the
fits are the MAP-only screening (fits.get_map_fits) instead of the Bayesian fits, with `profile_interval` also its
profile intervals of D_max."""
import logging

from . import counts, fits, utils

logger = logging.getLogger(__name__)


def main(filenames, cfg, map_only=False, profile_interval=False):
    n_files = len(filenames)
    bad_files = 0
    for filename in filenames:
        if not utils.file_is_valid(filename):
            bad_files += 1
            continue
        cfg.add_filename(filename)
        df_counts = counts.load_counts(cfg)
        if not utils.is_df_counts_accepted(df_counts, cfg):
            continue
        if map_only and profile_interval:
            fits.get_map_fits(df_counts, cfg, profile_interval=True)
        elif map_only:
            fits.get_map_fits(df_counts, cfg)
        else:
            fits.get_fits(df_counts, cfg)
        logger.debug("End of loop")
    if bad_files == n_files:
        raise Exception("All files were bad!")
