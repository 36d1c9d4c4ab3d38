"""Host-side configuration and DataFrame helpers of the `metadamage fit` path.

Mirrors the parts of the reference's utils.py that the hot path's callers need
(Config utils.py:43-184, SubstitutionBases 186-201, extract_name 219-224, file_is_valid 227-238,
downcast_dataframe 329-356, metadata_is_similar 362-377), plus the options this build adds:
`max_position` (documented in the reference's README.md:121 but never wired, cli.py:105) and
`gpus`.
"""
from dataclasses import asdict, dataclass, field
from enum import Enum
import logging
import os
from pathlib import Path
from typing import Optional

import numpy as np
import pandas as pd

logger = logging.getLogger(__name__)


class SubstitutionBases(str, Enum):
    """The twelve mismatches (utils.py:186-201)."""

    AC = "AC"
    AG = "AG"
    AT = "AT"
    CA = "CA"
    CG = "CG"
    CT = "CT"
    GA = "GA"
    GC = "GC"
    GT = "GT"
    TA = "TA"
    TC = "TC"
    TG = "TG"


def _available_cores():
    try:
        import psutil

        return psutil.cpu_count(logical=True) or 1
    except Exception:  # psutil is optional here
        return os.cpu_count() or 1


@dataclass
class Config:
    out_dir: Path
    max_fits: Optional[int]
    max_cores: int
    min_alignments: int
    min_y_sum: int
    substitution_bases_forward: str
    substitution_bases_reverse: str
    forced: bool
    version: str
    max_position: int = 15
    gpus: int = 1
    seed: int = 0
    filename: Optional[Path] = None
    shortname: Optional[str] = None
    N_filenames: Optional[int] = None
    N_fits: Optional[int] = None
    N_cores: int = field(init=False)

    def __post_init__(self):
        # same clipping rules as utils.py:70-85
        available = _available_cores()
        if self.max_cores > available:
            self.N_cores = available - 1
        elif self.max_cores < 0:
            self.N_cores = available - abs(self.max_cores)
        else:
            self.N_cores = self.max_cores
        if not 1 <= int(self.max_position) <= 64:
            raise ValueError("max_position must be in [1, 64]")

    def add_filenames(self, filenames):
        self.N_filenames = len(filenames)

    def add_filename(self, filename):
        self.filename = filename
        self.shortname = extract_name(filename)

    def _out(self, sub):
        if self.shortname is None:
            raise AssertionError("call cfg.add_filename(filename) before asking for output paths")
        return Path(self.out_dir) / sub / f"{self.shortname}.parquet"

    @property
    def filename_counts(self):
        return self._out("counts")

    @property
    def filename_fit_results(self):
        return self._out("fit_results")

    @property
    def filename_fit_predictions(self):
        return self._out("fit_predictions")

    @property
    def filename_fit_map(self):
        return self._out("fit_map")

    @property
    def filename_map_results(self):
        return self._out("map_results")

    def set_number_of_fits(self, df_counts):
        self.N_tax_ids = len(pd.unique(df_counts.tax_id))
        if self.max_fits is not None and self.max_fits > 0:
            self.N_fits = min(self.max_fits, self.N_tax_ids)
        else:
            self.N_fits = self.N_tax_ids
        logger.info("Setting number_of_fits to %s", self.N_fits)

    def to_dict(self):
        d = asdict(self)
        for key, val in d.items():
            if isinstance(val, Path):
                d[key] = str(val)
        return d


def extract_name(filename, max_length=60):
    shortname = Path(filename).stem.split(".")[0]
    if len(shortname) > max_length:
        shortname = shortname[:max_length] + "..."
    logger.info("Running new file: %s", shortname)
    return shortname


def file_is_valid(filename):
    """Existing, non-empty file. A missing file raises FileNotFoundError like the reference,
    whose error message stats the file (utils.py:231-232)."""
    path = Path(filename)
    if path.exists() and path.stat().st_size > 0:
        return True
    exists = path.exists()
    valid_size = path.stat().st_size > 0  # raises for a missing file, as upstream does
    logger.error("%s is not a valid file (exists=%s, size>0=%s). Skipping for now.", filename, exists, valid_size)
    return False


def is_df_counts_accepted(df_counts, cfg):
    if len(df_counts) > 0:
        return True
    logger.warning("%s: no TaxID passed the cuts; skipping the fits.", cfg.shortname)
    return False


def downcast_dataframe(df, categories, fully_automatic=False):
    """categories -> 'category'; integers -> uint32 (position -> int8); floats -> float32
    (utils.py:329-356, with the dtypes the pinned pandas 1.2 produced)."""
    categories = [c for c in categories if c in df.columns]
    out = df.astype({c: "category" for c in categories})
    int_cols = list(out.select_dtypes(include=["integer"]).columns)
    if int_cols and out[int_cols].max().max() > np.iinfo("uint32").max:
        raise AssertionError("Dataframe contains too large values.")
    for col in int_cols:
        if fully_automatic:
            out[col] = pd.to_numeric(out[col], downcast="integer")
        else:
            out[col] = out[col].astype("int8" if col == "position" else "uint32")
    for col in out.select_dtypes(include=["float"]).columns:
        out[col] = pd.to_numeric(out[col], downcast="float") if fully_automatic else out[col].astype("float32")
    return out


def metadata_is_similar(metadata_file, metadata_cfg, include=None):
    if include is None:
        if set(metadata_file.keys()) != set(metadata_cfg.keys()):
            return False
        include = set(metadata_file.keys())
    differing = [key for key in include if metadata_file.get(key) != metadata_cfg.get(key)]
    if differing:
        logger.info("The files' metadata are not the same, differing here: %s", differing)
        return False
    return True
