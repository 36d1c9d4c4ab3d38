"""ctypes / numpy mirrors of the structs declared in include/mdg.h.

Pure layout description (no compute): shared by the product binding (`_lib.py`) and, as test
infrastructure, by the oracle wrapper under `oracle/`.
"""
import ctypes as C

import numpy as np

NUM_RUNS = 6
RUN_NAMES = ("pmd_all", "null_all", "pmd_fwd", "null_fwd", "pmd_rev", "null_rev")
MAX_POSITION = 64

MDG_OK = 0
MDG_HOST = 0
MDG_DEVICE = 1

FIT_FAILED = 0x1
FIT_MAP_NOT_CONVERGED = 0x2
FIT_HAS_DIVERGENCES = 0x4
FIT_BUDGET_EXCEEDED = 0x8
FIT_COV_INVALID = 0x10


class FitConfig(C.Structure):
    """mdg_fit_config (include/mdg.h)."""

    _fields_ = [
        ("num_warmup", C.c_int32),
        ("num_samples", C.c_int32),
        ("max_tree_depth", C.c_int32),
        ("do_map", C.c_int32),
        ("do_fwd_rev", C.c_int32),
        ("find_heuristic_step_size", C.c_int32),
        ("reference_quirks", C.c_int32),
        ("pack_half_warps", C.c_int32),
        ("target_accept", C.c_double),
        ("init_step_size", C.c_double),
        ("max_delta_energy", C.c_double),
        ("init_radius", C.c_double),
        ("hpdi_prob", C.c_double),
        ("seed", C.c_uint64),
        ("q_prior_a", C.c_double),
        ("q_prior_b", C.c_double),
        ("A_prior_a", C.c_double),
        ("A_prior_b", C.c_double),
        ("c_prior_a", C.c_double),
        ("c_prior_b", C.c_double),
        ("phi_prior_rate", C.c_double),
        ("phi_min", C.c_double),
        ("max_leapfrogs_per_run", C.c_int32),
        ("reserved0", C.c_int32),
    ]

    def copy(self, **changes):
        out = FitConfig.from_buffer_copy(bytes(self))
        for key, val in changes.items():
            if not hasattr(out, key):
                raise AttributeError(f"mdg_fit_config has no field {key!r}")
            setattr(out, key, val)
        return out


class Timings(C.Structure):
    """mdg_timings (include/mdg.h)."""

    _fields_ = [
        ("counts_ms", C.c_float),
        ("map_ms", C.c_float),
        ("nuts_ms", C.c_float),
        ("ppc_ms", C.c_float),
        ("assemble_ms", C.c_float),
        ("total_ms", C.c_float),
        ("n_launches", C.c_uint32),
        ("reserved", C.c_uint32),
        ("leapfrogs", C.c_uint64 * NUM_RUNS),
        ("nuts_union_ms", C.c_float),
        ("nuts_begin_ms", C.c_float),
        ("nuts_end_ms", C.c_float),
        ("reserved1", C.c_float),
    ]


RUN_DIAG_DTYPE = np.dtype(
    [
        ("step_size", "<f8"),
        ("mean_accept", "<f8"),
        ("n_leapfrog", "<u4"),
        ("n_divergent", "<u4"),
        ("waic", "<f8"),
        ("lppd", "<f8"),
    ],
    align=True,
)

_REFERENCE_FLOAT_FIELDS = (
    "D_max",
    "n_sigma",
    "D_max_lower_hpdi",
    "D_max_upper_hpdi",
    "q_mean",
    "concentration_mean",
    "D_max_marginalized_mean",
    "n_sigma_forward",
    "D_max_forward",
    "q_mean_forward",
    "n_sigma_reverse",
    "D_max_reverse",
    "q_mean_reverse",
    "asymmetry",
    "normalized_noise",
    "normalized_noise_forward",
    "normalized_noise_reverse",
)
_REFERENCE_INT_FIELDS = (
    "N_z1_forward",
    "N_z1_reverse",
    "N_sum_forward",
    "N_sum_reverse",
    "N_sum_total",
    "y_sum_forward",
    "y_sum_reverse",
    "y_sum_total",
)
_EXTRA_FLOAT_FIELDS = (
    "map_A",
    "map_q",
    "map_c",
    "map_phi",
    "map_D_max",
    "map_logp",
    "map_null_q",
    "map_null_phi",
    "map_null_logp",
    "A_mean",
    "c_mean",
    "D_max_marginalized_std",
    "q_std",
    "concentration_std",
)

FIT_RESULT_DTYPE = np.dtype(
    [("tax_id", "<i8"), ("status", "<u4"), ("map_iters", "<u4")]
    + [(name, "<f8") for name in _REFERENCE_FLOAT_FIELDS]
    + [(name, "<u8") for name in _REFERENCE_INT_FIELDS]
    + [(name, "<f8") for name in _EXTRA_FLOAT_FIELDS]
    + [("run", RUN_DIAG_DTYPE, (NUM_RUNS,))],
    align=True,
)

MAP_RUN_DTYPE = np.dtype(
    [(name, "<f8") for name in ("q", "A", "c", "phi", "q_std", "A_std", "c_std", "phi_std", "cov_Ac", "logp", "loglik")]
    + [("iters", "<u4"), ("n_eval", "<u4"), ("flags", "<u4"), ("reserved", "<u4")],
    align=True,
)

MAP_RESULT_DTYPE = np.dtype(
    [("tax_id", "<i8"), ("status", "<u4"), ("reserved", "<u4")]
    + [(name, "<f8") for name in (
        "D_max", "D_max_std", "significance", "rho_Ac", "lambda_LR", "lambda_LR_P", "lambda_LR_z",
        "forward_D_max", "forward_D_max_std", "forward_lambda_LR", "reverse_D_max", "reverse_D_max_std", "reverse_lambda_LR",
        "normalized_noise", "normalized_noise_forward", "normalized_noise_reverse")]
    + [(name, "<u8") for name in _REFERENCE_INT_FIELDS]
    + [("run", MAP_RUN_DTYPE, (NUM_RUNS,))],
    align=True,
)


def ptr(arr, ctype=None):
    """Raw pointer of a C-contiguous numpy array (None -> NULL)."""
    if arr is None:
        return None
    if not arr.flags["C_CONTIGUOUS"]:
        raise ValueError("array passed to the C-ABI must be C-contiguous")
    return arr.ctypes.data_as(C.c_void_p if ctype is None else C.POINTER(ctype))
