"""ctypes binding of libmdgb200.so (include/mdg.h). There is NO CPU fallback: if the CUDA
library is missing or no B200 is visible, every compute entry point raises."""
import ctypes as C
import os

from ._abi import FitConfig, Timings

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MDG_LIB_PATH") or os.path.join(_HERE, "libmdgb200.so")  # override: kernel A/B experiments

# every symbol include/mdg.h declares
EXPORTED_SYMBOLS = (
    "mdg_version",
    "mdg_last_error",
    "mdg_device_count",
    "mdg_ctx_create",
    "mdg_ctx_destroy",
    "mdg_ctx_set_stream",
    "mdg_ctx_synchronize",
    "mdg_ctx_get_timings",
    "mdg_fit_config_default",
    "mdg_counts_reduce",
    "mdg_counts_order",
    "mdg_tsv_parse",
    "mdg_fit_batch",
    "mdg_fit_batch_submit",
    "mdg_fit_batch_wait",
    "mdg_map_batch",
    "mdg_map_profile",
    "mdg_select_top",
    "mdg_test_lgamma_digamma",
    "mdg_test_logp_grad",
    "mdg_test_exp_log",
    "mdg_test_philox",
    "mdg_test_betabinom_draws",
    "mdg_measure_fp64_peak",
)


class MdgError(RuntimeError):
    """Raised when a C-ABI call returns a non-zero status."""

    def __init__(self, code, message):
        super().__init__(f"libmdgb200 error {code}: {message}")
        self.code = code


_lib = None


def load():
    """Load the CUDA library; raises if it has not been built (see metadamage_b200/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m metadamage_b200.build` "
            "(or __graft_entry__.build()). metadamage_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64
    lib.mdg_version.restype = i32
    lib.mdg_last_error.restype = C.c_char_p
    lib.mdg_device_count.restype = i32
    lib.mdg_ctx_create.argtypes = [i32, C.POINTER(vp)]
    lib.mdg_ctx_destroy.argtypes = [vp]
    lib.mdg_ctx_destroy.restype = None
    lib.mdg_ctx_set_stream.argtypes = [vp, vp]
    lib.mdg_ctx_synchronize.argtypes = [vp]
    lib.mdg_ctx_get_timings.argtypes = [vp, C.POINTER(Timings)]
    lib.mdg_fit_config_default.argtypes = [C.POINTER(FitConfig)]
    lib.mdg_fit_config_default.restype = None
    lib.mdg_counts_reduce.argtypes = (
        [vp, i32, i64, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, i32, u32, u64] + [vp] * 13 + [i64, C.POINTER(i64)]
    )
    lib.mdg_counts_order.argtypes = [vp, i32, i64, vp, vp, vp, i64, vp, vp, vp, i64, C.POINTER(i64)]
    lib.mdg_tsv_parse.argtypes = [vp, i32, C.c_char_p, i64, i64, vp, vp, vp, vp, vp, i64, vp, vp, C.POINTER(i64), C.POINTER(C.c_int32)]
    lib.mdg_fit_batch.argtypes = [vp, i32, i64, i32, vp, vp, vp, vp, vp, C.POINTER(FitConfig)] + [vp] * 7
    lib.mdg_fit_batch_submit.argtypes = lib.mdg_fit_batch.argtypes + [C.POINTER(i64)]
    lib.mdg_fit_batch_wait.argtypes = [vp, i64, C.POINTER(Timings)]
    lib.mdg_map_batch.argtypes = [vp, i32, i64, i32, vp, vp, vp, vp, vp, C.POINTER(FitConfig), vp]
    lib.mdg_map_profile.argtypes = [vp, i32, i64, i32, vp, vp, C.POINTER(FitConfig), vp, C.c_double, vp]
    lib.mdg_select_top.argtypes = [vp, i32, i64, vp, vp, vp, i64, vp, vp, i64, vp, vp, C.POINTER(i64)]
    lib.mdg_test_lgamma_digamma.argtypes = [vp, i64, vp, vp, vp]
    lib.mdg_test_exp_log.argtypes = [vp, i64, vp, vp, vp]
    lib.mdg_test_logp_grad.argtypes = [vp, i32, vp, vp, C.POINTER(FitConfig), i32, i32, i32, i64, vp, vp, vp, vp]
    lib.mdg_test_philox.argtypes = [vp, i64, vp, vp, vp]
    lib.mdg_test_betabinom_draws.argtypes = [vp, u64, i64, C.c_double, C.c_double, C.c_double, vp]
    lib.mdg_measure_fp64_peak.argtypes = [vp, C.POINTER(C.c_double)]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise MdgError(rc, load().mdg_last_error().decode("utf-8", "replace"))


def default_config(**changes):
    cfg = FitConfig()
    load().mdg_fit_config_default(C.byref(cfg))
    return cfg.copy(**changes) if changes else cfg
