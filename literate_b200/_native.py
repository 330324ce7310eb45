"""ctypes binding of include/literate_b200.h.

Loading fails loudly if the shared library is missing; nothing in this package falls back to a
CPU implementation.  ``load(build_if_missing=True)`` compiles it in-tree with nvcc first.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "_lib", "libliterate_b200.so")

LR_ABI_VERSION = 1
LR_ACC_ROWS = 8
LR_KMAX = 30
LR_REC_DOUBLES = 144
LR_NCOUNTERS = 10
LR_TREND_REC_HEAD = 16
LR_TREND_STATE_DOUBLES = 12
LR_DD_NPAR = 11
LR_DD_REC_HEAD = 24
LR_DD_STATE_DOUBLES = 24
LR_OK = 0

# every symbol include/literate_b200.h declares (checked by the CPU tests)
EXPORTS = [
    "lr_abi_version", "lr_last_error", "lr_create", "lr_destroy", "lr_info", "lr_sync",
    "lr_acc_stride", "lr_bin_accumulate", "lr_bin_finalize", "lr_bin_stats", "lr_bin_stats_host",
    "lr_bin_accumulate_i32", "lr_bin_stats_host_i32", "lr_fe_ref_of_jitter", "lr_bin_table_hint", "lr_bin_last_build",
    "lr_dataset_create", "lr_dataset_create_host", "lr_dataset_create_general_host", "lr_dataset_destroy", "lr_state_eval_host", "lr_proposal_eval_host", "lr_loglik_direct",
    "lr_chains_create", "lr_chains_destroy", "lr_chains_records_per_run", "lr_chains_run", "lr_chains_run_host",
    "lr_imputation_envelope", "lr_chains_counters_host", "lr_chains_team_stats_host", "lr_chains_get_state_host", "lr_chains_set_state_host", "lr_chains_set_beta_host",
    "lr_chains_swap_info", "lr_chains_swap_apply", "lr_chains_swap_step", "lr_summarize_records", "lr_marginal_rates",
    "lr_trend_create", "lr_trend_create_host", "lr_trend_destroy", "lr_trend_record_doubles", "lr_trend_records_per_run",
    "lr_trend_run", "lr_trend_run_host", "lr_trend_eval_host", "lr_trend_state_host",
    "lr_trend_set_beta_host", "lr_trend_swap_info", "lr_trend_swap_apply", "lr_trend_swap_step", "lr_trend_temper_host",
    "lr_dd_create", "lr_dd_create_host", "lr_dd_destroy", "lr_dd_record_doubles", "lr_dd_records_per_run",
    "lr_dd_run", "lr_dd_run_host", "lr_dd_eval_host", "lr_dd_state_host",
    "lr_dd_set_beta_host", "lr_dd_swap_info", "lr_dd_swap_apply", "lr_dd_swap_step", "lr_dd_temper_host",
    "lr_column_hpd", "lr_chain_diagnostics", "lr_rank_transform", "lr_rank_diagnostics",
    "lr_dataset_bin_terms", "lr_predictive_check", "lr_loo",
]


class ChainConfig(C.Structure):
    """lr_chain_config"""
    _fields_ = [("model_BDI", C.c_int32), ("const_rates", C.c_int32), ("const_death_rate", C.c_int32),
                ("use_rate_HP", C.c_int32), ("poisson_prior", C.c_double), ("update_fraction", C.c_double),
                ("real_move_shift", C.c_int32), ("loop_variant", C.c_int32), ("beta", C.c_double)]


class NativeError(RuntimeError):
    pass


_lib = None


def load(build_if_missing=False):
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        # (re)build when the library is missing or older than its sources; a no-op when the digest stamp matches
        from . import build as _b
        try:
            _b.build()
        except Exception as e:
            # a library that does not match its sources is not silently used: the ABI version alone would not notice
            if not os.path.exists(LIB_PATH) or not os.environ.get("LR_ALLOW_STALE_LIB"):
                raise NativeError("rebuilding libliterate_b200.so failed (%s); set LR_ALLOW_STALE_LIB=1 to load the existing, "
                                  "possibly stale library" % e) from e
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} is missing. Build it with `python -m literate_b200.build` (needs nvcc); "
            "literate_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
    P = C.POINTER

    def sig(name, res, *args):
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = list(args)

    sig("lr_abi_version", C.c_int)
    sig("lr_last_error", C.c_char_p)
    sig("lr_create", C.c_int, C.c_int, P(vp))
    sig("lr_destroy", C.c_int, vp)
    sig("lr_info", C.c_int, vp, P(i32), P(i64), P(i32))
    sig("lr_sync", C.c_int, vp)
    sig("lr_acc_stride", i64, i32)
    sig("lr_bin_accumulate", C.c_int, vp, vp, vp, i64, i64, i32, i64, i32, f64, i32, f64, vp, vp)
    sig("lr_bin_finalize", C.c_int, vp, vp, i32, i32, f64, vp, vp, vp, vp)
    sig("lr_bin_stats", C.c_int, vp, vp, vp, i64, i64, i32, i64, i32, f64, i32, f64, vp, vp, vp, vp)
    sig("lr_bin_stats_host", C.c_int, vp, vp, vp, i64, i64, i32, i64, i32, f64, i32, f64, vp, vp, vp)
    sig("lr_bin_accumulate_i32", C.c_int, vp, vp, vp, i64, i64, i32, i64, i32, f64, i32, f64, vp, vp)
    sig("lr_bin_stats_host_i32", C.c_int, vp, vp, vp, i64, i64, i32, i64, i32, f64, i32, f64, vp, vp, vp)
    sig("lr_fe_ref_of_jitter", C.c_double, f64)
    sig("lr_bin_table_hint", C.c_int, vp, P(i32))
    sig("lr_bin_last_build", C.c_int, vp, P(i32))
    sig("lr_dataset_create", C.c_int, vp, i32, i32, i32, f64, f64, vp, vp, vp, vp, vp, vp, P(vp))
    sig("lr_dataset_create_host", C.c_int, vp, i32, i32, i32, f64, f64, vp, vp, vp, vp, vp, P(vp))
    sig("lr_dataset_create_general_host", C.c_int, vp, i32, i32, i32, f64, f64, vp, vp, vp, vp, vp, vp, vp, P(vp))
    sig("lr_dataset_destroy", C.c_int, vp)
    sig("lr_dataset_bin_terms", C.c_int, vp, vp, vp)
    sig("lr_state_eval_host", C.c_int, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("lr_proposal_eval_host", C.c_int, vp, i32, *([vp] * 24))
    sig("lr_loglik_direct", C.c_int, vp, vp, vp, i64, i64, i32, vp, vp, i32, vp, vp)
    sig("lr_chains_create", C.c_int, vp, vp, i32, P(ChainConfig), u64, i64, vp, P(vp))
    sig("lr_chains_destroy", C.c_int, vp)
    sig("lr_chains_records_per_run", i64, vp, i64, i64)
    sig("lr_chains_run", C.c_int, vp, i64, i64, vp, vp)
    sig("lr_chains_run_host", C.c_int, vp, i64, i64, vp)
    sig("lr_chains_counters_host", C.c_int, vp, vp)
    sig("lr_imputation_envelope", C.c_int, vp, vp, vp, vp, i32, i32, vp, vp)
    sig("lr_chains_team_stats_host", C.c_int, vp, vp)
    sig("lr_chains_get_state_host", C.c_int, vp, vp)
    sig("lr_chains_set_state_host", C.c_int, vp, vp)
    sig("lr_chains_set_beta_host", C.c_int, vp, vp)
    sig("lr_chains_swap_info", C.c_int, vp, vp, vp)
    sig("lr_chains_swap_apply", C.c_int, vp, vp, i64, i64, i32, u64, vp)
    sig("lr_chains_swap_step", C.c_int, vp, i32, u64)
    sig("lr_summarize_records", C.c_int, vp, vp, i64, f64, i32, vp, vp, vp, vp)
    sig("lr_marginal_rates", C.c_int, vp, vp, i64, f64, i32, i32, i32, vp, vp, vp)
    sig("lr_column_hpd", C.c_int, vp, vp, i64, i64, i32, i32, vp, vp, vp, vp, f64, vp, vp, vp, vp, vp)
    sig("lr_chain_diagnostics", C.c_int, vp, vp, i64, i64, i32, i32, i64, i32, vp, vp, vp, vp, vp, vp, vp)
    sig("lr_rank_transform", C.c_int, vp, vp, i64, i64, i32, i32, i64, i32, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("lr_rank_diagnostics", C.c_int, vp, vp, i64, i64, i32, i32, i64, i32, vp, vp, vp, vp, vp, vp, vp)
    sig("lr_predictive_check", C.c_int, vp, vp, i64, i64, i32, i32, i64, i32, i32, f64, i32, vp, i32, vp, i64, u64,
        vp, vp, vp, vp, vp, vp, vp)
    sig("lr_loo", C.c_int, vp, vp, i64, i64, i32, i32, i64, i32, i32, f64, i32, vp, vp, vp, vp, vp)
    sig("lr_trend_create", C.c_int, vp, i32, i32, vp, vp, vp, vp, i32, i32, i32, u64, i64, vp, vp, P(vp))
    sig("lr_trend_create_host", C.c_int, vp, i32, i32, vp, vp, vp, vp, i32, i32, i32, u64, i64, vp, P(vp))
    sig("lr_trend_destroy", C.c_int, vp)
    sig("lr_trend_record_doubles", i64, i32)
    sig("lr_trend_records_per_run", i64, vp, i64, i64)
    sig("lr_trend_run", C.c_int, vp, i64, i64, vp, vp)
    sig("lr_trend_run_host", C.c_int, vp, i64, i64, vp)
    sig("lr_trend_eval_host", C.c_int, vp, i32, *([vp] * 11))
    sig("lr_trend_state_host", C.c_int, vp, vp)
    sig("lr_dd_create", C.c_int, vp, i32, i32, vp, vp, vp, f64, f64, i32, i32, vp, vp, i32, i32, u64, i64, vp, vp, P(vp))
    sig("lr_dd_create_host", C.c_int, vp, i32, i32, vp, vp, vp, f64, f64, i32, i32, vp, vp, i32, i32, u64, i64, vp, P(vp))
    sig("lr_dd_destroy", C.c_int, vp)
    sig("lr_dd_record_doubles", i64, i32)
    sig("lr_dd_records_per_run", i64, vp, i64, i64)
    sig("lr_dd_run", C.c_int, vp, i64, i64, vp, vp)
    sig("lr_dd_run_host", C.c_int, vp, i64, i64, vp)
    sig("lr_dd_eval_host", C.c_int, vp, i32, *([vp] * 12))
    sig("lr_dd_state_host", C.c_int, vp, vp)
    for p in ("trend", "dd"):
        sig("lr_%s_set_beta_host" % p, C.c_int, vp, vp)
        sig("lr_%s_swap_info" % p, C.c_int, vp, vp, vp)
        sig("lr_%s_swap_apply" % p, C.c_int, vp, vp, i64, i64, i32, u64, vp)
        sig("lr_%s_swap_step" % p, C.c_int, vp, i32, u64)
        sig("lr_%s_temper_host" % p, C.c_int, vp, vp, vp)
    if lib.lr_abi_version() != LR_ABI_VERSION:
        raise NativeError("libliterate_b200.so ABI version mismatch; rebuild with `python -m literate_b200.build --force`")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != LR_OK:
        msg = load().lr_last_error().decode(errors="replace")
        raise NativeError(f"{what or 'literate_b200'} failed (status {rc}): {msg}")


def np_ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)
