"""ctypes binding of ``libcql_b200.so`` (``include/cql_b200.h``).

There is NO fallback: if the library is not built, cannot be loaded, or no
CUDA device is present, the product path raises.  (The CPU oracle under
``oracle/`` is test infrastructure and is never imported from here.)
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

# CQL_LIB: load another build of the same library (A/B measurements of compile-time variants); never a fallback
LIB_PATH = Path(os.environ["CQL_LIB"]) if os.environ.get("CQL_LIB") else Path(__file__).resolve().parent / "libcql_b200.so"

PREC_FP32, PREC_TF32X3, PREC_BF16, PREC_F16X3 = 0, 1, 2, 3
SQUASH_EPS, SQUASH_SOFTPLUS = 0, 1
SCORE_Q, SCORE_POLICY = 0, 1
BUF_SCALAR_GRADS, BUF_CRITIC_GRADS, BUF_ACTOR_GRADS, BUF_METRICS, BUF_PARAMS, BUF_ALL_GRADS, BUF_NOISE, BUF_BATCH = range(8)
MAX_TOPK = 1024
MAX_N_STEPS = 64                                     # CQL_MAX_N_STEPS: longest n-step TD horizon
MAX_CRITICS = 10                                     # CQL_MAX_CRITICS: largest critic ensemble (n_critics)
MAX_ACTION_SAMPLES = 32                              # CQL_MAX_ACTION_SAMPLES: most action samples (n_action_samples)
DT_I32, DT_I64, DT_F32, DT_F64 = 0, 1, 2, 3          # cql_mdp_append chunk dtypes
SCALER_NONE, SCALER_MIN_MAX, SCALER_STANDARD = 0, 1, 2   # cql_preprocessing kinds


class CqlConfig(C.Structure):
    """Mirror of ``struct cql_config`` (include/cql_b200.h)."""

    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32), ("batch_size", C.c_int32),
        ("n_critics", C.c_int32), ("n_action_samples", C.c_int32), ("precision", C.c_int32),
        ("squash", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32),
        ("gamma", C.c_float), ("tau", C.c_float),
        ("actor_lr", C.c_float), ("critic_lr", C.c_float), ("temp_lr", C.c_float), ("alpha_lr", C.c_float),
        ("initial_temperature", C.c_float), ("initial_alpha", C.c_float),
        ("alpha_threshold", C.c_float), ("conservative_weight", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
        ("seed", C.c_uint64),
    ]


class ColumnStats(C.Structure):
    """Mirror of ``struct cql_column_stats``."""

    _fields_ = [("count", C.c_int64), ("min", C.c_double), ("max", C.c_double), ("mean", C.c_double), ("m2", C.c_double)]


class TableStats(C.Structure):
    """Mirror of ``struct cql_table_stats``: col = obs.x, obs.y, act, rew."""

    _fields_ = [("col", ColumnStats * 4), ("rew_available", C.c_int32), ("pad", C.c_int32)]


class Preprocessing(C.Structure):
    """Mirror of ``struct cql_preprocessing``."""

    _fields_ = [
        ("obs_kind", C.c_int32), ("act_kind", C.c_int32), ("rew_kind", C.c_int32), ("pad", C.c_int32),
        ("obs_a", C.c_float * 2), ("obs_b", C.c_float * 2),
        ("act_a", C.c_float), ("act_b", C.c_float), ("rew_a", C.c_float), ("rew_b", C.c_float),
    ]


class OfflineSums(C.Structure):
    """Mirror of ``struct cql_offline_sums``."""

    _fields_ = [
        ("td_error", C.c_double), ("discounted_advantage", C.c_double), ("value", C.c_double),
        ("value_std", C.c_double), ("initial_value", C.c_double), ("action_diff", C.c_double),
        ("success_q", C.c_double), ("all_q", C.c_double),
        ("n_rows", C.c_int64), ("n_episodes", C.c_int64), ("n_success_rows", C.c_int64),
    ]


_P = C.c_void_p
_F = C.POINTER(C.c_float)
_I32 = C.POINTER(C.c_int32)
_I64 = C.POINTER(C.c_int64)

# name -> (restype, argtypes); every symbol declared in include/cql_b200.h
SIGNATURES = {
    "cql_abi_version": (C.c_int, []),
    "cql_create": (C.c_int, [C.POINTER(CqlConfig), C.POINTER(_P)]),
    "cql_destroy": (None, [_P]),
    "cql_last_error": (C.c_char_p, [_P]),
    "cql_state_floats": (C.c_int64, [_P]),
    "cql_set_weights": (C.c_int, [_P, _P, C.c_int64]),
    "cql_get_weights": (C.c_int, [_P, _P, C.c_int64]),
    "cql_set_optimizer": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64]),
    "cql_get_optimizer": (C.c_int, [_P, _P, _P, C.c_int64, _I64]),
    "cql_load_transitions": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64]),
    "cql_num_transitions": (C.c_int64, [_P]),
    "cql_build_mdp": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_float, _P, _P, _P, _P, _P]),
    "cql_sample_rows": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P]),
    "cql_update": (C.c_int, [_P, C.c_int64, _P, _P]),
    "cql_update_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cql_update_batches": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "cql_step_phase": (C.c_int, [_P, C.c_int, _P]),
    "cql_upload_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "cql_seen_csr": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "cql_dp_attach": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, C.c_int64, C.c_int64]),
    "cql_dp_allreduce": (C.c_int, [_P, C.c_int, _P]),
    "cql_dp_error": (C.c_int, [_P, _P]),
    "cql_dp_mode": (C.c_int, [_P, _P]),
    "cql_device_buffer": (C.c_int, [_P, C.c_int, C.POINTER(_P), _I64]),
    "cql_score_topk": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "cql_score_topk_dev": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "cql_score_pairs": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P]),
    "cql_rank_metrics": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "cql_topk_filter_dev": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P, _P, _P, C.c_int32, _P, _P, _P]),
    "cql_timed_update": (C.c_int, [_P, _P, _P]),
    "cql_mma_bench": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "cql_synth_table": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, C.c_uint64]),
    "cql_set_table_sharded": (C.c_int, [_P, C.c_int32]),
    "cql_set_n_steps": (C.c_int, [_P, C.c_int32]),
    "cql_set_table_rows": (C.c_int, [_P, _P, C.c_int64]),
    "cql_update_batch_rows": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "cql_get_table_stats": (C.c_int, [_P, C.POINTER(TableStats)]),
    "cql_set_preprocessing": (C.c_int, [_P, C.POINTER(Preprocessing)]),
    "cql_get_preprocessing": (C.c_int, [_P, C.POINTER(Preprocessing)]),
    "cql_mdp_begin": (C.c_int, [_P, C.c_int64]),
    "cql_mdp_append": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int64]),
    "cql_mdp_finish": (C.c_int, [_P, C.c_int32, C.c_float, _P, _P, _P, _P, _P]),
    "cql_selftest_umma": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, _P]),
    "cql_offline_eval": (C.c_int, [_P, C.c_float, C.POINTER(OfflineSums), _P]),
    "cql_launch_count": (C.c_int64, [_P]),
    "cql_fqe_enable": (C.c_int, [_P, C.c_int32]),
    "cql_fqe_update": (C.c_int, [_P, C.c_int64, _P, _P]),
    "cql_fqe_update_rows": (C.c_int, [_P, _P, _P, _P, _P]),
    "cql_copy_table": (C.c_int, [_P, _P, _P]),
    "cql_predict_value": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P]),
    "cql_sample_action": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P]),
}

_lib = None


class CqlLibraryError(RuntimeError):
    """The CUDA library is missing/unloadable, or a call into it failed."""


class CqlArgumentError(CqlLibraryError, ValueError):
    """A call into the library rejected an argument or the call sequence (return code 3)."""


def load() -> C.CDLL:
    """Load the C-ABI library (once).  Raises ``CqlLibraryError`` -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CqlLibraryError(
            f"{LIB_PATH} is not built; run `python -m replay_cql_b200.build` "
            "(needs nvcc).  replay_cql_b200 has no CPU fallback."
        )
    try:
        lib = C.CDLL(str(LIB_PATH))
    except OSError as exc:  # pragma: no cover - depends on the box
        raise CqlLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise CqlLibraryError(f"{LIB_PATH} does not export {name}") from exc
        fn.restype = res
        fn.argtypes = args
    if lib.cql_abi_version() != 2:
        raise CqlLibraryError("libcql_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(handle, rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cql_last_error(handle)
        err = CqlArgumentError if rc == 3 else CqlLibraryError
        raise err(f"{what} failed: {msg.decode() if msg else rc}")
