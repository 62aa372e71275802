"""ctypes binding of libml2048_b200.so (the C ABI declared in include/ml2048_b200.h).

There is no CPU fallback: if the CUDA library is missing or cannot be loaded the import of the
environment fails loudly.
"""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ML2048_LIB selects another build of the SAME sources (A/B experiments with -D switches, tools/variants.sh); it must export
# the full ABI like the default library
LIB_PATH = os.environ.get("ML2048_LIB") or os.path.join(_HERE, "libml2048_b200.so")

ABI_VERSION = 12
STATS_REPLICAS = 64
STATS_WORDS = 24  # 20 histogram bins + episodes, score_sum, step_sum, score_max (unsigned long long each)

REWARD_NORMAL, REWARD_IMPROVED, REWARD_RANK, REWARD_MAXCELL = 0, 1, 2, 3
RNG_REPLAY, RNG_PHILOX = 0, 1
ACT_U8, ACT_I32, ACT_I64 = 0, 1, 2
ACTIONS_GIVEN, ACTIONS_RANDOM_VALID, ACTIONS_FROM_LOGITS = 0, 1, 2
ONEHOT_NONE, ONEHOT_F32, ONEHOT_BF16, ONEHOT_U8 = 0, 1, 2, 3

ERRORS = {-1: "null pointer", -2: "misaligned pointer", -3: "bad size", -4: "bad enum", -5: "struct size mismatch",
          -6: "unsupported (no CUDA driver or device, or no such feature on it)"}
E_UNSUPPORTED = -6
COMPRESSIBLE_MAX_CHUNKS = 64


class StepArgs(C.Structure):
    """ml2048_step_args"""

    _fields_ = [
        ("struct_size", C.c_uint32),
        ("reward_kind", C.c_int32),
        ("rng_mode", C.c_int32),
        ("action_dtype", C.c_int32),
        ("action_mode", C.c_int32),
        ("onehot_dtype", C.c_int32),
        ("num_games", C.c_int64),
        ("slot_base", C.c_int64),
        ("board_in", C.c_void_p),
        ("board_out", C.c_void_p),
        ("valid_in", C.c_void_p),
        ("valid_out", C.c_void_p),
        ("actions", C.c_void_p),
        ("actions_out", C.c_void_p),
        ("step", C.c_void_p),
        ("score", C.c_void_p),
        ("reward", C.c_void_p),
        ("terminated", C.c_void_p),
        ("invalid", C.c_void_p),
        ("merged", C.c_void_p),
        ("onehot_out", C.c_void_p),
        ("randperm_keys", C.c_void_p),
        ("rand_seed", C.c_int64),
        ("two_mask", C.c_uint32),
        ("two_threshold", C.c_uint32),
        ("philox_seed", C.c_uint64),
        ("philox_counter", C.c_uint64),
        ("stats", C.c_void_p),
        ("sched", C.c_void_p),
        ("sched_cursor", C.c_void_p),
        ("sched_cursor_next", C.c_void_p),
        ("table_stride", C.c_int64),
        ("id", C.c_void_p),
        ("episode_id_base", C.c_int64),
        ("episode_capacity", C.c_int64),
        ("episode_steps", C.c_void_p),
        ("episode_score", C.c_void_p),
        ("episode_max_tile", C.c_void_p),
        ("logits", C.c_void_p),
        ("log_prob_out", C.c_void_p),
        ("tr_state", C.c_void_p),
        ("tr_valid_actions", C.c_void_p),
        ("tr_action", C.c_void_p),
        ("tr_reward", C.c_void_p),
        ("tr_next_state", C.c_void_p),
        ("tr_next_valid_actions", C.c_void_p),
        ("tr_step", C.c_void_p),
        ("tr_terminated", C.c_void_p),
        ("age", C.c_void_p),
        ("traj_id_base", C.c_int64),
        ("traj_capacity", C.c_int64),
        ("traj_max_rows", C.c_int64),
        ("traj_state", C.c_void_p),
        ("traj_action", C.c_void_p),
        ("traj_score", C.c_void_p),
        ("traj_rows", C.c_void_p),
        ("reset_rank", C.c_void_p),
        ("reset_chunk_base", C.c_void_p),
        ("reset_id_base", C.c_void_p),
        ("reset_indices", C.c_void_p),
        ("randperm", C.c_void_p),
        ("rand_base", C.c_int64),
        ("prepare_philox_counter", C.c_uint64),
    ]


class PrepareArgs(C.Structure):
    """ml2048_prepare_args"""

    _fields_ = [
        ("struct_size", C.c_uint32),
        ("rng_mode", C.c_int32),
        ("onehot_dtype", C.c_int32),
        ("reserved0", C.c_int32),
        ("num_games", C.c_int64),
        ("slot_base", C.c_int64),
        ("board", C.c_void_p),
        ("valid", C.c_void_p),
        ("id", C.c_void_p),
        ("step", C.c_void_p),
        ("score", C.c_void_p),
        ("reward", C.c_void_p),
        ("terminated", C.c_void_p),
        ("invalid", C.c_void_p),
        ("merged", C.c_void_p),
        ("onehot", C.c_void_p),
        ("randperm", C.c_void_p),
        ("rand_base", C.c_int64),
        ("two_mask", C.c_uint32),
        ("two_threshold", C.c_uint32),
        ("philox_seed", C.c_uint64),
        ("philox_counter", C.c_uint64),
        ("game_count", C.c_void_p),
        ("id_offset", C.c_void_p),
        ("reset_count", C.c_void_p),
        ("reset_indices", C.c_void_p),
        ("scratch", C.c_void_p),
        ("sched", C.c_void_p),
        ("sched_cursor", C.c_void_p),
        ("table_stride", C.c_int64),
        ("age", C.c_void_p),
    ]


class Compressible(C.Structure):
    """ml2048_compressible"""

    _fields_ = [
        ("ptr", C.c_uint64),
        ("size", C.c_uint64),
        ("granted", C.c_uint64),
        ("device", C.c_int32),
        ("chunks", C.c_int32),
        ("handles", C.c_uint64 * COMPRESSIBLE_MAX_CHUNKS),
    ]


class Pcg64(C.Structure):
    """ml2048_pcg64"""

    _fields_ = [
        ("state_hi", C.c_uint64),
        ("state_lo", C.c_uint64),
        ("inc_hi", C.c_uint64),
        ("inc_lo", C.c_uint64),
        ("has_uint32", C.c_int32),
        ("uinteger", C.c_uint32),
    ]


# every symbol include/ml2048_b200.h declares: (name, restype, argtypes)
_VP, _I64, _I32, _U64, _U32 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint32
SYMBOLS = {
    "ml2048_abi_version": (C.c_int, []),
    "ml2048_prepare_scratch_ints": (_I64, [_I64]),
    "ml2048_step": (C.c_int, [C.POINTER(StepArgs), _VP]),
    "ml2048_prepare": (C.c_int, [C.POINTER(PrepareArgs), _VP]),
    "ml2048_prepare_count": (C.c_int, [C.POINTER(PrepareArgs), _VP]),
    "ml2048_prepare_apply": (C.c_int, [C.POINTER(PrepareArgs), _VP]),
    "ml2048_autoreset_scratch_ints": (_I64, [_I64]),
    "ml2048_autoreset_scan": (C.c_int, [_VP, _VP, _VP, _I64, _VP, _VP, _VP, _VP, _VP, _VP]),
    "ml2048_reset_state": (C.c_int, [_VP] * 11 + [_I64, _VP]),
    "ml2048_encode_onehot": (C.c_int, [_VP, _VP, _I32, _I64, _VP]),
    "ml2048_valid_actions": (C.c_int, [_VP, _VP, _I64, _VP]),
    "ml2048_afterstates": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _I32, _I64, _VP]),
    "ml2048_ntuple_value": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_ntuple_greedy": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _I64, _VP]),
    "ml2048_ntuple_td_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_expectimax": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _I32, _I32, C.c_double] + [_VP] * 6 + [_I64, _VP]),
    "ml2048_tc_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_lambda_td_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP, _I64,
                                          _VP]),
    "ml2048_lambda_tc_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP, _I32,
                                          _VP, _I64, _VP]),
    "ml2048_staged_value": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_staged_greedy": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _I64, _VP]),
    "ml2048_staged_td_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_staged_tc_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_staged_lambda_td_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP,
                                                 _I32, _VP, _I64, _VP]),
    "ml2048_staged_lambda_tc_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP,
                                                 _I32, _VP, _I32, _VP, _I64, _VP]),
    "ml2048_staged_expectimax": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _I32, _I32, C.c_double] + [_VP] * 6 + [_I64, _VP]),
    "ml2048_promoted_value": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _VP, _I64, _VP]),
    "ml2048_promoted_greedy": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _I32, _VP, _VP, _VP, _VP, _VP, _I64, _VP]),
    "ml2048_promoted_td_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _VP, _I64, _VP]),
    "ml2048_promoted_tc_update": (C.c_int, [_VP, _VP, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _VP, _I64,
                                            _VP]),
    "ml2048_promoted_lambda_td_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _I64, _VP, _VP, _I32, _VP,
                                                   _I32, _VP, _VP, _I64, _VP]),
    "ml2048_promoted_lambda_tc_update": (C.c_int, [_VP, _VP, _VP, _I32, _I32, C.c_float, _VP, C.c_float, _VP, _VP, _VP, _I64, _VP, _VP,
                                                   _I32, _VP, _I32, _VP, _VP, _I64, _VP]),
    "ml2048_promoted_expectimax": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _I32, _VP, _I32, _VP, _I32, _I32, C.c_double] + [_VP] * 6
                                   + [_I64, _VP]),
    "ml2048_max_tile_hist": (C.c_int, [_VP, _VP, _I64, _VP, _VP]),
    "ml2048_copy_async": (C.c_int, [_VP, _VP, _I64, _VP]),
    "ml2048_stream_wait": (C.c_int, [_VP]),
    "ml2048_alloc_compressible": (C.c_int, [_I32, _I64, C.POINTER(Compressible)]),
    "ml2048_free_compressible": (C.c_int, [C.POINTER(Compressible)]),
    "ml2048_pack_flags": (C.c_int, [_VP, _VP, _VP, _VP, _I64, _VP]),
    "ml2048_unpack_flags": (None, [_VP, _I64, _VP, _VP, _VP, _I32]),
    "ml2048_unpack_flags_sliced": (C.c_int, [_VP, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _I32]),
    "ml2048_sample_random_valid": (C.c_int, [_VP, _VP, _I64, _I64, _U64, _U64, _VP]),
    "ml2048_sample_masked_categorical": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _I64, _I64, _U64, _U64, _VP]),
    "ml2048_gae": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _I64, _I64, _I64, C.c_float, C.c_float, _VP]),
    "ml2048_two_mask": (_U32, [_VP, C.c_double]),
    "ml2048_two_threshold": (_U32, [C.c_double]),
    "ml2048_philox_epoch_draws": (None, [_U64, _U64, C.c_double, C.POINTER(_U32), C.POINTER(_U32)]),
    "ml2048_philox4x32_10": (None, [_VP, _VP, _VP]),
    "ml2048_philox2x32_10": (None, [_VP, _U32, _VP]),
    "ml2048_pack_randperm_keys": (C.c_int, [_VP, _VP, _I64]),
    "ml2048_pcg64_random": (C.c_double, [C.POINTER(Pcg64)]),
    "ml2048_pcg64_integers": (_I64, [C.POINTER(Pcg64), _I64]),
    "ml2048_pcg64_random_f32": (None, [C.POINTER(Pcg64), _VP, _I64]),
    "ml2048_pcg64_permuted_rows_u8": (None, [C.POINTER(Pcg64), _VP, _I64, _I64]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raise (never fall back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m ml2048_b200.build` (nvcc, sm_100a). "
            "ml2048_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.ml2048_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libml2048_b200.so ABI {got} != expected {ABI_VERSION}: rebuild it")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f"{what}: argument error {rc} ({ERRORS.get(rc, '?')})")
    raise RuntimeError(f"{what}: CUDA error {rc}")
