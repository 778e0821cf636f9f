"""ctypes loader for libtwixt_b200.so (the C ABI of include/twixt_b200.h).

The library is the product: there is no Python or CPU implementation behind
it.  If it is missing it is built with nvcc (sm_100a cross-compiles without a
GPU); if that fails the import fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os


_lib = None


class GameInfo(C.Structure):
    _fields_ = [
        ("board_size", C.c_int32),
        ("num_distinct_actions", C.c_int32),
        ("num_players", C.c_int32),
        ("max_game_length", C.c_int32),
        ("obs_shape", C.c_int32 * 3),
        ("obs_size", C.c_int32),
        ("max_legal_actions", C.c_int32),
        ("record_words", C.c_int32),
        ("min_utility", C.c_double),
        ("max_utility", C.c_double),
        ("utility_sum", C.c_double),
    ]


class StepResult(C.Structure):
    _fields_ = [
        ("status", C.c_int32),
        ("current_player", C.c_int32),
        ("is_terminal", C.c_int32),
        ("num_legal", C.c_int32),
        ("returns", C.c_float * 2),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("plies", C.c_int64),
        ("games", C.c_int64),
        ("red_wins", C.c_int64),
        ("blue_wins", C.c_int64),
        ("draws", C.c_int64),
        ("swaps", C.c_int64),
        ("max_length", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("debug_violations", C.c_int64),
    ]


# every symbol include/twixt_b200.h declares: (name, restype, argtypes)
_P = C.c_void_p
_I64 = C.c_int64
SYMBOLS = [
    ("twixt_last_error", C.c_char_p, []),
    ("twixt_version", C.c_char_p, []),
    ("twixt_game_info_for", C.c_int, [C.c_int, C.POINTER(GameInfo)]),
    ("twixt_create", C.c_int, [C.c_int, _I64, C.c_int, C.c_uint64, C.POINTER(_P)]),
    ("twixt_destroy", None, [_P]),
    ("twixt_get_info", C.c_int, [_P, C.POINTER(GameInfo)]),
    ("twixt_num_envs", _I64, [_P]),
    ("twixt_set_stream", C.c_int, [_P, C.c_size_t]),
    ("twixt_get_stream", C.c_size_t, [_P]),
    ("twixt_synchronize", C.c_int, [_P]),
    ("twixt_set_seed", C.c_int, [_P, C.c_uint64]),
    ("twixt_set_stream_base", C.c_int, [_P, C.c_uint64]),
    ("twixt_reset", C.c_int, [_P, _I64, _I64]),
    ("twixt_clone", C.c_int, [_P, _I64, _I64, _I64]),
    ("twixt_clone_gather", C.c_int, [_P, _P, _I64, _I64]),
    ("twixt_clone_from", C.c_int, [_P, _I64, _P, _I64, _I64]),
    ("twixt_legal_actions", C.c_int, [_P, _I64, _I64, _P, C.c_int32, _I64, _P]),
    ("twixt_legal_mask", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_apply", C.c_int, [_P, _I64, _I64, _P, _P]),
    ("twixt_current_player", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_is_terminal", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_returns", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_observation", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_observation_and_mask", C.c_int, [_P, _I64, _I64, _P, _P]),
    ("twixt_replay", C.c_int, [_P, _I64, _I64, _P, _I64, _P, _P]),
    ("twixt_playout", C.c_int, [_P, _I64, _I64, C.c_int32, _P, _P, _P, _P, C.c_int32]),
    ("twixt_export_state", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_import_state", C.c_int, [_P, _I64, _I64, _P]),
    ("twixt_step", C.c_int, [_P, _I64, C.c_int32, C.POINTER(StepResult), _P]),
    ("twixt_set_validation", C.c_int, [_P, C.c_int]),
    ("twixt_shard_range", C.c_int, [_I64, C.c_int32, C.c_int32, C.POINTER(_I64), C.POINTER(_I64)]),
    ("twixt_stats_accumulate", C.c_int, [C.POINTER(Stats), C.POINTER(Stats)]),
    ("twixt_get_stats", C.c_int, [_P, C.POINTER(Stats)]),
    ("twixt_stats_reset", C.c_int, [_P]),
    ("twixt_mcts_create", C.c_int, [_P, _I64, C.c_int32, C.c_int32, C.c_double, C.POINTER(_P)]),
    ("twixt_mcts_destroy", None, [_P]),
    ("twixt_mcts_begin", C.c_int, [_P, _I64, _I64]),
    ("twixt_mcts_run", C.c_int, [_P, C.c_int32]),
    ("twixt_mcts_select", C.c_int, [_P, _I64, _P]),
    ("twixt_mcts_backup", C.c_int, [_P, _P]),
    ("twixt_mcts_root_stats", C.c_int, [_P, _P, _P, _P]),
    ("twixt_mcts_create_puct", C.c_int, [_P, _I64, C.c_int32, C.c_int32, C.c_double, C.POINTER(_P)]),
    ("twixt_mcts_backup_priors", C.c_int, [_P, _P, _P]),
    ("twixt_mcts_create_ex", C.c_int, [_P, _I64, C.c_int32, C.c_int32, C.c_double, C.c_uint32, C.POINTER(_P)]),
    ("twixt_mcts_solver_stats", C.c_int, [_P, _P, _P, _P, _P]),
    ("twixt_mcts_create_parallel", C.c_int, [_P, _I64, C.c_int32, C.c_int32, C.c_double, C.c_uint32, C.c_int32,
                                             C.c_double, C.POINTER(_P)]),
    ("twixt_mcts_advance", C.c_int, [_P, _P, C.c_int32, _P]),
    ("twixt_mcts_set_root_priors", C.c_int, [_P, _P]),
    ("twixt_mcts_create_gumbel", C.c_int, [_P, _I64, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                           C.POINTER(_P)]),
    ("twixt_mcts_set_root_gumbel", C.c_int, [_P, _P]),
    ("twixt_mcts_gumbel_stats", C.c_int, [_P, _P, _P]),
]

OK, EINVAL, ECUDA, EILLEGAL, ENOMEM = 0, -1, -2, -3, -4


def library_path() -> str:
    from . import build as _build  # lazily: `python -m twixt_for_open_spiel_b200.build` imports this package first
    return _build.LIB


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("TWIXT_B200_LIB")  # tests only: a variant build of the same sources
    if override:
        lib = C.CDLL(override)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
        return lib
    from . import build as _build
    if not os.path.exists(_build.LIB) or (os.environ.get("TWIXT_B200_REBUILD") == "1"):
        _build.build(force=True)
    elif _build.needs_build():
        try:
            _build.nvcc_path()
        except RuntimeError:
            pass  # no compiler on this machine: the present library is all there is
        else:
            _build.build()  # a compile or link error in edited sources must surface, not hide behind a stale binary
    lib = C.CDLL(_build.LIB)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib
