"""ctypes binding of the C ABI declared in include/cattus_b200.h.

This is the Python counterpart of the Rust FFI stub shown in INTEGRATION.md: same symbols, same argument meaning.
The library is mandatory: importing this module on a machine without libcattus_b200.so raises, and `create`
fails with ENODEV when no sm_100 device is present.  There is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

OK, EINVAL, ENODEV, ECUDA, ENOMEM, ERANGE, EDEVICE = 0, -1, -2, -3, -4, -5, -6
GAME_TTT, GAME_HEX, GAME_CHESS = 0, 1, 2
PRECISION_BF16, PRECISION_FP32_CHECK, PRECISION_FP8 = 0, 1, 2
PRECISION_IDS = {"bf16": PRECISION_BF16, "fp32-check": PRECISION_FP32_CHECK, "fp8": PRECISION_FP8}
TRUNK_PER_LAYER, TRUNK_FUSED, TRUNK_SMALL, TRUNK_FP32, TRUNK_DENSE = 0, 1, 2, 3, 4
TRUNK_PATH_NAMES = {TRUNK_PER_LAYER: "per-layer", TRUNK_FUSED: "fused", TRUNK_SMALL: "small", TRUNK_FP32: "fp32-check", TRUNK_DENSE: "dense"}
GAME_IDS = {"ttt": GAME_TTT, "hex": GAME_HEX, "chess": GAME_CHESS}


class Desc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("game", C.c_uint32), ("board_size", C.c_uint32), ("planes", C.c_uint32),
        ("moves", C.c_uint32), ("filters", C.c_uint32), ("blocks", C.c_uint32), ("value_channels", C.c_uint32),
        ("policy_channels", C.c_uint32), ("device", C.c_int32), ("max_batch", C.c_uint32), ("n_streams", C.c_uint32),
        ("precision", C.c_uint32), ("flags", C.c_uint32), ("weights_path", C.c_char_p),
    ]


class Metrics(C.Structure):
    _fields_ = [
        ("activation_count", C.c_uint64), ("positions", C.c_uint64), ("run_duration_last", C.c_double),
        ("run_duration_ema", C.c_double), ("mean_batch_fill", C.c_double), ("kernel_launches", C.c_uint64),
    ]


class Info(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in (
        "game", "board_size", "planes", "moves", "filters", "blocks", "value_channels", "policy_channels",
        "words_per_plane", "legal_bitmap_bytes", "max_batch", "n_streams", "precision", "sm_count",
        "kernels_per_batch", "trunk_path")]


class SelfPlayCfg(C.Structure):
    """cattus_b200_selfplay_cfg (include/cattus_b200_selfplay.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("game", C.c_uint32), ("board_size", C.c_uint32), ("sim_num", C.c_uint32),
        ("explore_factor", C.c_float), ("temperature_moves", C.POINTER(C.c_uint32)), ("temperature_values", C.POINTER(C.c_float)),
        ("n_temperatures", C.c_uint32), ("prior_noise_alpha", C.c_float), ("prior_noise_epsilon", C.c_float),
        ("cache_size", C.c_uint32), ("threads", C.c_uint32), ("games_per_thread", C.c_uint32), ("leaf_queue", C.c_uint32),
        ("games_num", C.c_uint32), ("first_game", C.c_uint32), ("game_stride", C.c_uint32), ("seed", C.c_uint64),
        ("out_dir1", C.c_char_p), ("out_dir2", C.c_char_p), ("keep_records", C.c_uint32), ("groups_per_thread", C.c_uint32),
        ("max_moves", C.c_uint32), ("speculate", C.c_uint32), ("device_games", C.c_uint32), ("device_tree_kwords", C.c_uint32),
        ("device_waves_in_flight", C.c_uint32),
    ]


class SelfPlaySummary(C.Structure):
    _fields_ = [
        ("player1_wins", C.c_uint32), ("player2_wins", C.c_uint32), ("draws", C.c_uint32), ("games", C.c_uint32),
        ("simulations", C.c_uint64), ("searches", C.c_uint64), ("evaluations", C.c_uint64), ("cache_hits", C.c_uint64),
        ("cache_misses", C.c_uint64), ("batches", C.c_uint64), ("terminal_leaves", C.c_uint64), ("seconds", C.c_double),
        ("search_duration", C.c_double), ("eval_wait_seconds", C.c_double), ("speculative_evaluations", C.c_uint64),
    ]


class ChessSearchStats(C.Structure):
    """cattus_b200_chess_search_stats (include/cattus_b200_selfplay.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("root_children", C.c_uint32), ("best_visits", C.c_uint32), ("speculative_evaluations", C.c_uint32),
        ("simulations", C.c_uint64), ("evaluations", C.c_uint64), ("cache_hits", C.c_uint64), ("terminal_leaves", C.c_uint64),
        ("seconds", C.c_double),
    ]


class ChessInfo(C.Structure):
    """cattus_b200_chess_info (include/cattus_b200_chess.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("turn", C.c_uint32), ("status", C.c_uint32), ("fifty_rule_count", C.c_uint32),
        ("in_check", C.c_uint32), ("n_legal", C.c_uint32), ("planes", C.c_uint64 * 18), ("legal_bitmap", C.c_uint8 * 235),
        ("pad", C.c_uint8), ("moves", C.c_uint16 * 224), ("nn_index", C.c_uint16 * 224),
    ]


class AnalysisPosition(C.Structure):
    """cattus_b200_analysis_position (include/cattus_b200_analysis.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("status", C.c_uint32), ("n_children", C.c_uint32), ("pv_len", C.c_uint32),
        ("simulations", C.c_uint32), ("best_move", C.c_uint16), ("pad", C.c_uint16), ("q", C.c_float),
    ]


class AnalysisOpts(C.Structure):
    """cattus_b200_analysis_opts (include/cattus_b200_analysis.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("search_batch", C.c_uint32)]


class SelfPlayOpts(C.Structure):
    """cattus_b200_selfplay_opts (include/cattus_b200_selfplay.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("search_batch", C.c_uint32)]


class MatchOpts(C.Structure):
    """cattus_b200_match_opts (include/cattus_b200_match.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("search_batch_a", C.c_uint32), ("search_batch_b", C.c_uint32)]


class MatchSide(C.Structure):
    """cattus_b200_match_side (include/cattus_b200_match.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("sim_num", C.c_uint32), ("explore_factor", C.c_float)]


class MatchSummary(C.Structure):
    """cattus_b200_match_summary (include/cattus_b200_match.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("a_wins", C.c_uint32), ("b_wins", C.c_uint32), ("draws", C.c_uint32), ("games", C.c_uint32),
        ("openings", C.c_uint32), ("skipped", C.c_uint32), ("pairs", C.c_uint32 * 5), ("simulations", C.c_uint64),
        ("evaluations", C.c_uint64), ("seconds", C.c_double),
    ]


class MatchGame(C.Structure):
    """cattus_b200_match_game (include/cattus_b200_match.h)."""
    _fields_ = [(n, C.c_uint32) for n in ("struct_size", "opening", "a_is_player1", "winner", "termination", "n_moves")]


class SessionOpts(C.Structure):
    """cattus_b200_session_opts (include/cattus_b200_session.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("search_batch", C.c_uint32), ("tree_kwords", C.c_uint32)]


class SessionLimits(C.Structure):
    """cattus_b200_session_limits (include/cattus_b200_session.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("nodes", C.c_uint32), ("minibatches", C.c_uint32), ("pad", C.c_uint32), ("deadline_us", C.c_uint64)]


class SessionSnapshot(C.Structure):
    """cattus_b200_session_snapshot (include/cattus_b200_session.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("valid", C.c_uint32), ("searching", C.c_uint32), ("simulations", C.c_uint32), ("minibatches", C.c_uint32),
        ("collisions", C.c_uint32), ("best_move", C.c_uint16), ("pv_len", C.c_uint16), ("q", C.c_float), ("seconds", C.c_double),
        ("pv", C.c_uint16 * 16),
    ]


class SessionStats(C.Structure):
    """cattus_b200_session_stats (include/cattus_b200_session.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("stop_reason", C.c_uint32), ("reused_visits", C.c_uint32), ("pad", C.c_uint32), ("seconds", C.c_double)]


SESSION_RUNNING = 1

# every symbol include/*.h declares: name -> (restype, argtypes)
_H = C.c_void_p
_u16p = C.POINTER(C.c_uint16)
_u64p, _u8p, _f32p, _u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_uint32)
SYMBOLS = {
    "cattus_b200_create": (C.c_int, [C.POINTER(Desc), C.POINTER(_H)]),
    "cattus_b200_create_from_memory": (C.c_int, [C.POINTER(Desc), C.c_void_p, C.c_size_t, C.POINTER(_H)]),
    "cattus_b200_destroy": (None, [_H]),
    "cattus_b200_get_info": (C.c_int, [_H, C.POINTER(Info)]),
    "cattus_b200_eval": (C.c_int, [_H, _u64p, _u8p, _f32p, C.c_uint32, _u32p, _f32p]),
    "cattus_b200_eval_batch": (C.c_int, [_H, _u64p, _u8p, C.c_uint32, _f32p, C.c_size_t, _u32p, _f32p]),
    "cattus_b200_eval_batch_submit": (C.c_int, [_H, _u64p, _u8p, C.c_uint32, C.c_int, C.POINTER(C.c_int32)]),
    "cattus_b200_eval_batch_wait": (C.c_int, [_H, C.c_int32, _f32p, C.c_size_t, _u32p, _f32p]),
    "cattus_b200_encode": (C.c_int, [_H, _u64p, C.c_uint32, C.c_uint32, _f32p]),
    "cattus_b200_run_dense": (C.c_int, [_H, _f32p, C.c_uint32, _f32p, _f32p]),
    "cattus_b200_resident_upload": (C.c_int, [_H, _u64p, _u8p, C.c_uint32]),
    "cattus_b200_eval_resident": (C.c_int, [_H, C.c_uint32, C.c_void_p]),
    "cattus_b200_resident_download": (C.c_int, [_H, C.c_uint32, _f32p, C.c_size_t, _u32p, _f32p]),
    "cattus_b200_time_stage": (C.c_int, [_H, C.c_uint32, C.c_uint32, C.c_uint32, _f32p]),
    "cattus_b200_time_sustained": (C.c_int, [_H, _u64p, _u8p, C.c_uint32, C.c_uint32, C.c_uint32, _f32p]),
    "cattus_b200_get_metrics": (C.c_int, [_H, C.POINTER(Metrics)]),
    "cattus_b200_last_error": (C.c_char_p, []),
    "cattus_b200_abi_version": (C.c_uint32, []),
    # include/cattus_b200_selfplay.h
    "cattus_b200_selfplay_run": (C.c_int, [_H, _H, C.POINTER(SelfPlayCfg), C.POINTER(_H)]),
    "cattus_b200_selfplay_run_with": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SelfPlayCfg), C.POINTER(_H)]),
    "cattus_b200_selfplay_run_opts": (C.c_int, [_H, _H, C.POINTER(SelfPlayCfg), C.POINTER(SelfPlayOpts), C.POINTER(_H)]),
    "cattus_b200_selfplay_summary_get": (C.c_int, [_H, C.POINTER(SelfPlaySummary)]),
    "cattus_b200_selfplay_batches": (C.c_int, [_H, _u64p, _u64p]),
    "cattus_b200_selfplay_game_count": (C.c_int, [_H, _u32p]),
    "cattus_b200_selfplay_game_info": (C.c_int, [_H, C.c_uint32, _u32p, _u32p, _u32p]),
    "cattus_b200_selfplay_game_moves": (C.c_int, [_H, C.c_uint32, _u8p, C.c_uint32]),
    "cattus_b200_selfplay_game_moves16": (C.c_int, [_H, C.c_uint32, _u16p, C.c_uint32]),
    "cattus_b200_selfplay_entry": (C.c_int, [_H, C.c_uint32, C.c_uint32, _u8p, C.c_size_t, C.POINTER(C.c_size_t), _u32p]),
    "cattus_b200_selfplay_free": (None, [_H]),
    "cattus_b200_selfplay_last_error": (C.c_char_p, []),
    "cattus_b200_chess_search_create": (C.c_int, [_H, C.POINTER(SelfPlayCfg), C.POINTER(_H)]),
    "cattus_b200_chess_search_create_with": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(SelfPlayCfg), C.POINTER(_H)]),
    "cattus_b200_chess_search_go": (C.c_int, [_H, C.c_char_p, _u16p, C.c_uint32, _u16p, C.POINTER(ChessSearchStats)]),
    "cattus_b200_chess_search_destroy": (None, [_H]),
    # include/cattus_b200_analysis.h
    "cattus_b200_analyse": (C.c_int, [_H, C.POINTER(SelfPlayCfg), C.c_uint32, C.POINTER(C.c_char_p), _u16p, _u32p, C.POINTER(_H)]),
    "cattus_b200_analysis_count": (C.c_int, [_H, _u32p]),
    "cattus_b200_analysis_get": (C.c_int, [_H, C.c_uint32, C.POINTER(AnalysisPosition)]),
    "cattus_b200_analysis_children": (C.c_int, [_H, C.c_uint32, _u16p, _u32p, _f32p, _f32p, C.c_uint32]),
    "cattus_b200_analysis_pv": (C.c_int, [_H, C.c_uint32, _u16p, C.c_uint32]),
    "cattus_b200_analyse_opts": (C.c_int, [_H, C.POINTER(SelfPlayCfg), C.POINTER(AnalysisOpts), C.c_uint32, C.POINTER(C.c_char_p), _u16p, _u32p,
                                           C.POINTER(_H)]),
    "cattus_b200_analysis_batches": (C.c_int, [_H, C.c_uint32, _u32p, _u32p]),
    "cattus_b200_analysis_free": (None, [_H]),
    # include/cattus_b200_match.h
    "cattus_b200_match_run": (C.c_int, [_H, _H, C.POINTER(SelfPlayCfg), C.POINTER(MatchSide), C.c_uint32, C.POINTER(C.c_char_p), _u16p, _u32p,
                                        C.POINTER(_H)]),
    "cattus_b200_match_run_opts": (C.c_int, [_H, _H, C.POINTER(SelfPlayCfg), C.POINTER(MatchSide), C.POINTER(MatchOpts), C.c_uint32,
                                             C.POINTER(C.c_char_p), _u16p, _u32p, C.POINTER(_H)]),
    "cattus_b200_match_summary_get": (C.c_int, [_H, C.POINTER(MatchSummary)]),
    "cattus_b200_match_batches": (C.c_int, [_H, C.c_uint32, _u64p, _u64p]),
    "cattus_b200_match_opening_status": (C.c_int, [_H, C.c_uint32, _u32p]),
    "cattus_b200_match_game_get": (C.c_int, [_H, C.c_uint32, C.POINTER(MatchGame)]),
    "cattus_b200_match_game_moves": (C.c_int, [_H, C.c_uint32, _u16p, C.c_uint32]),
    "cattus_b200_match_free": (None, [_H]),
    # include/cattus_b200_session.h
    "cattus_b200_session_create": (C.c_int, [_H, C.POINTER(SelfPlayCfg), C.POINTER(SessionOpts), C.POINTER(_H)]),
    "cattus_b200_session_set_position": (C.c_int, [_H, C.c_char_p, _u16p, C.c_uint32]),
    "cattus_b200_session_new_game": (C.c_int, [_H]),
    "cattus_b200_session_go": (C.c_int, [_H, C.POINTER(SessionLimits)]),
    "cattus_b200_session_stop": (C.c_int, [_H]),
    "cattus_b200_session_info": (C.c_int, [_H, C.POINTER(SessionSnapshot)]),
    "cattus_b200_session_wait": (C.c_int, [_H, C.c_uint32, C.POINTER(_H)]),
    "cattus_b200_session_result_stats": (C.c_int, [_H, C.POINTER(SessionStats)]),
    "cattus_b200_session_destroy": (None, [_H]),
    # include/cattus_b200_chess.h
    "cattus_b200_chess_position": (C.c_int, [C.c_char_p, _u16p, C.c_uint32, C.POINTER(ChessInfo)]),
    "cattus_b200_chess_perft": (C.c_int, [C.c_char_p, C.c_uint32, C.POINTER(C.c_uint64)]),
    "cattus_b200_chess_nn_table": (C.c_int, [_u16p, C.c_uint32]),
    "cattus_b200_chess_last_error": (C.c_char_p, []),
}

EVAL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, _u64p, _u8p, C.c_uint32, _f32p, C.c_size_t, _u32p, _f32p)

_lib = None


def library_path() -> Path:
    return _build.LIB


def load() -> C.CDLL:
    """Loads (building first if the sources are newer) the shared library and types every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build()
    lib = C.CDLL(str(path))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class CattusB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"cattus_b200 error {code}: {message}")
        self.code = code


def check(rc: int) -> None:
    if rc != OK:
        raise CattusB200Error(rc, (load().cattus_b200_last_error() or b"").decode(errors="replace"))
