"""ctypes wrapper of tests/emul/libmatch_emul.so (TEST INFRASTRUCTURE): match play from openings over the host emulation
of the device-resident search, with Python evaluator callbacks."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

from cattus_b200 import _lib
from cattus_b200.analysis import encode_positions
from cattus_b200.match import collect, side_struct
from cattus_b200.selfplay import SelfPlayRunner, _eval_thunk, parse_game

HERE = Path(__file__).resolve().parent
SO = HERE / "libmatch_emul.so"
SRC = HERE / "match_emul.cpp"
CSRC = HERE.parent.parent / "cattus_b200" / "csrc"


def build() -> Path:
    deps = [SRC, HERE / "dsearch_emul.cpp"] + sorted(CSRC.glob("*.hpp")) + sorted((HERE.parent.parent / "include").glob("*.h"))
    if SO.exists() and all(d.stat().st_mtime <= SO.stat().st_mtime for d in deps):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-fno-strict-aliasing", "-o", str(SO), str(SRC)],
                   check=True)
    return SO


_cached = None


def load():
    global _cached
    if _cached is None:
        lib = C.CDLL(str(build()))
        lib.match_emul_run.restype = C.c_void_p
        lib.match_emul_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_char_p), C.POINTER(C.c_uint16),
                                       C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        lib.match_emul_error.restype = C.c_char_p
        lib.match_emul_error.argtypes = [C.c_void_p]
        lib.match_emul_summary.argtypes = [C.c_void_p, C.POINTER(_lib.MatchSummary)]
        lib.match_emul_opening_status.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        lib.match_emul_game.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_lib.MatchGame)]
        lib.match_emul_game_moves.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16), C.c_uint32]
        lib.match_emul_free.argtypes = [C.c_void_p]
        _cached = lib
    return _cached


def play(game: str, openings, cfg: dict, eval_a, eval_b=None, *, sim_num_b=None, explore_factor_b=None, n_slots: int, pool_words: int = 1 << 16,
         depth: int = 2, roots_cap: int = 0):
    """-> MatchResult; raises RuntimeError with the driver's message.  eval_b None: one evaluator (and cache) for both
    sides.  depth: dsearch_emul_run's knobs (waves in flight | 256 begin overlapped | 512 two populations); roots_cap:
    history positions one wave uploads."""
    lib = load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    g, s = parse_game(game)
    chess = g == _lib.GAME_CHESS
    words = 18 if chess else 3 * ((s * s + 63) // 64)
    errors: list = []
    ta = _eval_thunk(eval_a, words, chess, errors)
    tb = _eval_thunk(eval_b, words, chess, errors) if eval_b is not None else None
    n, fa, ma, oa = encode_positions(game, openings)
    side = side_struct(sim_num_b, explore_factor_b)
    h = lib.match_emul_run(C.cast(ta, C.c_void_p), C.cast(tb, C.c_void_p) if tb else None, C.byref(c), C.byref(side) if side is not None else None,
                           n, fa, ma, oa, n_slots, pool_words, depth, roots_cap)
    try:
        if errors:
            raise errors[0]
        err = lib.match_emul_error(h)
        if err:
            raise RuntimeError(err.decode())
        return collect(lib.match_emul_summary, lib.match_emul_opening_status, lib.match_emul_game, lib.match_emul_game_moves, h)
    finally:
        lib.match_emul_free(h)
