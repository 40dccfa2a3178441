"""ctypes wrapper of tests/emul/libselfplay_batch_emul.so (TEST INFRASTRUCTURE): self-play and match play with per-side
minibatches under virtual loss over the host emulation of the device-resident search, with Python evaluator callbacks."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

from cattus_b200 import _lib
from cattus_b200.analysis import encode_positions
from cattus_b200.match import collect, opts_struct, side_struct
from cattus_b200.selfplay import GameRecord, SelfPlayRunner, _eval_thunk, parse_game

HERE = Path(__file__).resolve().parent
SO = HERE / "libselfplay_batch_emul.so"
SRC = HERE / "selfplay_batch_emul.cpp"
CSRC = HERE.parent.parent / "cattus_b200" / "csrc"


def build() -> Path:
    deps = [SRC, HERE / "match_emul.cpp", HERE / "dsearch_emul.cpp"] + sorted(CSRC.glob("*.hpp")) + sorted((HERE.parent.parent / "include").glob("*.h"))
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
        lib.selfplay_batch_emul_run.restype = C.c_void_p
        lib.selfplay_batch_emul_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                                C.POINTER(C.c_int)]
        lib.selfplay_batch_emul_batches.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        lib.dsearch_emul_error.restype = C.c_char_p
        lib.dsearch_emul_error.argtypes = [C.c_void_p]
        lib.dsearch_emul_game_count.restype = C.c_uint32
        lib.dsearch_emul_game_count.argtypes = [C.c_void_p]
        lib.dsearch_emul_counters.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        lib.dsearch_emul_game_info.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        lib.dsearch_emul_game_moves.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16)]
        lib.dsearch_emul_entry.restype = C.c_uint32
        lib.dsearch_emul_entry.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint8), C.c_uint32, C.POINTER(C.c_uint32)]
        lib.dsearch_emul_free.argtypes = [C.c_void_p]
        lib.match_batch_emul_run.restype = C.c_void_p
        lib.match_batch_emul_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                             C.POINTER(C.c_char_p), C.POINTER(C.c_uint16), C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32,
                                             C.c_uint32, C.POINTER(C.c_int)]
        lib.match_batch_emul_batches.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        lib.match_emul_error.restype = C.c_char_p
        lib.match_emul_error.argtypes = [C.c_void_p]
        lib.match_emul_summary.argtypes = [C.c_void_p, C.POINTER(_lib.MatchSummary)]
        lib.match_emul_opening_status.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        lib.match_emul_game.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_lib.MatchGame)]
        lib.match_emul_game_moves.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16), C.c_uint32]
        lib.match_emul_free.argtypes = [C.c_void_p]
        _cached = lib
    return _cached


class EmulError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


def _words(game):
    g, s = parse_game(game)
    chess = g == _lib.GAME_CHESS
    return (18 if chess else 3 * ((s * s + 63) // 64)), chess


def selfplay(game: str, cfg: dict, eval1, eval2, games_num: int, *, search_batch=None, opts_size: int = 0, max_batch: int = 4096,
             pool_words: int = 1 << 16, depth: int = 2):
    """-> (counters dict with per-model "minibatches" / "collisions" pairs, [GameRecord]); raises EmulError(code, message).
    search_batch None passes no options (NULL); opts_size overrides their struct_size.  The slots are cfg's device_games
    checked against max_batch; depth: dsearch_emul_run's knobs (waves in flight | 256 begin overlapped)."""
    lib = load()
    c = SelfPlayRunner(game, cfg)._fill(games_num, None, None, True, 0, 1)
    words, chess = _words(game)
    errors: list = []
    t1 = _eval_thunk(eval1, words, chess, errors)
    t2 = _eval_thunk(eval2, words, chess, errors) if eval2 is not None else None
    opts = None
    if search_batch is not None:
        opts = _lib.SelfPlayOpts()
        opts.struct_size = opts_size or C.sizeof(_lib.SelfPlayOpts)
        opts.search_batch = search_batch
    code = C.c_int(0)
    h = lib.selfplay_batch_emul_run(C.cast(t1, C.c_void_p), C.cast(t2, C.c_void_p) if t2 else None, C.byref(c),
                                    C.byref(opts) if opts is not None else None, max_batch, pool_words, depth, C.byref(code))
    try:
        if errors:
            raise errors[0]
        err = lib.dsearch_emul_error(h)
        if err:
            raise EmulError(code.value, err.decode())
        cnt = (C.c_uint64 * 8)()
        lib.dsearch_emul_counters(h, cnt)
        counters = dict(zip(("simulations", "evaluations", "terminal", "searches", "cache_hits", "w1", "w2", "draws"), [int(x) for x in cnt]))
        mb = (C.c_uint64 * 4)()
        lib.selfplay_batch_emul_batches(h, mb)
        counters["minibatches"], counters["collisions"] = (int(mb[0]), int(mb[1])), (int(mb[2]), int(mb[3]))
        records = []
        for k in range(lib.dsearch_emul_game_count(h)):
            gi, w, nm = C.c_uint32(), C.c_uint32(), C.c_uint32()
            lib.dsearch_emul_game_info(h, k, C.byref(gi), C.byref(w), C.byref(nm))
            mv = (C.c_uint16 * max(1, nm.value))()
            lib.dsearch_emul_game_moves(h, k, mv)
            entries, dirs = [], []
            for pi in range(nm.value):
                d = C.c_uint32()
                nb = lib.dsearch_emul_entry(h, k, pi, None, 0, C.byref(d))
                buf = (C.c_uint8 * nb)()
                lib.dsearch_emul_entry(h, k, pi, buf, nb, C.byref(d))
                entries.append(bytes(buf))
                dirs.append(d.value)
            records.append(GameRecord(gi.value, w.value or None, list(mv)[: nm.value], entries, dirs))
        return counters, records
    finally:
        lib.dsearch_emul_free(h)


def match(game: str, openings, cfg: dict, eval_a, eval_b=None, *, sim_num_b=None, explore_factor_b=None, search_batch=None, search_batch_b=None,
          opts_size: int = 0, max_batch: int = 4096, pool_words: int = 1 << 16, depth: int = 2, roots_cap: int = 0):
    """-> MatchResult with per-side minibatches / collisions; raises EmulError(code, message).  The options are
    match.play's (none given: NULL); eval_b None: one evaluator for both sides."""
    lib = load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    words, chess = _words(game)
    errors: list = []
    ta = _eval_thunk(eval_a, words, chess, errors)
    tb = _eval_thunk(eval_b, words, chess, errors) if eval_b is not None else None
    n, fa, ma, oa = encode_positions(game, openings)
    side = side_struct(sim_num_b, explore_factor_b)
    opts = opts_struct(search_batch, search_batch_b)
    if opts is not None and opts_size:
        opts.struct_size = opts_size
    code = C.c_int(0)
    h = lib.match_batch_emul_run(C.cast(ta, C.c_void_p), C.cast(tb, C.c_void_p) if tb else None, C.byref(c),
                                 C.byref(side) if side is not None else None, C.byref(opts) if opts is not None else None, max_batch, n, fa, ma,
                                 oa, pool_words, depth, roots_cap, C.byref(code))
    try:
        if errors:
            raise errors[0]
        err = lib.match_emul_error(h)
        if err:
            raise EmulError(code.value, err.decode())
        return collect(lib.match_emul_summary, lib.match_emul_opening_status, lib.match_emul_game, lib.match_emul_game_moves, h,
                       lib.match_batch_emul_batches)
    finally:
        lib.match_emul_free(h)
