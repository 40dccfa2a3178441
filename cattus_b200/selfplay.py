"""Host-side mirror of the reference's self-play executable over include/cattus_b200_selfplay.h.

    {game}_self_player --model1-path .. --model2-path .. --games-num N --out-dir1 .. --out-dir2 .. \
        --summary-file .. --config-file cfg.json            (training/self-play/src/self_play_cmd.rs:14-31)
                          ->  SelfPlayRunner(game, cfg).generate_data(model1, model2, games_num, out_dir1, out_dir2)

`cfg` is the same JSON object the reference executable reads (self_play_cmd.rs:34-53; written by
training/cattus_train/self_play.py): {"model": {"batch_size", "inference"}, "mcts": {"sim_num", "explore_factor",
"temperature_policy", "prior_noise_alpha", "prior_noise_epsilon", "cache_size"}, "threads"} plus the optional keys
"games_per_thread", "groups_per_thread", "leaf_queue", "max_moves", "speculate" and "seed" that only this backend
understands (include/cattus_b200_selfplay.h documents each; none of them changes a game except "seed" and "max_moves").  The returned summary has the layout of
the reference's summary file (self_play_cmd.rs:131-149) with the metric keys the trainer reads
(training/cattus_train/train_process.py:176-186).

The MCTS, the rules, the cache and the .traindata writers run in C++ (csrc/selfplay.cpp); network evaluations go to
the GPU through `cattus_b200_eval_batch` / `cattus_b200_eval`.  `run_with` binds an arbitrary evaluator callback instead
(the reference's `dyn ValueFunction`); it is what the CPU tests and the bench's CPU-baseline leg use.
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import SelfPlayCfg, SelfPlaySummary


def parse_game(game: str) -> Tuple[int, int]:
    """'hex5' -> (GAME_HEX, 5); 'ttt' / 'tictactoe' -> (GAME_TTT, 3); 'chess' -> (GAME_CHESS, 8)."""
    if game in ("ttt", "tictactoe"):
        return _lib.GAME_TTT, 3
    if game == "chess":
        return _lib.GAME_CHESS, 8
    m = re.fullmatch(r"hex(\d+)?", game)
    if m:
        return _lib.GAME_HEX, int(m.group(1) or 11)
    raise ValueError(f"unknown game {game!r} (hex<S>, ttt, chess)")


@dataclass
class GameRecord:
    game_idx: int
    winner: Optional[int]  # None, 1, 2
    moves: List[int]       # hex / ttt: cell index; chess: from | to << 6 | promotion << 12 (cattus_b200_chess.h)
    entries: List[bytes]   # exact .traindata bytes per position
    entry_dirs: List[int]  # 1 -> out_dir1, 2 -> out_dir2


class SelfPlayError(RuntimeError):
    pass


def _check(lib, rc: int) -> None:
    if rc != 0:
        raise SelfPlayError(f"cattus_b200_selfplay error {rc}: {(lib.cattus_b200_selfplay_last_error() or b'').decode(errors='replace')}")


def _eval_thunk(fn: Callable, words: int, chess: bool, errors: list):
    """Wraps a Python evaluator as a cattus_b200_eval_fn (keep the returned object alive while C may call it)."""

    def thunk(_ctx, planes, legal, n, probs_out, probs_cap, prob_offsets, values_out):
        try:
            w = np.ctypeslib.as_array(planes, shape=(n, words)).copy()
            if chess:
                probs, values = fn(w, n, np.ctypeslib.as_array(legal, shape=(n, 235)).copy())
            else:
                probs, values = fn(w, n)
            off = 0
            for i in range(n):
                p = np.asarray(probs[i], dtype=np.float32)
                if off + len(p) > probs_cap:
                    return _lib.ERANGE
                prob_offsets[i] = off
                for k, x in enumerate(p):
                    probs_out[off + k] = float(x)
                off += len(p)
                values_out[i] = float(np.float32(values[i]))
            prob_offsets[n] = off
            return 0
        except Exception as e:  # never let an exception cross the C boundary
            errors.append(e)
            return _lib.EINVAL

    return _lib.EVAL_FN(thunk)


class SelfPlayRunner:
    def __init__(self, game: str, cfg: dict):
        self._lib = _lib.load()
        self.game = game
        self.cfg = cfg
        mc = cfg["mcts"]
        c = SelfPlayCfg()
        c.struct_size = C.sizeof(SelfPlayCfg)
        c.game, c.board_size = parse_game(game)
        c.sim_num = int(mc["sim_num"])
        c.explore_factor = float(mc.get("explore_factor", 2.0 ** 0.5))
        policy = list(mc.get("temperature_policy", [[0, 1.0]]))
        assert policy, "temperature_policy must not be empty (self_play_cmd.rs:68)"
        self._tm = (C.c_uint32 * len(policy))(*[int(p[0]) for p in policy])
        self._tv = (C.c_float * len(policy))(*[float(p[1]) for p in policy])
        c.temperature_moves = C.cast(self._tm, C.POINTER(C.c_uint32))
        c.temperature_values = C.cast(self._tv, C.POINTER(C.c_float))
        c.n_temperatures = len(policy)
        c.prior_noise_alpha = float(mc.get("prior_noise_alpha", 0.0))
        c.prior_noise_epsilon = float(mc.get("prior_noise_epsilon", 0.0))
        c.cache_size = int(mc.get("cache_size", 0))
        c.threads = int(cfg.get("threads", 1))
        c.games_per_thread = int(cfg.get("games_per_thread", 1))
        c.leaf_queue = int(cfg.get("leaf_queue", 0))
        c.groups_per_thread = int(cfg.get("groups_per_thread", 0))
        c.max_moves = int(cfg.get("max_moves", 0))
        c.speculate = int(cfg.get("speculate", 0))
        c.device_games = int(cfg.get("device_games", 0))
        c.device_tree_kwords = int(cfg.get("device_tree_kwords", 0))
        c.device_waves_in_flight = int(cfg.get("device_waves_in_flight", 0))
        c.seed = int(cfg.get("seed", 0)) & 0xFFFFFFFFFFFFFFFF
        self._c = c
        # descents per minibatch under virtual loss (DESIGN.md section 16); absent or 1: one leaf in flight, the reference's
        # search.  Needs device_games > 0, and its games are not the reference's.
        self._opts = None
        if "search_batch" in cfg:
            self._opts = _lib.SelfPlayOpts()
            self._opts.struct_size = C.sizeof(_lib.SelfPlayOpts)
            self._opts.search_batch = int(cfg["search_batch"])

    def _fill(self, games_num, out_dir1, out_dir2, keep_records, first_game, game_stride):
        c = self._c
        c.games_num = int(games_num)
        c.first_game = int(first_game)
        c.game_stride = int(game_stride)
        c.out_dir1 = None if out_dir1 is None else str(out_dir1).encode()
        c.out_dir2 = None if out_dir2 is None else str(out_dir2).encode()
        c.keep_records = 1 if keep_records else 0
        return c

    # ---------------------------------------------------------------- entry points
    def generate_data(self, model1, model2, games_num: int, out_dir1=None, out_dir2=None, *, keep_records: bool = False,
                      first_game: int = 0, game_stride: int = 1):
        """model1 / model2: CudaNetwork instances (model2 may be None or the same object: one evaluator, one cache)."""
        c = self._fill(games_num, out_dir1, out_dir2, keep_records, first_game, game_stride)
        h = C.c_void_p()
        h2 = model2._h if (model2 is not None and model2 is not model1) else None
        opts = C.byref(self._opts) if self._opts is not None else None
        _check(self._lib, self._lib.cattus_b200_selfplay_run_opts(model1._h, h2, C.byref(c), opts, C.byref(h)))
        return self._collect(h, keep_records)

    def run_with(self, eval1: Callable, eval2: Optional[Callable], games_num: int, out_dir1=None, out_dir2=None, *,
                 keep_records: bool = False, first_game: int = 0, game_stride: int = 1):
        """eval(planes u64 [n, words], n) -> (list of n probability arrays over the legal moves ascending, values[n]);
        for chess eval(planes, n, legal u8 [n, 235]) with the legal-move bitmaps over the nn indices."""
        if self._opts is not None and self._opts.search_batch > 1:
            raise SelfPlayError("search_batch > 1 needs the device-resident search of generate_data (device_games > 0)")
        c = self._fill(games_num, out_dir1, out_dir2, keep_records, first_game, game_stride)
        g, s = parse_game(self.game)
        chess = g == _lib.GAME_CHESS
        words = 18 if chess else 3 * ((s * s + 63) // 64)
        errors: list = []

        def thunk_for(fn):
            return _eval_thunk(fn, words, chess, errors)

        t1 = thunk_for(eval1)
        t2 = thunk_for(eval2) if eval2 is not None else None
        h = C.c_void_p()
        rc = self._lib.cattus_b200_selfplay_run_with(C.cast(t1, C.c_void_p), None, C.cast(t2, C.c_void_p) if t2 else None, None, C.byref(c), C.byref(h))
        if errors:
            raise errors[0]
        _check(self._lib, rc)
        return self._collect(h, keep_records)

    # ---------------------------------------------------------------- results
    def _collect(self, h, keep_records: bool):
        lib = self._lib
        try:
            s = SelfPlaySummary()
            _check(lib, lib.cattus_b200_selfplay_summary_get(h, C.byref(s)))
            mb, co = C.c_uint64(), C.c_uint64()
            _check(lib, lib.cattus_b200_selfplay_batches(h, C.byref(mb), C.byref(co)))
            summary = {
                "player1_wins": s.player1_wins, "player2_wins": s.player2_wins, "draws": s.draws,
                "metrics": {
                    "cache.hits": s.cache_hits, "cache.misses": s.cache_misses, "mcts.search_duration": s.search_duration,
                    "model.activation_count": s.batches,
                    "selfplay.games": s.games, "selfplay.simulations": s.simulations, "selfplay.searches": s.searches,
                    "selfplay.evaluations": s.evaluations, "selfplay.terminal_leaves": s.terminal_leaves,
                    "selfplay.seconds": s.seconds, "selfplay.eval_wait_seconds": s.eval_wait_seconds,
                    "selfplay.speculative_evaluations": s.speculative_evaluations,
                    "selfplay.minibatches": mb.value, "selfplay.collisions": co.value,
                    "selfplay.sims_per_sec": (s.simulations / s.seconds) if s.seconds > 0 else 0.0,
                },
            }
            records: List[GameRecord] = []
            if keep_records:
                n = C.c_uint32()
                _check(lib, lib.cattus_b200_selfplay_game_count(h, C.byref(n)))
                for k in range(n.value):
                    gi, w, nm = C.c_uint32(), C.c_uint32(), C.c_uint32()
                    _check(lib, lib.cattus_b200_selfplay_game_info(h, k, C.byref(gi), C.byref(w), C.byref(nm)))
                    mv = (C.c_uint16 * max(1, nm.value))()
                    _check(lib, lib.cattus_b200_selfplay_game_moves16(h, k, mv, nm.value))
                    entries, dirs = [], []
                    for pi in range(nm.value):
                        nb, od = C.c_size_t(), C.c_uint32()
                        _check(lib, lib.cattus_b200_selfplay_entry(h, k, pi, None, 0, C.byref(nb), C.byref(od)))
                        buf = (C.c_uint8 * nb.value)()
                        _check(lib, lib.cattus_b200_selfplay_entry(h, k, pi, buf, nb.value, C.byref(nb), C.byref(od)))
                        entries.append(bytes(buf))
                        dirs.append(od.value)
                    records.append(GameRecord(gi.value, w.value or None, list(mv)[: nm.value], entries, dirs))
            return summary, records
        finally:
            lib.cattus_b200_selfplay_free(h)


# ---------------------------------------------------------------------------------------------------------------------
# one chess search at a time: the player of the reference's UCI loop (engine/src/chess/uci.rs)
# ---------------------------------------------------------------------------------------------------------------------
_PROMO = (None, "q", "n", "r", "b")


def move_to_lan(m: int) -> str:
    """from | to << 6 | promotion << 12 -> 'e2e4' / 'e7e8q' (the crate's ChessMove Display, which the UCI loop prints)."""
    sq = lambda x: "abcdefgh"[x & 7] + "12345678"[x >> 3]  # noqa: E731
    return sq(m & 63) + sq((m >> 6) & 63) + (_PROMO[m >> 12] or "")


def move_from_lan(lan: str) -> int:
    """ChessMove::from_lan (chess/core.rs:24-51)."""
    if len(lan) not in (4, 5):
        raise ValueError(f"Invalid LAN length: {lan!r}")
    f = (ord(lan[1]) - 49) * 8 + ord(lan[0]) - 97
    t = (ord(lan[3]) - 49) * 8 + ord(lan[2]) - 97
    if not (0 <= f < 64 and 0 <= t < 64):
        raise ValueError(f"bad squares in {lan!r}")
    promo = 0
    if len(lan) == 5:
        if lan[4] not in "qnrb":
            raise ValueError(f"Unknown promotion char: {lan[4]!r} in lan str {lan!r}")
        promo = _PROMO.index(lan[4])
    return f | (t << 6) | (promo << 12)


class ChessSearch:
    """MctsPlayer<ChessGame> over include/cattus_b200_selfplay.h's cattus_b200_chess_search_*: `ChessSearch(cfg, model)`
    is `ucinewgame`, `go(fen, moves)` is `position ...` + `go` and returns (bestmove as LAN, stats)."""

    def __init__(self, cfg: dict, model=None, eval_fn: Optional[Callable] = None):
        self._lib = _lib.load()
        self._runner = SelfPlayRunner("chess", cfg)  # fills the mcts.* fields of the C struct
        c = self._runner._fill(2, None, None, False, 0, 1)
        self._errors: list = []
        h = C.c_void_p()
        if model is not None:
            self._thunk = None
            _check(self._lib, self._lib.cattus_b200_chess_search_create(model._h, C.byref(c), C.byref(h)))
        else:
            assert eval_fn is not None, "either a CudaNetwork or an evaluator callback"
            self._thunk = _eval_thunk(eval_fn, 18, True, self._errors)
            _check(self._lib, self._lib.cattus_b200_chess_search_create_with(C.cast(self._thunk, C.c_void_p), None, C.byref(c), C.byref(h)))
        self._h = h

    def go(self, fen: Optional[str] = None, moves=()):
        mv = [move_from_lan(m) if isinstance(m, str) else int(m) for m in moves]
        arr = (C.c_uint16 * max(1, len(mv)))(*mv)
        best = C.c_uint16()
        st = _lib.ChessSearchStats()
        st.struct_size = C.sizeof(_lib.ChessSearchStats)
        rc = self._lib.cattus_b200_chess_search_go(self._h, None if fen is None else fen.encode(), arr, len(mv), C.byref(best), C.byref(st))
        if self._errors:
            raise self._errors.pop()
        _check(self._lib, rc)
        return move_to_lan(best.value), {"simulations": st.simulations, "evaluations": st.evaluations, "cache_hits": st.cache_hits,
                                         "terminal_leaves": st.terminal_leaves, "seconds": st.seconds, "root_children": st.root_children,
                                         "best_visits": st.best_visits, "speculative_evaluations": st.speculative_evaluations}

    def close(self):
        if self._h:
            self._lib.cattus_b200_chess_search_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
