"""Batched MCTS analysis of given positions on the device-resident search (include/cattus_b200_analysis.h).

    analyse(model, "chess", [(fen, ["e2e4", "e7e5"]), None, ...], cfg) -> [PositionAnalysis, ...]

Each position is searched as a fresh MctsPlayer with no root noise searches it (engine/src/mcts/mod.rs:335-385), thousands
at a time with the search trees in HBM: the visit counts and the best move are those `ChessSearch.go` returns with noise
off and temperature 0, and no result depends on `device_games`, `device_waves_in_flight`, the cache or the order of the
positions.  `cfg` is the self-play JSON config: "mcts" (sim_num, explore_factor, cache_size; prior_noise_epsilon must be
0) and the top-level "device_games", "device_tree_kwords" and "device_waves_in_flight".

`search_batch` L > 1 searches each tree in minibatches of L descents under virtual loss (DESIGN.md section 15), so the
evaluator sees up to L leaves of one tree at once: the mode for one position, or a few, searched deeply.  Its results
are deterministic (position, history, network, sim_num, explore_factor and L decide them) but differ from one leaf in
flight; `minibatches` and `collisions` count its rounds and the descents that ended on an already claimed leaf.
`device_games` 0 then means min(n, max_batch / L), and device_games x L above max_batch is ERANGE.

A position is `(fen, moves)`, a bare move list (from the initial position) or a FEN string (chess); `fen` None is the
initial position and is the only choice for hex and tic-tac-toe.  Moves: chess LAN strings ("e7e8q") or
from | to << 6 | promotion << 12 integers; hex and tic-tac-toe cell indices.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

from . import _lib
from ._lib import AnalysisOpts
from .selfplay import SelfPlayRunner, move_from_lan, parse_game

STATUS_NAMES = {0: "searched", 1: "player1 won", 2: "player2 won", 3: "draw"}


@dataclass
class PositionAnalysis:
    status: int                # 0 searched; 1 / 2 the game is over and that player won; 3 draw -- not searched
    best_move: Optional[int]   # None when not searched
    simulations: int
    q: float                   # the side to move's mean score over the search, in [-1, 1]
    moves: List[int] = field(default_factory=list)      # root children in edges() order (calc_moves_probabilities' order)
    visits: List[int] = field(default_factory=list)
    w: List[float] = field(default_factory=list)        # score_w, from the side to move at the root
    priors: List[float] = field(default_factory=list)   # init_score: the network's policy
    pv: List[int] = field(default_factory=list)         # principal variation, most visited child at every ply
    minibatches: int = 0       # rounds of descents (one leaf in flight: one per simulation); 0 when not searched
    collisions: int = 0        # descents that ended on a leaf an earlier descent of their minibatch had claimed

    @property
    def best_visits(self) -> int:
        return self.visits[self.moves.index(self.best_move)] if self.best_move is not None else 0


def encode_positions(game: str, positions: Sequence):
    """-> (n, fens array, moves array, offsets array) for cattus_b200_analyse (keep the arrays alive while C reads them)."""
    chess = parse_game(game)[0] == _lib.GAME_CHESS
    fens: List[Optional[bytes]] = []
    flat: List[int] = []
    offsets = [0]
    for p in positions:
        if p is None:
            fen, mv = None, ()
        elif isinstance(p, str):
            fen, mv = p, ()
        elif isinstance(p, tuple) and len(p) == 2 and (p[0] is None or isinstance(p[0], str)):
            fen, mv = p
        else:
            fen, mv = None, p
        fens.append(None if fen is None else fen.encode())
        for m in mv:
            flat.append(move_from_lan(m) if (chess and isinstance(m, str)) else int(m))
        offsets.append(len(flat))
    n = len(fens)
    fa = (C.c_char_p * max(1, n))(*fens)
    ma = (C.c_uint16 * max(1, len(flat)))(*flat)
    oa = (C.c_uint32 * (n + 1))(*offsets)
    return n, fa, ma, oa


def collect(count, get, children, pv, h, batches=None) -> List[PositionAnalysis]:
    """Reads a result object through its accessors (the library's, or the test emulation's of the same signatures);
    `batches` (optional) reads the minibatch counts."""
    n = C.c_uint32()
    count(h, C.byref(n))
    out = []
    for k in range(n.value):
        s = _lib.AnalysisPosition()
        s.struct_size = C.sizeof(_lib.AnalysisPosition)
        if get(h, k, C.byref(s)) != 0:
            raise RuntimeError(f"analysis result {k} cannot be read")
        nc = s.n_children
        mv, vi = (C.c_uint16 * max(1, nc))(), (C.c_uint32 * max(1, nc))()
        w, pr = (C.c_float * max(1, nc))(), (C.c_float * max(1, nc))()
        pva = (C.c_uint16 * 16)()
        if children(h, k, mv, vi, w, pr, nc) != 0 or pv(h, k, pva, 16) != 0:
            raise RuntimeError(f"analysis result {k} cannot be read")
        searched = s.status == 0
        a = PositionAnalysis(int(s.status), int(s.best_move) if searched else None, int(s.simulations), float(s.q),
                             list(mv)[:nc], list(vi)[:nc], list(w)[:nc], list(pr)[:nc], list(pva)[: s.pv_len])
        if batches is not None:
            mb, co = C.c_uint32(), C.c_uint32()
            if batches(h, k, C.byref(mb), C.byref(co)) != 0:
                raise RuntimeError(f"analysis result {k} cannot be read")
            a.minibatches, a.collisions = int(mb.value), int(co.value)
        out.append(a)
    return out


def analyse(model, game: str, positions: Sequence, cfg: dict, search_batch: int = 1) -> List[PositionAnalysis]:
    """model: a CudaNetwork of the game (any precision).  search_batch: descents per minibatch (1: one leaf in flight).
    Raises CattusB200Error (EINVAL for a bad FEN or an illegal move, naming the position index; ERANGE when the tree
    memory runs out or device_games x search_batch exceeds the model's batch)."""
    lib = _lib.load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    n, fa, ma, oa = encode_positions(game, positions)
    h = C.c_void_p()
    if search_batch == 1:
        _lib.check(lib.cattus_b200_analyse(model._h, C.byref(c), n, fa, ma, oa, C.byref(h)))
    else:
        opts = AnalysisOpts(C.sizeof(AnalysisOpts), int(search_batch))
        _lib.check(lib.cattus_b200_analyse_opts(model._h, C.byref(c), C.byref(opts), n, fa, ma, oa, C.byref(h)))
    try:
        return collect(lib.cattus_b200_analysis_count, lib.cattus_b200_analysis_get, lib.cattus_b200_analysis_children,
                       lib.cattus_b200_analysis_pv, h, lib.cattus_b200_analysis_batches)
    finally:
        lib.cattus_b200_analysis_free(h)
