"""Colour-balanced match play between two networks from an opening suite on the device-resident search
(include/cattus_b200_match.h).

    play(model_a, model_b, "chess", [(fen, ["e2e4", "e7e5"]), None, ...], cfg, sim_num_b=800) -> MatchResult

Opening k is played twice: game 2k with A as player 1, game 2k + 1 with B as player 1.  Each game is a self-play game
(the config's temperature policy and root noise, per-game random stream from (seed, game index), tree reuse, threefold
repetition, "max_moves" adjudication) started from the opening; repetition looks back into the opening's positions and
the temperature policy counts moves from the opening.  With every opening the initial position, the games are those of
`SelfPlayRunner.generate_data(A, B, 2n)` with the same seed.  `cfg` is the self-play JSON config: "mcts" (sim_num,
explore_factor, temperature_policy, prior noise, cache_size) and the top-level "seed", "max_moves", "device_games",
"device_tree_kwords" and "device_waves_in_flight".  Side B may play with its own sim_num / explore_factor.

Openings take the forms `analysis.analyse` takes: `(fen, moves)`, a bare move list, a FEN string (chess) or None.

The statistics are pentanomial: each opening's two games give A p in {0, 1/4, 1/2, 3/4, 1}; s = mean p,
sigma^2 = mean (p - s)^2 / N_pairs, Elo(x) = -400 log10(1 / x - 1) at s with the 95 % interval
[Elo(s - 1.96 sigma), Elo(s + 1.96 sigma)], arguments clipped to [0, 1] where Elo is -inf / +inf.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

from . import _lib
from .analysis import encode_positions
from .selfplay import SelfPlayRunner

TERMINATIONS = {1: "rules", 2: "repetition", 3: "max_moves"}


@dataclass
class MatchGame:
    opening: int
    a_is_player1: bool
    winner: Optional[int]  # None: draw; 1 / 2: that player (chess: white / black)
    termination: str       # "rules", "repetition" (threefold) or "max_moves" (adjudicated)
    moves: List[int]       # from the opening position; chess from | to << 6 | promotion << 12, hex / ttt cell index

    @property
    def a_points(self) -> float:
        if self.winner is None:
            return 0.5
        return 1.0 if (self.winner == 1) == self.a_is_player1 else 0.0


@dataclass
class Elo:
    elo: float                # math.inf / -math.inf when s is 1 / 0
    lo: float                 # 95 % interval, likewise possibly infinite
    hi: float
    score: float              # s: A's mean points per game
    stderr: float             # sigma of s
    pairs: int


def elo_of(x: float) -> float:
    """-400 log10(1 / x - 1) on [0, 1], -inf at 0 and +inf at 1."""
    if x <= 0.0:
        return -math.inf
    if x >= 1.0:
        return math.inf
    return -400.0 * math.log10(1.0 / x - 1.0)


def pentanomial(pair_points: Sequence[float]) -> List[int]:
    """Counts of pairs in which A scored 0, 1/2, 1, 3/2, 2 points (pair_points are in points per pair, 0 .. 2)."""
    out = [0] * 5
    for p in pair_points:
        out[int(round(2 * p))] += 1
    return out


def elo_from_pairs(pairs: Sequence[int]) -> Optional[Elo]:
    """The pentanomial estimate from the five counts; None without a pair."""
    n = sum(pairs)
    if n == 0:
        return None
    ps = [j / 4.0 for j in range(5)]
    s = sum(c * p for c, p in zip(pairs, ps)) / n
    var = sum(c * (p - s) ** 2 for c, p in zip(pairs, ps)) / n / n
    sd = math.sqrt(var)
    return Elo(elo_of(s), elo_of(s - 1.96 * sd), elo_of(s + 1.96 * sd), s, sd, n)


def fmt_elo(x: float):
    """A JSON-safe Elo: a number rounded to 0.01, or "+inf" / "-inf"."""
    return round(x, 2) if math.isfinite(x) else ("+inf" if x > 0 else "-inf")


@dataclass
class MatchResult:
    games: List[MatchGame]
    opening_status: List[int]  # per opening: 0 played; 1 / 2 already won by that player, 3 already drawn -- not played
    a_wins: int
    b_wins: int
    draws: int
    pairs: List[int]           # pentanomial counts
    simulations: int
    evaluations: int
    seconds: float
    # per side (A, B): rounds of descents (one leaf in flight: one per simulation) and descents that collided with an
    # earlier one of their minibatch
    minibatches: Tuple[int, int] = (0, 0)
    collisions: Tuple[int, int] = (0, 0)

    @property
    def skipped(self) -> int:
        return sum(1 for s in self.opening_status if s != 0)

    def elo(self) -> Optional[Elo]:
        return elo_from_pairs(self.pairs)


def side_struct(sim_num_b: Optional[int], explore_factor_b: Optional[float]):
    if sim_num_b is None and explore_factor_b is None:
        return None
    s = _lib.MatchSide()
    s.struct_size = C.sizeof(_lib.MatchSide)
    s.sim_num = int(sim_num_b or 0)
    s.explore_factor = -1.0 if explore_factor_b is None else float(explore_factor_b)
    return s


def collect(summary_get, opening_status, game_get, game_moves, h, batches=None) -> MatchResult:
    """Reads a match result through its accessors (the library's, or the test emulation's of the same signatures);
    `batches` (optional) reads each side's minibatch and collision counts."""
    s = _lib.MatchSummary()
    s.struct_size = C.sizeof(_lib.MatchSummary)
    if summary_get(h, C.byref(s)) != 0:
        raise RuntimeError("match summary cannot be read")
    status = []
    for k in range(s.openings):
        st = C.c_uint32()
        if opening_status(h, k, C.byref(st)) != 0:
            raise RuntimeError(f"match opening {k} cannot be read")
        status.append(int(st.value))
    games = []
    for k in range(s.games):
        g = _lib.MatchGame()
        g.struct_size = C.sizeof(_lib.MatchGame)
        mv = None
        if game_get(h, k, C.byref(g)) == 0:
            mv = (C.c_uint16 * max(1, g.n_moves))()
        if mv is None or game_moves(h, k, mv, g.n_moves) != 0:
            raise RuntimeError(f"match game {k} cannot be read")
        games.append(MatchGame(int(g.opening), bool(g.a_is_player1), int(g.winner) or None, TERMINATIONS[g.termination], list(mv)[: g.n_moves]))
    res = MatchResult(games, status, int(s.a_wins), int(s.b_wins), int(s.draws), list(s.pairs), int(s.simulations), int(s.evaluations),
                      float(s.seconds))
    if batches is not None:
        mb, co = [], []
        for side in (0, 1):
            m, c = C.c_uint64(), C.c_uint64()
            if batches(h, side, C.byref(m), C.byref(c)) != 0:
                raise RuntimeError("match minibatch counts cannot be read")
            mb.append(int(m.value))
            co.append(int(c.value))
        res.minibatches, res.collisions = tuple(mb), tuple(co)
    return res


def opts_struct(search_batch: Optional[int], search_batch_b: Optional[int]):
    """cattus_b200_match_opts: search_batch for both sides, search_batch_b overriding B's; None when neither is given."""
    if search_batch is None and search_batch_b is None:
        return None
    o = _lib.MatchOpts()
    o.struct_size = C.sizeof(_lib.MatchOpts)
    o.search_batch_a = int(search_batch or 1)
    o.search_batch_b = int(search_batch_b if search_batch_b is not None else (search_batch or 1))
    return o


def play(model_a, model_b, game: str, openings: Sequence, cfg: dict, sim_num_b: Optional[int] = None,
         explore_factor_b: Optional[float] = None, search_batch: Optional[int] = None, search_batch_b: Optional[int] = None) -> MatchResult:
    """model_a / model_b: CudaNetworks of the game (any precision each); model_b None or model_a: one handle, one
    evaluator and one cache.  search_batch: descents per minibatch under virtual loss of both sides (DESIGN.md section
    16; None or 1: one leaf in flight, the reference's search); search_batch_b overrides B's.  A side with L > 1 does not
    play the reference's games.  Raises CattusB200Error (EINVAL for a bad FEN or an illegal move, naming the opening
    index; ERANGE when the tree memory runs out or device_games x L exceeds a model's max_batch)."""
    lib = _lib.load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    n, fa, ma, oa = encode_positions(game, openings)
    side = side_struct(sim_num_b, explore_factor_b)
    opts = opts_struct(search_batch, search_batch_b)
    hb = model_b._h if (model_b is not None and model_b is not model_a) else None
    h = C.c_void_p()
    _lib.check(lib.cattus_b200_match_run_opts(model_a._h, hb, C.byref(c), C.byref(side) if side is not None else None,
                                              C.byref(opts) if opts is not None else None, n, fa, ma, oa, C.byref(h)))
    try:
        return collect(lib.cattus_b200_match_summary_get, lib.cattus_b200_match_opening_status, lib.cattus_b200_match_game_get,
                       lib.cattus_b200_match_game_moves, h, lib.cattus_b200_match_batches)
    finally:
        lib.cattus_b200_match_free(h)
