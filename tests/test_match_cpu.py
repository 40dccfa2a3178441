"""CPU tests of match play from openings (cattus_b200/csrc/dsearch_match.hpp over ds::Driver and dsearch_core.hpp).

The match driver and the per-slot search code are compiled for the host with a one-lane warp (tests/emul) and driven by
deterministic Python evaluators.  From the initial position a match must play exactly the emulated self-play games of
(A, B); from real openings every game must equal oracle/mcts.py's self-play game loop started from the same history
(play_from below).  Also the pentanomial statistics, the PGN writer and the input errors.
"""
from __future__ import annotations

import math
import re

import pytest

from cattus_b200 import match as M
from cattus_b200 import san as S
from cattus_b200.selfplay import move_from_lan
from oracle import chess as oc
from oracle import mcts as om
from tests.emul import emul
from tests.emul import match_emul as me
from tests.test_analysis_cpu import REPEAT_CHILD, chess_history, chess_positions, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, _params, chess_cb, chess_cfg, chess_fake_net, chess_oracle_fn
from tests.test_selfplay_cpu import cb_for, cfg_with, fake_net, oracle_net_fn

NOISY = dict(prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[4, 1.0], [9999, 0.0]])


def small_cb(game, net):
    return chess_cb(net) if game == "chess" else cb_for(net, 1)


def nets(game):
    if game == "chess":
        return chess_fake_net("hash"), chess_fake_net("hash", salt=99)
    return fake_net("hash"), fake_net("hash", salt=99)


@pytest.mark.parametrize("game,sim_num,pairs", [("hex5", 30, 4), ("ttt", 40, 3), ("chess", 16, 2)])
def test_initial_position_openings_play_the_self_play_games(game, sim_num, pairs):
    """Openings = the initial position x n: game for game the emulated self-play Driver with (A, B), noise and temperature on."""
    a, b = nets(game)
    mk = chess_cfg if game == "chess" else cfg_with
    cfg = mk(sim_num=sim_num, seed=13, max_moves=24 if game == "chess" else 0, **NOISY)
    counters, ref = emul.run(game, cfg, small_cb(game, a), small_cb(game, b), 2 * pairs, n_slots=3, pool_words=1 << 16)
    got = me.play(game, [None] * pairs, cfg, small_cb(game, a), small_cb(game, b), n_slots=3)
    assert len(got.games) == len(ref) == 2 * pairs
    for r, g in zip(ref, got.games):
        assert (g.opening, g.a_is_player1) == (r.game_idx // 2, r.game_idx % 2 == 0)
        assert g.moves == r.moves and g.winner == r.winner, r.game_idx
    assert (got.a_wins, got.b_wins, got.draws) == (counters["w1"], counters["w2"], counters["draws"])
    assert got.simulations == counters["simulations"] and got.skipped == 0


def small_history(game, moves):
    p = om.HexPosition.new(5) if game == "hex5" else om.TttPosition.new()
    h = [p]
    for m in moves:
        h.append(h[-1].moved_position(m))
    return h


def play_from(game_idx: int, history, params1, params2, eval1, eval2, base_seed: int, max_moves: int = 0) -> om.GameRecord:
    """oracle/mcts.py's play_game (self_play.rs:179-246) started after `history` (an opening, oldest first) instead of the
    initial position, built from the same oracle pieces: repetition counts the opening's positions; the temperature policy
    gets the history from the opening position on, and max_moves counts the moves played after it."""
    rng = om.SplitMix64(om.game_seed(base_seed, game_idx))
    player1 = om.MctsPlayer(params1, eval1, rng)
    player2 = om.MctsPlayer(params2, eval2, rng)
    history = list(history)
    base = len(history) - 1
    entries, moves = [], []
    limit = getattr(type(history[0]), "REPETITION_LIMIT", None)
    seen = None
    if limit:
        seen = {}
        for p in history:
            seen[p] = seen.get(p, 0) + 1
    while True:
        st, winner = history[-1].status()
        if seen is not None and seen[history[-1]] >= limit:
            st, winner = "finished", None
        if st != "finished" and max_moves and len(moves) >= max_moves:
            st, winner = "finished", None
        if st == "finished":
            break
        who = history[-1].turn
        if game_idx % 2 == 1:
            who = om.opposite(who)
        player = player1 if who == om.P1 else player2
        probs = player.calc_moves_probabilities(history)
        mv = player.choose_move_from_probabilities(history[base:], probs)
        entries.append((history[-1], probs))
        moves.append(mv)
        history.append(history[-1].moved_position(mv))
        if seen is not None:
            seen[history[-1]] = seen.get(history[-1], 0) + 1
    return om.GameRecord(game_idx, winner, moves, entries, player1.sims_done + player2.sims_done,
                         player1.terminal_leaves + player2.terminal_leaves, player1.repetition_hits + player2.repetition_hits)


def test_play_from_the_initial_position_is_the_oracle_game():
    """The helper above is play_game when the history is the initial position alone."""
    n1, n2 = fake_net("hash"), fake_net("hash", salt=99)
    cfg = cfg_with(sim_num=20, seed=4, **NOISY)
    mc = cfg["mcts"]
    params = om.MctsParams(mc["sim_num"], mc["explore_factor"], om.TemperaturePolicy.from_config(mc["temperature_policy"]),
                           mc["prior_noise_alpha"], mc["prior_noise_epsilon"])
    e1, e2 = om.Evaluator(oracle_net_fn(n1), None), om.Evaluator(oracle_net_fn(n2), None)
    for g in range(2):
        ref = om.play_game(g, lambda: om.HexPosition.new(5), params, params, e1, e2, 4)
        got = play_from(g, [om.HexPosition.new(5)], params, params, e1, e2, 4)
        assert (got.moves, got.winner, got.sims) == (ref.moves, ref.winner, ref.sims)


def oracle_match(game, histories, cfg, net_a, net_b, sim_num_b=None, explore_factor_b=None):
    """Every played opening's two games by the oracle's game loop (play_from) from the opening's history."""
    if game == "chess":
        params_a = _params(cfg)
        ea, eb = om.Evaluator(chess_oracle_fn(net_a), None), om.Evaluator(chess_oracle_fn(net_b), None)
    else:
        mc = cfg["mcts"]
        params_a = om.MctsParams(mc["sim_num"], mc["explore_factor"], om.TemperaturePolicy.from_config(mc["temperature_policy"]),
                                 mc["prior_noise_alpha"], mc["prior_noise_epsilon"])
        ea, eb = om.Evaluator(oracle_net_fn(net_a), None), om.Evaluator(oracle_net_fn(net_b), None)
    params_b = om.MctsParams(**dict(params_a.__dict__, sim_num=sim_num_b or params_a.sim_num,
                                    explore_factor=params_a.explore_factor if explore_factor_b is None else explore_factor_b))
    out = {}
    for k, h in enumerate(histories):
        if h is None:
            continue
        for c in (0, 1):
            out[(k, c == 0)] = play_from(2 * k + c, h, params_a, params_b, ea, eb, cfg["seed"], cfg.get("max_moves", 0))
    return out


def check_against_oracle(got, ref, to_move=lambda m: m):
    assert [(g.opening, g.a_is_player1) for g in got.games] == sorted(ref, key=lambda x: (x[0], not x[1]))
    for g in got.games:
        o = ref[(g.opening, g.a_is_player1)]
        assert g.moves == [to_move(m) for m in o.moves], (g.opening, g.a_is_player1)
        assert g.winner == o.winner


@pytest.mark.parametrize("game,sim_num", [("hex5", 30), ("ttt", 30)])
def test_openings_equal_oracle_play_game_hex_ttt(game, sim_num):
    na, nb = nets(game)
    openings = hex_positions(5, 6, 7) if game == "hex5" else ttt_positions(6, 8)
    cfg = cfg_with(sim_num=sim_num, seed=3, **NOISY)
    got = me.play(game, openings, cfg, cb_for(na, 1), cb_for(nb, 1), sim_num_b=sim_num + 12, n_slots=4)
    ref = oracle_match(game, [small_history(game, m) for m in openings], cfg, na, nb, sim_num_b=sim_num + 12)
    check_against_oracle(got, ref)
    assert got.simulations == sum(o.sims for o in ref.values())


# the position after REPEAT_CHILD has occurred twice: black's f6g8 repeats the start position a third time
SHUFFLE = (None, REPEAT_CHILD)
# the rooks leave white's king one move at a time (a2 <-> a1); the opening's rook shuffle has seen the FEN's position
# twice, so white's forced Ka2 completes a threefold repetition
FORCED = ("1r5k/8/8/8/8/2r5/K7/8 b - - 0 1", ["c3d3", "a2a1", "d3c3", "a1a2", "c3d3", "a2a1", "d3c3"])
FINISHED = [(None, ["f2f3", "e7e5", "g2g4", "d8h4"]), (None, REPEAT_CHILD + ["f6g8"]), ("7k/5Q2/6K1/8/8/8/8/8 b - -", [])]


def test_chess_openings_equal_oracle_play_game():
    """FEN openings, a repetition set up by the opening and completed by the game, finished openings; two evaluators and a
    different sim_num for B; noise and temperature on."""
    na, nb = chess_fake_net("uniform"), chess_fake_net("hash", salt=99)
    openings = [FORCED, (KIWIPETE, ["e1g1"]), FINISHED[0], SHUFFLE, (KIWIPETE, [])] + chess_positions(6, 31)[2:] + FINISHED[1:]
    cfg = chess_cfg(sim_num=14, seed=5, max_moves=30, **NOISY)
    got = me.play("chess", openings, cfg, chess_cb(na), chess_cb(nb), sim_num_b=22, n_slots=5)
    assert got.opening_status[2] == 2 and got.opening_status[-2:] == [3, 3]
    assert got.skipped == 3 and sum(got.opening_status[k] == 0 for k in range(len(openings))) == len(openings) - 3
    hist = [None if st else chess_history(f, m) for (f, m), st in zip(openings, got.opening_status)]
    ref = oracle_match("chess", hist, cfg, na, nb, sim_num_b=22)
    check_against_oracle(got, ref, oc.move_to_u16)
    assert [(g.moves, g.termination) for g in got.games if g.opening == 0] == [([move_from_lan("a1a2")], "repetition")] * 2
    assert {g.termination for g in got.games} >= {"repetition", "max_moves"}
    assert got.a_wins + got.b_wins + got.draws == len(got.games) == 2 * (len(openings) - 3)


def test_results_do_not_depend_on_slots_waves_cache_populations_or_order():
    na, nb = chess_fake_net("hash"), chess_fake_net("hash", salt=99)
    openings = chess_positions(10, 3) + [SHUFFLE]
    cfg = chess_cfg(sim_num=12, seed=2, max_moves=16, **NOISY)
    ref = me.play("chess", openings, cfg, chess_cb(na), chess_cb(nb), n_slots=1, depth=1)
    for n_slots, depth, cache, roots_cap in ((3, 1, 0, 0), (22, 3, 0, 0), (4, 3 | 256, 5000, 0), (16, 2 | 256 | 512, 5000, 0), (8, 2 | 256, 64, 1)):
        got = me.play("chess", openings, chess_cfg(sim_num=12, seed=2, max_moves=16, cache_size=cache, **NOISY), chess_cb(na), chess_cb(nb),
                      n_slots=n_slots, depth=depth, roots_cap=roots_cap)
        assert got.games == ref.games and got.pairs == ref.pairs, (n_slots, depth, cache)
    # reversed openings: the same game for each (opening, colour).  Without noise and at temperature 0, since with them a
    # game's random stream is seeded from its game index 2k + c, which follows the opening's place in the input
    quiet = chess_cfg(sim_num=12, seed=2, max_moves=16)
    fwd = me.play("chess", openings, quiet, chess_cb(na), chess_cb(nb), n_slots=4)
    rev = me.play("chess", openings[::-1], quiet, chess_cb(na), chess_cb(nb), n_slots=5)
    n = len(openings)
    assert sorted(((n - 1 - g.opening, g.a_is_player1, g.moves, g.winner) for g in rev.games)) == \
        sorted(((g.opening, g.a_is_player1, g.moves, g.winner) for g in fwd.games))
    # one evaluator on both sides (one handle): the same games as two evaluators of the same net
    one = me.play("chess", openings, cfg, chess_cb(na), None, n_slots=6)
    two = me.play("chess", openings, cfg, chess_cb(na), chess_cb(na), n_slots=6)
    assert one.games == two.games
    hnet = fake_net("hash")
    hpos = hex_positions(5, 8, 4)
    hcfg = cfg_with(sim_num=24, seed=6, **NOISY)
    href = me.play("hex5", hpos, hcfg, cb_for(hnet, 1), None, n_slots=1, depth=1)
    for n_slots, depth, cache in ((3, 1, 0), (16, 3, 1000), (5, 2 | 256 | 512, 100)):
        got = me.play("hex5", hpos, cfg_with(sim_num=24, seed=6, cache_size=cache, **NOISY), cb_for(hnet, 1), None, n_slots=n_slots, depth=depth)
        assert got.games == href.games


def test_summary_counts_equal_a_direct_count():
    na, nb = fake_net("hash"), fake_net("coarse", salt=5)
    got = me.play("hex5", hex_positions(5, 12, 2), cfg_with(sim_num=20, seed=1, **NOISY), cb_for(na, 1), cb_for(nb, 1), n_slots=6)
    by_opening = {}
    for g in got.games:
        by_opening[g.opening] = by_opening.get(g.opening, 0.0) + g.a_points
    assert got.pairs == M.pentanomial(by_opening.values())
    assert got.a_wins == sum(g.a_points == 1.0 for g in got.games) and got.b_wins == sum(g.a_points == 0.0 for g in got.games)
    assert got.draws == sum(g.a_points == 0.5 for g in got.games)
    e = got.elo()
    assert e.pairs == 12 and e.score == pytest.approx(sum(g.a_points for g in got.games) / len(got.games))


# --------------------------------------------------------------------------------------------------------------
# statistics on hand-made pair lists
# --------------------------------------------------------------------------------------------------------------
def test_pentanomial_elo():
    e = M.elo_from_pairs(M.pentanomial([1.0] * 10))  # every pair 1-1
    assert e.elo == 0.0 and e.lo == 0.0 and e.hi == 0.0 and e.stderr == 0.0
    e = M.elo_from_pairs(M.pentanomial([1.5] * 8))  # s = 0.75
    assert e.elo == pytest.approx(190.85, abs=0.005) and e.lo == e.hi == e.elo
    e = M.elo_from_pairs(M.pentanomial([2.0, 1.0, 1.5, 1.0]))  # s = 0.6875
    assert e.elo == pytest.approx(-400 * math.log10(1 / 0.6875 - 1)) and e.lo < e.elo < e.hi
    p = [0.0, 0.25, 0.5, 0.75, 1.0]
    pairs = [1, 2, 3, 4, 5]
    n = sum(pairs)
    s = sum(c * q for c, q in zip(pairs, p)) / n
    sd = math.sqrt(sum(c * (q - s) ** 2 for c, q in zip(pairs, p)) / n / n)
    e = M.elo_from_pairs(pairs)
    assert e.score == pytest.approx(s) and e.stderr == pytest.approx(sd)
    assert e.lo == pytest.approx(M.elo_of(s - 1.96 * sd)) and e.hi == pytest.approx(M.elo_of(s + 1.96 * sd))
    w = M.elo_from_pairs([0, 0, 0, 0, 7])  # all wins
    assert w.elo == math.inf and w.lo == math.inf and w.hi == math.inf
    assert M.fmt_elo(w.elo) == "+inf" and M.fmt_elo(M.elo_from_pairs([3, 0, 0, 0, 0]).elo) == "-inf"
    assert M.elo_from_pairs([0, 0, 0, 1, 2]).hi == math.inf  # the interval reaches s = 1: infinite, not a number
    assert M.elo_from_pairs([0] * 5) is None
    assert M.pentanomial([0.0, 0.5, 1.0, 1.5, 2.0, 2.0]) == [1, 1, 1, 1, 2]


# --------------------------------------------------------------------------------------------------------------
# PGN (cattus_b200/san.py)
# --------------------------------------------------------------------------------------------------------------
def parse_movetext(fen, pgn: str):
    """The moves of a PGN game's movetext, read back with san.move_from_san."""
    body = "\n".join(line for line in pgn.splitlines() if not line.startswith("["))
    body = re.sub(r"\{[^}]*\}", " ", body)
    played = []
    for tok in body.split():
        if re.fullmatch(r"\d+\.(\.\.)?", tok) or tok in ("1-0", "0-1", "1/2-1/2", "*"):
            continue
        played.append(S.move_from_san(fen, played, tok))
    return played


def test_pgn_movetext_parses_back_to_the_moves():
    na = chess_fake_net("hash")
    openings = [(None, ["e2e4", "c7c5"]), (KIWIPETE, ["e1g1"]), SHUFFLE, ("7k/5Q2/6K1/8/8/8/8/8 b - -", [])]
    res = me.play("chess", openings, chess_cfg(sim_num=10, seed=4, max_moves=40, **NOISY), chess_cb(na), None, n_slots=3)
    assert res.opening_status == [0, 0, 0, 3]
    for g in res.games:
        fen, lans = openings[g.opening]
        opening = [move_from_lan(m) for m in lans]
        text = S.pgn_game(fen, opening, g.moves, g.winner, g.termination, white="A" if g.a_is_player1 else "B",
                          black="B" if g.a_is_player1 else "A", round_=f"{g.opening + 1}.{0 if g.a_is_player1 else 1}")
        assert parse_movetext(fen, text) == opening + g.moves
        result = {None: "1/2-1/2", 1: "1-0", 2: "0-1"}[g.winner]
        assert f'[Result "{result}"]' in text and text.rstrip().endswith(result)
        assert ('[SetUp "1"]' in text and f'[FEN "{fen}' in text) == (fen is not None)
        assert '[Termination "' + ("adjudication" if g.termination == "max_moves" else "normal") + '"]' in text
    # black to move first: the movetext starts "N..." and the move numbers follow the FEN's fullmove field
    text = S.pgn_game("4k3/8/8/8/8/8/4P3/4K3 b - - 0 17", [], [move_from_lan("e8d8"), move_from_lan("e2e4")], None, "max_moves")
    assert "17... Kd8 18. e4" in text


# --------------------------------------------------------------------------------------------------------------
# errors
# --------------------------------------------------------------------------------------------------------------
def test_bad_input_is_einval_naming_the_opening_or_field():
    net = chess_fake_net("hash")
    with pytest.raises(RuntimeError, match="opening 1: bad FEN"):
        me.play("chess", [None, "not a fen"], chess_cfg(sim_num=8), chess_cb(net), None, n_slots=2)
    with pytest.raises(RuntimeError, match="opening 2: move 1 is not legal"):
        me.play("chess", [None, (None, ["e2e4"]), (None, ["e2e4", "e2e4"])], chess_cfg(sim_num=8), chess_cb(net), None, n_slots=2)
    with pytest.raises(RuntimeError, match="opening 0: a FEN is only accepted for chess"):
        me.play("hex5", [(KIWIPETE, [])], cfg_with(sim_num=8), cb_for(fake_net("hash"), 1), None, n_slots=1)
    with pytest.raises(RuntimeError, match="sim_num must be > 1"):
        me.play("chess", [None], chess_cfg(sim_num=1), chess_cb(net), None, n_slots=1)
    with pytest.raises(RuntimeError, match="side B's sim_num must be > 1"):
        me.play("chess", [None], chess_cfg(sim_num=8), chess_cb(net), None, sim_num_b=1, n_slots=1)
    with pytest.raises(RuntimeError, match="error bits"):  # tree memory running out mid-search
        me.play("hex5", [[], [1]], cfg_with(sim_num=200), cb_for(fake_net("hash"), 1), None, n_slots=2, pool_words=2048)
    # every opening finished: nothing to play, and no evaluator call
    calls = []
    res = me.play("chess", FINISHED, chess_cfg(sim_num=8), lambda *a: calls.append(1), None, n_slots=2)
    assert res.games == [] and res.opening_status == [2, 3, 3] and res.elo() is None and calls == []


def test_side_b_settings_apply_to_b_only():
    """B's sim_num and explore_factor change B's searches alone, as the oracle with those settings for B plays them."""
    na = fake_net("hash")
    opening = hex_positions(5, 3, 1)
    cfg = cfg_with(sim_num=20, seed=2)
    same = me.play("hex5", opening, cfg, cb_for(na, 1), None, n_slots=2)
    odds = me.play("hex5", opening, cfg, cb_for(na, 1), None, sim_num_b=50, explore_factor_b=0.5, n_slots=2)
    ref = oracle_match("hex5", [small_history("hex5", m) for m in opening], cfg, na, na, sim_num_b=50, explore_factor_b=0.5)
    check_against_oracle(odds, ref)
    assert odds.simulations == sum(o.sims for o in ref.values()) != same.simulations
    assert [g.moves for g in odds.games] != [g.moves for g in same.games]


def test_play_match_reads_openings(tmp_path):
    from cattus_b200.play_match import read_openings

    (tmp_path / "c.txt").write_text("# comment\n\nstartpos\nstartpos moves e2e4 e7e5\n" + KIWIPETE + ' bm Qxf6; id "kiwi";\n'
                                    + KIWIPETE + " 0 1\n" + KIWIPETE + " moves e1g1\n" + KIWIPETE + "\n")
    assert read_openings(tmp_path / "c.txt", True) == [(None, []), (None, [move_from_lan("e2e4"), move_from_lan("e7e5")]), (KIWIPETE, []),
                                                       (KIWIPETE + " 0 1", []), (KIWIPETE, [move_from_lan("e1g1")]), (KIWIPETE, [])]
    (tmp_path / "h.txt").write_text("startpos\n3 7 12\n")
    assert read_openings(tmp_path / "h.txt", False) == [(None, []), (None, [3, 7, 12])]
