"""CPU tests of the batched analysis of given positions (cattus_b200/csrc/dsearch_analysis.hpp over dsearch_core.hpp).

The analysis driver and the per-slot search code are compiled for the host with a one-lane warp (tests/emul) and driven
by a deterministic Python evaluator; every position's children, visit counts, best move and principal variation must
equal a fresh oracle MctsPlayer's search of the same history with noise off.  Also the SAN / EPD helpers of the CLI.
"""
from __future__ import annotations

import random

import pytest

from cattus_b200 import san as S
from cattus_b200.selfplay import move_from_lan, move_to_lan
from oracle import chess as oc
from oracle import mcts as om
from tests.emul import analysis_emul as ae
from tests.test_chess_cpu import KIWIPETE, PERFT, chess_cb, chess_cfg, chess_fake_net, chess_oracle_fn
from tests.test_selfplay_cpu import cb_for, cfg_with, fake_net, oracle_net_fn

# one root child (g1f3 ... f6g8) completes a threefold repetition of the start position
REPEAT_CHILD = ["g1f3", "g8f6", "f3g1", "f6g8", "g1f3", "g8f6", "f3g1"]


def oracle_search(history, evaluator, sim_num):
    """A fresh MctsPlayer with noise off: (children moves, visits, best move, PV) of its search of history[-1]."""
    params = om.MctsParams(sim_num=sim_num, explore_factor=1.41421, temperature=om.TemperaturePolicy.from_config([[9999, 0.0]]))
    player = om.MctsPlayer(params, evaluator, om.SplitMix64(0))
    probs = player.calc_moves_probabilities(history)
    best = player.choose_move_from_probabilities(history, probs)
    edges = list(reversed(player.root.children))
    pv, node = [], player.root
    while node.children and len(pv) < 16:  # most visits; equal counts -> smallest insertion index
        top = max(c.n for c in node.children)
        e = next(c for c in node.children if c.n == top)
        pv.append(e.m)
        node = e.target
    return [e.m for e in edges], [e.n for e in edges], best, pv


def hex_positions(s, count, seed):
    rng = random.Random(seed)
    out = []
    while len(out) < count:
        pos, moves = om.HexPosition.new(s), []
        for _ in range(rng.randrange(0, s * s - 2)):
            legal = pos.legal_moves()
            m = rng.choice(legal)
            nxt = pos.moved_position(m)
            if nxt.is_finished():
                break
            pos, moves = nxt, moves + [m]
        out.append(moves)
    return out


def ttt_positions(count, seed):
    rng = random.Random(seed)
    out = []
    while len(out) < count:
        pos, moves = om.TttPosition.new(), []
        for _ in range(rng.randrange(0, 7)):
            m = rng.choice(pos.legal_moves())
            nxt = pos.moved_position(m)
            if nxt.is_finished():
                break
            pos, moves = nxt, moves + [m]
        out.append(moves)
    return out


def chess_positions(count, seed):
    """(fen, LAN moves) from seeded random playouts, some from FENs, and the repetition case."""
    rng = random.Random(seed)
    out = [(None, REPEAT_CHILD), (KIWIPETE, ["e1g1", "e8c8"])]
    fens = [None, KIWIPETE] + [f for f, _ in PERFT[2:]]
    while len(out) < count:
        fen = rng.choice(fens)
        pos = oc.ChessPosition.from_fen(fen) if fen else oc.ChessPosition.new()
        moves = []
        for _ in range(rng.randrange(0, 30)):
            legal = pos.legal_moves()
            m = rng.choice(legal)
            nxt = pos.moved_position(m)
            if nxt.is_finished():
                break
            pos, moves = nxt, moves + [oc.move_to_lan(m)]
        out.append((fen, moves))
    return out


def chess_history(fen, moves):
    h = [oc.ChessPosition.from_fen(fen) if fen else oc.ChessPosition.new()]
    for lan in moves:
        h.append(h[-1].moved_position(next(m for m in h[-1].legal_moves() if oc.move_to_lan(m) == lan)))
    return h


def check_against_oracle(results, histories, evaluator, sim_num, to_move=lambda m: m):
    for k, (a, hist) in enumerate(zip(results, histories)):
        moves, visits, best, pv = oracle_search(hist, evaluator, sim_num)
        assert a.status == 0 and a.simulations == sim_num
        assert a.moves == [to_move(m) for m in moves], k
        assert a.visits == visits, k
        assert a.best_move == to_move(best), k
        assert a.pv == [to_move(m) for m in pv], k
        assert a.pv[0] == a.best_move
        assert abs(a.q - sum(a.w) / sum(a.visits)) < 1e-6


@pytest.mark.parametrize("game,kind,sim_num", [("hex5", "hash", 60), ("hex5", "uniform", 40), ("ttt", "coarse", 50)])
def test_analysis_equals_fresh_oracle_player_hex_ttt(game, kind, sim_num):
    net = fake_net(kind)
    cfg = cfg_with(sim_num=sim_num)
    positions = hex_positions(5, 20, 3) if game == "hex5" else ttt_positions(20, 4)
    got = ae.analyse(game, positions, cfg, cb_for(net, 1), n_slots=6)
    if game == "hex5":
        hists = []
        for mv in positions:
            p = om.HexPosition.new(5)
            for m in mv:
                p = p.moved_position(m)
            hists.append([p])
    else:
        hists = []
        for mv in positions:
            p = om.TttPosition.new()
            for m in mv:
                p = p.moved_position(m)
            hists.append([p])
    check_against_oracle(got, hists, om.Evaluator(oracle_net_fn(net), None), sim_num)


@pytest.mark.parametrize("kind", ["hash", "uniform"])
def test_analysis_equals_fresh_oracle_player_chess(kind):
    net = chess_fake_net(kind)
    positions = chess_positions(20, 11)
    got = ae.analyse("chess", positions, chess_cfg(sim_num=40), chess_cb(net), n_slots=5)
    hists = [chess_history(f, m) for f, m in positions]
    check_against_oracle(got, hists, om.Evaluator(chess_oracle_fn(net), None), 40, oc.move_to_u16)
    # the repetition case: the child that repeats the start position a third time is scored as a draw inside the search
    rep = [a for a, (f, m) in zip(got, positions) if m == REPEAT_CHILD][0]
    assert move_from_lan("f6g8") in rep.moves


def test_results_do_not_depend_on_slots_waves_cache_or_order():
    net = chess_fake_net("hash")
    positions = chess_positions(24, 5)
    cfg = chess_cfg(sim_num=30)
    ref = ae.analyse("chess", positions, cfg, chess_cb(net), n_slots=1, depth=1)
    for n_slots, depth, cache, roots_cap in ((3, 1, 0, 0), (16, 3, 0, 0), (3, 3 | 256, 5000, 0), (16, 1, 64, 0), (4, 2 | 256 | 512, 5000, 0),
                                             (16, 2 | 256, 0, 1)):
        got = ae.analyse("chess", positions, chess_cfg(sim_num=30, cache_size=cache), chess_cb(net), n_slots=n_slots, depth=depth, roots_cap=roots_cap)
        assert got == ref, (n_slots, depth, cache)
    rev = ae.analyse("chess", positions[::-1], cfg, chess_cb(net), n_slots=7)
    assert rev[::-1] == ref
    hnet = fake_net("hash")
    hpos = hex_positions(5, 16, 9)
    href = ae.analyse("hex5", hpos, cfg_with(sim_num=40), cb_for(hnet, 1), n_slots=1, depth=1)
    for n_slots, depth, cache in ((3, 1, 0), (16, 3, 1000), (5, 2 | 256 | 512, 100)):
        assert ae.analyse("hex5", hpos, cfg_with(sim_num=40, cache_size=cache), cb_for(hnet, 1), n_slots=n_slots, depth=depth) == href


def test_finished_roots_are_reported_without_a_search():
    net = chess_fake_net("hash")
    calls = []

    def counting(words, n, legal):
        calls.append(n)
        return chess_cb(net)(words, n, legal)

    positions = [(None, ["f2f3", "e7e5", "g2g4", "d8h4"]),                 # mate: black (player 2) won
                 ("7k/5Q2/6K1/8/8/8/8/8 b - -", []),                      # stalemate
                 (None, REPEAT_CHILD + ["f6g8"]),                         # threefold repetition in the given history
                 (None, ["e2e4"])]
    only = ae.analyse("chess", positions[:3], chess_cfg(sim_num=20), counting, n_slots=2)
    assert [a.status for a in only] == [2, 3, 3] and calls == []
    got = ae.analyse("chess", positions, chess_cfg(sim_num=20), counting, n_slots=2)
    assert [a.status for a in got] == [2, 3, 3, 0]
    for a in got[:3]:
        assert a.moves == [] and a.pv == [] and a.best_move is None and a.simulations == 0
    assert got[3].simulations == 20 and calls
    rng = random.Random(1)
    p, won = om.HexPosition.new(5), []
    while not p.is_finished():
        won.append(rng.choice(p.legal_moves()))
        p = p.moved_position(won[-1])
    got = ae.analyse("hex5", [won, []], cfg_with(sim_num=10), cb_for(fake_net("hash"), 1), n_slots=2)
    assert got[0].status == p.status()[1] and got[0].moves == [] and got[1].status == 0


def test_bad_input_is_einval_naming_the_position_or_field():
    net = chess_fake_net("hash")
    with pytest.raises(RuntimeError, match="position 1: bad FEN"):
        ae.analyse("chess", [None, "not a fen"], chess_cfg(sim_num=8), chess_cb(net), n_slots=2)
    with pytest.raises(RuntimeError, match="position 2: move 1 is not legal"):
        ae.analyse("chess", [None, (None, ["e2e4"]), (None, ["e2e4", "e2e4"])], chess_cfg(sim_num=8), chess_cb(net), n_slots=2)
    with pytest.raises(RuntimeError, match="prior_noise_epsilon"):
        ae.analyse("chess", [None], chess_cfg(sim_num=8, prior_noise_alpha=0.3, prior_noise_epsilon=0.25), chess_cb(net), n_slots=1)
    with pytest.raises(RuntimeError, match="position 0: a FEN is only accepted for chess"):
        ae.analyse("hex5", [(KIWIPETE, [])], cfg_with(sim_num=8), cb_for(fake_net("hash"), 1), n_slots=1)
    with pytest.raises(RuntimeError, match="position 1: move 0 is not legal"):
        ae.analyse("hex5", [[3], [99]], cfg_with(sim_num=8), cb_for(fake_net("hash"), 1), n_slots=1)


def test_tree_pool_exhaustion_is_an_error_not_a_result():
    with pytest.raises(RuntimeError, match="error bits"):
        ae.analyse("hex5", [[], [1]], cfg_with(sim_num=200), cb_for(fake_net("hash"), 1), n_slots=2, pool_words=2048)


# --------------------------------------------------------------------------------------------------------------
# SAN and EPD (cattus_b200/san.py)
# --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fen", [f for f, _ in PERFT])
def test_san_is_unique_and_round_trips_on_the_perft_positions(fen):
    legal = S.legal_moves(fen)
    sans = [S.move_to_san(fen, [], m) for m in legal]
    assert len(set(sans)) == len(sans)
    for m, s in zip(legal, sans):
        assert S.move_from_san(fen, [], s) == m
        assert S.move_from_san(fen, [], s + "!?") == m


def test_san_hand_checked_cases():
    assert S.move_to_san(KIWIPETE, [], move_from_lan("e1g1")) == "O-O"
    assert S.move_to_san(KIWIPETE, [], move_from_lan("e1c1")) == "O-O-O"
    assert S.move_from_san(KIWIPETE, [], "0-0-0") == move_from_lan("e1c1")
    ep = "4k3/8/8/3pP3/8/8/8/4K3 w - d6"
    assert S.move_to_san(ep, [], move_from_lan("e5d6")) == "exd6"
    assert S.board(ep, [move_from_lan("e5d6")]).get(35) is None  # the d5 pawn is gone
    promo = "8/P6k/8/8/8/8/8/4K3 w - -"
    assert S.move_to_san(promo, [], move_from_lan("a7a8q")) == "a8=Q"
    assert S.move_to_san(promo, [], move_from_lan("a7a8n")) == "a8=N"
    assert S.move_from_san(promo, [], "a8=R") == move_from_lan("a7a8r")
    # file and rank disambiguation
    knights = "4k3/8/8/8/8/8/8/1N2K1N1 w - -"
    rooks = "4k3/8/8/8/8/8/4K3/R6R w - -"
    assert S.move_to_san(rooks, [], move_from_lan("a1d1")) == "Rad1"
    assert S.move_to_san(rooks, [], move_from_lan("h1f1")) == "Rhf1"
    stacked = "4k3/8/8/R7/8/8/8/R3K3 w - -"
    assert S.move_to_san(stacked, [], move_from_lan("a1a3")) == "R1a3"
    assert S.move_to_san(stacked, [], move_from_lan("a5a3")) == "R5a3"
    assert S.move_from_san(knights, [], "Nd2") == move_from_lan("b1d2")
    mate = S.move_to_san(None, [move_from_lan(x) for x in ("f2f3", "e7e5", "g2g4")], move_from_lan("d8h4"))
    assert mate == "Qh4#"
    with pytest.raises(ValueError):
        S.move_from_san(rooks, [], "Rd1")  # two rooks reach d1
    with pytest.raises(ValueError):
        S.move_from_san(None, [], "e5")


def test_epd_and_fen_lines():
    rec = S.parse_epd('r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - bm Qxf6 Nxf7; am O-O; id "kiwi; pete";')
    assert rec.fen == KIWIPETE and rec.id == "kiwi; pete"
    assert rec.ops["bm"] == ["Qxf6", "Nxf7"] and rec.ops["am"] == ["O-O"]
    assert {S.move_from_san(rec.fen, [], m) for m in rec.ops["bm"]} == {move_from_lan("f3f6"), move_from_lan("e5f7")}
    assert S.parse_epd("8/8/8/8/8/8/8/K6k w - -").ops == {}
    assert S.parse_fen_line("startpos moves e2e4 e7e5") == (None, ["e2e4", "e7e5"])
    assert S.parse_fen_line(KIWIPETE + " 0 1 moves e1g1") == (KIWIPETE + " 0 1", ["e1g1"])
    assert S.parse_fen_line(KIWIPETE) == (KIWIPETE, [])
    assert move_to_lan(S.move_from_san(None, [], "Nf3")) == "g1f3"
