"""CPU tests of the minibatched search under virtual loss (DESIGN.md section 15).

The per-slot code (dsearch_core.hpp's batch_select_slot / batch_expand_slot) and the analysis driver run on the host
with a one-lane warp (tests/emul/search_batch_emul.cpp) and must equal tests/batch_oracle.py -- a plain sequential
statement of the definition over oracle/mcts.py's MctsPlayer -- exactly: children, visits, W bits, best move, PV,
minibatches and collisions.
"""
from __future__ import annotations

from collections import Counter

import numpy as np
import pytest

from oracle import chess as oc
from oracle import mcts as om
from tests import batch_oracle as bo
from tests.emul import analysis_emul as ae
from tests.emul import search_batch_emul as se
from tests.test_analysis_cpu import REPEAT_CHILD, chess_history, chess_positions, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, chess_cb, chess_cfg, chess_fake_net, chess_oracle_fn
from tests.test_selfplay_cpu import cb_for, cfg_with, fake_net, oracle_net_fn

EINVAL, ERANGE = -1, -5
# black to move and mate (Qh4#): many descents of one minibatch end on the same finished position
FOOLS = (None, ["f2f3", "e7e5", "g2g4"])


def bits(xs):
    return np.asarray(xs, dtype=np.float32).view(np.uint32).tolist()


def small_history(game, moves):
    p = om.HexPosition.new(5) if game == "hex5" else om.TttPosition.new()
    for m in moves:
        p = p.moved_position(m)
    return [p]


def check(results, histories, evaluator, sim_num, L, to_move=lambda m: m):
    for k, (a, hist) in enumerate(zip(results, histories)):
        player, moves, visits, w, best, pv = bo.search(hist, evaluator, sim_num, L)
        assert a.status == 0 and a.simulations == sim_num, k
        assert a.moves == [to_move(m) for m in moves], k
        assert a.visits == visits, k
        assert bits(a.w) == bits(w), k
        assert a.best_move == to_move(best), k
        assert a.pv == [to_move(m) for m in pv], k
        assert (a.minibatches, a.collisions) == (player.minibatches, player.collisions), k


# ------------------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("game", ["hex5", "ttt", "chess"])
def test_oracle_search_batch_1_is_mcts_player(game):
    if game == "chess":
        net = chess_fake_net("hash")
        ev = om.Evaluator(chess_oracle_fn(net), None)
        hists = [chess_history(f, m) for f, m in chess_positions(4, 2)]
    else:
        net = fake_net("hash")
        ev = om.Evaluator(oracle_net_fn(net), None)
        hists = [small_history(game, m) for m in (hex_positions(5, 4, 1) if game == "hex5" else ttt_positions(4, 1))]
    params = om.MctsParams(sim_num=30, explore_factor=1.41421, temperature=om.TemperaturePolicy.from_config([[9999, 0.0]]))
    for h in hists:
        ref = om.MctsPlayer(params, ev, om.SplitMix64(0))
        ref_probs = ref.calc_moves_probabilities(h)
        got = bo.BatchedPlayer(params, ev, om.SplitMix64(0), 1)
        assert got.calc_moves_probabilities(h) == ref_probs
        assert [(e.m, e.n, float(e.w)) for e in got.root.children] == [(e.m, e.n, float(e.w)) for e in ref.root.children]
        assert (got.minibatches, got.collisions) == (30, 0)


def _ttt_player(prior, L, sim_num):
    """Tic-tac-toe from the empty board with a fixed evaluator: `prior(cell)` for every legal cell, value 0."""

    def net(pos):
        return [np.float32(prior(m)) for m in pos.legal_moves()], np.float32(0.0)

    params = om.MctsParams(sim_num=sim_num, explore_factor=1.41421, temperature=om.TemperaturePolicy.from_config([[9999, 0.0]]))
    player = bo.BatchedPlayer(params, om.Evaluator(net, None), om.SplitMix64(0), L)
    player.calc_moves_probabilities([om.TttPosition.new()])
    return player


def test_oracle_hand_worked_first_minibatch_is_one_simulation_and_collisions():
    # the root is unexpanded: descent 1 claims it, descents 2..4 end there too
    p = _ttt_player(lambda m: 1.0 / 9.0, 4, 4)
    assert p.choices[0] == [-1, -1, -1, -1]
    assert (p.minibatches, p.collisions, p.sims_done) == (2, 3, 4)
    assert p.choices[1] == [0, 1, 2]  # the second minibatch: k = min(4, 4 - 1) = 3


def test_oracle_hand_worked_second_minibatch_spreads_over_the_root():
    ef = np.float32(1.41421)

    def score(prior, n, v, simcount):  # select's heuristic with n' = n + v, w' = -v (value 0 everywhere)
        n2, w2 = n + v, np.float32(-v)
        exploit = np.float32(0.0) if n2 == 0 else np.float32(w2 / np.float32(n2))
        return np.float32(exploit + np.float32(np.float32(ef * np.float32(prior)) * np.float32(np.sqrt(np.float32(simcount)) / np.float32(1 + n2))))

    # centre prior 0.6, others 0.05: descent 1 takes the centre (1.41421 * 0.6 = 0.85 against 0.07); descent 2 sees it at
    # n' = 1, w' = -1: -1 + 0.85 * sqrt(2) / 2 = -0.40 < 0.05 * 1.41421 * sqrt(2) = 0.10, so cell 0 (ties: the first
    # inserted); descents 3, 4 take cells 1, 2 the same way
    prior = lambda m: 0.6 if m == 4 else 0.05  # noqa: E731
    want, v = [], {m: 0 for m in range(9)}
    for j in range(4):
        simcount = 1 + sum(v.values())
        s = [score(prior(m), 0, v[m], simcount) for m in range(9)]
        top = max(s)
        pick = min(m for m in range(9) if s[m] == top)
        want.append(pick)
        v[pick] += 1
    assert want == [4, 0, 1, 2]
    p = _ttt_player(prior, 4, 5)
    assert p.choices[1] == want and p.collisions == 3
    # nine children, twelve descents: each child claimed once, the last three descents collide
    p = _ttt_player(lambda m: 1.0 / 9.0, 12, 13)
    assert sorted(p.choices[1][:9]) == list(range(9)) and p.collisions == 11 + 3


# ------------------------------------------------------------------------------------------------------------ emulation
@pytest.mark.parametrize("L", [2, 3, 7, 32, 256])
@pytest.mark.parametrize("game", ["hex5", "ttt"])
def test_emulation_equals_oracle_hex_ttt(game, L):
    net = fake_net("hash" if L != 7 else "coarse")
    sim_num = 61
    positions = hex_positions(5, 6, L) if game == "hex5" else ttt_positions(8, L)
    got = se.analyse(game, positions, cfg_with(sim_num=sim_num, device_games=3), cb_for(net, 1), search_batch=L)
    check(got, [small_history(game, m) for m in positions], om.Evaluator(oracle_net_fn(net), None), sim_num, L)


@pytest.mark.parametrize("L", [2, 3, 7, 32, 256])
def test_emulation_equals_oracle_chess(L):
    net = chess_fake_net("hash")
    sim_num = 97 if L < 256 else 301
    positions = [FOOLS, (None, REPEAT_CHILD), (KIWIPETE, [])] + chess_positions(4, L)[2:]
    got = se.analyse("chess", positions, chess_cfg(sim_num=sim_num, device_games=2), chess_cb(net), search_batch=L,
                      pool_words=1 << 18)
    hists = [chess_history(f, m) for f, m in positions]
    check(got, hists, om.Evaluator(chess_oracle_fn(net), None), sim_num, L, oc.move_to_u16)
    # the mate is found, and descents of one minibatch pile onto it and onto the repetition
    assert oc.move_to_u16(next(m for m in chess_history(*FOOLS)[-1].legal_moves() if oc.move_to_lan(m) == "d8h4")) == got[0].best_move


def piled(player):
    """Most descents of one minibatch that were scored on the same node."""
    return max(max(Counter(i for k, i in mb if k == "score").values(), default=0) for mb in player.kinds)


def test_descents_piling_onto_a_terminal_or_a_repetition_are_backed_up_not_collided():
    # several descents of one minibatch end on the same finished position or complete the same threefold repetition:
    # neither is a claim, so each is backed up with its value
    net = fake_net("hash")
    hist = small_history("ttt", [0, 4, 1])  # O to move must block at 2
    ev = om.Evaluator(oracle_net_fn(net), None)
    player, *_ = bo.search(hist, ev, 50, 16)
    assert piled(player) >= 2
    check(se.analyse("ttt", [[0, 4, 1]], cfg_with(sim_num=50), cb_for(net, 1), search_batch=16), [hist], ev, 50, 16)
    cnet = chess_fake_net("hash")
    cev = om.Evaluator(chess_oracle_fn(cnet), None)
    for pos, sims in ((FOOLS, 97), ((None, REPEAT_CHILD), 120)):
        hist = chess_history(*pos)
        player, *_ = bo.search(hist, cev, sims, 32)
        assert piled(player) >= 2, pos
        check(se.analyse("chess", [pos], chess_cfg(sim_num=sims), chess_cb(cnet), search_batch=32), [hist], cev, sims, 32, oc.move_to_u16)


def test_results_do_not_depend_on_slots_waves_cache_or_order():
    net = chess_fake_net("hash")
    positions = chess_positions(12, 8)
    ref = se.analyse("chess", positions, chess_cfg(sim_num=45, device_games=1), chess_cb(net), search_batch=7, depth=1)
    assert all(a.minibatches > 0 for a in ref if a.status == 0)
    for games, depth, cache in ((3, 1, 0), (16, 3, 0), (3, 3 | 256, 5000), (16, 1, 64), (4, 2 | 256, 5000)):
        got = se.analyse("chess", positions, chess_cfg(sim_num=45, device_games=games, cache_size=cache), chess_cb(net), search_batch=7, depth=depth)
        assert got == ref, (games, depth, cache)
    rev = se.analyse("chess", positions[::-1], chess_cfg(sim_num=45, device_games=5), chess_cb(net), search_batch=7)
    assert rev[::-1] == ref
    hnet = fake_net("hash")
    hpos = hex_positions(5, 10, 9)
    href = se.analyse("hex5", hpos, cfg_with(sim_num=50, device_games=1), cb_for(hnet, 1), search_batch=16, depth=1)
    for games, depth, cache in ((3, 1, 0), (16, 3, 1000), (5, 2 | 256, 100)):
        assert se.analyse("hex5", hpos, cfg_with(sim_num=50, device_games=games, cache_size=cache), cb_for(hnet, 1), search_batch=16,
                          depth=depth) == href


@pytest.mark.parametrize("search_batch", [0, 1])
def test_search_batch_1_is_the_one_leaf_analysis(search_batch):
    net = chess_fake_net("hash")
    positions = chess_positions(10, 3)
    ref = ae.analyse("chess", positions, chess_cfg(sim_num=30), chess_cb(net), n_slots=4)
    got = se.analyse("chess", positions, chess_cfg(sim_num=30, device_games=4), chess_cb(net), search_batch=search_batch)
    for a, r in zip(got, ref):
        assert (a.minibatches, a.collisions) == ((30, 0) if a.status == 0 else (0, 0))
        a.minibatches = a.collisions = 0
    assert got == ref


def test_slots_times_search_batch_beyond_max_batch_is_erange_and_bad_opts_einval():
    net = chess_fake_net("hash")
    with pytest.raises(se.EmulError, match="max_batch") as e:
        se.analyse("chess", [None], chess_cfg(sim_num=8, device_games=5), chess_cb(net), search_batch=64, max_batch=256)
    assert e.value.code == ERANGE
    with pytest.raises(se.EmulError, match="max_batch") as e:
        se.analyse("chess", [None], chess_cfg(sim_num=8), chess_cb(net), search_batch=512, max_batch=256)
    assert e.value.code == ERANGE
    with pytest.raises(se.EmulError, match="struct_size") as e:
        se.analyse("chess", [None], chess_cfg(sim_num=8), chess_cb(net), search_batch=4, opts_size=4)
    assert e.value.code == EINVAL
    # device_games 0 takes max_batch / search_batch slots: 4 positions over 2 slots give the same results
    got = se.analyse("chess", [None] * 4, chess_cfg(sim_num=20), chess_cb(net), search_batch=64, max_batch=128)
    assert got == se.analyse("chess", [None] * 4, chess_cfg(sim_num=20, device_games=1), chess_cb(net), search_batch=64, max_batch=128)
