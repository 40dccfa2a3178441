"""CPU tests of self-play and match play with minibatches under virtual loss per side (DESIGN.md section 16).

The self-play / match driver and the minibatch kernels' per-slot code run on the host with a one-lane warp
(tests/emul/selfplay_batch_emul.cpp) and must equal, move for move and byte for byte, tests/batch_game_oracle.py's game
loop whose players are tests/batch_oracle.py's BatchedPlayer(L) -- a plain sequential statement of the minibatched search over oracle/mcts.py.
"""
from __future__ import annotations

import pytest

from oracle import chess as oc
from oracle import mcts as om
from tests import batch_game_oracle as bo
from tests.emul import emul
from tests.emul import match_emul as me
from tests.emul import selfplay_batch_emul as sbe
from tests.test_analysis_cpu import REPEAT_CHILD, chess_history, chess_positions, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, _params, chess_cb, chess_cfg, chess_fake_net, chess_oracle_fn
from tests.test_match_cpu import FORCED, SHUFFLE, small_history
from tests.test_selfplay_cpu import cb_for, cfg_with, fake_net, oracle_net_fn

EINVAL, ERANGE = -1, -5
NOISY = dict(prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[4, 1.0], [9999, 0.0]])


def setup(game, salt_b=None):
    """(net A, net B or None, callback factory, oracle evaluator factory, params from cfg, initial position)."""
    if game == "chess":
        na = chess_fake_net("hash")
        nb = chess_fake_net("hash", salt=salt_b) if salt_b is not None else None
        return na, nb, chess_cb, lambda n: om.Evaluator(chess_oracle_fn(n), None), _params, oc.ChessPosition.new
    na = fake_net("hash")
    nb = fake_net("hash", salt=salt_b) if salt_b is not None else None
    wpp = 1 if game == "ttt" else (int(game[3:]) ** 2 + 63) // 64
    new = om.TttPosition.new if game == "ttt" else (lambda: om.HexPosition.new(int(game[3:])))
    return na, nb, (lambda n: cb_for(n, wpp)), (lambda n: om.Evaluator(oracle_net_fn(n), None)), _params, new


def oracle_selfplay(game, cfg, L, games_num, na, nb, ev, params, new):
    ea = ev(na)
    eb = ea if nb is None else ev(nb)
    p = params(cfg)
    out = []
    for g in range(games_num):
        out.append(bo.play_from(g, [new()], p, p, ea, eb, cfg["seed"], cfg.get("max_moves", 0), (L, L)))
    return out


def check_selfplay(game, cfg, L, counters, records, ref, chess):
    to_move = oc.move_to_u16 if chess else (lambda m: m)
    assert len(records) == len(ref)
    mb, co = [0, 0], [0, 0]
    for rec, (o, p1, p2) in zip(records, ref):
        assert rec.game_idx == o.game_idx
        assert rec.moves == [to_move(m) for m in o.moves], (L, rec.game_idx)
        assert rec.winner == o.winner
        assert len(rec.entries) == len(o.entries)
        for k, (pos, probs) in enumerate(o.entries):
            assert rec.entries[k] == om.data_entry_bytes(pos, probs, o.winner), (L, rec.game_idx, k)
        m1, m2 = p1, p2  # play_from's player1 is model 1's player in every game, whichever colour it has
        mb[0] += m1.minibatches
        mb[1] += m2.minibatches
        co[0] += m1.collisions
        co[1] += m2.collisions
    assert counters["simulations"] == sum(o.sims for o, _, _ in ref) == counters["searches"] * cfg["mcts"]["sim_num"]
    assert counters["terminal"] == sum(o.terminal_leaves for o, _, _ in ref)
    assert counters["minibatches"] == tuple(mb) and counters["collisions"] == tuple(co)


# ------------------------------------------------------------------------------------------------------------ the reference
@pytest.mark.parametrize("game", ["hex5", "chess"])
def test_reference_with_l1_is_the_oracle_play_game(game):
    na, nb, _, ev, params, new = setup(game, salt_b=99)
    mk = chess_cfg if game == "chess" else cfg_with
    cfg = mk(sim_num=14 if game == "chess" else 24, seed=4, max_moves=12 if game == "chess" else 0, **NOISY)
    ea, eb = ev(na), ev(nb)
    for g in range(2):
        ref = om.play_game(g, new, params(cfg), params(cfg), ea, eb, cfg["seed"], cfg.get("max_moves", 0))
        got, p1, p2 = bo.play_from(g, [new()], params(cfg), params(cfg), ea, eb, cfg["seed"], cfg.get("max_moves", 0))
        assert (got.moves, got.winner, got.sims) == (ref.moves, ref.winner, ref.sims)
        assert [(p, [(m, float(x)) for m, x in q]) for p, q in got.entries] == [(p, [(m, float(x)) for m, x in q]) for p, q in ref.entries]
        assert p1.collisions == p2.collisions == 0


# ------------------------------------------------------------------------------------------------------------ self-play
@pytest.mark.parametrize("L", [2, 7, 32])
@pytest.mark.parametrize("game", ["hex5", "ttt", "chess"])
def test_selfplay_equals_the_reference(game, L):
    """Noise and temperature on; every game's first search expands its root inside a minibatch (the noise of that
    root); later searches reuse their trees; chess games run into max_moves and into repetitions inside minibatches."""
    na, nb, cb, ev, params, new = setup(game, salt_b=99)
    if game == "chess":
        cfg = chess_cfg(sim_num=24, seed=7, max_moves=14, device_games=3, **NOISY)
    else:
        cfg = cfg_with(sim_num=30 if game == "hex5" else 20, seed=7, device_games=3, **NOISY)
    games_num = 4
    counters, records = sbe.selfplay(game, cfg, cb(na), cb(nb), games_num, search_batch=L)
    ref = oracle_selfplay(game, cfg, L, games_num, na, nb, ev, params, new)
    check_selfplay(game, cfg, L, counters, records, ref, game == "chess")
    assert sum(counters["collisions"]) > 0


def test_selfplay_chess_repetition_scored_inside_minibatches():
    # a deterministic net at temperature 0 shuffles pieces: the searches see threefold repetitions inside minibatches
    na, _, cb, ev, params, new = setup("chess")
    cfg = chess_cfg(sim_num=12, seed=5, device_games=2)
    counters, records = sbe.selfplay("chess", cfg, cb(na), None, 2, search_batch=4)
    ref = oracle_selfplay("chess", cfg, 4, 2, na, None, ev, params, new)
    check_selfplay("chess", cfg, 4, counters, records, ref, True)
    assert sum(p1.repetition_hits + p2.repetition_hits for _, p1, p2 in ref) > 0


# ------------------------------------------------------------------------------------------------------------ match play
def oracle_match(game, histories, cfg, na, nb, ev, params, La, Lb, sim_num_b=None):
    pa = params(cfg)
    pb = om.MctsParams(**dict(pa.__dict__, sim_num=sim_num_b or pa.sim_num))
    ea, eb = ev(na), ev(nb)
    out = {}
    for k, h in enumerate(histories):
        if h is None:
            continue
        for c in (0, 1):
            out[(k, c == 0)] = bo.play_from(2 * k + c, h, pa, pb, ea, eb, cfg["seed"], cfg.get("max_moves", 0), (La, Lb))
    return out


def check_match(got, ref, to_move=lambda m: m):
    assert [(g.opening, g.a_is_player1) for g in got.games] == sorted(ref, key=lambda x: (x[0], not x[1]))
    mb, co = [0, 0], [0, 0]
    for g in got.games:
        o, p1, p2 = ref[(g.opening, g.a_is_player1)]
        assert g.moves == [to_move(m) for m in o.moves], (g.opening, g.a_is_player1)
        assert g.winner == o.winner
        a, b = p1, p2  # A is model 1
        mb[0] += a.minibatches
        mb[1] += b.minibatches
        co[0] += a.collisions
        co[1] += b.collisions
    assert got.simulations == sum(o.sims for o, _, _ in ref.values())
    assert got.minibatches == tuple(mb) and got.collisions == tuple(co)


@pytest.mark.parametrize("La,Lb", [(1, 16), (8, 3)])
def test_match_hex_ttt_equals_the_reference(La, Lb):
    for game, openings in (("hex5", hex_positions(5, 3, 7)), ("ttt", ttt_positions(3, 8))):
        na, nb, cb, ev, params, _ = setup(game, salt_b=99)
        cfg = cfg_with(sim_num=26, seed=3, **NOISY)
        got = sbe.match(game, openings, cfg, cb(na), cb(nb), sim_num_b=34, search_batch=La, search_batch_b=Lb)
        ref = oracle_match(game, [[*small_history(game, m)] for m in openings], cfg, na, nb, ev, params, La, Lb, sim_num_b=34)
        check_match(got, ref)


@pytest.mark.parametrize("La,Lb", [(1, 16), (8, 3)])
def test_match_chess_openings_equal_the_reference(La, Lb):
    """FEN openings and the repetition opening; two evaluators and a different sim_num for B."""
    na, nb, cb, ev, params, _ = setup("chess", salt_b=99)
    openings = [FORCED, (KIWIPETE, ["e1g1"]), SHUFFLE] + chess_positions(2, 31)[1:]
    cfg = chess_cfg(sim_num=16, seed=5, max_moves=12, **NOISY)
    got = sbe.match("chess", openings, cfg, cb(na), cb(nb), sim_num_b=22, search_batch=La, search_batch_b=Lb)
    ref = oracle_match("chess", [chess_history(f, m) for f, m in openings], cfg, na, nb, ev, params, La, Lb, sim_num_b=22)
    check_match(got, ref, oc.move_to_u16)
    assert {g.termination for g in got.games} >= {"repetition", "max_moves"}


# ------------------------------------------------------------------------------------------------------------ invariance
def test_results_do_not_depend_on_slots_waves_begin_cache_handles_or_order():
    na = chess_fake_net("hash")
    openings = chess_positions(5, 3) + [SHUFFLE]
    cfg = chess_cfg(sim_num=14, seed=2, max_moves=10, **NOISY)
    ref = sbe.match("chess", openings, dict(cfg, device_games=1), chess_cb(na), None, search_batch=1, search_batch_b=9, depth=1)
    assert ref.collisions[1] > 0 and ref.collisions[0] == 0
    for slots, depth, cache in ((3, 1, 0), (16, 3, 0), (3, 3 | 256, 5000), (16, 2 | 256, 64)):
        got = sbe.match("chess", openings, chess_cfg(sim_num=14, seed=2, max_moves=10, cache_size=cache, device_games=slots, **NOISY), chess_cb(na),
                        None, search_batch=1, search_batch_b=9, depth=depth)
        assert (got.games, got.pairs, got.minibatches, got.collisions) == (ref.games, ref.pairs, ref.minibatches, ref.collisions), (slots, depth)
    two = sbe.match("chess", openings, cfg, chess_cb(na), chess_cb(na), search_batch=1, search_batch_b=9)
    assert (two.games, two.minibatches, two.collisions) == (ref.games, ref.minibatches, ref.collisions)
    # reversed openings, noise off: the same game for each (opening, colour)
    quiet = chess_cfg(sim_num=14, seed=2, max_moves=10)
    fwd = sbe.match("chess", openings, dict(quiet, device_games=4), chess_cb(na), None, search_batch=5)
    rev = sbe.match("chess", openings[::-1], dict(quiet, device_games=5), chess_cb(na), None, search_batch=5)
    n = len(openings)
    assert sorted((n - 1 - g.opening, g.a_is_player1, g.moves, g.winner) for g in rev.games) == \
        sorted((g.opening, g.a_is_player1, g.moves, g.winner) for g in fwd.games)
    # self-play
    hnet = fake_net("hash")
    hcfg = cfg_with(sim_num=24, seed=6, **NOISY)
    hc, href = sbe.selfplay("hex5", dict(hcfg, device_games=1), cb_for(hnet, 1), None, 6, search_batch=6, depth=1)
    for slots, depth, cache in ((3, 1, 0), (16, 3, 1000), (5, 2 | 256, 100)):
        c, got = sbe.selfplay("hex5", cfg_with(sim_num=24, seed=6, cache_size=cache, device_games=slots, **NOISY), cb_for(hnet, 1), None, 6,
                              search_batch=6, depth=depth)
        assert got == href and (c["minibatches"], c["collisions"]) == (hc["minibatches"], hc["collisions"]), (slots, depth)


# ------------------------------------------------------------------------------------------------------------ L = 1
def test_l1_through_the_new_entries_is_the_existing_driver():
    hnet, hnet2 = fake_net("hash"), fake_net("hash", salt=99)
    cfg = cfg_with(sim_num=20, seed=9, device_games=3, **NOISY)
    ref_c, ref = emul.run("hex5", cfg, cb_for(hnet, 1), cb_for(hnet2, 1), 4, n_slots=3, pool_words=1 << 16)
    for sb in (None, 0, 1):
        c, got = sbe.selfplay("hex5", cfg, cb_for(hnet, 1), cb_for(hnet2, 1), 4, search_batch=sb)
        assert got == ref
        assert c["simulations"] == ref_c["simulations"] and sum(c["minibatches"]) == ref_c["simulations"] and c["collisions"] == (0, 0)
    na, nb = chess_fake_net("hash"), chess_fake_net("hash", salt=99)
    openings = chess_positions(4, 2) + [SHUFFLE]
    ccfg = chess_cfg(sim_num=12, seed=2, max_moves=10, **NOISY)
    mref = me.play("chess", openings, ccfg, chess_cb(na), chess_cb(nb), n_slots=5)
    for a, b in ((None, None), (1, 1), (1, None)):
        got = sbe.match("chess", openings, dict(ccfg, device_games=5), chess_cb(na), chess_cb(nb), search_batch=a, search_batch_b=b)
        assert (got.games, got.pairs, got.simulations, got.evaluations) == (mref.games, mref.pairs, mref.simulations, mref.evaluations)
        if a is not None:
            assert sum(got.minibatches) == got.simulations and got.collisions == (0, 0)


# ------------------------------------------------------------------------------------------------------------ errors
def test_errors():
    net = chess_fake_net("hash")
    cb = chess_cb(net)
    with pytest.raises(sbe.EmulError, match="max_batch") as e:  # device_games x L above max_batch
        sbe.selfplay("chess", chess_cfg(sim_num=8, device_games=5), cb, None, 2, search_batch=64, max_batch=256)
    assert e.value.code == ERANGE
    with pytest.raises(sbe.EmulError, match="max_batch") as e:  # the larger side decides
        sbe.match("chess", [None], chess_cfg(sim_num=8, device_games=4), cb, None, search_batch=1, search_batch_b=128, max_batch=256)
    assert e.value.code == ERANGE
    with pytest.raises(sbe.EmulError, match="search_batch") as e:  # the host-tree driver keeps one leaf in flight
        sbe.selfplay("chess", chess_cfg(sim_num=8, device_games=0), cb, None, 2, search_batch=4)
    assert e.value.code == EINVAL
    with pytest.raises(sbe.EmulError, match="struct_size") as e:
        sbe.selfplay("chess", chess_cfg(sim_num=8, device_games=2), cb, None, 2, search_batch=4, opts_size=4)
    assert e.value.code == EINVAL
    with pytest.raises(sbe.EmulError, match="struct_size") as e:
        sbe.match("chess", [None], chess_cfg(sim_num=8), cb, None, search_batch=4, opts_size=8)
    assert e.value.code == EINVAL
    # device_games 0 in a match takes max_batch / L slots
    got = sbe.match("chess", [None, (None, ["e2e4"])], chess_cfg(sim_num=12, max_moves=4), cb, None, search_batch=64, max_batch=128)
    ref = sbe.match("chess", [None, (None, ["e2e4"])], chess_cfg(sim_num=12, max_moves=4, device_games=1), cb, None, search_batch=64, max_batch=128)
    assert got.games == ref.games


def test_host_tree_driver_rejects_minibatches_through_the_library():
    from cattus_b200.selfplay import SelfPlayError, SelfPlayRunner

    net = fake_net("hash")
    with pytest.raises(SelfPlayError, match="search_batch"):
        SelfPlayRunner("hex5", cfg_with(sim_num=8, search_batch=4)).run_with(cb_for(net, 1), None, 2)
