"""CPU tests of persistent device search sessions (DESIGN.md section 17).

The session's begin, minibatch kernels and host driver (dsearch_session.hpp, thread included) run on the host with a
one-lane warp (tests/emul/session_emul.cpp) and must equal tests/session_oracle.py -- one BatchedPlayer kept across
searches -- exactly: children, visits, W bits, best move, PV, minibatches, collisions, new simulations, kept visits.
"""
from __future__ import annotations

import io
import threading
import time

import numpy as np
import pytest

from cattus_b200 import _lib
from cattus_b200.uci import UCI, time_budget_ms
from oracle import chess as oc
from oracle import mcts as om
from tests import session_oracle as so
from tests.emul import search_batch_emul as se
from tests.emul import session_emul as sx
from tests.test_analysis_cpu import chess_history
from tests.test_chess_cpu import KIWIPETE, chess_cb, chess_cfg, chess_fake_net, chess_oracle_fn
from tests.test_search_batch_cpu import small_history
from tests.test_selfplay_cpu import cb_for, cfg_with, fake_net, oracle_net_fn


def bits(xs):
    return np.asarray(xs, dtype=np.float32).view(np.uint32).tolist()


def setup(game):
    if game == "chess":
        net = chess_fake_net("hash")
        return net, om.Evaluator(chess_oracle_fn(net), None), chess_cb(net), chess_cfg(sim_num=64), oc.move_to_u16, chess_history
    net = fake_net("hash")
    return net, om.Evaluator(oracle_net_fn(net), None), cb_for(net, 1), cfg_with(sim_num=64), (lambda m: m), (lambda f, m: small_history(game, m))


def same(r, o, to_move):
    a = r.analysis
    assert a.moves == [to_move(m) for m in o["moves"]]
    assert a.visits == o["visits"]
    assert bits(a.w) == bits(o["w"])
    assert a.best_move == to_move(o["best"])
    assert a.pv == [to_move(m) for m in o["pv"]]
    assert (a.minibatches, a.collisions, a.simulations, r.reused_visits) == (o["minibatches"], o["collisions"], o["simulations"], o["reused"])


# a line of play per game: each search extends the previous position by 0, 1 or 2 plies (reuse), or by 3 or jumps (fresh)
LINES = {
    "hex5": [[], [12], [12, 7], [12, 7], [12, 7, 13, 6], [12, 7, 13, 6, 11, 8, 2], [3], [3, 9]],
    "ttt": [[], [4], [4, 0], [4, 0, 8, 2], [4, 0, 8, 2, 1, 7], [1], [1, 4, 0]],
    "chess": [(None, []), (None, ["e2e4"]), (None, ["e2e4", "e7e5"]), (None, ["e2e4", "e7e5", "g1f3", "b8c6"]),
              (None, ["e2e4", "e7e5", "g1f3", "b8c6"]), (None, ["e2e4", "e7e5", "g1f3", "b8c6", "f1b5", "a7a6", "b5a4"]), (KIWIPETE, []),
              (KIWIPETE, ["e1g1"])],
}


def fen_moves(game, pos):
    return pos if game == "chess" else (None, pos)


@pytest.mark.parametrize("L", [2, 7, 32])
@pytest.mark.parametrize("game", ["hex5", "ttt", "chess"])
def test_fresh_go_equals_analyse(game, L):
    net, ev, cb, cfg, to_move, hist = setup(game)
    pos = LINES[game][2]
    with sx.create(game, cfg, cb, L, tree_kwords=512) as s:
        s.set_position(*fen_moves(game, pos))
        r = s.search(nodes=64)
    ref = se.analyse(game, [fen_moves(game, pos)], dict(cfg, device_games=1), cb, search_batch=L)[0]
    assert r.stop_reason == "nodes" and r.reused_visits == 0
    assert r.analysis == ref


@pytest.mark.parametrize("L", [3, 16])
@pytest.mark.parametrize("game", ["hex5", "ttt", "chess"])
def test_sequence_with_reuse_equals_oracle(game, L):
    net, ev, cb, cfg, to_move, hist = setup(game)
    player = so.SessionPlayer(ev, L)
    reused = 0
    with sx.create(game, cfg, cb, L, tree_kwords=512) as s:
        for k, pos in enumerate(LINES[game]):
            fen, moves = fen_moves(game, pos)
            nodes = [40, 64, 23, None][k % 4]
            cap = 6 if nodes is None else None
            s.set_position(fen, moves)
            r = s.search(nodes=nodes, minibatches=cap)
            o = player.search(hist(fen, moves), nodes, cap)
            same(r, o, to_move)
            reused += r.reused_visits
    assert reused > 0


@pytest.mark.parametrize("game", ["hex5", "chess"])
def test_minibatch_cap_and_stop_after_wave_replay(game):
    net, ev, cb, cfg, to_move, hist = setup(game)
    fen, moves = fen_moves(game, LINES[game][1])
    with sx.create(game, cfg, cb, 8, tree_kwords=512) as s:
        s.set_position(fen, moves)
        r = s.search(minibatches=5)
    assert r.stop_reason == "minibatches" and r.analysis.minibatches == 5
    same(r, so.SessionPlayer(ev, 8).search(hist(fen, moves), None, 5), to_move)
    for after in (1, 4):
        with sx.create(game, cfg, cb, 8, tree_kwords=512, stop_after_waves=after, depth=1) as s:
            s.set_position(fen, moves)
            r = s.search()
        # the word is written after wave `after`'s boundary, so the next minibatch's boundary sees it
        assert r.stop_reason == "stop" and r.analysis.minibatches == after + 1
        same(r, so.SessionPlayer(ev, 8).search(hist(fen, moves), None, r.analysis.minibatches), to_move)


def test_capacity_stop_is_replayable():
    net, ev, cb, cfg, to_move, hist = setup("hex5")
    with sx.create("hex5", cfg, cb, 8, tree_kwords=4) as s:
        s.set_position(None, [])
        r = s.search()
        assert r.stop_reason == "capacity" and r.analysis.minibatches > 1
        same(r, so.SessionPlayer(ev, 8).search(hist(None, []), None, r.analysis.minibatches), to_move)
        s.set_position(None, [])  # the same root: the full tree gives way to a fresh one
        r2 = s.search(nodes=30)
        assert r2.reused_visits == 0
        same(r2, so.SessionPlayer(ev, 8).search(hist(None, []), 30), to_move)


@pytest.mark.parametrize("depth,cache", [(1, 0), (3, 0), (3, 5000), (1, 64)])
def test_waves_in_flight_and_cache_change_nothing(depth, cache):
    net, ev, cb, cfg, to_move, hist = setup("chess")
    out = []
    for d, c in ((2, 0), (depth, cache)):
        with sx.create("chess", dict(cfg, mcts=dict(cfg["mcts"], cache_size=c)), cb, 16, tree_kwords=512, depth=d) as s:
            got = []
            for pos in LINES["chess"][:5]:
                s.set_position(*pos)
                got.append(s.search(nodes=50))
            out.append([(g.analysis, g.reused_visits, g.stop_reason) for g in got])
    assert out[0] == out[1]


def test_info_snapshots_are_monotone_and_the_last_is_the_result():
    net, ev, cb, cfg, to_move, hist = setup("hex5")
    snaps = []
    with sx.create("hex5", cfg, cb, 4, tree_kwords=512) as s:
        s.set_position(None, [12])
        s.go(nodes=3000, on_info=snaps.append, info_interval_ms=1)
        r = s.wait()
        last = s.info()
    assert [x.simulations for x in snaps] == sorted(x.simulations for x in snaps)
    assert not last.searching and last.valid
    assert (last.simulations, last.minibatches, last.collisions, last.best_move, last.pv) == (
        r.analysis.simulations, r.analysis.minibatches, r.analysis.collisions, r.analysis.best_move, r.analysis.pv)


def test_explicit_stop_from_another_thread():
    net, ev, cb, cfg, to_move, hist = setup("hex5")
    with sx.create("hex5", cfg, cb, 4, tree_kwords=2048) as s:
        s.set_position(None, [])
        s.go()
        time.sleep(0.05)
        threading.Thread(target=s.stop).start()
        r = s.wait(timeout=60)
    assert r is not None and r.stop_reason == "stop" and r.analysis.minibatches >= 1
    same(r, so.SessionPlayer(ev, 4).search(hist(None, []), None, r.analysis.minibatches), to_move)


def test_errors():
    net, ev, cb, cfg, to_move, hist = setup("chess")
    with pytest.raises(_lib.CattusB200Error, match="search_batch") as e:
        sx.create("chess", cfg, cb, 1)
    assert e.value.code == _lib.EINVAL
    with pytest.raises(_lib.CattusB200Error, match="struct_size"):
        sx.create("chess", cfg, cb, 4, opts_size=8)
    with pytest.raises(_lib.CattusB200Error, match="max_batch"):
        sx.create("chess", cfg, cb, 512, max_batch=256)
    with pytest.raises(_lib.CattusB200Error, match="tree_kwords"):
        sx.create("chess", cfg, cb, 64, tree_kwords=8)
    with sx.create("chess", cfg, cb, 4, tree_kwords=512) as s:
        with pytest.raises(_lib.CattusB200Error, match="before set_position"):
            s.go(nodes=10)
        with pytest.raises(_lib.CattusB200Error, match="bad FEN") as e:
            s.set_position("not a fen", [])
        assert e.value.code == _lib.EINVAL
        with pytest.raises(_lib.CattusB200Error, match="move 1 is not legal"):
            s.set_position(None, ["e2e4", "e2e4"])
        s.set_position(None, ["e2e4"])
        s.go()
        with pytest.raises(_lib.CattusB200Error, match="go while a search runs"):
            s.go(nodes=5)
        s.stop()
        assert s.wait().stop_reason == "stop"
    h = sx.create("ttt", cfg_with(sim_num=8), cb_for(fake_net("hash"), 1), 4, tree_kwords=64)
    lim = _lib.SessionLimits(4, 10, 0, 0, 0)
    assert sx.load().session_emul_go(h._h, lim) == _lib.EINVAL
    h.set_position(None, [0, 3, 1, 4, 2])  # finished: no search
    r = h.search(nodes=10)
    assert r.analysis.status == 1 and r.stop_reason == "finished"
    h.close()


def test_time_budget():
    assert time_budget_ms(60000, 1000, None, 30) == min(30000, 60000 / 30 + 750) - 30
    assert time_budget_ms(1000, 0, 1, 30) == 500 - 30
    assert time_budget_ms(20, 0, None, 30) == 0
    assert time_budget_ms(10000, 5000, 5, 0) == min(5000, 2000 + 3750)


# ------------------------------------------------------------------------------------------------------------ UCI
class Lines(io.StringIO):
    def lines(self):
        return self.getvalue().splitlines()


def wait_for(out, word, timeout=60.0):
    t = time.time()
    while time.time() - t < timeout:
        if any(line.startswith(word) for line in out.lines()):
            return
        time.sleep(0.01)
    raise AssertionError(f"no {word!r} in {out.lines()}")


def uci_session():
    net = chess_fake_net("hash")
    cfg = {"mcts": {"sim_num": 64, "explore_factor": 1.41421}, "search_batch": 8, "device_session": True, "info_interval_ms": 20}
    out = Lines()
    u = UCI(cfg, out=out, session_factory=lambda c, L: sx.create("chess", c, chess_cb(net), L, tree_kwords=2048))
    return u, out


def test_uci_session_go_nodes_and_clock():
    u, out = uci_session()
    u.handle("uci")
    u.handle("position startpos moves e2e4")
    u.handle("go nodes 100")
    wait_for(out, "bestmove")
    u.handle("position startpos moves e2e4 e7e5")
    u.handle("go wtime 60000 btime 60000 winc 1000 binc 1000")
    u.handle("isready")
    assert "readyok" in out.lines()
    while sum(line.startswith("bestmove") for line in out.lines()) < 2:
        time.sleep(0.01)
    u.close()
    infos = [line for line in out.lines() if line.startswith("info depth")]
    assert infos and all(" nodes " in line and " pv " in line for line in infos)
    best = [line.split() for line in out.lines() if line.startswith("bestmove")]
    assert all(len(b) == 4 and b[2] == "ponder" for b in best)


def test_uci_session_infinite_stop_and_ponder():
    u, out = uci_session()
    u.handle("position startpos")
    u.handle("go infinite")
    time.sleep(0.1)
    u.handle("isready")
    assert "readyok" in out.lines() and not any(line.startswith("bestmove") for line in out.lines())
    u.handle("stop")
    wait_for(out, "bestmove")
    n = len(out.lines())
    u.handle("position startpos moves d2d4 d7d5")
    u.handle("go ponder wtime 2000 btime 2000")
    time.sleep(0.1)
    assert not any(line.startswith("bestmove") for line in out.lines()[n:])
    u.handle("ponderhit")
    t = time.time()
    while not any(line.startswith("bestmove") for line in out.lines()[n:]):
        time.sleep(0.01)
        assert time.time() - t < 60
    u.handle("quit")
    u.close()


def test_a_failed_search_leaves_the_session_usable():
    # an evaluator batch smaller than a minibatch's new leaves: the device reports kErrRows (ERANGE) mid-search; the next
    # search clears the error word and the virtual counts and starts from a fresh root
    net, ev, cb, cfg, to_move, hist = setup("chess")
    lib = sx.load()
    with sx.create("chess", cfg, cb, 16, tree_kwords=512) as s:
        s.set_position(None, ["e2e4"])
        lib.session_emul_set_max_rows(s._h, 2)
        with pytest.raises(_lib.CattusB200Error) as e:
            s.search(nodes=200)
        assert e.value.code == _lib.ERANGE
        lib.session_emul_set_max_rows(s._h, 16)
        player = so.SessionPlayer(ev, 16)
        for pos in ((None, ["e2e4"]), (None, ["e2e4", "e7e5"])):
            s.set_position(*pos)
            same(s.search(nodes=100), player.search(hist(*pos), 100), to_move)


def test_uci_ponderhit_starts_the_clock_at_once():
    # the info interval is long: the budget, not the next info line, decides when bestmove comes
    net = chess_fake_net("hash")
    cfg = {"mcts": {"sim_num": 64, "explore_factor": 1.41421}, "search_batch": 8, "device_session": True, "info_interval_ms": 5000}
    out = Lines()
    u = UCI(cfg, out=out, session_factory=lambda c, L: sx.create("chess", c, chess_cb(net), L, tree_kwords=2048))
    u.handle("position startpos moves e2e4")
    u.handle("go ponder wtime 3000 btime 3000")  # black to move: budget min(1500, 100) - 30 = 70 ms
    time.sleep(0.2)
    t0 = time.monotonic()
    u.handle("ponderhit")
    wait_for(out, "bestmove")
    took = (time.monotonic() - t0) * 1000.0
    u.close()
    assert u.last_stats["stop_reason"] == "stop"
    assert took < 70 + 400, took


def test_uci_failed_search_still_answers_bestmove():
    net = chess_fake_net("hash")
    cfg = {"mcts": {"sim_num": 64, "explore_factor": 1.41421}, "search_batch": 16, "device_session": True, "info_interval_ms": 20}
    out = Lines()
    u = UCI(cfg, out=out, session_factory=lambda c, L: sx.create("chess", c, chess_cb(net), L, tree_kwords=2048))
    u.handle("position startpos")
    u.handle("go nodes 1")
    wait_for(out, "bestmove")
    sx.load().session_emul_set_max_rows(u.session._h, 2)
    u.handle("position startpos moves d2d4")
    u.handle("go nodes 500")
    while sum(line.startswith("bestmove") for line in out.lines()) < 2:
        time.sleep(0.01)
    assert out.lines()[-1] == "bestmove 0000"
    sx.load().session_emul_set_max_rows(u.session._h, 16)
    u.handle("go nodes 100")
    while sum(line.startswith("bestmove") for line in out.lines()) < 3:
        time.sleep(0.01)
    u.close()
    assert out.lines()[-1] != "bestmove 0000"
