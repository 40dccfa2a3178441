"""GPU (-m gpu): persistent device search sessions (DESIGN.md section 17).

A session's searches must equal tests/session_oracle.py driven by the same CudaNetwork, bit for bit, across a line of
play with tree reuse; a stopped search must replay at its reported minibatch count; movetime must end near its
deadline; snapshots must be monotone and end at the result; an open session must leave the handle's self-play and
analysis results unchanged; and the UCI CLI must run in session mode end to end.
"""
from __future__ import annotations

import json
import subprocess
import sys
import time

import pytest

from cattus_b200.analysis import analyse
from cattus_b200.session import DeviceSearch
from oracle import chess as oc
from oracle import mcts as om
from tests import session_oracle as so
from tests.test_analysis_cpu import chess_history
from tests.test_chess_cpu import chess_cfg, chess_oracle_fn
from tests.test_search_batch_cpu import small_history
from tests.test_session_cpu import LINES, fen_moves, same
from tests.test_selfplay_cpu import cfg_with, oracle_net_fn
from tests.util import make_network

pytestmark = pytest.mark.gpu


def run_line(nw, game, ev, to_move, hist, L, positions, cfg):
    player = so.SessionPlayer(ev, L)
    reused = 0
    with DeviceSearch(nw, game, cfg, L, tree_kwords=8192) as s:
        for k, pos in enumerate(positions):
            fen, moves = fen_moves(game, pos)
            nodes = [300, 500, 123, None][k % 4]
            cap = 7 if nodes is None else None
            s.set_position(fen, moves)
            r = s.search(nodes=nodes, minibatches=cap)
            same(r, player.search(hist(fen, moves), nodes, cap), to_move)
            reused += r.reused_visits
    assert reused > 0


def test_session_equals_oracle_hex5():
    from tests.test_gpu_selfplay import gpu_net_fn

    with make_network("hex5", batch_size=64) as nw:
        ev = om.Evaluator(oracle_net_fn(gpu_net_fn(nw, 5)), None)
        run_line(nw, "hex5", ev, lambda m: m, lambda f, m: small_history("hex5", m), 16, LINES["hex5"], cfg_with(sim_num=64))


@pytest.mark.parametrize("name,precision", [("chess_dev", "bf16"), ("chess10x128", "bf16"), ("chess10x128", "fp8")])
def test_session_equals_oracle_chess(name, precision):
    from tests.test_gpu_selfplay import chess_gpu_net

    with make_network(name, precision=precision, batch_size=256) as nw:
        ev = om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None)
        run_line(nw, "chess", ev, oc.move_to_u16, chess_history, 64, LINES["chess"], chess_cfg(sim_num=64, cache_size=20000))


def test_fresh_session_equals_analyse_and_stopped_search_replays():
    pos = (None, ["e2e4", "c7c5"])
    with make_network("chess10x128", batch_size=256) as nw:
        ref = analyse(nw, "chess", [pos], chess_cfg(sim_num=3000), search_batch=256)[0]
        with DeviceSearch(nw, "chess", chess_cfg(), 256) as s:
            s.set_position(*pos)
            r = s.search(nodes=3000)
            a = r.analysis
            assert r.stop_reason == "nodes" and a == ref
            s.new_game()
            s.go()
            time.sleep(0.3)
            s.stop()
            r = s.wait(timeout=120)
            assert r.stop_reason == "stop" and r.reused_visits == 0 and r.analysis.minibatches >= 1
            s.new_game()
            r2 = s.search(minibatches=r.analysis.minibatches)
            assert r2.stop_reason == "minibatches" and r2.analysis == r.analysis


def test_movetime_and_snapshots():
    with make_network("chess10x128", batch_size=256) as nw:
        with DeviceSearch(nw, "chess", chess_cfg(), 256) as s:
            s.set_position(None, ["d2d4"])
            s.search(nodes=2000)  # warm-up
            s.new_game()
            snaps = []
            t0 = time.perf_counter()
            s.go(movetime_ms=200, on_info=snaps.append, info_interval_ms=10)
            r = s.wait(timeout=60)
            wall = (time.perf_counter() - t0) * 1000.0
            last = s.info()
    per_mb = r.seconds * 1000.0 / r.analysis.minibatches
    print(f"movetime 200 ms: search {r.seconds * 1000:.1f} ms (wall {wall:.1f} ms), {r.analysis.minibatches} minibatches of "
          f"{per_mb:.2f} ms, overrun {r.seconds * 1000 - 200:.1f} ms")
    assert r.stop_reason == "deadline"
    assert r.seconds * 1000.0 <= 200 + 3 * per_mb + 50
    assert snaps and [x.simulations for x in snaps] == sorted(x.simulations for x in snaps)
    assert [x.minibatches for x in snaps] == sorted(x.minibatches for x in snaps)
    assert (last.simulations, last.minibatches, last.best_move, last.pv) == (r.analysis.simulations, r.analysis.minibatches, r.analysis.best_move,
                                                                             r.analysis.pv)


def test_open_session_leaves_selfplay_and_analysis_unchanged():
    from cattus_b200.selfplay import SelfPlayRunner
    from tests.test_analysis_cpu import chess_positions

    base = dict(sim_num=24, prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[10, 1.0], [9999, 0.0]], seed=7, max_moves=16,
                device_games=8)
    positions = chess_positions(8, 4)
    with make_network("chess_dev", batch_size=512, n_streams=2) as nw:
        _, before = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        a_before = analyse(nw, "chess", positions, chess_cfg(sim_num=200, device_games=4), search_batch=16)
        with DeviceSearch(nw, "chess", chess_cfg(), 64) as s:
            s.set_position(None, ["e2e4"])
            s.go()
            _, after = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
            a_after = analyse(nw, "chess", positions, chess_cfg(sim_num=200, device_games=4), search_batch=16)
            s.stop()
            assert s.wait(timeout=120).stop_reason in ("stop", "capacity")
    assert [(r.moves, r.winner, r.entries) for r in after] == [(r.moves, r.winner, r.entries) for r in before]
    assert a_after == a_before


def test_one_stream_model_is_einval():
    from cattus_b200._lib import EINVAL, CattusB200Error

    with make_network("chess_dev", batch_size=64, n_streams=1) as nw:
        with pytest.raises(CattusB200Error, match="n_streams") as e:
            DeviceSearch(nw, "chess", chess_cfg(), 16)
        assert e.value.code == EINVAL


SCRIPT = ["uci", "isready", "ucinewgame", "position startpos moves e2e4 e7e5", "go wtime 60000 btime 60000 winc 1000 binc 1000",
          "position startpos moves e2e4 e7e5 g1f3 b8c6", "go infinite", "isready", "stop", "position startpos moves e2e4 e7e5 g1f3 b8c6 f1b5",
          "go ponder wtime 3000 btime 3000", "ponderhit", "isready"]


def test_uci_cli_session_mode(tmp_path):
    from tests.util import blob

    (tmp_path / "net.cb2").write_bytes(blob("chess10x128"))
    cfg = {"model": {"model_path": str(tmp_path / "net.cb2"), "batch_size": 256}, "mcts": {"sim_num": 1000, "explore_factor": 1.41421},
           "search_batch": 256, "device_session": True, "info_interval_ms": 100}
    (tmp_path / "cfg.json").write_text(json.dumps(cfg))
    p = subprocess.Popen([sys.executable, "-m", "cattus_b200.uci", "--config-file", str(tmp_path / "cfg.json")], stdin=subprocess.PIPE,
                         stdout=subprocess.PIPE, text=True)
    lines = []

    def until(word):
        while True:
            line = p.stdout.readline()
            assert line, lines
            lines.append(line.strip())
            if line.startswith(word):
                return line

    def send(cmd):
        p.stdin.write(cmd + "\n")
        p.stdin.flush()

    for cmd in SCRIPT[:5]:
        send(cmd)
    until("bestmove")
    send(SCRIPT[5])
    send(SCRIPT[6])
    time.sleep(0.5)
    send(SCRIPT[7])
    until("readyok")
    assert sum(x.startswith("bestmove") for x in lines) == 1  # go infinite holds its bestmove until stop
    send(SCRIPT[8])
    until("bestmove")
    send(SCRIPT[9])
    send(SCRIPT[10])
    time.sleep(0.3)
    send(SCRIPT[11])
    until("bestmove")
    send("quit")
    p.stdin.close()
    assert p.wait(timeout=120) == 0
    best = [x.split() for x in lines if x.startswith("bestmove")]
    assert len(best) == 3 and all(b[1] != "0000" and len(b) == 4 and b[2] == "ponder" for b in best)
    assert any(x.startswith("info depth") and " nodes " in x and " score cp " in x for x in lines)
    for b, hist in zip(best, ([["e2e4", "e7e5"]], [["e2e4", "e7e5", "g1f3", "b8c6"]], [["e2e4", "e7e5", "g1f3", "b8c6", "f1b5"]])):
        h = chess_history(None, hist[0])
        assert b[1] in [oc.move_to_lan(m) for m in h[-1].legal_moves()]
