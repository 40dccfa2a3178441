"""GPU (-m gpu): minibatched search under virtual loss on the device (DESIGN.md section 15).

Every result must equal tests/batch_oracle.py driven by the same CudaNetwork, bit for bit (children, visits, W, best
move, PV, minibatches, collisions); no result may depend on device_games, the waves in flight, the cache or the other
positions; a batched analysis must leave self-play and one-leaf analyses on the same handle unchanged; and the UCI
front end and the CLI run the mode end to end.
"""
from __future__ import annotations

import io
import json

import numpy as np
import pytest

from cattus_b200.analysis import analyse
from oracle import chess as oc
from oracle import mcts as om
from tests.test_analysis_cpu import REPEAT_CHILD, chess_history, chess_positions, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, chess_cfg, chess_oracle_fn
from tests.test_gpu_analysis import random_playouts
from tests.test_search_batch_cpu import FOOLS, check, small_history
from tests.test_selfplay_cpu import cfg_with, oracle_net_fn
from tests.util import make_network

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("L", [16, 256])
@pytest.mark.parametrize("name,game", [("hex5", "hex5"), ("ttt", "ttt")])
def test_device_minibatches_equal_oracle_hex_ttt(name, game, L):
    from tests.test_gpu_selfplay import gpu_net_fn

    positions = hex_positions(5, 6, 3) if game == "hex5" else ttt_positions(6, 4)
    with make_network(name, batch_size=3 * L) as nw:
        got = analyse(nw, game, positions, cfg_with(sim_num=300, device_games=3), search_batch=L)
        ev = om.Evaluator(oracle_net_fn(gpu_net_fn(nw, 5 if game == "hex5" else 3)), None)
        check(got, [small_history(game, m) for m in positions], ev, 300, L)


@pytest.mark.parametrize("L", [16, 256])
@pytest.mark.parametrize("name,precision", [("chess_dev", "bf16"), ("chess10x128", "bf16"), ("chess10x128", "fp8")])
def test_device_minibatches_equal_oracle_chess(name, precision, L):
    from tests.test_gpu_selfplay import chess_gpu_net

    positions = [FOOLS, (None, REPEAT_CHILD), (KIWIPETE, [])] + chess_positions(4, 17)[2:]
    with make_network(name, precision=precision, batch_size=4 * L) as nw:
        got = analyse(nw, "chess", positions, chess_cfg(sim_num=301, device_games=4, cache_size=10000), search_batch=L)
        ev = om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None)
        check(got, [chess_history(f, m) for f, m in positions], ev, 301, L, oc.move_to_u16)


def test_device_minibatches_deep_tree_equals_oracle():
    """One chess position at sim_num 4000 with L = 256: a deep tree with many collisions."""
    from tests.test_gpu_selfplay import chess_gpu_net

    pos = (None, ["e2e4", "e7e5", "g1f3"])
    with make_network("chess10x128", batch_size=256) as nw:
        got = analyse(nw, "chess", [pos], chess_cfg(sim_num=4000, cache_size=100000), search_batch=256)
        check(got, [chess_history(*pos)], om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None), 4000, 256, oc.move_to_u16)
    assert got[0].collisions > 100 and got[0].minibatches < 4000 // 100


def test_device_minibatches_invariance():
    """256 chess positions at L = 16: identical at device_games 256 / 100 / 7, 1 or 3 waves in flight, cache on and off,
    and analysed alone (a sample)."""
    positions = random_playouts(256, 31, 30)
    base = dict(sim_num=200)
    with make_network("chess_dev", batch_size=4096) as nw:
        ref = analyse(nw, "chess", positions, chess_cfg(device_games=256, **base), search_batch=16)
        runs = [analyse(nw, "chess", positions, chess_cfg(device_games=100, device_waves_in_flight=3, **base), search_batch=16),
                analyse(nw, "chess", positions, chess_cfg(device_games=7, device_waves_in_flight=1, cache_size=1 << 16, **base), search_batch=16),
                analyse(nw, "chess", positions, chess_cfg(device_games=256, device_waves_in_flight=3, cache_size=4096, **base), search_batch=16)]
        for r in runs:
            assert r == ref
        rng = np.random.default_rng(5)
        for k in rng.choice(len(positions), 6, replace=False):
            assert analyse(nw, "chess", [positions[k]], chess_cfg(**base), search_batch=16) == [ref[k]]
    assert sum(a.status == 0 for a in ref) > 240 and all(a.minibatches >= 200 // 16 for a in ref if a.status == 0)


def test_self_play_and_one_leaf_analysis_unchanged_by_a_batched_analysis():
    from cattus_b200.selfplay import SelfPlayRunner

    base = dict(sim_num=24, prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[10, 1.0], [9999, 0.0]], seed=7, max_moves=16,
                device_games=8)
    positions = chess_positions(12, 4)
    with make_network("chess_dev", batch_size=512) as nw:
        _, before = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        one_before = analyse(nw, "chess", positions, chess_cfg(sim_num=40, device_games=4))
        analyse(nw, "chess", positions, chess_cfg(sim_num=300, device_games=2, cache_size=5000), search_batch=256)
        _, after = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        one_after = analyse(nw, "chess", positions, chess_cfg(sim_num=40, device_games=4))
    assert [(r.moves, r.winner, r.entries) for r in after] == [(r.moves, r.winner, r.entries) for r in before]
    assert one_after == one_before


def test_uci_search_batch_bestmove_equals_the_analysis():
    from cattus_b200.selfplay import move_to_lan
    from cattus_b200.uci import UCI, q_to_cp

    moves = ["e2e4", "c7c5", "g1f3"]
    cfg = {"mcts": {"sim_num": 2000, "explore_factor": 1.41421, "cache_size": 0}, "search_batch": 256}
    with make_network("chess10x128", batch_size=256) as nw:
        a = analyse(nw, "chess", [(None, moves)], chess_cfg(sim_num=2000), search_batch=256)[0]
        out = io.StringIO()
        uci = UCI(cfg, model=nw, out=out)
        for line in ("uci", "isready", "ucinewgame", "position startpos moves " + " ".join(moves), "go wtime 1000"):
            uci.handle(line)
    lines = out.getvalue().splitlines()
    info = next(x for x in lines if x.startswith("info depth"))
    assert lines[-1] == f"bestmove {move_to_lan(a.best_move)}"
    w = info.split()
    assert w[w.index("depth") + 1] == str(len(a.pv)) and w[w.index("nodes") + 1] == "2000" and int(w[w.index("nps") + 1]) > 0
    assert w[w.index("cp") + 1] == str(q_to_cp(a.q)) and w[w.index("pv") + 1:] == [move_to_lan(m) for m in a.pv]
    assert uci.last_stats["minibatches"] == a.minibatches


def test_analyse_cli_search_batch(tmp_path):
    from cattus_b200.analyse import main
    from tests.util import blob

    (tmp_path / "net.cb2").write_bytes(blob("chess_dev"))
    (tmp_path / "cfg.json").write_text(json.dumps({"mcts": {"sim_num": 500}, "model": {"batch_size": 64}}))
    (tmp_path / "in.fen").write_text("startpos moves e2e4\n" + KIWIPETE + "\n")
    assert main(["--model-path", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--fen-file", str(tmp_path / "in.fen"),
                 "--search-batch", "64", "--out", str(tmp_path / "out.jsonl")]) == 0
    rows = [json.loads(x) for x in (tmp_path / "out.jsonl").read_text().splitlines()]
    assert len(rows) == 2 and all(r["simulations"] == 500 and r["minibatches"] >= 500 // 64 and r["collisions"] >= 0 for r in rows)
