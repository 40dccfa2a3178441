"""GPU (-m gpu): batched analysis of given positions on the device-resident search (include/cattus_b200_analysis.h).

Every position's root visit counts and principal variation must equal a fresh oracle MctsPlayer (noise off) driven by the
same CudaNetwork; best move and visits must equal a fresh ChessSearch.go; and no result may depend on device_games,
the waves in flight, the cache or the other positions of the call.
"""
from __future__ import annotations

import json

import numpy as np
import pytest

from cattus_b200 import _lib
from cattus_b200.analysis import analyse
from oracle import chess as oc
from oracle import mcts as om
from tests.test_analysis_cpu import REPEAT_CHILD, check_against_oracle, chess_history, chess_positions, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, chess_cfg, chess_oracle_fn
from tests.test_selfplay_cpu import cfg_with, oracle_net_fn
from tests.util import make_network

pytestmark = pytest.mark.gpu


def random_playouts(n: int, seed: int, max_plies: int = 40):
    """(None, LAN moves) of n seeded random playouts from the start position, on the library's own rules (fast enough for
    thousands); a playout stops before a finished position."""
    import random

    from cattus_b200 import san as S
    from cattus_b200.selfplay import move_to_lan

    rng = random.Random(seed)
    out = []
    for _ in range(n):
        moves = []
        for _ in range(rng.randrange(0, max_plies + 1)):
            m = rng.choice(S.legal_moves(None, moves))
            info = S.position_info(None, moves + [m])
            if info.status != 0:
                break
            moves.append(m)
        out.append((None, [move_to_lan(m) for m in moves]))
    return out


def _small_game_hist(game, positions):
    hists = []
    for mv in positions:
        p = om.HexPosition.new(5) if game == "hex5" else om.TttPosition.new()
        for m in mv:
            p = p.moved_position(m)
        hists.append([p])
    return hists


@pytest.mark.parametrize("name,game,sim_num", [("hex5", "hex5", 60), ("ttt", "ttt", 40)])
def test_device_analysis_equals_oracle_player_hex_ttt(name, game, sim_num):
    from tests.test_gpu_selfplay import gpu_net_fn

    positions = hex_positions(5, 10, 3) if game == "hex5" else ttt_positions(10, 4)
    with make_network(name, batch_size=64) as nw:
        got = analyse(nw, game, positions, cfg_with(sim_num=sim_num, device_games=4))
        ev = om.Evaluator(oracle_net_fn(gpu_net_fn(nw, 5 if game == "hex5" else 3)), None)
        check_against_oracle(got, _small_game_hist(game, positions), ev, sim_num)


@pytest.mark.parametrize("name,precision,sim_num,count", [("chess_dev", "bf16", 32, 8), ("chess10x128", "bf16", 24, 5), ("chess10x128", "fp8", 24, 5)])
def test_device_analysis_equals_oracle_player_chess(name, precision, sim_num, count):
    """FP8 too: the oracle is driven by the same FP8 handle, so the search must match it exactly."""
    from tests.test_gpu_selfplay import chess_gpu_net

    positions = chess_positions(count, 17)
    with make_network(name, precision=precision, batch_size=64) as nw:
        got = analyse(nw, "chess", positions, chess_cfg(sim_num=sim_num, device_games=3, cache_size=10000))
        ev = om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None)
        check_against_oracle(got, [chess_history(f, m) for f, m in positions], ev, sim_num, oc.move_to_u16)


def test_device_analysis_equals_fresh_uci_search():
    from cattus_b200.selfplay import ChessSearch, move_from_lan

    positions = chess_positions(8, 23) + [(None, REPEAT_CHILD)]
    cfg = chess_cfg(sim_num=100, cache_size=100000, device_games=16)
    with make_network("chess10x128", batch_size=64) as nw:
        got = analyse(nw, "chess", positions, cfg)
        for (fen, moves), a in zip(positions, got):
            with ChessSearch(chess_cfg(sim_num=100, cache_size=100000), model=nw) as search:
                best, stats = search.go(fen, moves)
            assert move_from_lan(best) == a.best_move
            # the UCI search reports the best child's visit share times sim_num, rounded, in f32
            share = np.float32(np.float32(a.best_visits) / np.float32(sum(a.visits)))
            assert stats["best_visits"] == int(share * np.float32(100) + np.float32(0.5))
            assert stats["simulations"] == a.simulations == 100
            assert stats["root_children"] == len(a.moves)


def test_device_analysis_invariance_at_scale():
    """4096 chess positions at sim_num 64: each result bit-identical among all 4096 at device_games 4096 and 64, with 1 or
    3 waves in flight, with the cache on and off, and analysed alone (a sample)."""
    positions = random_playouts(4096, 29, 30)
    base = dict(sim_num=64)
    with make_network("chess_dev", batch_size=4096, n_streams=2) as nw:
        ref = analyse(nw, "chess", positions, chess_cfg(device_games=4096, **base))
        runs = [analyse(nw, "chess", positions, chess_cfg(device_games=64, device_waves_in_flight=3, **base)),
                analyse(nw, "chess", positions, chess_cfg(device_games=4096, device_waves_in_flight=1, cache_size=1 << 20, **base)),
                analyse(nw, "chess", positions, chess_cfg(device_games=1000, device_waves_in_flight=3, cache_size=4096, **base))]
        for r in runs:
            assert r == ref
        rng = np.random.default_rng(3)
        for k in rng.choice(len(positions), 12, replace=False):
            assert analyse(nw, "chess", [positions[k]], chess_cfg(**base)) == [ref[k]]
    assert sum(a.status == 0 for a in ref) > 4000 and all(a.simulations == 64 for a in ref if a.status == 0)


def test_device_analysis_errors():
    with make_network("chess_dev", batch_size=16) as nw:
        with pytest.raises(_lib.CattusB200Error, match="max_batch") as e:
            analyse(nw, "chess", [None] * 64, chess_cfg(sim_num=8, device_games=64))
        assert e.value.code == _lib.ERANGE
        # a tree budget below what sim_num needs is refused before any search (a pool that runs out mid-search is ERANGE,
        # tests/test_analysis_cpu.py)
        with pytest.raises(_lib.CattusB200Error, match="do not fit") as e:
            analyse(nw, "chess", [None], chess_cfg(sim_num=64, device_tree_kwords=4))
        assert e.value.code == _lib.ENOMEM
        with pytest.raises(_lib.CattusB200Error, match="position 1: bad FEN") as e:
            analyse(nw, "chess", [None, "nonsense"], chess_cfg(sim_num=8))
        assert e.value.code == _lib.EINVAL
        with pytest.raises(_lib.CattusB200Error, match="prior_noise_epsilon"):
            analyse(nw, "chess", [None], chess_cfg(sim_num=8, prior_noise_alpha=0.3, prior_noise_epsilon=0.25))
        with pytest.raises(_lib.CattusB200Error, match="another game"):
            analyse(nw, "hex5", [[]], cfg_with(sim_num=8))
        # the handle still works
        assert analyse(nw, "chess", [(KIWIPETE, [])], chess_cfg(sim_num=8))[0].simulations == 8


def test_self_play_before_and_after_an_analysis_plays_the_same_games():
    from cattus_b200.selfplay import SelfPlayRunner

    base = dict(sim_num=24, prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[10, 1.0], [9999, 0.0]], seed=7, max_moves=16,
                device_games=8)
    with make_network("chess_dev", batch_size=64) as nw:
        _, before = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        analyse(nw, "chess", chess_positions(40, 2), chess_cfg(sim_num=30, device_games=16, cache_size=5000))
        _, after = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
    assert [(r.moves, r.winner, r.entries) for r in after] == [(r.moves, r.winner, r.entries) for r in before]


def test_analyse_cli_epd(tmp_path):
    from cattus_b200.analyse import main
    from tests.util import blob

    (tmp_path / "net.cb2").write_bytes(blob("chess_dev"))
    (tmp_path / "cfg.json").write_text(json.dumps({"mcts": {"sim_num": 32, "cache_size": 10000}, "model": {"batch_size": 64}}))
    (tmp_path / "in.epd").write_text(KIWIPETE + ' bm Qxf6; id "kiwi";\n' + '7k/5Q2/6K1/8/8/8/8/8 b - - id "stalemate";\n'
                                     + "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - am e4;\n")
    assert main(["--model-path", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--epd", str(tmp_path / "in.epd"),
                 "--out", str(tmp_path / "out.jsonl")]) == 0
    rows = [json.loads(x) for x in (tmp_path / "out.jsonl").read_text().splitlines()]
    assert [r["id"] for r in rows] == ["kiwi", "stalemate", "line3"]
    assert rows[1]["status"] == "draw" and "best" not in rows[1]
    assert rows[0]["status"] == "searched" and rows[0]["simulations"] == 32 and rows[0]["pv"][0] == rows[0]["best"]
    assert "solved" in rows[0] and "solved" in rows[2]
    (tmp_path / "in.fen").write_text("startpos moves e2e4\n" + KIWIPETE + " moves e1g1\n")
    assert main(["--model-path", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--fen-file", str(tmp_path / "in.fen"),
                 "--precision", "bf16", "--out", str(tmp_path / "out2.jsonl")]) == 0
    rows = [json.loads(x) for x in (tmp_path / "out2.jsonl").read_text().splitlines()]
    assert len(rows) == 2 and rows[0]["moves"] == ["e2e4"] and rows[1]["san"]
