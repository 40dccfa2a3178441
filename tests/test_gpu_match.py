"""GPU (-m gpu): match play from openings on the device-resident search (include/cattus_b200_match.h).

From the initial position a match must play the games of the real device self-play of (A, B); from real openings every
game must equal oracle/mcts.py's play_game driven by the same CudaNetworks; and no game may depend on device_games, the
waves in flight, the cache or whether both sides share one handle.
"""
from __future__ import annotations

import json
import re

import pytest

from cattus_b200 import _lib
from cattus_b200.match import play
from oracle import chess as oc
from oracle import mcts as om
from tests.test_analysis_cpu import chess_history, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, _params, chess_cfg, chess_oracle_fn
from tests.test_gpu_analysis import random_playouts
from tests.test_match_cpu import FINISHED, FORCED, NOISY, SHUFFLE, check_against_oracle, play_from, small_history
from tests.test_selfplay_cpu import cfg_with, oracle_net_fn
from tests.util import blob, make_network

pytestmark = pytest.mark.gpu


def network(name: str, seed: int, precision: str = "bf16", batch_size: int = 64):
    from cattus_b200 import CudaNetwork
    from oracle import net

    return CudaNetwork(blob(name, seed), net.CONFIGS[name].game, batch_size=batch_size, n_streams=2, precision=precision)


@pytest.mark.parametrize("name,game,sim_num,pairs", [("hex5", "hex5", 40, 6), ("chess_dev", "chess", 24, 4)])
def test_initial_position_match_equals_device_self_play(name, game, sim_num, pairs):
    from cattus_b200.selfplay import SelfPlayRunner

    mk = chess_cfg if game == "chess" else cfg_with
    cfg = mk(sim_num=sim_num, seed=11, max_moves=30 if game == "chess" else 0, cache_size=10000, device_games=5, **NOISY)
    with network(name, 0) as a, network(name, 1) as b:
        summary, recs = SelfPlayRunner(game, cfg).generate_data(a, b, 2 * pairs, keep_records=True)
        got = play(a, b, game, [None] * pairs, cfg)
    assert [(g.opening * 2 + (0 if g.a_is_player1 else 1), g.moves, g.winner) for g in got.games] == [(r.game_idx, r.moves, r.winner) for r in recs]
    assert (got.a_wins, got.b_wins, got.draws) == (summary["player1_wins"], summary["player2_wins"], summary["draws"])
    assert got.simulations == summary["metrics"]["selfplay.simulations"]


def _oracle(game, hists, cfg, net_a, net_b, sim_num_b):
    from tests.test_gpu_selfplay import chess_gpu_net, gpu_net_fn

    if game == "chess":
        params_a = _params(cfg)
        ea, eb = (om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None) for nw in (net_a, net_b))
    else:
        mc = cfg["mcts"]
        params_a = om.MctsParams(mc["sim_num"], mc["explore_factor"], om.TemperaturePolicy.from_config(mc["temperature_policy"]),
                                 mc["prior_noise_alpha"], mc["prior_noise_epsilon"])
        s = 5 if game == "hex5" else 3
        ea, eb = (om.Evaluator(oracle_net_fn(gpu_net_fn(nw, s)), None) for nw in (net_a, net_b))
    params_b = om.MctsParams(**dict(params_a.__dict__, sim_num=sim_num_b))
    out = {}
    for k, h in enumerate(hists):
        if h is not None:
            for c in (0, 1):
                out[(k, c == 0)] = play_from(2 * k + c, h, params_a, params_b, ea, eb, cfg["seed"], cfg.get("max_moves", 0))
    return out


@pytest.mark.parametrize("name,game,precision", [("hex5", "hex5", "bf16"), ("ttt", "ttt", "bf16"), ("chess_dev", "chess", "bf16"),
                                                 ("chess10x128", "chess", "bf16"), ("chess10x128", "chess", "fp8")])
def test_device_match_equals_oracle_play_game(name, game, precision):
    """Two networks, a different sim_num for B, noise and temperature on.  FP8 too: the oracle is driven by the same handles."""
    if game == "chess":
        openings = [FORCED, (KIWIPETE, ["e1g1"]), FINISHED[0], SHUFFLE] + random_playouts(2, 5, 20)
        cfg = chess_cfg(sim_num=12, seed=3, max_moves=8, device_games=4, **NOISY)
    else:
        openings = hex_positions(5, 3, 7) if game == "hex5" else ttt_positions(3, 8)
        cfg = cfg_with(sim_num=20, seed=3, device_games=4, **NOISY)
    sim_b = cfg["mcts"]["sim_num"] + 6
    with network(name, 0, precision) as a, network(name, 1, precision) as b:
        got = play(a, b, game, openings, cfg, sim_num_b=sim_b)
        hists = [None if st else (chess_history(*o) if game == "chess" else small_history(game, o)) for o, st in zip(openings, got.opening_status)]
        ref = _oracle(game, hists, cfg, a, b, sim_b)
    check_against_oracle(got, ref, oc.move_to_u16 if game == "chess" else (lambda m: m))
    if game == "chess":
        assert got.opening_status[2] == 2 and got.games[0].termination == "repetition"


def test_device_match_invariance_at_scale():
    """300 chess openings x 2 games: identical at device_games 512 / 100 / 16, with 1 and 3 waves in flight, with the cache
    on and off, and with one handle on both sides or two handles of one blob."""
    openings = random_playouts(300, 41, 16)
    base = dict(sim_num=32, seed=9, max_moves=20, **NOISY)
    with make_network("chess_dev", batch_size=512, n_streams=2) as nw, make_network("chess_dev", batch_size=512, n_streams=2) as nw2:
        ref = play(nw, None, "chess", openings, chess_cfg(device_games=512, **base))
        runs = [play(nw, None, "chess", openings, chess_cfg(device_games=100, device_waves_in_flight=3, cache_size=1 << 16, **base)),
                play(nw, None, "chess", openings, chess_cfg(device_games=16, device_waves_in_flight=1, **base)),
                play(nw, nw2, "chess", openings, chess_cfg(device_games=512, device_waves_in_flight=3, cache_size=4096, **base))]
    for r in runs:
        assert r.games == ref.games and r.pairs == ref.pairs
    assert len(ref.games) == 2 * (300 - ref.skipped) and ref.simulations > 0


def test_self_play_before_and_after_a_match_plays_the_same_games():
    from cattus_b200.selfplay import SelfPlayRunner

    base = dict(sim_num=24, seed=7, max_moves=16, device_games=8, **NOISY)
    with network("chess_dev", 0) as a, network("chess_dev", 1) as b:
        _, before = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(a, b, 8, keep_records=True)
        play(a, b, "chess", random_playouts(20, 3, 12), chess_cfg(sim_num=16, max_moves=12, device_games=16, cache_size=5000), sim_num_b=30)
        _, after = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(a, b, 8, keep_records=True)
    assert [(r.moves, r.winner, r.entries) for r in after] == [(r.moves, r.winner, r.entries) for r in before]


def test_device_match_errors():
    with network("chess_dev", 0, batch_size=16) as nw, make_network("hex5", batch_size=16) as hx:
        with pytest.raises(_lib.CattusB200Error, match="max_batch") as e:
            play(nw, None, "chess", [None] * 40, chess_cfg(sim_num=8, device_games=64))
        assert e.value.code == _lib.ERANGE
        with pytest.raises(_lib.CattusB200Error, match="opening 1: bad FEN") as e:
            play(nw, None, "chess", [None, "nonsense"], chess_cfg(sim_num=8))
        assert e.value.code == _lib.EINVAL
        with pytest.raises(_lib.CattusB200Error, match="another game") as e:
            play(nw, hx, "chess", [None], chess_cfg(sim_num=8))
        assert e.value.code == _lib.EINVAL
        with pytest.raises(_lib.CattusB200Error, match="sim_num must be > 1"):
            play(nw, None, "chess", [None], chess_cfg(sim_num=8), sim_num_b=1)
        assert len(play(nw, None, "chess", [(KIWIPETE, [])], chess_cfg(sim_num=8, max_moves=2)).games) == 2  # the handle still works


def test_play_match_cli(tmp_path):
    from cattus_b200 import san as S
    from cattus_b200.play_match import main
    from cattus_b200.selfplay import move_from_lan
    from tests.test_match_cpu import parse_movetext

    (tmp_path / "net.cb2").write_bytes(blob("chess10x128"))
    (tmp_path / "cfg.json").write_text(json.dumps({"mcts": {"sim_num": 16, "cache_size": 10000, "temperature_policy": [[4, 1.0], [9999, 0.0]]},
                                                   "model": {"batch_size": 64}, "max_moves": 12, "seed": 1}))
    (tmp_path / "open.txt").write_text("startpos moves e2e4 e7e5\n" + KIWIPETE + ' bm Qxf6; id "kiwi";\n' + FORCED[0] + " moves " + " ".join(FORCED[1])
                                       + "\n7k/5Q2/6K1/8/8/8/8/8 b - - 0 1\n")
    args = ["--model-a", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--openings", str(tmp_path / "open.txt"),
            "--precision-b", "fp8", "--sim-num-b", "20", "--out", str(tmp_path / "games.jsonl"), "--pgn", str(tmp_path / "games.pgn")]
    assert main(args) == 0
    rows = [json.loads(x) for x in (tmp_path / "games.jsonl").read_text().splitlines()]
    skipped = [r for r in rows if not r.get("played", True)]
    games = [r for r in rows if "moves" in r]
    assert [r["opening"] for r in skipped] == [3] and len(games) == 6
    assert [g["termination"] for g in games if g["opening"] == 2] == ["repetition"] * 2
    pgn = re.split(r"\n\n(?=\[Event )", (tmp_path / "games.pgn").read_text().strip())
    assert len(pgn) == 6
    for text, g in zip(pgn, games):
        fen = None if g["fen"] == S.START_FEN else g["fen"]
        assert parse_movetext(fen, text) == [move_from_lan(m) for m in g["opening_moves"] + g["moves"]]
    assert main(["--model-a", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--pairs", "2"]) == 0
