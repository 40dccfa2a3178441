"""GPU (-m gpu): self-play and match play with minibatches under virtual loss per side on the device (DESIGN.md
section 16).

Every game must equal tests/batch_game_oracle.py's game loop over BatchedPlayer(L), driven by the same CudaNetwork (moves,
winners, .traindata bytes, minibatches, collisions); no game may depend on device_games, the waves in flight or the
cache; a minibatched match must leave one-leaf self-play and analysis on the same handle unchanged; and the CLIs run
the mode end to end.
"""
from __future__ import annotations

import json

import pytest

from cattus_b200.analysis import analyse
from cattus_b200.match import play
from oracle import chess as oc
from oracle import mcts as om
from tests import batch_game_oracle as bo
from tests.test_analysis_cpu import chess_history, hex_positions, ttt_positions
from tests.test_chess_cpu import KIWIPETE, _params, chess_cfg, chess_oracle_fn
from tests.test_gpu_analysis import random_playouts
from tests.test_match_cpu import FORCED, NOISY, SHUFFLE, small_history
from tests.test_selfplay_cpu import cfg_with, oracle_net_fn
from tests.util import blob, make_network

pytestmark = pytest.mark.gpu


def evaluator(nw, game):
    from tests.test_gpu_selfplay import chess_gpu_net, gpu_net_fn

    if game == "chess":
        return om.Evaluator(chess_oracle_fn(chess_gpu_net(nw)), None)
    return om.Evaluator(oracle_net_fn(gpu_net_fn(nw, 5 if game == "hex5" else 3)), None)


def new_position(game):
    if game == "chess":
        return oc.ChessPosition.new()
    return om.TttPosition.new() if game == "ttt" else om.HexPosition.new(5)


CASES = [("hex5", "hex5", "bf16"), ("ttt", "ttt", "bf16"), ("chess_dev", "chess", "bf16"), ("chess10x128", "chess", "bf16"),
         ("chess10x128", "chess", "fp8")]


@pytest.mark.parametrize("L", [16, 64])
@pytest.mark.parametrize("name,game,precision", CASES)
def test_device_selfplay_equals_oracle(name, game, precision, L):
    from cattus_b200.selfplay import SelfPlayRunner

    mk = chess_cfg if game == "chess" else cfg_with
    cfg = mk(sim_num=40, seed=5, max_moves=10 if game == "chess" else 0, device_games=4, cache_size=4096, search_batch=L, **NOISY)
    games_num = 4
    with make_network(name, precision=precision, batch_size=4 * L) as nw:
        summary, recs = SelfPlayRunner(game, cfg).generate_data(nw, None, games_num, keep_records=True)
        ev = evaluator(nw, game)
        p = _params(cfg)
        ref = [bo.play_from(g, [new_position(game)], p, p, ev, ev, cfg["seed"], cfg.get("max_moves", 0), (L, L)) for g in range(games_num)]
    to_move = oc.move_to_u16 if game == "chess" else (lambda m: m)
    for r, (o, p1, p2) in zip(recs, ref):
        assert r.moves == [to_move(m) for m in o.moves] and r.winner == o.winner, r.game_idx
        assert r.entries == [om.data_entry_bytes(pos, probs, o.winner) for pos, probs in o.entries], r.game_idx
    m = summary["metrics"]
    assert m["selfplay.simulations"] == sum(o.sims for o, _, _ in ref)
    assert m["selfplay.minibatches"] == sum(p1.minibatches + p2.minibatches for _, p1, p2 in ref)
    assert m["selfplay.collisions"] == sum(p1.collisions + p2.collisions for _, p1, p2 in ref) > 0


@pytest.mark.parametrize("name,game,precision", CASES)
def test_device_match_l1_against_l16_equals_oracle(name, game, precision):
    if game == "chess":
        openings = [FORCED, (KIWIPETE, ["e1g1"]), SHUFFLE] + random_playouts(2, 5, 20)
        cfg = chess_cfg(sim_num=40, seed=3, max_moves=8, device_games=4, **NOISY)
        hist = lambda o: chess_history(*o)  # noqa: E731
    else:
        openings = hex_positions(5, 3, 7) if game == "hex5" else ttt_positions(3, 8)
        cfg = cfg_with(sim_num=40, seed=3, device_games=4, **NOISY)
        hist = lambda o: small_history(game, o)  # noqa: E731
    from tests.test_gpu_match import network

    with network(name, 0, precision, batch_size=64) as a, network(name, 1, precision, batch_size=64) as b:
        got = play(a, b, game, openings, cfg, sim_num_b=48, search_batch=1, search_batch_b=16)
        pa = _params(cfg)
        pb = om.MctsParams(**dict(pa.__dict__, sim_num=48))
        ea, eb = evaluator(a, game), evaluator(b, game)
        ref = {}
        for k, (o, st) in enumerate(zip(openings, got.opening_status)):
            if not st:
                for c in (0, 1):
                    ref[(k, c == 0)] = bo.play_from(2 * k + c, hist(o), pa, pb, ea, eb, cfg["seed"], cfg.get("max_moves", 0), (1, 16))
    to_move = oc.move_to_u16 if game == "chess" else (lambda m: m)
    for g in got.games:
        o, p1, p2 = ref[(g.opening, g.a_is_player1)]
        assert g.moves == [to_move(m) for m in o.moves] and g.winner == o.winner, (g.opening, g.a_is_player1)
    assert got.minibatches == (sum(r[1].minibatches for r in ref.values()), sum(r[2].minibatches for r in ref.values()))
    assert got.collisions == (0, sum(r[2].collisions for r in ref.values()))


def test_device_minibatched_match_invariance_at_scale():
    """200 chess openings x 2 games at L = 16: identical at several device_games, 1 / 3 waves, cache on and off."""
    openings = random_playouts(200, 43, 16)
    base = dict(sim_num=48, seed=9, max_moves=16, **NOISY)
    with make_network("chess_dev", batch_size=4096, n_streams=2) as nw:
        ref = play(nw, None, "chess", openings, chess_cfg(device_games=256, **base), search_batch=16)
        runs = [play(nw, None, "chess", openings, chess_cfg(device_games=100, device_waves_in_flight=3, cache_size=1 << 16, **base), search_batch=16),
                play(nw, None, "chess", openings, chess_cfg(device_games=17, device_waves_in_flight=1, **base), search_batch=16)]
    for r in runs:
        assert (r.games, r.pairs, r.minibatches, r.collisions) == (ref.games, ref.pairs, ref.minibatches, ref.collisions)
    assert sum(ref.collisions) > 0 and len(ref.games) == 2 * (200 - ref.skipped)


def test_one_handle_shares_state_cleanly():
    """L = 1 self-play and a one-leaf analysis give the same results before and after a minibatched match on the handle."""
    from cattus_b200.selfplay import SelfPlayRunner

    base = dict(sim_num=24, seed=7, max_moves=16, device_games=8, **NOISY)
    positions = random_playouts(8, 4, 12)
    with make_network("chess_dev", batch_size=1024) as nw:
        _, before = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        one_before = analyse(nw, "chess", positions, chess_cfg(sim_num=40, device_games=4))
        play(nw, None, "chess", random_playouts(20, 3, 12), chess_cfg(sim_num=60, max_moves=12, device_games=16, cache_size=5000),
             search_batch=64, search_batch_b=3)
        _, after = SelfPlayRunner("chess", chess_cfg(**base)).generate_data(nw, None, 8, keep_records=True)
        one_after = analyse(nw, "chess", positions, chess_cfg(sim_num=40, device_games=4))
    assert [(r.moves, r.winner, r.entries) for r in after] == [(r.moves, r.winner, r.entries) for r in before]
    assert one_after == one_before


def test_device_errors():
    from cattus_b200 import _lib
    from cattus_b200.selfplay import SelfPlayError, SelfPlayRunner

    with make_network("chess_dev", batch_size=64) as nw:
        with pytest.raises(_lib.CattusB200Error, match="max_batch") as e:
            play(nw, None, "chess", [None] * 4, chess_cfg(sim_num=8, device_games=8), search_batch_b=16)
        assert e.value.code == _lib.ERANGE
        with pytest.raises(SelfPlayError, match="max_batch"):
            SelfPlayRunner("chess", chess_cfg(sim_num=8, device_games=8, search_batch=16)).generate_data(nw, None, 8)
        with pytest.raises(SelfPlayError, match="search_batch"):
            SelfPlayRunner("chess", chess_cfg(sim_num=8, search_batch=16)).generate_data(nw, None, 2)
        assert len(play(nw, None, "chess", [(KIWIPETE, [])], chess_cfg(sim_num=8, max_moves=2)).games) == 2  # the handle still works


def test_self_player_cli_search_batch(tmp_path):
    from cattus_b200.self_player import main

    (tmp_path / "net.cb2").write_bytes(blob("chess_dev"))
    (tmp_path / "cfg.json").write_text(json.dumps({"mcts": {"sim_num": 64, "cache_size": 0, "temperature_policy": [[4, 1.0], [9999, 0.0]],
                                                            "prior_noise_alpha": 0.3, "prior_noise_epsilon": 0.25},
                                                   "model": {"batch_size": 64}, "threads": 1, "max_moves": 6, "search_batch": 32}))
    net = str(tmp_path / "net.cb2")
    assert main(["--model1-path", net, "--model2-path", net, "--games-num", "6", "--out-dir1", str(tmp_path / "d1"), "--out-dir2",
                 str(tmp_path / "d2"), "--summary-file", str(tmp_path / "s.json"), "--config-file", str(tmp_path / "cfg.json")]) == 0
    s = json.loads((tmp_path / "s.json").read_text())
    m = s["metrics"]
    assert s["player1_wins"] + s["player2_wins"] + s["draws"] == 6
    assert m["selfplay.simulations"] == m["selfplay.searches"] * 64 and m["selfplay.minibatches"] < m["selfplay.simulations"]
    files = sorted((tmp_path / "d1").glob("*.traindata")) + sorted((tmp_path / "d2").glob("*.traindata"))
    assert len(files) == m["selfplay.searches"] and all(f.stat().st_size == 18 * 8 + 235 + 225 * 4 + 1 for f in files)


def test_play_match_cli_search_batch_b(tmp_path, capsys):
    from cattus_b200.play_match import main

    (tmp_path / "net.cb2").write_bytes(blob("chess10x128"))
    (tmp_path / "cfg.json").write_text(json.dumps({"mcts": {"sim_num": 128}, "model": {"batch_size": 256}, "max_moves": 8, "seed": 1}))
    (tmp_path / "open.txt").write_text("startpos moves e2e4 e7e5\n" + KIWIPETE + "\n")
    assert main(["--model-a", str(tmp_path / "net.cb2"), "--config-file", str(tmp_path / "cfg.json"), "--openings", str(tmp_path / "open.txt"),
                 "--search-batch-b", "64", "--out", str(tmp_path / "games.jsonl"), "--pgn", str(tmp_path / "games.pgn")]) == 0
    summary = json.loads(capsys.readouterr().err.strip().splitlines()[-1])
    assert summary["games"] == 4 and summary["collisions"][0] == 0 and summary["collisions"][1] > 0
    assert summary["minibatches"][1] < summary["minibatches"][0]
    assert len((tmp_path / "games.jsonl").read_text().splitlines()) == 4 and (tmp_path / "games.pgn").read_text().count("[Event ") == 4
