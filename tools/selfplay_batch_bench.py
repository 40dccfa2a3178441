#!/usr/bin/env python
"""Self-play and match play with minibatches under virtual loss (DESIGN.md section 16) on one GPU.

Workload: chess 10x128 (random-init weights, seed 0, bf16), one handle.
  1. few-opening match: 32 openings (seeded random playouts) x 2 games, sim_num 4000, max_moves 40, both sides at
     search_batch L in --match-batches; L arms alternate over --rounds, medians of seconds per call, with sims/s,
     minibatches and collisions;
  2. trainer-sized self-play: 100 games at sim_num 600 (the chess_dev search settings: explore 1.41421, root noise
     0.3 / 0.25, temperature 1 for 30 moves) with max_moves 16, on the device at L in --selfplay-batches against the
     host-tree driver with speculation (8 threads, the self_player defaults), alternating, medians;
  3. virtual loss in games: A at L = 1 against B at L = 64 and at L = 256, equal sim_num 2000, --elo-openings openings
     x 2 games, --elo-max-moves; pentanomial counts and Elo with its 95 % interval.  A wave ends with its slowest warp,
     so A's one-leaf searches advance one simulation per wave of B's minibatches: keep this part small.  The net is random-init: this measures what the
     minibatches change in the search, not what they cost a trained net.
The GPU name, power limit and max SM clock are read in the same run and written beside the numbers.

    python tools/selfplay_batch_bench.py [--out profiles/r03e_selfplay_batch_chess10x128.json]
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from tools.fp8_bench import gpu_record  # noqa: E402

NOISY = {"prior_noise_alpha": 0.3, "prior_noise_epsilon": 0.25, "temperature_policy": [[30, 1.0], [9999, 0.0]]}


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--match-batches", default="1,16,64,256")
    ap.add_argument("--selfplay-batches", default="1,8,16,32")
    ap.add_argument("--match-sims", type=int, default=4000)
    ap.add_argument("--elo-openings", type=int, default=32)
    ap.add_argument("--elo-max-moves", type=int, default=16)
    ap.add_argument("--elo-sims", type=int, default=2000)
    ap.add_argument("--skip", default="", help="comma-separated parts to skip: match,selfplay,elo")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    skip = set(filter(None, args.skip.split(",")))

    from cattus_b200 import CudaNetwork
    from cattus_b200.match import fmt_elo, play
    from cattus_b200.selfplay import SelfPlayRunner
    from cattus_b200.export import export_blob
    from oracle import net
    from tests.test_gpu_analysis import random_playouts

    cfg_net = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg_net, 0), cfg_net.game)
    res = {"net": args.net + " (random-init weights, seed 0), bf16, one handle", "gpu_before": gpu_record()}

    with CudaNetwork(blob, "chess", batch_size=4096, n_streams=2, precision="bf16") as nw:
        # ------------------------------------------------------------------ 1. few-opening match
        if "match" not in skip:
            openings = random_playouts(32, 7, 12)
            Ls = [int(x) for x in args.match_batches.split(",")]
            cfg = {"mcts": {"sim_num": args.match_sims, "explore_factor": 1.41421, "cache_size": 1 << 20, **NOISY}, "max_moves": 40, "seed": 1}
            play(nw, None, "chess", openings[:2], dict(cfg, max_moves=2), search_batch=Ls[-1])  # warm-up
            runs = {L: [] for L in Ls}
            for _ in range(args.rounds):
                for L in Ls:
                    r, s = timed(lambda: play(nw, None, "chess", openings, cfg, search_batch=L))
                    runs[L].append((s, r))
                    print(json.dumps({"match": L, "seconds": round(s, 3), "sims": r.simulations}), flush=True)
            out = {}
            for L, rr in runs.items():
                sec = float(np.median([s for s, _ in rr]))
                r = rr[0][1]
                out[str(L)] = {"seconds_per_call": round(sec, 3), "sims_per_s": round(r.simulations / sec, 1), "games": len(r.games),
                               "simulations": r.simulations, "evaluations": r.evaluations, "minibatches": sum(r.minibatches),
                               "collisions": sum(r.collisions), "all_seconds": [round(s, 3) for s, _ in rr]}
            res["few_opening_match"] = {"openings": "32 random playouts of 0-12 plies, seed 7, x 2 games", "sim_num": args.match_sims,
                                        "max_moves": 40, "cache_size": 1 << 20, "device_games": "0 (min(64, 4096 / L))", "by_L": out}

        # ------------------------------------------------------------------ 2. trainer-sized self-play
        if "selfplay" not in skip:
            Ls = [int(x) for x in args.selfplay_batches.split(",")]
            mcts = {"sim_num": 600, "explore_factor": 1.41421, "cache_size": 100000, **NOISY}
            base = {"mcts": mcts, "max_moves": 16, "seed": 3}
            host = dict(base, threads=8, games_per_thread=64, groups_per_thread=2, speculate=14)
            arms = {f"device L={L}": dict(base, device_games=min(100, 4096 // L), search_batch=L) for L in Ls}
            arms["host trees, speculate 14"] = host
            for name, c in arms.items():  # warm-up
                SelfPlayRunner("chess", dict(c, max_moves=1)).generate_data(nw, None, 4)
            runs = {k: [] for k in arms}
            for _ in range(args.rounds):
                for name, c in arms.items():
                    (summary, _), s = timed(lambda: SelfPlayRunner("chess", c).generate_data(nw, None, 100))
                    runs[name].append((s, summary["metrics"]))
                    print(json.dumps({"selfplay": name, "seconds": round(s, 3)}), flush=True)
            out = {}
            for name, rr in runs.items():
                sec = float(np.median([s for s, _ in rr]))
                m = rr[0][1]
                out[name] = {"seconds": round(sec, 3), "sims_per_s": round(m["selfplay.simulations"] / sec, 1), "simulations": m["selfplay.simulations"],
                             "evaluations": m["selfplay.evaluations"], "minibatches": m["selfplay.minibatches"], "collisions": m["selfplay.collisions"],
                             "all_seconds": [round(s, 3) for s, _ in rr]}
            res["trainer_selfplay"] = {"games": 100, "sim_num": 600, "max_moves": 16, "noise": [0.3, 0.25], "cache_size": 100000,
                                       "host": "threads 8, games_per_thread 64, groups_per_thread 2, speculate 14 (self_player defaults)",
                                       "arms": out}

        # ------------------------------------------------------------------ 3. virtual loss in games
        if "elo" not in skip:
            openings = random_playouts(args.elo_openings, 11, 12)
            cfg = {"mcts": {"sim_num": args.elo_sims, "explore_factor": 1.41421, "cache_size": 1 << 20, **NOISY}, "max_moves": args.elo_max_moves,
                   "seed": 5}
            out = {}
            for Lb in (64, 256):
                r, s = timed(lambda: play(nw, None, "chess", openings, cfg, search_batch=1, search_batch_b=Lb))
                e = r.elo()
                out[f"A L=1 vs B L={Lb}"] = {"seconds": round(s, 3), "a_wins": r.a_wins, "draws": r.draws, "b_wins": r.b_wins, "pentanomial": r.pairs,
                                             "score_a": None if e is None else round(e.score, 4),
                                             "elo_a": None if e is None else fmt_elo(e.elo),
                                             "elo_a_95": None if e is None else [fmt_elo(e.lo), fmt_elo(e.hi)],
                                             "terminations": {t: sum(g.termination == t for g in r.games) for t in ("rules", "repetition", "max_moves")},
                                             "minibatches": list(r.minibatches), "collisions": list(r.collisions)}
                print(json.dumps({"elo": Lb, **out[f"A L=1 vs B L={Lb}"]}), flush=True)
            res["virtual_loss_in_games"] = {"openings": f"{args.elo_openings} random playouts of 0-12 plies, seed 11, x 2 games",
                                            "sim_num": args.elo_sims, "max_moves": args.elo_max_moves, "note": "random-init net: says nothing about a trained net",
                                            "matches": out}
    res["gpu_after"] = gpu_record()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
