#!/usr/bin/env python
"""Match play from openings (include/cattus_b200_match.h) on one GPU: bf16 against FP8 handles of the same blob.

Workload: chess 10x128 (random-init weights, seed 0), `--openings` openings from seeded random playouts (0-40 plies from
the start position, finished positions never reached), each played twice, sim_num 600 for both sides, max_moves 60,
temperature 0 after the first 8 moves (1 before), no root noise, the HBM cache on, device_games = all games at once.
Turns alternate which precision is side A (bf16-as-A, fp8-as-A, ...), after one warm-up match; games/s and sims/s of
every turn are recorded and the medians reported.  The W/D/L, pentanomial counts and Elo of each turn are from the bf16
handle's side.  The GPU name, power limit and clocks are read in the same run and written beside the numbers.

    python tools/match_bench.py [--openings 2048] [--out profiles/r03c_match_chess10x128.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--openings", type=int, default=2048)
    ap.add_argument("--sim-num", type=int, default=600)
    ap.add_argument("--max-moves", type=int, default=60)
    ap.add_argument("--turns", type=int, default=4)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    from cattus_b200 import CudaNetwork
    from cattus_b200.export import export_blob
    from cattus_b200.match import elo_from_pairs, fmt_elo, play
    from oracle import net
    from tests.test_gpu_analysis import random_playouts

    cfg_net = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg_net, 0), cfg_net.game)
    openings = random_playouts(args.openings, args.seed, 40)
    games = 2 * args.openings
    cfg = {"mcts": {"sim_num": args.sim_num, "explore_factor": 1.41421, "temperature_policy": [[8, 1.0], [9999, 0.0]], "cache_size": 1000000},
           "max_moves": args.max_moves, "seed": 5, "device_games": games}
    res = {"net": args.net, "openings": args.openings, "games": games, "sim_num": args.sim_num, "max_moves": args.max_moves,
           "mcts": cfg["mcts"], "device_games": games,
           "opening_source": f"random playouts of 0-40 plies from the start position, seed {args.seed}", "gpu_before": gpu_record()}
    with CudaNetwork(blob, cfg_net.game, batch_size=games, n_streams=2, precision="bf16") as nb, \
            CudaNetwork(blob, cfg_net.game, batch_size=games, n_streams=2, precision="fp8") as n8:
        # warm-up: module loads, graph capture, first-touch of the pinned buffers
        play(nb, n8, "chess", openings[:128], dict(cfg, device_games=256, max_moves=4, mcts=dict(cfg["mcts"], sim_num=16)))
        turns = []
        for t in range(args.turns):
            a_name = "bf16" if t % 2 == 0 else "fp8"
            a, b = (nb, n8) if a_name == "bf16" else (n8, nb)
            t0 = time.perf_counter()
            r = play(a, b, "chess", openings, cfg)
            secs = time.perf_counter() - t0
            bf16_pairs = r.pairs if a_name == "bf16" else r.pairs[::-1]
            wins, losses = (r.a_wins, r.b_wins) if a_name == "bf16" else (r.b_wins, r.a_wins)
            e = elo_from_pairs(bf16_pairs)
            turn = {"a": a_name, "seconds": secs, "games_per_sec": len(r.games) / secs, "sims_per_sec": r.simulations / secs,
                    "simulations": r.simulations, "evaluations": r.evaluations, "moves": sum(len(g.moves) for g in r.games),
                    "terminations": {k: sum(g.termination == k for g in r.games) for k in ("rules", "repetition", "max_moves")},
                    "bf16_wins": wins, "draws": r.draws, "bf16_losses": losses, "bf16_pentanomial": bf16_pairs,
                    "bf16_score": e.score, "bf16_elo": fmt_elo(e.elo), "bf16_elo_95": [fmt_elo(e.lo), fmt_elo(e.hi)]}
            turns.append(turn)
            print(json.dumps(turn), flush=True)
    res["turns"] = turns
    res["median"] = {k: float(np.median([t[k] for t in turns])) for k in ("games_per_sec", "sims_per_sec", "seconds")}
    res["gpu_after"] = gpu_record()
    print(json.dumps({"median": res["median"]}), flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
