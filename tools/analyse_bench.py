#!/usr/bin/env python
"""Batched analysis (include/cattus_b200_analysis.h) on one GPU: bf16 and FP8 handles of the same blob, in turns.

Workload: chess 10x128 (random-init weights, seed 0), `--positions` positions from seeded random playouts (0-40 plies from
the start position, finished ones skipped), sim_num 600, device_games = positions, the HBM cache on.  Each precision is
run `--rounds` times alternately after one warm-up call; positions/s and sims/s of every turn are recorded and the medians
reported.  Then the search-level agreement of the two precisions over the same positions: the fraction with the same
best move and the mean total variation distance between the two root visit distributions.  The GPU name, power limit
and clocks are read in the same run and written beside the numbers.

    python tools/analyse_bench.py [--positions 4096] [--out profiles/r03b_analyse_chess10x128.json]
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


def playout_positions(n: int, seed: int):
    from tests.test_gpu_analysis import random_playouts

    return random_playouts(n, seed, 40)


def visit_tv(a, b) -> float:
    """Total variation distance between two root visit distributions over the same children."""
    pa = dict(zip(a.moves, np.asarray(a.visits, dtype=np.float64) / max(1, sum(a.visits))))
    pb = dict(zip(b.moves, np.asarray(b.visits, dtype=np.float64) / max(1, sum(b.visits))))
    return 0.5 * sum(abs(pa.get(m, 0.0) - pb.get(m, 0.0)) for m in set(pa) | set(pb))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--positions", type=int, default=4096)
    ap.add_argument("--sim-num", type=int, default=600)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    from cattus_b200 import CudaNetwork
    from cattus_b200.analysis import analyse
    from cattus_b200.export import export_blob
    from oracle import net

    cfg_net = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg_net, 0), cfg_net.game)
    positions = playout_positions(args.positions, args.seed)
    cfg = {"mcts": {"sim_num": args.sim_num, "explore_factor": 1.41421, "cache_size": 1000000}, "device_games": args.positions}
    res = {"net": args.net, "positions": args.positions, "sim_num": args.sim_num, "device_games": args.positions, "cache_size": 1000000,
           "position_source": f"random playouts of 0-40 plies from the start position, seed {args.seed}", "gpu_before": gpu_record()}
    precs = ("bf16", "fp8")
    results = {}
    with CudaNetwork(blob, cfg_net.game, batch_size=args.positions, n_streams=2, precision="bf16") as nb, \
            CudaNetwork(blob, cfg_net.game, batch_size=args.positions, n_streams=2, precision="fp8") as n8:
        nws = {"bf16": nb, "fp8": n8}
        for p in precs:  # warm-up: module loads, graph capture, first-touch of the pinned buffers
            analyse(nws[p], "chess", positions[:256], dict(cfg, device_games=256, mcts=dict(cfg["mcts"], sim_num=16)))
        runs = {p: [] for p in precs}
        for _ in range(args.rounds):
            for p in precs:
                t0 = time.perf_counter()
                out = analyse(nws[p], "chess", positions, cfg)
                secs = time.perf_counter() - t0
                sims = sum(a.simulations for a in out)
                run = {"seconds": secs, "positions_per_sec": len(out) / secs, "sims_per_sec": sims / secs}
                runs[p].append(run)
                results[p] = out
                print(json.dumps({"precision": p, **run}), flush=True)
        res["runs"] = runs
        res["median"] = {p: {k: float(np.median([r[k] for r in runs[p]])) for k in ("positions_per_sec", "sims_per_sec", "seconds")} for p in precs}
        res["fp8_speedup"] = res["median"]["fp8"]["sims_per_sec"] / res["median"]["bf16"]["sims_per_sec"]
    res["gpu_after"] = gpu_record()
    a, b = results["bf16"], results["fp8"]
    searched = [(x, y) for x, y in zip(a, b) if x.status == 0]
    same = sum(x.best_move == y.best_move for x, y in searched)
    tvs = [visit_tv(x, y) for x, y in searched]
    res["agreement"] = {"searched_positions": len(searched), "same_best_move": same, "same_best_move_fraction": same / max(1, len(searched)),
                        "mean_visit_tv": float(np.mean(tvs)) if tvs else 0.0, "median_visit_tv": float(np.median(tvs)) if tvs else 0.0,
                        "same_pv_first_2": sum(x.pv[:2] == y.pv[:2] for x, y in searched)}
    print(json.dumps({"agreement": res["agreement"], "median": res["median"]}), flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
