#!/usr/bin/env python
"""Minibatched search under virtual loss (DESIGN.md section 15) on one GPU: a few chess positions searched deeply.

Workload: chess 10x128 (random-init weights, seed 0), bf16 and FP8 handles of the same blob.  Positions: one (after
1. e4 e5 2. Nf3) and a set of 16 from seeded random playouts.  Every analysis call searches them at sim_num 10000 with
search_batch L in --batches (L = 1 is the one-leaf analysis); bf16 and FP8 alternate, --rounds turns each after a
warm-up, and the medians are reported with minibatches and collisions.  Also:
  * the per-call set-up floor: the same call at sim_num 2;
  * the host UCI search (ChessSearch.go, speculate 31, a fresh search per position) on the same positions;
  * the crossover: 4096 positions at L = 1 against 64 positions at L = 64, both at --cross-sims;
  * agreement of L = 256 with L = 1 on the 16 positions: best move, first two PV plies, visit total variation;
  * where the time of one L = 256 call goes, from torch.profiler in a run of its own: CUDA time per kernel name.
The GPU name, power limit and max SM clock are read in the same run and written beside the numbers.

    python tools/search_batch_bench.py [--out profiles/r03d_search_batch_chess10x128.json]
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

from tools.analyse_bench import visit_tv  # noqa: E402
from tools.fp8_bench import gpu_record  # noqa: E402

ONE = (None, ["e2e4", "e7e5", "g1f3"])


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--sim-num", type=int, default=10000)
    ap.add_argument("--batches", default="1,16,64,256,1024")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cross-sims", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    from cattus_b200 import CudaNetwork
    from cattus_b200.analysis import analyse
    from cattus_b200.export import export_blob
    from cattus_b200.selfplay import ChessSearch
    from oracle import net
    from tests.test_gpu_analysis import random_playouts

    cfg_net = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg_net, 0), cfg_net.game)
    sets = {"one": [ONE], "sixteen": random_playouts(16, args.seed, 30)}
    batches = [int(x) for x in args.batches.split(",")]
    mcts = {"sim_num": args.sim_num, "explore_factor": 1.41421, "cache_size": 1 << 20}
    res = {"net": args.net + " (random-init weights, seed 0)", "sim_num": args.sim_num, "cache_size": mcts["cache_size"],
           "positions": {"one": "startpos moves e2e4 e7e5 g1f3", "sixteen": f"random playouts of 0-30 plies, seed {args.seed}"},
           "gpu_before": gpu_record()}
    precs = ("bf16", "fp8")

    def cfg(sim_num, games=0):
        c = {"mcts": dict(mcts, sim_num=sim_num)}
        if games:
            c["device_games"] = games
        return c

    with CudaNetwork(blob, "chess", batch_size=4096, n_streams=2, precision="bf16") as nb, \
            CudaNetwork(blob, "chess", batch_size=4096, n_streams=2, precision="fp8") as n8:
        nws = {"bf16": nb, "fp8": n8}
        for p in precs:  # warm-up: module loads, graph captures, first touch of the pinned buffers
            for L in batches:
                analyse(nws[p], "chess", sets["sixteen"], cfg(64), search_batch=L)
        # the set-up floor of one call: two simulations
        floor = {p: [] for p in precs}
        for _ in range(args.rounds):
            for p in precs:
                floor[p].append(timed(lambda: analyse(nws[p], "chess", [ONE], cfg(2), search_batch=256))[1])
        res["setup_floor_seconds_sim2"] = {p: float(np.median(v)) for p, v in floor.items()}
        print(json.dumps({"setup_floor": res["setup_floor_seconds_sim2"]}), flush=True)
        # the timed grid
        runs: dict = {}
        results: dict = {}
        for _ in range(args.rounds):
            for name, pos in sets.items():
                for L in batches:
                    for p in precs:
                        out, secs = timed(lambda: analyse(nws[p], "chess", pos, cfg(args.sim_num), search_batch=L))
                        key = f"{p}/{name}/L{L}"
                        sims = sum(a.simulations for a in out)
                        mb = [a.minibatches for a in out if a.status == 0]
                        co = [a.collisions for a in out if a.status == 0]
                        runs.setdefault(key, []).append({"seconds": secs, "sims_per_sec": sims / secs, "minibatches_mean": float(np.mean(mb)),
                                                         "collisions_mean": float(np.mean(co)),
                                                         "collisions_per_minibatch": float(np.sum(co) / max(1, np.sum(mb)))})
                        results[key] = out
                        print(json.dumps({key: runs[key][-1]}), flush=True)
        res["grid_runs"] = runs
        res["grid_median"] = {k: {f: float(np.median([r[f] for r in v])) for f in v[0]} for k, v in runs.items()}
        # the host UCI search with speculate 31, a fresh search per position
        host = {p: {name: [] for name in sets} for p in precs}
        for _ in range(args.rounds):
            for p in precs:
                for name, pos in sets.items():
                    per = []
                    for fen, moves in pos:
                        with ChessSearch({"mcts": dict(mcts), "speculate": 31}, model=nws[p]) as s:
                            per.append(timed(lambda: s.go(fen, moves))[1])
                    host[p][name].append(float(np.mean(per)))
        res["host_go_speculate31_seconds_per_go"] = {p: {n: float(np.median(v)) for n, v in d.items()} for p, d in host.items()}
        print(json.dumps({"host_go": res["host_go_speculate31_seconds_per_go"]}), flush=True)
        # crossover: many positions one leaf each against a few positions many leaves each
        wide = random_playouts(4096, args.seed + 1, 30)
        cross = {}
        for p in precs:
            out, s1 = timed(lambda: analyse(nws[p], "chess", wide, cfg(args.cross_sims, 4096), search_batch=1))
            sims1 = sum(a.simulations for a in out)
            out, s64 = timed(lambda: analyse(nws[p], "chess", wide[:64], cfg(args.cross_sims, 64), search_batch=64))
            sims64 = sum(a.simulations for a in out)
            cross[p] = {"L1_4096_positions": {"seconds": s1, "sims_per_sec": sims1 / s1},
                        "L64_64_positions": {"seconds": s64, "sims_per_sec": sims64 / s64}}
        res["crossover"] = {"sim_num": args.cross_sims, **cross}
        print(json.dumps({"crossover": cross}), flush=True)
        # agreement of L = 256 with one leaf in flight
        agree = {}
        for p in precs:
            a1, a256 = results.get(f"{p}/sixteen/L1"), results.get(f"{p}/sixteen/L256")
            if a1 is None or a256 is None:
                continue
            pairs = [(x, y) for x, y in zip(a1, a256) if x.status == 0]
            agree[p] = {"positions": len(pairs), "same_best_move": sum(x.best_move == y.best_move for x, y in pairs),
                        "same_pv_first_2": sum(x.pv[:2] == y.pv[:2] for x, y in pairs),
                        "mean_visit_tv": float(np.mean([visit_tv(x, y) for x, y in pairs]))}
        res["agreement_L256_vs_L1"] = agree
        print(json.dumps({"agreement": agree}), flush=True)
        # where the time of one L = 256 call goes (a separate, traced run)
        import torch
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            out, secs = timed(lambda: analyse(nb, "chess", [ONE], cfg(args.sim_num), search_batch=256))
            torch.cuda.synchronize()
        kern: dict = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                k = kern.setdefault(ev.name, [0, 0.0])
                k[0] += 1
                k[1] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        waves = out[0].minibatches
        res["trace_bf16_one_L256"] = {"seconds_traced": secs, "minibatches": waves, "collisions": out[0].collisions,
                                      "kernels_us_total": {k: round(v[1], 1) for k, v in sorted(kern.items(), key=lambda kv: -kv[1][1])[:16]},
                                      "kernels_launches": {k: v[0] for k, v in sorted(kern.items(), key=lambda kv: -kv[1][1])[:16]},
                                      "gpu_busy_us_per_minibatch": round(sum(v[1] for v in kern.values()) / max(1, waves), 1)}
        print(json.dumps({"trace": res["trace_bf16_one_L256"]}), flush=True)
    res["gpu_after"] = gpu_record()
    text = json.dumps(res, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
