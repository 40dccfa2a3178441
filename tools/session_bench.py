#!/usr/bin/env python
"""Persistent device search sessions (DESIGN.md section 17) on one GPU, chess 10x128 (random-init weights, seed 0).

  * seconds per `go nodes 10000` at L = 256, bf16 and FP8, in alternating turns: a fresh analyse() call, a session
    search from a fresh root, and a session search reusing the tree after 2 plies;
  * the fraction of visits reused over a 30-ply line (each search at nodes 10000, the position advanced by the best move);
  * achieved time and overrun of movetime 100 / 500 / 2000;
  * stop latency: from stop() to the end of the search, on an infinite search;
  * the capacity in nodes: an unlimited search until the 2^26-word tree buffer is full.
The GPU name, power limit and max SM clock are read in the same run and written beside the numbers.

    python tools/session_bench.py [--out profiles/r03f_session_chess10x128.json]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from tools.fp8_bench import gpu_record  # noqa: E402

LINE = ["e2e4", "e7e5", "g1f3", "b8c6"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--nodes", type=int, default=10000)
    ap.add_argument("--L", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--plies", type=int, default=30)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    from cattus_b200 import CudaNetwork
    from cattus_b200.analysis import analyse
    from cattus_b200.export import export_blob
    from cattus_b200.selfplay import move_to_lan
    from cattus_b200.session import DeviceSearch
    from oracle import net

    cfg_net = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg_net, 0), cfg_net.game)
    mcts = {"sim_num": args.nodes, "explore_factor": 1.41421, "cache_size": 1 << 20}
    cfg = {"mcts": mcts}
    res = {"net": args.net + " (random-init weights, seed 0)", "nodes": args.nodes, "search_batch": args.L, "cache_size": mcts["cache_size"],
           "gpu_before": gpu_record()}
    L = args.L
    with CudaNetwork(blob, "chess", batch_size=L, n_streams=2, precision="bf16") as nb, \
            CudaNetwork(blob, "chess", batch_size=L, n_streams=2, precision="fp8") as n8:
        nws = {"bf16": nb, "fp8": n8}
        sess = {p: DeviceSearch(nws[p], "chess", cfg, L) for p in nws}

        def fresh_analyse(p):
            t0 = time.perf_counter()
            analyse(nws[p], "chess", [(None, LINE)], cfg, search_batch=L)
            return time.perf_counter() - t0

        def session_fresh(p):
            s = sess[p]
            s.new_game()
            s.set_position(None, LINE)
            t0 = time.perf_counter()
            s.search(nodes=args.nodes)
            return time.perf_counter() - t0

        def session_reuse(p):
            s = sess[p]
            s.new_game()
            s.set_position(None, LINE[:2])
            r0 = s.search(nodes=args.nodes)
            s.set_position(None, LINE[:2] + [move_to_lan(m) for m in r0.analysis.pv[:2]])
            t0 = time.perf_counter()
            r = s.search(nodes=args.nodes)
            return time.perf_counter() - t0, r.reused_visits

        for p in nws:  # warm-up
            fresh_analyse(p)
            session_fresh(p)
            session_reuse(p)
        times = {p: {"analyse": [], "session_fresh": [], "session_reuse": [], "reused_visits": []} for p in nws}
        for _ in range(args.rounds):
            for p in nws:
                times[p]["analyse"].append(fresh_analyse(p))
                times[p]["session_fresh"].append(session_fresh(p))
                t, reused = session_reuse(p)
                times[p]["session_reuse"].append(t)
                times[p]["reused_visits"].append(reused)
        res["go_nodes_seconds"] = {p: {k: (statistics.median(v) if k != "reused_visits" else v) for k, v in d.items()} | {"all": d}
                                   for p, d in times.items()}

        # reuse over a line of play
        s = sess["bf16"]
        s.new_game()
        moves, total_reused, total_visits = [], 0, 0
        for _ in range(args.plies):
            s.set_position(None, moves)
            r = s.search(nodes=args.nodes)
            if r.analysis.status != 0:
                break
            total_reused += r.reused_visits
            total_visits += sum(r.analysis.visits)
            moves.append(move_to_lan(r.analysis.best_move))
        res["reuse_line"] = {"plies": len(moves), "reused_visits": total_reused, "root_visits": total_visits,
                             "fraction_reused": total_reused / max(1, total_visits)}

        # movetime
        mt = {}
        for ms in (100, 500, 2000):
            runs = []
            for _ in range(3):
                s.new_game()
                s.set_position(None, LINE)
                t0 = time.perf_counter()
                r = s.search(movetime_ms=ms)
                wall = time.perf_counter() - t0
                runs.append({"search_ms": r.seconds * 1000, "wall_ms": wall * 1000, "overrun_ms": r.seconds * 1000 - ms, "minibatches": r.analysis.minibatches,
                             "ms_per_minibatch": r.seconds * 1000 / r.analysis.minibatches, "stop_reason": r.stop_reason})
            mt[str(ms)] = runs
        res["movetime"] = mt

        # stop latency
        lat = []
        for _ in range(5):
            s.new_game()
            s.set_position(None, LINE)
            s.go()
            time.sleep(0.25)
            t0 = time.perf_counter()
            s.stop()
            r = s.wait()
            lat.append({"stop_to_result_ms": (time.perf_counter() - t0) * 1000, "minibatches": r.analysis.minibatches,
                        "ms_per_minibatch": r.seconds * 1000 / r.analysis.minibatches})
        res["stop_latency"] = lat

        # capacity
        s.new_game()
        s.set_position(None, LINE)
        t0 = time.perf_counter()
        r = s.search()
        res["capacity"] = {"stop_reason": r.stop_reason, "simulations": r.analysis.simulations, "root_visits": sum(r.analysis.visits),
                           "minibatches": r.analysis.minibatches, "collisions": r.analysis.collisions, "seconds": time.perf_counter() - t0}
        for x in sess.values():
            x.close()
    res["gpu_after"] = gpu_record()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
