#!/usr/bin/env python
"""BF16 vs FP8 (CATTUS_B200_PRECISION_FP8) on one GPU, two handles of the same blob in the same process, measured in turns.

  * trunk stage (time_stage 1: encode + stem + residual blocks + head convs, one trunk_fused launch; CUDA events, L2 flushed
    before every iteration) at B = 1024 / 2048 / 4096, with its TFLOP/s as a share of the measured bf16 figure and of the FP8
    data-sheet rate (a kernel's share, not a reached peak);
  * the whole captured graph (time_stage 4) over a batch sweep;
  * device-resident evaluation (resident_upload once, eval_resident back to back, one synchronise) in positions/s;
  * time_sustained (4 distinct resident batches rotated back to back, no flush);
  * device-resident chess self-play (sim_num 600, 16 moves, 4096 games in flight).
The GPU name, power limit and clocks are read in the same run and written beside the numbers.

    python tools/fp8_bench.py [--net chess10x128] [--out profiles/fp8_bench.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

FP8_DATASHEET_TFLOPS = 4500.0  # HGX B200 data sheet, one GPU, dense FP8
BF16_DATASHEET_TFLOPS = 2250.0


def gpu_record() -> dict:
    q = "name,power.limit,clocks.max.sm,clocks.sm,power.draw,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:  # recorded, not hidden
        return {"error": repr(e)}


def trunk_flops(cfg) -> int:
    """Dense MACs x 2 of what trunk_fused computes per position: stem, residual blocks and both 1x1 head convs (unpadded)."""
    s2 = cfg.board_size ** 2
    f = cfg.filters
    return 2 * s2 * (9 * cfg.planes * f + cfg.blocks * 2 * 9 * f * f + f * (cfg.value_channels + cfg.policy_channels))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", default="chess10x128")
    ap.add_argument("--rounds", type=int, default=5, help="alternating bf16 / fp8 rounds per measurement")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--selfplay-games", type=int, default=4096)
    ap.add_argument("--no-selfplay", action="store_true")
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    from bench import load_peaks
    from cattus_b200 import CudaNetwork
    from cattus_b200.export import export_blob
    from cattus_b200.selfplay import SelfPlayRunner
    from oracle import net
    from tests.util import synth_inputs

    cfg = net.CONFIGS[args.net]
    blob = export_blob(net.make_state_dict(cfg, 0), cfg.game)
    peaks = load_peaks()
    res = {"net": args.net, "gpu_before": gpu_record(), "bf16_measured_tflops": peaks["bf16_tflops"], "bf16_measured_source": peaks["source"],
           "fp8_datasheet_tflops": FP8_DATASHEET_TFLOPS, "bf16_datasheet_tflops": BF16_DATASHEET_TFLOPS}
    words, bitmaps, _ = synth_inputs(args.net, 4 * 4096, 7)
    precs = ("bf16", "fp8")
    with CudaNetwork(blob, cfg.game, batch_size=4096, n_streams=4, precision="bf16") as nb, \
            CudaNetwork(blob, cfg.game, batch_size=4096, n_streams=4, precision="fp8") as n8:
        nws = {"bf16": nb, "fp8": n8}
        assert nb.trunk_path == n8.trunk_path == "fused"

        def alternate(fn):
            """fn(nw) -> list of samples; rounds of bf16 then fp8; returns the medians."""
            got = {p: [] for p in precs}
            for _ in range(args.rounds):
                for p in precs:
                    got[p] += list(fn(nws[p]))
            return {p: float(np.median(got[p])) for p in precs}

        # ---- trunk stage
        fl = trunk_flops(cfg)
        res["trunk"] = []
        for b in (1024, 2048, 4096):
            for p in precs:
                nws[p].resident_upload(words[:b], bitmaps[:b])
                nws[p].time_stage(1, b, 5)  # warm-up
            med = alternate(lambda nw: nw.time_stage(1, b, args.iters))
            row = {"batch": b}
            for p in precs:
                tf = fl * b / (med[p] * 1e-3) / 1e12
                row[p] = {"ms": med[p], "tflops": tf, "share_of_measured_bf16": tf / peaks["bf16_tflops"], "share_of_fp8_datasheet": tf / FP8_DATASHEET_TFLOPS}
            row["fp8_speedup"] = med["bf16"] / med["fp8"]
            res["trunk"].append(row)
            print(json.dumps({"trunk": row}), flush=True)

        # ---- whole graph, batch sweep
        res["graph_sweep"] = []
        for b in (1, 8, 64, 256, 1024, 4096):
            for p in precs:
                nws[p].resident_upload(words[:b], bitmaps[:b])
                nws[p].time_stage(4, b, 5)
            med = alternate(lambda nw: nw.time_stage(4, b, args.iters))
            row = {"batch": b, **{p: {"ms": med[p], "positions_per_sec": b / (med[p] * 1e-3)} for p in precs}, "fp8_speedup": med["bf16"] / med["fp8"]}
            res["graph_sweep"].append(row)
            print(json.dumps({"graph": row}), flush=True)

        # ---- device-resident evaluation, back to back (no flush)
        b, reps = 4096, 200

        def resident(nw):
            nw.resident_upload(words[:b], bitmaps[:b])
            nw.eval_resident(b)
            nw.resident_download(b)
            t0 = time.perf_counter()
            for _ in range(reps):
                nw.eval_resident(b)
            nw.resident_download(b)  # synchronises the device
            return [b * reps / (time.perf_counter() - t0)]

        med = alternate(resident)
        res["resident_evals_per_sec"] = {"batch": b, **med, "fp8_speedup": med["fp8"] / med["bf16"]}
        print(json.dumps({"resident": res["resident_evals_per_sec"]}), flush=True)

        # ---- time_sustained: 4 distinct batches of 4096 rotated, back to back
        for p in precs:
            nws[p].time_sustained(words, bitmaps, 4096, 4, 20)
        med = alternate(lambda nw: [4096 * 400 / (nw.time_sustained(words, bitmaps, 4096, 4, 400) * 1e-3)])
        res["sustained_positions_per_sec"] = {"batch": 4096, **med, "fp8_speedup": med["fp8"] / med["bf16"],
                                              "trunk_tflops_bound_from_positions": {p: fl * med[p] / 1e12 for p in precs}}
        print(json.dumps({"sustained": res["sustained_positions_per_sec"]}), flush=True)
        res["gpu_after_evaluator_legs"] = gpu_record()

    # ---- device-resident chess self-play, one precision at a time (each handle sized for the games in flight)
    if not args.no_selfplay and cfg.game == "chess":
        mc = {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[30, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
              "prior_noise_epsilon": 0.25, "cache_size": 1000000}
        dg = args.selfplay_games
        res["selfplay"] = {"sim_num": 600, "max_moves": 16, "device_games": dg}
        for p in ("bf16", "fp8", "bf16", "fp8"):  # two turns each; the second of each is reported, the first too
            with CudaNetwork(blob, cfg.game, batch_size=dg, n_streams=2, precision=p) as nw:
                SelfPlayRunner("chess", {"mcts": dict(mc, sim_num=16), "seed": 1, "max_moves": 2, "device_games": 64}).generate_data(nw, None, 64)
                s, _ = SelfPlayRunner("chess", {"mcts": mc, "seed": 1, "max_moves": 16, "device_games": dg}).generate_data(nw, None, dg)
            m = s["metrics"]
            run = {"sims_per_sec": m["selfplay.simulations"] / m["selfplay.seconds"], "seconds": m["selfplay.seconds"],
                   "waves": m["model.activation_count"], "ms_per_wave": 1e3 * m["selfplay.seconds"] / max(1, m["model.activation_count"])}
            res["selfplay"].setdefault(p, []).append(run)
            print(json.dumps({"selfplay": p, **run}), flush=True)
        res["gpu_after_selfplay"] = gpu_record()

    text = json.dumps(res, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")
    print(json.dumps({"summary": {"trunk_speedup": {r["batch"]: round(r["fp8_speedup"], 3) for r in res["trunk"]},
                                  "graph_speedup": {r["batch"]: round(r["fp8_speedup"], 3) for r in res["graph_sweep"]}}}), flush=True)


if __name__ == "__main__":
    main()
