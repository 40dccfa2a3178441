#!/usr/bin/env python
"""bench.py -- NN evals/s of the batched leaf-evaluation hot path (BASELINE.json metric) on N B200s.

One "step" = one pass of the hot path (encode -> conv trunk -> heads -> mask/softmax/tanh) over `positions_per_step`
synthetic positions (SURVEY.md section 8d generator, random-init ConvNetV1 weights of the named architecture).

  value     whole-job positions/s with the packed positions already resident in HBM, device time from CUDA events on
            the evaluator stream, L2 flushed (256 MiB memset) before every device batch, max over ranks.
  e2e       the same metric through the reference-facing C-ABI call `cattus_b200_eval_batch` with HOST buffers:
            pack into the pinned block, cudaMemcpyAsync H2D, graph, D2H of probabilities and values, every step.
  roofline  conv trunk (stem + residual blocks, the dense contraction) timed alone on the same stream:
            algorithmic FLOP (2*MAC, unpadded) / average duration vs the measured bf16 peak of MEASURED_PEAKS.json.
  cpu_baseline  the oracle's restatement of the reference's torch-py CPU engine on the box's host cores (rank 0, N=1).

`--dump-outputs DIR` writes what `value` and `e2e` returned in their last timed step.  Weights and positions are seeded, so
two builds run with the same arguments can be compared output for output.

`--impl reference` times that CPU path alone (the reference has no GPU code of its own and its Rust engines cannot be
built here: no cargo/rustc, no ONNX Runtime / tract / ExecuTorch wheels -- see DESIGN.md).

Multi-GPU: replicas only -- one process per GPU (torchrun), each with its own evaluator, queue and positions; no
collective on the data path (self-play games are independent).  torch.distributed is used for the barrier and the
max-over-ranks of the timings only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree this runs from may be read-only: the bench writes nothing there

WORKLOADS = {
    # name: (oracle config, device batch, device batches per step)
    "chess10x128": ("chess10x128", 4096, 4),
    "chess_dev": ("chess_dev", 4096, 4),
    # widths outside the two whole-trunk kernels (per-layer tensor-core path; cattus_b200_info.trunk_path says which)
    "chess_4x64": ("chess_4x64", 4096, 4),
    "chess_4x256": ("chess_4x256", 4096, 4),
    "chess20x256": ("chess20x256", 4096, 4),
    # 16-filter nets: a 4096-position batch is ONE round per CTA, so per-CTA setup and the 64-CTA FC launch are not
    # amortised; 16384 runs 4 rounds per CTA (hex5: 66.6 -> 93 M positions/s)
    "hex5": ("hex5", 16384, 4),
    "hex7": ("hex7", 16384, 4),
    "hex4": ("hex4", 16384, 4),
    "hex9": ("hex9", 16384, 4),
    "hex11": ("hex11", 8192, 4),
}
DEFAULT_WORKLOAD = "chess10x128"
CONFIG_NOTES = {
    "chess10x128": "BASELINE.json configs[3]: chess, random-init AlphaZero-style ResNet 10 blocks x 128 filters (heads 32/32), bf16; "
                   "the configuration the north star's tensor-core target is quoted on; fits one GPU",
    "hex5": "BASELINE.json configs[1]: hex 5x5, ConvNetV1 7x16 (heads 16/16) random-init (shipped model/hex5 is an LFS stub)",
    "hex7": "BASELINE.json configs[2]: hex 7x7, ConvNetV1 7x16 (heads 16/16) random-init",
    "hex4": "BASELINE.json configs[0]: hex 4x4, ConvNetV1 7x16 (heads 16/16) random-init",
    "chess_dev": "training/config/chess_dev.yaml: chess, ConvNetV1 7x16 (heads 8/8) random-init",
    "chess_4x64": "chess, ConvNetV1 4 x 64 (heads 8/8): a width training/config/chess_dev.yaml:30-37 recommends, outside the whole-trunk kernels",
    "chess_4x256": "chess, ConvNetV1 4 x 256 (heads 16/16): the widest net chess_dev.yaml:30-37 recommends, per-layer path",
    "chess20x256": "chess, ConvNetV1 20 x 256 (heads 32/32): the top of the range chess_dev.yaml:30-37 recommends, per-layer path",
    "hex9": "hex 9x9 (training/self-play/src/bin/hex9_self_player.rs), ConvNetV1 7x16 (heads 16/16) random-init",
    "hex11": "hex 11x11, the reference's standard board (engine/src/hex/core.rs:341), ConvNetV1 7x16 (heads 16/16) random-init",
}


def workload_config(workload: str, batch: int, per_step: int, cpu_sample: int) -> dict:
    """The `config` object BOTH arms print (identical by construction): what is evaluated, not how."""
    from oracle import net

    cfg_name, _, _ = WORKLOADS[workload]
    cfg = net.CONFIGS[cfg_name]
    return {"workload": workload, "note": CONFIG_NOTES.get(workload, ""), "net": cfg.to_dict(),
            "weights": "random-init (numpy PCG64 seed 0), BN folded", "positions": "synthetic (SURVEY.md section 8d generator)",
            "positions_per_step": {"cattus_b200": batch * per_step, "reference": cpu_sample,
                                   "why": "the reference arm times a bounded sample of the same workload on the host cores"},
            "device_batch": batch,
            "l2": "cattus_b200 arm: 256 MiB memset before every timed device batch (inputs are far smaller than L2); reference arm: CPU, n/a",
            "parallelism": "replicas, one evaluator per GPU, no collective on the data path"}


def cpu_sample_for(args, cfg) -> int:
    return args.cpu_sample or (256 if cfg.filters >= 64 else 2048)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock, power and throttle reasons DURING the timed regions (B200_PROFILING.md recipe: the fields of its nvidia-smi
    line).  Read through NVML in this process (what nvidia-smi itself calls; no start-up latency, which on an 8-GPU box was
    longer than the timed region) and ONLY while a measurement window is open: polling the driver all the time was measured
    to slow small kernels down (batch-1 graph 0.124 -> 0.148 ms with a 20 ms nvidia-smi loop running throughout).  Falls
    back to an nvidia-smi child process if NVML cannot be loaded."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.samples = []  # (monotonic time, sm MHz, max MHz, W, [reasons])
        self.active = False
        self.stopping = False
        self.t_open = 0.0
        self.nvml = None
        self.proc = None
        self.thread = None

    def start(self):
        if os.environ.get("CATTUS_B200_BENCH_NO_CLOCKS"):  # A/B knob: does reading the clocks change what is measured?
            return self
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.device]) if visible and all(v.strip().isdigit() for v in visible.split(",")) else self.device
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None
            try:  # the recipe's own command, sampled for the whole run at its 200 ms period
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.device)],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.thread = threading.Thread(target=self._read_smi, daemon=True)
                self.thread.start()
                t0 = time.monotonic()
                while not self.samples and time.monotonic() - t0 < 6.0:
                    time.sleep(0.02)
            except Exception:
                self.proc = None
        return self

    def _sample_nvml(self):
        n = self.nvml
        try:
            sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
            try:
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:
                mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            self.samples.append((time.monotonic(), sm, self.max_mhz, power, [k for k, bit in self.REASONS.items() if mask & bit]))
        except Exception:
            pass

    def _poll_nvml(self):
        while not self.stopping:
            if self.active:
                self._sample_nvml()
                # dense at the start of a window (short kernels loops), sparse in seconds-long legs
                time.sleep(0.01 if time.monotonic() - self.t_open < 0.5 else 0.2)
            else:
                time.sleep(0.002)

    def _read_smi(self):
        names = list(self.REASONS)
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                self.samples.append((time.monotonic(), float(f[1]), float(f[2]), float(f[3]),
                                     [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue

    def begin(self):
        """Opens a measurement window (NVML: sampling starts now)."""
        self.t_open = time.monotonic()
        self.active = True
        return self.t_open

    def end(self, t0: float = None) -> dict:
        """Closes the window opened at t0 (default: the last begin()) and summarises its samples: median SM clock, max power,
        union of the throttle reasons."""
        t1 = time.monotonic()
        if self.nvml is not None and self.active:
            self._sample_nvml()  # at least one sample inside even the shortest window
        self.active = False
        t0 = self.t_open if t0 is None else t0
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi / NVML unavailable"]}
        inside = [s for s in self.samples if t0 <= s[0] <= t1 + 0.03]
        note = None
        if not inside and self.samples:  # nvidia-smi fallback and a region shorter than its period
            mid = 0.5 * (t0 + t1)
            inside = [min(self.samples, key=lambda s: abs(s[0] - mid))]
            note = "region shorter than the sampling period: nearest sample"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "power_w_max": None, "samples": 0, "reasons": []}
        out = {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": max(s[2] for s in inside),
               "power_w_max": max(s[3] for s in inside), "samples": len(inside), "reasons": sorted({r for s in inside for r in s[4]}),
               "source": "NVML" if self.nvml is not None else "nvidia-smi -lms 200"}
        if note:
            out["note"] = note
        return out

    def close(self):
        self.stopping = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.proc = None


def make_inputs(cfg, n, seed):
    from oracle import games

    if cfg.game == "chess":
        return games.synth_chess_positions(n, seed)
    words, _ = games.synth_hex_positions(n, cfg.board_size, seed)
    return words, None


DUMP_BYTES = 60 << 20  # what --dump-outputs writes in all stays under 64 MB with the .npy headers


def dump_outputs(out_dir, outputs):
    """Writes each (probs, offsets, values) triple of `outputs` ({prefix: what eval_batch returns}) as
    out_dir/<prefix>_{probs,offsets,values,positions}.npy: probs and values float32, offsets and position indices float64
    (exact).  If all of it would exceed DUMP_BYTES, every triple is cut to the same share of its positions, a fixed seeded
    sample, and offsets index the sampled probabilities."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    total = sum(p.size * 4 + o.size * 8 + v.size * 4 + v.size * 8 for p, o, v in outputs.values())
    share = min(1.0, DUMP_BYTES / max(1, total))
    for prefix, (probs, offsets, values) in outputs.items():
        n = len(values)
        offsets = offsets.astype(np.int64)
        pos = np.arange(n)
        if share < 1.0:
            pos = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * share)), replace=False))
            probs = np.concatenate([probs[offsets[i]:offsets[i + 1]] for i in pos])
            offsets = np.concatenate([[0], np.cumsum(np.diff(offsets)[pos])])
        np.save(out_dir / f"{prefix}_probs.npy", np.asarray(probs, dtype=np.float32))
        np.save(out_dir / f"{prefix}_offsets.npy", offsets.astype(np.float64))
        np.save(out_dir / f"{prefix}_values.npy", np.asarray(values[pos], dtype=np.float32))
        np.save(out_dir / f"{prefix}_positions.npy", pos.astype(np.float64))


def cpu_reference_step(model, cfg, words, bitmaps, liboracle):
    """One pass of the reference's CPU path over a sample: planes_to_tensor (C restatement of net/mod.rs:121-156) ->
    torch-py engine restated (model.rs:68-84) -> clamp + calc_moves_probs (C restatement of net/mod.rs:57-61,106-119)."""
    import ctypes as C

    n = len(words)
    x = np.empty((n, cfg.planes, cfg.board_size, cfg.board_size), dtype=np.float32)
    w = np.ascontiguousarray(words, dtype=np.uint64)
    liboracle.oracle_planes_to_tensor(w.ctypes.data_as(C.c_void_p), n, n, cfg.planes, cfg.board_size, x.ctypes.data_as(C.c_void_p))
    logits, values = model.run(x)
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    if bitmaps is None:  # hex: legal = empty cells
        wpp = (cfg.board_size ** 2 + 63) // 64
        ww = w.reshape(n, cfg.planes, wpp)
        empty = ww[:, 2] & ~(ww[:, 0] | ww[:, 1])
        bm = np.ascontiguousarray(empty.view(np.uint8).reshape(n, wpp * 8))
    else:
        bm = np.ascontiguousarray(bitmaps, dtype=np.uint8)
    probs = np.empty(n * cfg.moves, dtype=np.float32)
    offsets = np.empty(n + 1, dtype=np.uint32)
    liboracle.oracle_policy_batch(logits.ctypes.data_as(C.c_void_p), n, cfg.moves, bm.ctypes.data_as(C.c_void_p), bm.shape[1],
                                  probs.ctypes.data_as(C.c_void_p), offsets.ctypes.data_as(C.c_void_p))
    return probs[: offsets[n]], values


def time_cpu_reference(cfg, sample_n, budget_s, steps=None, warmup=1, seed=1234):
    """Returns (positions/s, cores, description).  Bounded: `steps` passes if given, else as many as fit in budget_s."""
    import ctypes as C

    from oracle import net

    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle")], check=True)
    liboracle = C.CDLL(str(ROOT / "oracle" / "_build" / "liboracle.so"))
    cores = len(os.sched_getaffinity(0))
    sd = net.make_state_dict(cfg, 0)
    model = net.TorchCpuModel(sd, cfg, sample_n, cores)
    words, bitmaps = make_inputs(cfg, sample_n, seed)
    for _ in range(max(1, warmup)):
        cpu_reference_step(model, cfg, words, bitmaps, liboracle)
    done, t0 = 0, time.perf_counter()
    while True:
        cpu_reference_step(model, cfg, words, bitmaps, liboracle)
        done += 1
        el = time.perf_counter() - t0
        if (steps is not None and done >= steps) or (steps is None and el >= budget_s):
            break
    return done * sample_n / el, cores, el / done, f"{done} passes over {sample_n} positions, torch {cores} threads fp32 (reference torch-py engine restated) + C restatement of planes_to_tensor/calc_moves_probs"


def time_cpu_run_duration_batch1(cfg, calls=200, seed=4321):
    """model.run_duration of the reference's own bench (bench/inference_engine/main.py: batch_size 1, threads 1): median
    seconds of one torch-py Model::run on one position."""
    from oracle import games as og, net

    sd = net.make_state_dict(cfg, 0)
    model = net.TorchCpuModel(sd, cfg, 1, 1)
    words, _ = make_inputs(cfg, 8, seed)
    x = og.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    for i in range(10):
        model.run(x[i % 8:i % 8 + 1])
    t = np.empty(calls)
    for i in range(calls):
        t0 = time.perf_counter()
        model.run(x[i % 8:i % 8 + 1])
        t[i] = time.perf_counter() - t0
    return float(np.median(t))


SELFPLAY_CFG = {
    # training/config/hex5_cfg.yaml / hex7_cfg.yaml: engine.mcts with the self_play.engine_overrides applied
    "hex5": {"sim_num": 1400, "explore_factor": 1.41421, "temperature_policy": [[10, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
             "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    "hex7": {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[10, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
             "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    "hex9": {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[10, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
             "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    "hex11": {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[10, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
              "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    "hex4": {"sim_num": 100, "explore_factor": 1.41421, "temperature_policy": [[4, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
             "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    # training/config/chess_dev.yaml (engine.mcts + self_play.engine_overrides) on BASELINE config 4's 10 x 128 net and on the yaml's own net
    "chess10x128": {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[30, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
                    "prior_noise_epsilon": 0.25, "cache_size": 1000000},
    "chess_dev": {"sim_num": 600, "explore_factor": 1.41421, "temperature_policy": [[30, 1.0], [9999, 0.0]], "prior_noise_alpha": 0.03,
                  "prior_noise_epsilon": 0.25, "cache_size": 1000000},
}


def selfplay_max_moves(args, game: str) -> int:
    if args.selfplay_max_moves >= 0:
        return args.selfplay_max_moves
    return 16 if game.startswith("chess") else 0


def cpu_selfplay_max_moves(args, game: str) -> int:
    """The CPU arm's bounded sample: a chess 10 x 128 leaf costs ~10 ms on one core, so one 600-simulation search per game."""
    return 1 if game.startswith("chess") else selfplay_max_moves(args, game)


def runner_game(name: str) -> str:
    """SelfPlayRunner's game name for a net configuration name."""
    return "chess" if name.startswith("chess") else name


def selfplay_summary_to_dict(game, mcts_cfg, summary, games, threads, gpt, extra=None, max_moves=0):
    m = summary["metrics"]
    yaml = "chess_dev.yaml" if game.startswith("chess") else f"{game}_cfg.yaml"
    d = {"metric": "selfplay_sims_per_sec", "unit": "sims/s", "workload": f"{game} self-play, sim_num {mcts_cfg['sim_num']}, noise + temperature as "
         f"training/config/{yaml}" + (f", games stopped after {max_moves} moves" if max_moves else ""), "games": games, "threads": threads, "games_per_thread": gpt, "simulations": m["selfplay.simulations"],
         "seconds": m["selfplay.seconds"], "evaluations": m["selfplay.evaluations"], "evaluator_calls": m["model.activation_count"],
         "mean_batch": m["selfplay.evaluations"] / max(1, m["model.activation_count"]),
         "cache_hit_rate": m["cache.hits"] / max(1, m["cache.hits"] + m["cache.misses"]),
         "eval_wait_frac": m["selfplay.eval_wait_seconds"] / max(1e-9, m["selfplay.seconds"] * threads),
         "player1_wins": summary["player1_wins"], "player2_wins": summary["player2_wins"], "draws": summary["draws"]}
    if extra:
        d.update(extra)
    return d


def time_cpu_selfplay(game, games, threads, max_moves=0):
    """The reference's arrangement on the host cores: `threads` OS threads with one tree each (hex5_cfg.yaml: threads 8),
    per-leaf evaluation by the reference's torch-py CPU engine restated (model.rs:68-84; calls are serialised like its
    Mutex<Model>), same MCTS parameters.  Bounded sample: `games` games."""
    from cattus_b200.selfplay import SelfPlayRunner
    from oracle import games as og, net

    cfg = net.CONFIGS[game]
    sd = net.make_state_dict(cfg, 0)
    cores = len(os.sched_getaffinity(0))
    model = net.TorchCpuModel(sd, cfg, 1, 1)  # batch-1 evaluations of a 70 k-parameter net: one intra-op thread is the fastest setting
    s = cfg.board_size

    def cb(words, n, bitmaps=None):
        x = og.planes_to_tensor_fast(words, s, cfg.planes)
        probs, values = [], []
        for i in range(n):
            logits, v = model.run(x[i:i + 1])
            if bitmaps is not None:  # chess: the legal moves come as a bitmap over the nn indices
                legal = og.legal_from_bitmap(bitmaps[i], cfg.moves)
            else:
                ww = words[i].reshape(cfg.planes, -1)
                legal = [k for k in range(s * s) if not ((int(ww[0][k >> 6]) | int(ww[1][k >> 6])) >> (k & 63)) & 1]
            probs.append(og.calc_moves_probs(legal, og.clamp_non_finite(np.asarray(logits[0], dtype=np.float32))))
            values.append(float(np.asarray(v).reshape(-1)[0]))
        return probs, values

    mc = SELFPLAY_CFG[game]
    runner = SelfPlayRunner(runner_game(game), {"mcts": mc, "threads": threads, "games_per_thread": 1, "seed": 1, "max_moves": max_moves})
    summary, _ = runner.run_with(cb, None, games)
    return selfplay_summary_to_dict(game, mc, summary, games, threads, 1, max_moves=max_moves, extra={
        "value": summary["metrics"]["selfplay.sims_per_sec"], "cores": cores, "kind": "port",
        "sample": f"repo driver + CPU evaluator: {games} games, {threads} threads x 1 tree each, one leaf at a time (the reference's thread "
                  f"arrangement; its Mutex<Model> serialises evaluations, so more threads add nothing), per-leaf torch-CPU fp32 evaluation "
                  f"with 1 intra-op thread"})


def cpu_batch_sweep(cfg, batches=(1, 8, 64, 256, 1024), seconds_each=1.2, seed=99):
    """BASELINE.md section 4: the CPU path at the batch sizes the shipped configs use and beyond (bounded: ~1 s per point)."""
    import ctypes as C

    from oracle import net

    liboracle = C.CDLL(str(ROOT / "oracle" / "_build" / "liboracle.so"))
    cores = len(os.sched_getaffinity(0))
    sd = net.make_state_dict(cfg, 0)
    out = []
    for b in batches:
        model = net.TorchCpuModel(sd, cfg, b, 1 if b == 1 else cores)
        words, bitmaps = make_inputs(cfg, b, seed)
        cpu_reference_step(model, cfg, words, bitmaps, liboracle)
        done, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds_each:
            cpu_reference_step(model, cfg, words, bitmaps, liboracle)
            done += 1
        el = time.perf_counter() - t0
        out.append({"batch": b, "ms": el / done * 1e3, "positions_per_sec": done * b / el, "threads": 1 if b == 1 else cores})
    return out


def run_reference_arm(args, rank, world):
    """The reference's CPU inference path on the host cores.  Nothing of the repo's library is loaded into this process:
    the headline uses torch + oracle/ only, and the self-play legs (which need a search driver around the CPU evaluator) run
    in a child process (`--impl reference-selfplay`)."""
    from oracle import net

    if rank != 0:
        return
    cfg_name, batch, per_step = WORKLOADS[args.workload]
    if args.batch:
        batch = args.batch
    cfg = net.CONFIGS[cfg_name]
    sample_n = cpu_sample_for(args, cfg)
    value, cores, sec_per_step, desc = time_cpu_reference(cfg, sample_n, budget_s=0, steps=max(1, args.steps), warmup=max(1, args.warmup))
    line = {
        "impl": "reference", "metric": "nn_evals_per_sec", "value": value, "unit": "positions/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, batch, per_step, sample_n),
        "reference": "CPU inference path of the reference (host cores only; the reference has no GPU kernels): torch-py engine restated "
                     "(engine/src/net/model.rs:68-84) + C restatement of planes_to_tensor / calc_moves_probs",
        "cpu_baseline": {"value": value, "unit": "positions/s", "cores": cores, "kind": "port", "sample": desc,
                         "model_run_duration_batch1_us": time_cpu_run_duration_batch1(cfg) * 1e6},
        "e2e": {"value": value, "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    line["batch_sweep"] = cpu_batch_sweep(cfg)
    if args.workload == DEFAULT_WORKLOAD and not args.no_other_workloads:
        # BASELINE configs[0]: hex 4x4 on the current CPU inference backend ("runs today on CPU")
        hcfg = net.CONFIGS["hex4"]
        hv, hcores, _, hdesc = time_cpu_reference(hcfg, 2048, budget_s=2.0)
        line["other_workloads"] = [{"workload": "hex4", "note": CONFIG_NOTES["hex4"], "value": hv, "unit": "positions/s", "cores": hcores, "sample": hdesc}]
    if not args.no_selfplay:
        cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference-selfplay", "--selfplay-game", *args.selfplay_game,
               "--selfplay-max-moves", str(args.selfplay_max_moves)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        legs = None
        for ln in res.stdout.splitlines():
            if ln.startswith("{"):
                legs = json.loads(ln)["legs"]
        if legs:
            line["selfplay"] = legs[0]
            line["selfplay_others"] = legs[1:]
        else:
            line["selfplay"] = {"unavailable": (res.stderr or "no output")[-400:]}
    print(json.dumps(line), flush=True)


def run_reference_selfplay(args):
    """Child process of the reference arm: the repo's search driver bound to the reference's CPU evaluator (one tree per OS
    thread, one leaf at a time -- the reference's arrangement).  This is 'repo driver + CPU evaluator', the closest runnable
    stand-in for the reference's Rust self-play executable (no cargo here)."""
    legs = [time_cpu_selfplay(g, 2, 2, cpu_selfplay_max_moves(args, g)) for g in args.selfplay_game]
    print(json.dumps({"legs": legs}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cattus_b200", choices=["cattus_b200", "reference", "reference-selfplay"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="device batch (positions per launch sequence); default per workload")
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline work (rank 0, N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the self-play sims/s leg")
    ap.add_argument("--no-other-workloads", action="store_true", help="skip the brief hex5 evals/s leg of the default run")
    ap.add_argument("--selfplay-game", nargs="+", default=["hex5", "hex7", "chess10x128"], choices=sorted(SELFPLAY_CFG),
                    help="self-play legs: the first is reported as `selfplay` (BASELINE configs[1]), the rest under `selfplay_others` "
                         "(configs[2] hex7, configs[3] chess 10x128)")
    ap.add_argument("--device-games", type=int, default=0,
                    help="concurrent device-resident games per GPU in a self-play leg (0 = 16384 for the 16-filter nets, 4096 for chess 10x128)")
    ap.add_argument("--no-host-driver", action="store_true", help="skip the host-tree driver's sims/s (kept beside the device-resident number)")
    ap.add_argument("--sustained-seconds", type=float, default=2.2, help="length of the sustained leg (0 = skip)")
    ap.add_argument("--selfplay-games", type=int, default=0, help="games per GPU in a self-play leg (0 = 8192; chess: one wave, threads x games per thread)")
    ap.add_argument("--selfplay-threads", type=int, default=0, help="worker threads per GPU (0 = host cores / GPUs)")
    ap.add_argument("--selfplay-gpt", type=int, default=0, help="concurrent games per worker thread (0 = 512; chess 1024)")
    ap.add_argument("--selfplay-groups", type=int, default=2, help="slot groups per worker thread (one batch in flight per group)")
    ap.add_argument("--selfplay-max-moves", type=int, default=-1,
                    help="stop self-play games after this many moves (0 = play to the end as the reference does; default: 0 for hex, 16 for chess, "
                         "whose random-net games run for hundreds of moves)")
    ap.add_argument("--no-single-search", dest="single_search", action="store_false",
                    help="skip the one-tree search at sim_num 10000 (BASELINE configs[4]) that each self-play leg adds")
    ap.add_argument("--single-search", action="store_true", default=True,
                    help="also time ONE tree searching with --sim-num 10000 (BASELINE configs[4]'s UCI setting, on the self-play game): "
                         "two games, one thread, one leaf at a time through cattus_b200_eval")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed paths returned in their last step (rank 0): resident_* from the device-resident "
                         "batch of `value`, e2e_* from the host-buffer call of `e2e`, as DIR/<name>.npy (float32 / float64, < 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cattus_b200":
        ap.error("--dump-outputs applies to --impl cattus_b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.impl == "reference-selfplay":
        run_reference_selfplay(args)
        return
    args.warmup = max(args.warmup, 3)

    import torch

    from cattus_b200 import CudaNetwork
    from cattus_b200.export import export_blob
    from oracle import net  # only for NetConfig / the seeded weight + position generators and the cpu_baseline leg

    from cattus_b200 import replicas

    rep = replicas.init_from_env("nccl")

    def barrier():
        rep.barrier()
        torch.cuda.synchronize(local_rank)

    max_over_ranks = rep.max_over_ranks

    cfg_name, batch, per_step = WORKLOADS[args.workload]
    if args.batch:
        batch = args.batch
    cfg = net.CONFIGS[cfg_name]
    peaks = load_peaks()
    sd = net.make_state_dict(cfg, 0)
    nw = CudaNetwork(export_blob(sd, cfg.game), cfg.game, device=local_rank, batch_size=batch, n_streams=args.streams, precision="bf16")
    positions_per_step = batch * per_step
    words, bitmaps = make_inputs(cfg, positions_per_step, seed=replicas.rank_seed(0xCA7705, rank))

    # ---------------- batch-size sweep (BASELINE configs[4]): whole graph, inputs resident, L2 flushed, CUDA events.  The small-batch
    # and per-leaf latencies are taken FIRST, at the clocks an idle GPU boosts to: after the long full-batch loops below the
    # GPU sits in its power-capped state (1.6-1.7 GHz) for a while, which is not what a single UCI search sees.
    sweep = []
    if rank == 0:
        for nb in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192):  # every power of two (BASELINE configs[4]: 1-4096)
            if nb >= batch:
                continue
            nw.resident_upload(words[:nb], None if bitmaps is None else bitmaps[:nb])
            nw.time_stage(4, nb, 3)
            ms = float(np.mean(nw.time_stage(4, nb, 10)))
            sweep.append({"batch": nb, "ms": ms, "positions_per_sec": nb / (ms * 1e-3)})
    # ---------------- per-leaf latency: one blocking cattus_b200_eval at a time (what a single-tree UCI search sees;
    # BASELINE configs[4], `--sim-num 10000`: NN part of one search = 10000 x this)
    leaf = None
    if rank == 0 and world == 1:
        k = min(2000, positions_per_step)
        for i in range(50):
            nw.eval_planes(words[i], None if bitmaps is None else bitmaps[i])
        lat = np.empty(k)
        for i in range(k):
            t0 = time.perf_counter()
            nw.eval_planes(words[i], None if bitmaps is None else bitmaps[i])
            lat[i] = time.perf_counter() - t0
        leaf = {"api": "cattus_b200_eval (one blocking leaf at a time, host buffers)", "calls": int(k), "median_us": float(np.median(lat) * 1e6),
                # the score of the reference's own bench (bench/inference_engine/main.py:103: summary["metrics"]["model.run_duration"],
                # RunningAverage(0.99) of the seconds around one Model::run at batch_size 1)
                "model_run_duration_us": float(nw.metrics()["model.run_duration"] * 1e6),
                "p90_us": float(np.percentile(lat, 90) * 1e6), "evals_per_sec": float(k / lat.sum()),
                "nn_seconds_per_10000_sim_search": float(np.median(lat) * 10000)}
    # ---------------- device-resident throughput (value) and the trunk roofline
    nw.resident_upload(words[:batch], None if bitmaps is None else bitmaps[:batch])
    nw.time_stage(4, batch, args.warmup * per_step)
    sampler = ClockSampler(local_rank).start()  # runs for the whole process; every measurement reads its own window
    launches0 = nw.metrics()["model.kernel_launches"]
    barrier()
    sampler.begin()
    ms_all = nw.time_stage(4, batch, args.steps * per_step)
    barrier()
    clocks = sampler.end()
    t_value = max_over_ranks(float(ms_all.sum()) * 1e-3)
    dumped = {}
    if args.dump_outputs and rank == 0:
        dumped["resident"] = nw.resident_download(batch)
    if rank == 0:
        sweep.append({"batch": batch, "ms": float(np.mean(ms_all)), "positions_per_sec": batch / (float(np.mean(ms_all)) * 1e-3)})

    def timed_with_clocks(fn):
        """One clock record per measurement: the power-cap state drifts between loops."""
        t0 = sampler.begin()
        out = fn()
        c = sampler.end(t0)
        return out, {"sm_mhz": c.get("sm_mhz"), "power_w_max": c.get("power_w_max"), "samples": c.get("samples"), "reasons": c.get("reasons")}

    stage_iters = max(40, 2 * args.steps)  # tens of milliseconds per stage measurement: a stable mean and a few clock samples per window
    # the stages of ONE pass (no L2 flush between them, as inside the graph): they must add up to the graph
    nw.time_stage(5, batch, 3)
    ms_split, clocks_split = timed_with_clocks(lambda: nw.time_stage(5, batch, stage_iters))
    # the trunk stage alone, L2 flushed (the roofline's kernel), at the north star's batch sizes
    trunk_alone = {}
    for nb in sorted({b_ for b_ in (1024, 2048, 4096, batch) if b_ <= batch}):
        nw.resident_upload(words[:nb], None if bitmaps is None else bitmaps[:nb])
        nw.time_stage(1, nb, 8)
        ms_nb, c_nb = timed_with_clocks(lambda nb=nb: nw.time_stage(1, nb, stage_iters))
        trunk_alone[nb] = (float(np.mean(ms_nb)), c_nb)
    nw.resident_upload(words[:batch], None if bitmaps is None else bitmaps[:batch])
    barrier()

    # ---------------- end to end through the C ABI with host buffers
    for _ in range(args.warmup):
        nw.eval_batch(words, bitmaps)
    barrier()
    t_e2e0 = sampler.begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        probs, offsets, values = nw.eval_batch(words, bitmaps)
    torch.cuda.synchronize(local_rank)
    t_e2e_local = time.perf_counter() - t0
    barrier()
    clocks_e2e = sampler.end(t_e2e0)
    t_e2e = max_over_ranks(t_e2e_local)
    if args.dump_outputs and rank == 0:
        dumped["e2e"] = (probs, offsets, values)
        dump_outputs(args.dump_outputs, dumped)
    launches = nw.metrics()["model.kernel_launches"] - launches0
    # per position: 8-byte prefix (probability offset, #legal) + packed planes (+ the legal bitmap padded to 8 B for chess)
    rec_bytes = 8 + cfg.planes * ((cfg.board_size ** 2 + 63) // 64) * 8 + (((cfg.moves + 31) // 32 * 4 + 7) // 8 * 8 if bitmaps is not None else 0)
    h2d = positions_per_step * rec_bytes + 16 * per_step
    d2h = int(offsets[-1]) * 4 + positions_per_step * 4
    kernels_per_batch = nw.info.kernels_per_batch
    fused, small, trunk_path = nw.fused_trunk, nw.small_trunk, nw.trunk_path
    # ---------------- sustained: >= 2 s of device batches back to back, rotating over 4 distinct resident batches (no L2 flush
    # needed).  LAST of the evaluator legs: it leaves the GPU in its 1 kW power-capped clock state for a while, which would
    # otherwise colour the latency measurements above.
    sustained = None
    if args.sustained_seconds > 0 and args.streams >= 4 and per_step >= 4:
        iters = max(50, int(args.sustained_seconds / (float(np.mean(ms_all)) * 1e-3)))
        nw.time_sustained(words, bitmaps, batch, 4, 20)
        barrier()
        ms_sus, clocks_sus = timed_with_clocks(lambda: nw.time_sustained(words, bitmaps, batch, 4, iters))
        barrier()
        sustained = {"device_batches": iters, "distinct_resident_batches": 4, "seconds": ms_sus * 1e-3, "ms_per_device_batch": ms_sus / iters,
                     "positions_per_sec": world * iters * batch / (max_over_ranks(ms_sus * 1e-3)), "clocks": clocks_sus}
    barrier()
    nw.close()

    # ---------------- HBM-bound kernels (north star: "achieved HBM GB/s for encode and softmax against B200 peak").
    # On the production path both are fused away (encode into the trunk kernels, mask/softmax into the policy FC
    # epilogue), so the standalone kernels of the unfused comparison path (flags bit 0) are timed here as evidence.
    hbm_kernels = []
    if rank == 0 and world == 1 and not args.no_other_workloads:
        # at a size where the launch latency does not dominate (round 1 timed 4096 positions: 21 us of which ~5 us are launch)
        hb = min(65536, 16 * batch)
        hwords = np.concatenate([words] * (hb // len(words) + 1))[:hb]
        hbitmaps = None if bitmaps is None else np.concatenate([bitmaps] * (hb // len(bitmaps) + 1))[:hb]
        with CudaNetwork(export_blob(sd, cfg.game), cfg.game, device=local_rank, batch_size=hb, n_streams=1, precision="bf16", fused_trunk=False) as unf:
            unf.resident_upload(hwords, hbitmaps)
            for st in (0, 3):
                unf.time_stage(st, hb, 3)
            t_enc = float(np.mean(unf.time_stage(0, hb, 10))) * 1e-3
            t_tail = float(np.mean(unf.time_stage(3, hb, 10))) * 1e-3
        s2 = cfg.board_size ** 2
        wpp = (s2 + 63) // 64
        enc_alg = cfg.planes * wpp * 8 + cfg.planes * s2 * 2           # packed planes in + unpadded bf16 activations out (SURVEY 8d)
        enc_act = cfg.planes * wpp * 8 + s2 * 64 * 2                   # what the kernel really writes: channels padded to 64
        legal_mean = float(offsets[-1]) / positions_per_step
        tail_alg = 2 * 4 * cfg.moves + (cfg.moves + 7) // 8 + 512       # logits read (twice counted in SURVEY 8d) + mask + value hidden row
        for name_k, t_k, alg, act in (("encode_nhwc_bf16_kernel", t_enc, enc_alg, enc_act),
                                      ("value_tail_kernel + policy_tail_kernel", t_tail, tail_alg, 4 * cfg.moves + (cfg.moves + 7) // 8 + 512 + 4 * legal_mean)):
            hbm_kernels.append({"kernel": name_k, "bound": "hbm", "ms": t_k * 1e3, "positions_per_launch": hb, "algorithmic_bytes_per_position": alg,
                                "actual_bytes_per_position": act, "achieved": hb * alg / t_k / 1e9, "achieved_actual": hb * act / t_k / 1e9,
                                "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hb * alg / t_k / 1e9 / peaks["hbm_gbs"],
                                "frac_actual": hb * act / t_k / 1e9 / peaks["hbm_gbs"],
                                "note": "unfused comparison path (flags bit 0); fused away on the production path"})

    # ---------------- the other single-GPU configuration of BASELINE.json (configs[1], hex5) in the same line, briefly
    others = []
    if args.workload == DEFAULT_WORKLOAD and not args.no_other_workloads:
        for oname in ("hex5",):
            ocfg_name, obatch, oper = WORKLOADS[oname]
            ocfg = net.CONFIGS[ocfg_name]
            owords, _ = make_inputs(ocfg, obatch * oper, seed=replicas.rank_seed(0xCA7705, rank))
            with CudaNetwork(export_blob(net.make_state_dict(ocfg, 0), ocfg.game), ocfg.game, device=local_rank, batch_size=obatch, n_streams=args.streams,
                             precision="bf16") as onw:
                onw.resident_upload(owords[:obatch])
                onw.time_stage(4, obatch, 3)
                barrier()
                oms = onw.time_stage(4, obatch, 3 * oper)
                barrier()
                ot = max_over_ranks(float(oms.sum()) * 1e-3)
                for _ in range(2):
                    onw.eval_batch(owords)
                barrier()
                t0 = time.perf_counter()
                for _ in range(3):
                    onw.eval_batch(owords)
                ote = max_over_ranks(time.perf_counter() - t0)
                barrier()
                olaunches = 3 * oper * onw.info.kernels_per_batch + 5 * oper * onw.info.kernels_per_batch
            others.append({"workload": oname, "note": CONFIG_NOTES[oname], "device_batch": obatch, "value": world * 3 * oper * obatch / ot,
                           "e2e": world * 3 * oper * obatch / ote, "unit": "positions/s", "ms_per_device_batch": float(np.mean(oms)),
                           "gpu_launches": int(olaunches)})

    # ---------------- self-play MCTS sims/s (second half of the BASELINE metric).  Headline arrangement: DEVICE-RESIDENT search
    # (trees in HBM, one warp per game, leaves written straight into the evaluator's device batch; csrc/dsearch_core.hpp) --
    # the host only acts once per move, so sims/s no longer depends on the host cores per GPU.  The host-tree driver's
    # number on the same evaluator is kept beside it.
    selfplay_legs = []
    for sp_game in ([] if args.no_selfplay else args.selfplay_game):
        from cattus_b200.selfplay import SelfPlayRunner

        sp_cfg = net.CONFIGS[sp_game]
        cores = len(os.sched_getaffinity(0))
        chess_sp = sp_cfg.game == "chess"
        mc = SELFPLAY_CFG[sp_game]
        sp_max_moves = selfplay_max_moves(args, sp_game)
        sp_blob = export_blob(net.make_state_dict(sp_cfg, 0), sp_cfg.game)
        dg = args.device_games or (4096 if sp_cfg.filters >= 64 else 16384)
        games_total = max(2, (args.selfplay_games or dg) * world // 2 * 2)
        with CudaNetwork(sp_blob, sp_cfg.game, device=local_rank, batch_size=dg, n_streams=2, precision="bf16") as sp_nw:  # two lanes: two slot populations take waves in turn
            runner = SelfPlayRunner(runner_game(sp_game), {"mcts": mc, "seed": 1, "max_moves": sp_max_moves, "device_games": dg})
            SelfPlayRunner(runner_game(sp_game), {"mcts": dict(mc, sim_num=16), "seed": 1, "max_moves": 2, "device_games": 64}).generate_data(
                sp_nw, None, 64 * world, first_game=rank, game_stride=world)  # warm-up: the evaluator's launch sequence, the allocator
            l0 = sp_nw.metrics()["model.kernel_launches"]
            barrier()
            t_sp0 = sampler.begin()
            summary, _ = runner.generate_data(sp_nw, None, games_total, first_game=rank, game_stride=world)
            sp_clocks = sampler.end(t_sp0)
            barrier()
            sp_launches = sp_nw.metrics()["model.kernel_launches"] - l0
        m = summary["metrics"]
        sims_all = rep.sum_over_ranks(float(m["selfplay.simulations"]))
        secs = max_over_ranks(float(m["selfplay.seconds"]))
        selfplay = selfplay_summary_to_dict(sp_game, mc, summary, games_total, 1, dg, max_moves=sp_max_moves, extra={
            "value": sims_all / secs, "n_gpus": world, "host_cores": cores, "gpu_launches": int(sp_launches),
            "arrangement": "device-resident search: trees in HBM, one warp per game, one host thread per GPU acting once per move",
            "device_games": dg, "clocks": sp_clocks, "waves": m["model.activation_count"], "ms_per_wave": 1e3 * m["selfplay.seconds"] / max(1, m["model.activation_count"]),
            "note": "rank 0's counters shown; value = simulations of all ranks / max seconds (the whole call: allocation, all games to their end "
                    "incl. the tail where finished games leave slots empty); games partitioned by index across GPUs, no collective"})
        del selfplay["threads"], selfplay["games_per_thread"], selfplay["eval_wait_frac"], selfplay["cache_hit_rate"]
        if not args.no_host_driver:
            # the host-tree driver (round 1's arrangement) on the same evaluator: bound by the host cores per GPU
            threads = args.selfplay_threads or max(1, cores // max(1, world))
            gpt = args.selfplay_gpt or (1024 if chess_sp else 512)
            h_games = max(2, (threads * gpt if chess_sp else min(8192, threads * gpt)) * world // 2 * 2)
            h_max_moves = sp_max_moves  # the same games as the device-resident leg (the host cache's hit rate depends on how far games go)
            with CudaNetwork(sp_blob, sp_cfg.game, device=local_rank, batch_size=max(64, min(4096, gpt)),
                             n_streams=max(4, min(32, threads * args.selfplay_groups)), precision="bf16") as h_nw:
                h_runner = SelfPlayRunner(runner_game(sp_game), {"mcts": mc, "threads": threads, "games_per_thread": gpt,
                                                                 "groups_per_thread": args.selfplay_groups, "seed": 1, "max_moves": h_max_moves})
                h_runner.generate_data(h_nw, None, 2 * threads, first_game=rank, game_stride=world)
                hl0 = h_nw.metrics()["model.kernel_launches"]
                barrier()
                h_sum, _ = h_runner.generate_data(h_nw, None, h_games, first_game=rank, game_stride=world)
                barrier()
                selfplay["gpu_launches"] += int(h_nw.metrics()["model.kernel_launches"] - hl0)
            hm = h_sum["metrics"]
            selfplay["host_driver"] = selfplay_summary_to_dict(sp_game, mc, h_sum, h_games, threads, gpt, max_moves=h_max_moves, extra={
                "value": rep.sum_over_ranks(float(hm["selfplay.simulations"])) / max_over_ranks(float(hm["selfplay.seconds"])),
                "arrangement": "trees on the host: worker threads x games per thread, batched leaves (csrc/selfplay.cpp)", "host_cores": cores})
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            selfplay["cpu_baseline"] = time_cpu_selfplay(sp_game, 2, 2, cpu_selfplay_max_moves(args, sp_game))
        extras = rank == 0 and world == 1 and sp_game in (args.selfplay_game[0], "chess10x128")  # once per game family, at N = 1 only
        if extras:
            # The job the trainer actually submits (self_play.games_num 100, engine.threads 8 in the shipped configs): a dozen
            # leaves in flight per worker, so the device batches are nearly empty -- with and without speculative rows.
            with CudaNetwork(export_blob(net.make_state_dict(sp_cfg, 0), sp_cfg.game), sp_cfg.game, device=local_rank, batch_size=256, n_streams=16,
                             precision="bf16") as tr_nw:
                trainer = []
                for speculate in (0, 14):
                    tr_runner = SelfPlayRunner(runner_game(sp_game), {"mcts": mc, "threads": 8, "games_per_thread": 64, "seed": 1, "groups_per_thread": 2,
                                                                     "max_moves": sp_max_moves, "speculate": speculate})
                    tr_runner.generate_data(tr_nw, None, 16)  # warm-up: graphs of the small buckets
                    tr_sum, _ = tr_runner.generate_data(tr_nw, None, 100)
                    tm = tr_sum["metrics"]
                    trainer.append({"speculate": speculate, "sims_per_sec": tm["selfplay.sims_per_sec"], "seconds": tm["selfplay.seconds"],
                                    "evaluator_calls": tm["model.activation_count"], "evaluations": tm["selfplay.evaluations"],
                                    "speculative_evaluations": tm["selfplay.speculative_evaluations"],
                                    "outcome": [tr_sum["player1_wins"], tr_sum["player2_wins"], tr_sum["draws"]]})
                assert trainer[0]["outcome"] == trainer[1]["outcome"], "speculation changed game outcomes"
                selfplay["trainer_sized_job"] = {"games": 100, "threads": 8, "runs": trainer,
                                                 "note": "100 games over 8 worker threads (2 slot groups each) as the shipped training configs ask for; speculate = rows per game "
                                                         "evaluated ahead into the cache in the otherwise nearly empty device batches (same games)"}
        if extras and args.single_search:
            with CudaNetwork(export_blob(net.make_state_dict(sp_cfg, 0), sp_cfg.game), sp_cfg.game, device=local_rank, batch_size=64, n_streams=1,
                             precision="bf16") as ss_nw:
                ss_mc = dict(mc, sim_num=10000)
                if sp_cfg.game == "chess":
                    # BASELINE config 5: the UCI loop's `position` + `go` (cattus_b200/uci.py), a new player per position
                    from cattus_b200.selfplay import ChessSearch

                    per = []
                    for speculate in (0, 31):
                        for fen in (None, "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq -"):
                            with ChessSearch({"mcts": ss_mc, "seed": 1, "speculate": speculate}, model=ss_nw) as search:
                                best, st = search.go(fen, [])
                            per.append({"position": fen or "startpos", "speculate": speculate, "bestmove": best, "seconds": st["seconds"],
                                        "evaluations": st["evaluations"], "speculative_evaluations": st["speculative_evaluations"],
                                        "cache_hits": st["cache_hits"], "sims_per_sec": st["simulations"] / st["seconds"]})
                    assert all(a["bestmove"] == b["bestmove"] for a, b in zip(per[:2], per[2:])), "speculation changed a search result"
                    selfplay["single_search"] = {"sim_num": 10000, "searches": per,
                                                 "seconds_per_search": float(np.mean([p["seconds"] for p in per if p["speculate"] == 0])),
                                                 "seconds_per_search_speculating": float(np.mean([p["seconds"] for p in per if p["speculate"]])),
                                                 "note": "UCI `go` at sim_num 10000: one tree, one leaf in flight (the reference's arrangement); speculate = 31 lets "
                                                         "up to 31 likely next leaves ride in the same evaluator call into the cache (same moves, fewer round "
                                                         "trips); cache hits without speculation are transpositions inside the one search"}
                else:
                    per = {}
                    for speculate in (0, 31):
                        ss_sum, ss_rec = SelfPlayRunner(sp_game, {"mcts": ss_mc, "threads": 1, "games_per_thread": 1, "leaf_queue": 1, "seed": 1,
                                                                  "speculate": speculate}).generate_data(ss_nw, None, 2, keep_records=True)
                        per[speculate] = (ss_sum["metrics"], [r.moves for r in ss_rec])
                    assert per[0][1] == per[31][1], "speculation changed a game"
                    sm, sm_spec = per[0][0], per[31][0]
                    selfplay["single_search"] = {"sim_num": 10000, "searches": sm["selfplay.searches"],
                                                 "seconds_per_search": sm["selfplay.seconds"] / max(1, sm["selfplay.searches"]),
                                                 "seconds_per_search_speculating": sm_spec["selfplay.seconds"] / max(1, sm_spec["selfplay.searches"]),
                                                 "sims_per_sec": sm["selfplay.sims_per_sec"], "evaluations": sm["selfplay.evaluations"],
                                                 "evaluator_calls": sm["model.activation_count"], "evaluator_calls_speculating": sm_spec["model.activation_count"],
                                                 "note": "two whole games of one tree, one leaf in flight (the reference's UCI arrangement), per-leaf "
                                                         "cattus_b200_eval; speculating: up to 31 likely next leaves ride along into the cache (same games)"}
        selfplay_legs.append(selfplay)
    selfplay = selfplay_legs[0] if selfplay_legs else None

    total_positions = world * positions_per_step * args.steps
    value = total_positions / t_value
    e2e_value = total_positions / t_e2e
    s2 = cfg.board_size ** 2
    stem_flops = 2 * 9 * cfg.planes * cfg.filters * s2
    trunk_flops = stem_flops + cfg.trunk_flops_per_position
    t_trunk, clocks_trunk = trunk_alone[batch][0] * 1e-3, trunk_alone[batch][1]
    achieved = batch * trunk_flops / t_trunk / 1e12
    traffic = None
    try:  # DRAM bytes of the same kernel from the committed `ncu --set full` capture (per launch, same workload and batch)
        tj = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        kname = "trunk_fused_kernel" if fused else "trunk_small_kernel" if small else ""
        te = tj.get(f"{kname}@{args.workload}") or tj.get(kname)
        if te and te["workload"] == args.workload and te["positions_per_launch"] == batch:
            traffic = {"bytes": te["dram_bytes_read"] + te["dram_bytes_write"], "dram_bytes_read": te["dram_bytes_read"],
                       "dram_bytes_write": te["dram_bytes_write"], "source": te["source"]}
    except Exception:
        traffic = None
    split = np.mean(ms_split, axis=0)
    split_sum, all_graph = float(split.sum()), float(np.mean(ms_all))
    rel = abs(split_sum - all_graph) / all_graph
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
                "traffic": traffic, "kernel": (f"trunk_fused_kernel<{cfg.filters}> (encode + stem + residual blocks + head convs, one launch)" if fused else
                           "trunk_small_kernel (encode + stem + residual blocks + head convs, one launch)" if small else
                           "tc_gemm_kernel x (1 + 2R) conv layers (stem + residual blocks)"),
                "trunk_path": trunk_path,
                "peak_source": peaks["source"] + ", burst figure (stage timed alone)", "flop_per_position": trunk_flops, "positions_per_launch": batch,
                "ms": t_trunk * 1e3, "clocks": clocks_trunk,
                # the north star's bar: >= 50 % of the bf16 peak on the trunk at batch >= 1024 -- the trunk stage alone (L2 flushed) per batch size
                "by_batch": [{"positions_per_launch": nb, "ms": ms_nb, "achieved": nb * trunk_flops / (ms_nb * 1e-3) / 1e12,
                              "frac": nb * trunk_flops / (ms_nb * 1e-3) / 1e12 / peaks["bf16_tflops"], "clocks": c_nb}
                             for nb, (ms_nb, c_nb) in sorted(trunk_alone.items())],
                # stages of ONE pass of the launch sequence (events between the stages, no L2 flush inside the pass)
                "stages_ms": {"encode_trunk": float(split[0]), "heads": float(split[1]), "tail": float(split[2]), "sum": split_sum,
                              "all_graph": all_graph, "rel_diff": rel, "clocks": clocks_split,
                              "trusted": "both (within 3 %)" if rel <= 0.03 else "all_graph (the captured graph, which `value` is made of; the split pass "
                                                                                 "adds an event record between stages and ran in another power-cap state)"},
                "whole_net_tflops": batch * cfg.flops_per_position / (all_graph * 1e-3) / 1e12}
    if sustained is not None:
        tf = batch * cfg.flops_per_position / (sustained["ms_per_device_batch"] * 1e-3) / 1e12
        sustained.update({"whole_net_tflops": tf, "peak": peaks["bf16_tflops_sustained"], "frac": tf / peaks["bf16_tflops_sustained"],
                          # the trunk's share of a pass (split timing) applied to the sustained time per device batch
                          "trunk_tflops_estimate": batch * trunk_flops / (sustained["ms_per_device_batch"] * 1e-3 * float(split[0]) / split_sum) / 1e12,
                          "peak_source": peaks["source"] + ", sustained figure (kernels timed inside a seconds-long run)",
                          "note": "frac = whole-network algorithmic FLOP (trunk + heads) / wall time of the run vs the sustained cuBLAS bf16 peak"})
    roofline["sustained"] = sustained

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample_n = args.cpu_sample or (256 if cfg.filters >= 64 else 2048)
        v, cores, _, desc = time_cpu_reference(cfg, sample_n, budget_s=args.cpu_budget)
        cpu_baseline = {"value": v, "unit": "positions/s", "cores": cores, "kind": "port", "sample": desc,
                        "model_run_duration_batch1_us": time_cpu_run_duration_batch1(cfg) * 1e6}

    if rank == 0:
        line = {
            "metric": "nn_evals_per_sec", "value": value, "unit": "positions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_value / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": workload_config(args.workload, batch, per_step, cpu_sample_for(args, cfg)),
            "run": {"streams": args.streams, "replicas": world, "kernels_per_device_batch": kernels_per_batch, "trunk_path": trunk_path,
                    "positions_per_step": positions_per_step},
            "clocks": clocks,
            "clocks_e2e": clocks_e2e,
            "e2e": {"value": e2e_value, "unit": "positions/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": t_e2e / args.steps * 1e3, "api": "cattus_b200_eval_batch (host buffers -> pinned block -> H2D -> graph -> D2H)"},
            "gpu_launches": int(launches) + sum(leg["gpu_launches"] for leg in selfplay_legs) + sum(o["gpu_launches"] for o in others),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "batch_sweep": sweep,
            "leaf_latency": leaf,
            "hbm_kernels": hbm_kernels,
            "other_workloads": others,
            "selfplay": selfplay,
            "selfplay_others": selfplay_legs[1:],
        }
        print(json.dumps(line), flush=True)
    sampler.close()
    rep.close()


if __name__ == "__main__":
    main()
