"""Drop-in for the reference's `{game}_self_player` executables with the B200 evaluator behind it.

Same command line (training/self-play/src/self_play_cmd.rs:14-31) and same JSON config file (:34-53), as the trainer
invokes it (training/cattus_train/train_process.py:159-170, :341-352):

    python -m cattus_b200.self_player --model1-path M1.cb2 --model2-path M2.cb2 --games-num N \
        --out-dir1 D1 --out-dir2 D2 [--summary-file S.json] --config-file cfg.json

* the game and board size are read from the model blob's header (the reference has one binary per game);
* `config.model.inference` may carry `{"engine": "cuda-b200", "device": 0, "precision": "bf16", "streams": 4}`;
  `precision` is "bf16" (default), "fp32-check" or the opt-in "fp8" (8x8 nets with 64 / 128 / 256 filters only);
  `config.model.batch_size` is the evaluator's max batch; the optional top-level keys `games_per_thread`, `leaf_queue`
  and `seed` select this backend's many-games-per-thread arrangement (default 64 games per worker thread);
* with few games per worker thread (`games_num / threads` <= 96) `speculate` defaults on: likely next leaves are evaluated
  ahead into the value-function cache in the otherwise nearly empty batches -- same games, several times fewer round trips;
* the optional top-level key `search_batch` L > 1 runs every search in minibatches of L descents under virtual loss on
  the device-resident search (DESIGN.md section 16): a hundred games then fill the evaluator's batch.  Such games are not
  the reference's; `device_games` defaults to min(games_num, 4096 / L) and the evaluator's batch holds device_games x L;
* `.traindata` files are byte-for-byte what the reference's serializers write (hex, tic-tac-toe and chess:
  serialize/{hex,ttt,chess}.rs), named `{game_idx:08}_{pos_idx:03}`;
* the summary file has the reference's layout (:131-149): player1_wins, player2_wins, draws and the metric keys the
  trainer reads -- model.activation_count, model.run_duration, mcts.search_duration, cache.hits, cache.misses -- and
  selfplay.minibatches / selfplay.collisions among the others.

With `torchrun` / `--gpus N` style partitioning use `--first-game r --game-stride n --device r` per process.
"""
from __future__ import annotations

import argparse
import json
import struct
import sys
from pathlib import Path

from . import _lib
from .network import CudaNetwork
from .selfplay import SelfPlayRunner


def game_of_blob(path: Path):
    """('hex5', 'hex') / ('ttt', 'ttt') / ('chess', 'chess') from the .cb2 header (export.py)."""
    with open(path, "rb") as f:
        h = struct.unpack("<16I", f.read(64))
    if h[0] != 0x00324243:
        raise ValueError(f"{path}: not a .cb2 weight blob (export it with cattus_b200.export.export_model)")
    game_id, s = h[2], h[3]
    if game_id == _lib.GAME_HEX:
        return f"hex{s}", "hex"
    if game_id == _lib.GAME_TTT:
        return "ttt", "ttt"
    if game_id == _lib.GAME_CHESS:
        return "chess", "chess"
    raise ValueError(f"{path}: unknown game id {game_id}")


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="cattus_b200.self_player", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--model1-path", required=True, type=Path)
    ap.add_argument("--model2-path", required=True, type=Path)
    ap.add_argument("--games-num", required=True, type=int)
    ap.add_argument("--out-dir1", required=True, type=Path)
    ap.add_argument("--out-dir2", required=True, type=Path)
    ap.add_argument("--summary-file", type=Path, default=None)
    ap.add_argument("--config-file", required=True, type=Path)
    ap.add_argument("--device", type=int, default=None, help="CUDA ordinal (default: config.model.inference.device or 0)")
    ap.add_argument("--first-game", type=int, default=0)
    ap.add_argument("--game-stride", type=int, default=1)
    args = ap.parse_args(argv)

    cfg = json.loads(args.config_file.read_text())
    inference = (cfg.get("model") or {}).get("inference") or {}
    engine = inference.get("engine", "cuda-b200")
    if engine != "cuda-b200":
        raise SystemExit(f"this executable is the cuda-b200 engine; config.model.inference.engine is {engine!r} (there is no CPU fallback)")
    device = args.device if args.device is not None else int(inference.get("device", 0))
    game, family = game_of_blob(args.model1_path)
    if game_of_blob(args.model2_path)[0] != game:
        raise SystemExit("model1 and model2 are for different games")
    # Big jobs run the DEVICE-RESIDENT search (trees in HBM, one warp per game, DESIGN.md section 7a): sims/s then no longer
    # depends on the host cores.  "device_games" in the config file decides; without it, jobs of >= 2048 games take it on
    # their own (same games either way).  Small jobs keep their trees on the host, where speculative rows hide the latency.
    with open(args.model1_path, "rb") as f:
        filters = struct.unpack("<16I", f.read(64))[6]
    search_batch = int(cfg.get("search_batch", 1) or 1)
    if "device_games" not in cfg and search_batch > 1:  # minibatches run on the device-resident search only
        cfg["device_games"] = max(1, min(args.games_num, 4096 // search_batch))
    if "device_games" not in cfg and args.games_num >= 2048:
        cfg["device_games"] = min(args.games_num, 4096 if filters >= 64 else 16384)
    device_games = int(cfg.get("device_games", 0))
    cfg.setdefault("games_per_thread", 64)
    # A trainer-sized job (self_play.games_num 100, threads 8) keeps only a dozen leaves in flight per worker, far below the
    # ~256 positions a device batch can hold at no extra latency: let likely next leaves ride along into the cache (same games,
    # fewer round trips).  Big jobs fill their batches with real leaves and need none.
    slots = max(1, min(int(cfg["games_per_thread"]), -(-args.games_num // max(1, int(cfg.get("threads", 1))))))
    if (cfg.get("mcts") or {}).get("cache_size"):
        cfg.setdefault("speculate", min(31, 192 // slots) if slots <= 96 else 0)
    cfg.setdefault("groups_per_thread", 2)  # a worker simulates one half of its games while the other half's leaves are on the GPU
    max_batch = max(int(cfg["model"].get("batch_size", 64)), min(4096, int(cfg["games_per_thread"])), 256 if cfg.get("speculate") else 1,
                    device_games * search_batch)
    kw = dict(device=device, batch_size=max_batch, n_streams=int(inference.get("streams", 4)), precision=inference.get("precision", "bf16"))
    if args.summary_file is not None and args.summary_file.exists():
        raise SystemExit(f"{args.summary_file} exists")  # File::create_new (self_play_cmd.rs:150)

    nw1 = CudaNetwork(args.model1_path, family, **kw)
    same = args.model1_path == args.model2_path  # self_play_cmd.rs:93: one network, one cache
    nw2 = nw1 if same else CudaNetwork(args.model2_path, family, **kw)
    try:
        runner = SelfPlayRunner(game, cfg)
        summary, _ = runner.generate_data(nw1, None if same else nw2, args.games_num, args.out_dir1, args.out_dir2,
                                          first_game=args.first_game, game_stride=args.game_stride)
        m1 = nw1.metrics()
        summary["metrics"]["model.activation_count"] = m1["model.activation_count"] + (0 if same else nw2.metrics()["model.activation_count"])
        summary["metrics"]["model.run_duration"] = m1["model.run_duration"]
    finally:
        nw1.close()
        if not same:
            nw2.close()
    if args.summary_file is not None:
        args.summary_file.write_text(json.dumps(summary))
    return 0


if __name__ == "__main__":
    sys.exit(main())
