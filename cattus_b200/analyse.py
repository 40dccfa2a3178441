"""Analyse a file of chess positions on the B200 with the device-resident search.

    python -m cattus_b200.analyse --model-path NET.cb2 --config-file cfg.json [--precision bf16|fp8] \\
        (--epd FILE | --fen-file FILE) [--search-batch L] [--out results.jsonl]

--epd:      EPD records -- the four FEN fields, then operations; `bm` / `am` (best / avoid moves in SAN) and `id` are read.
--fen-file: one position per line, `<FEN> [moves <LAN> ...]` or `startpos [moves ...]`.
Blank lines and lines starting with # are skipped.

cfg.json is the self-play config: "mcts" (sim_num, explore_factor, cache_size; prior_noise_epsilon must be 0) and the
optional top-level "device_games", "device_tree_kwords", "device_waves_in_flight"; "model.batch_size" sizes the
evaluator (default 4096).  One JSON line per position goes to --out (default stdout): id, fen, moves, status, best move in
UCI LAN and SAN, its visits, simulations, Q (the side to move's mean score) and the principal variation.  With EPD bm / am
operations the solve count is printed to stderr.

--search-batch L > 1 searches every tree in minibatches of L descents under virtual loss (DESIGN.md section 15): for
deep searches of a few positions.  The evaluator batch is sized to hold device_games x L rows.  Each JSON line of a
searched position also carries `minibatches` and `collisions`.
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path
from typing import List, Optional

from . import san as S
from .analysis import STATUS_NAMES, analyse
from .selfplay import move_from_lan, move_to_lan


def read_positions(path: Path, epd: bool):
    """-> list of (id, fen or None, [moves], bm set or None, am set or None)."""
    out = []
    for k, line in enumerate(path.read_text().splitlines()):
        if not line.strip() or line.lstrip().startswith("#"):
            continue
        if epd:
            rec = S.parse_epd(line)
            bm = {S.move_from_san(rec.fen, [], m) for m in rec.ops["bm"]} if "bm" in rec.ops else None
            am = {S.move_from_san(rec.fen, [], m) for m in rec.ops["am"]} if "am" in rec.ops else None
            out.append((rec.id or f"line{k + 1}", rec.fen, [], bm, am))
        else:
            fen, lans = S.parse_fen_line(line)
            out.append((f"line{k + 1}", fen, [move_from_lan(m) for m in lans], None, None))
    return out


def report(pid: str, fen: Optional[str], moves: List[int], a) -> dict:
    r = {"id": pid, "fen": fen or S.START_FEN, "moves": [move_to_lan(m) for m in moves], "status": STATUS_NAMES[a.status]}
    if a.status == 0:
        r.update(best=move_to_lan(a.best_move), san=S.move_to_san(fen, moves, a.best_move), visits=a.best_visits, simulations=a.simulations,
                 q=round(a.q, 6), pv=[move_to_lan(m) for m in a.pv], pv_san=S.san_line(fen, moves, a.pv), minibatches=a.minibatches,
                 collisions=a.collisions)
    return r


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="cattus_b200.analyse", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--model-path", required=True, type=Path)
    ap.add_argument("--config-file", required=True, type=Path)
    ap.add_argument("--precision", default="bf16", choices=("bf16", "fp8"))
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--epd", type=Path)
    src.add_argument("--fen-file", type=Path)
    ap.add_argument("--out", type=Path)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--search-batch", type=int, default=1, help="descents per minibatch under virtual loss (1: one leaf in flight)")
    args = ap.parse_args(argv)
    cfg = json.loads(args.config_file.read_text())
    items = read_positions(args.epd or args.fen_file, args.epd is not None)
    from .network import CudaNetwork

    batch = int((cfg.get("model") or {}).get("batch_size", 4096))
    if args.search_batch > 1:
        batch = max(batch, args.search_batch * max(1, int(cfg.get("device_games", 1))))
    with CudaNetwork(args.model_path, "chess", device=args.device, batch_size=batch, n_streams=1, precision=args.precision) as nw:
        t0 = time.perf_counter()
        res = analyse(nw, "chess", [(fen, moves) for _, fen, moves, _, _ in items], cfg, search_batch=args.search_batch)
        secs = time.perf_counter() - t0
    out = args.out.open("w") if args.out else sys.stdout
    solved = graded = 0
    try:
        for (pid, fen, moves, bm, am), a in zip(items, res):
            r = report(pid, fen, moves, a)
            if bm is not None or am is not None:
                ok = a.best_move is not None and (bm is None or a.best_move in bm) and (am is None or a.best_move not in am)
                r["solved"] = ok
                graded += 1
                solved += ok
            out.write(json.dumps(r) + "\n")
    finally:
        if args.out:
            out.close()
    sims = sum(a.simulations for a in res)
    print(f"{len(res)} positions in {secs:.2f} s ({sims / max(secs, 1e-9):.0f} simulations/s)", file=sys.stderr)
    if graded:
        print(f"solved {solved} / {graded}", file=sys.stderr)
    return 0


if __name__ == "__main__":
    sys.exit(main())
