"""Play a colour-balanced match between two networks on the B200 with the device-resident search.

    python -m cattus_b200.play_match --model-a A.cb2 --model-b B.cb2 --config-file cfg.json [--game chess] \\
        [--precision-a bf16|fp8] [--precision-b bf16|fp8] [--sim-num-b N] [--explore-factor-b X] \\
        [--search-batch L] [--search-batch-b L] (--openings FILE | --pairs N) [--out games.jsonl] [--pgn games.pgn]

Each opening is played twice, A as player 1 in the first game and B in the second.  --model-b defaults to --model-a,
so `--precision-b fp8` alone plays a blob's bf16 against its FP8 handle.  --sim-num-b / --explore-factor-b give B its
own search settings (a search-odds match); everything else comes from cfg.json, the self-play config: "mcts" (sim_num,
explore_factor, temperature_policy, prior noise, cache_size), "seed", "max_moves" and the device_* keys; "model.batch_size"
sizes the evaluators (default 4096).  --search-batch L runs both sides' searches in minibatches of L descents under
virtual loss (DESIGN.md section 16), --search-batch-b B's alone: a side with L > 1 does not play the reference's search,
so `--search-batch-b 64` against the same net measures what the minibatches cost in games.

--openings: chess lines are EPD records (the four FEN fields, operations ignored), `<FEN> [moves <LAN> ...]` or
`startpos [moves ...]`; hex and tic-tac-toe lines are cell indices (`startpos` or an empty move list: the initial
position).  Blank lines and lines starting with # are skipped.  Without --openings the initial position is played
--pairs times.

Output: one JSON line per game to --out (default stdout), then a summary line on stderr (W/D/L from A's side, the
pentanomial counts, score, Elo with its 95 % interval, games/s, simulations/s and each side's minibatches and
collisions).  --pgn writes the chess games.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path
from typing import List, Optional, Tuple

from . import _lib
from . import san as S
from .analysis import STATUS_NAMES
from .match import fmt_elo, play
from .selfplay import move_from_lan, move_to_lan, parse_game


def read_openings(path: Path, chess: bool) -> List[Tuple[Optional[str], List[int]]]:
    out = []
    for line in path.read_text().splitlines():
        s = line.strip()
        if not s or s.startswith("#"):
            continue
        if not chess:
            out.append((None, [] if s == "startpos" else [int(x) for x in s.replace(",", " ").split()]))
        elif s.startswith("startpos") or " moves" in s:
            fen, lans = S.parse_fen_line(s)
            out.append((fen, [move_from_lan(m) for m in lans]))
        else:
            fields = s.split()
            is_fen = len(fields) == 4 or (len(fields) == 6 and fields[4].isdigit() and fields[5].isdigit())
            out.append((s if is_fen else S.parse_epd(s).fen, []))
    return out


def game_row(g, openings, chess: bool) -> dict:
    fen, opening = openings[g.opening]
    enc = move_to_lan if chess else int
    row = {"opening": g.opening, "a_is_player1": g.a_is_player1, "winner": g.winner, "a_points": g.a_points, "termination": g.termination,
           "moves": [enc(m) for m in g.moves]}
    if chess:
        row.update(fen=fen or S.START_FEN, opening_moves=[move_to_lan(m) for m in opening])
    else:
        row["opening_moves"] = list(opening)
    return row


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="cattus_b200.play_match", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--model-a", required=True, type=Path)
    ap.add_argument("--model-b", type=Path, help="default: --model-a")
    ap.add_argument("--precision-a", default="bf16", choices=("bf16", "fp8"))
    ap.add_argument("--precision-b", default="bf16", choices=("bf16", "fp8"))
    ap.add_argument("--sim-num-b", type=int)
    ap.add_argument("--explore-factor-b", type=float)
    ap.add_argument("--search-batch", type=int, help="descents per minibatch of both sides (default 1: one leaf in flight)")
    ap.add_argument("--search-batch-b", type=int, help="descents per minibatch of B (default: --search-batch)")
    ap.add_argument("--config-file", required=True, type=Path)
    ap.add_argument("--game", default="chess")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--openings", type=Path)
    src.add_argument("--pairs", type=int)
    ap.add_argument("--out", type=Path)
    ap.add_argument("--pgn", type=Path)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args(argv)
    game_id = parse_game(args.game)[0]
    chess = game_id == _lib.GAME_CHESS
    if args.pgn and not chess:
        ap.error("--pgn is for chess")
    cfg = json.loads(args.config_file.read_text())
    openings = read_openings(args.openings, chess) if args.openings else [(None, [])] * args.pairs
    from .network import CudaNetwork

    batch = int((cfg.get("model") or {}).get("batch_size", 4096))
    model_b = args.model_b or args.model_a
    net_game = {v: k for k, v in _lib.GAME_IDS.items()}[game_id]
    with CudaNetwork(args.model_a, net_game, device=args.device, batch_size=batch, n_streams=1, precision=args.precision_a) as na:
        if model_b == args.model_a and args.precision_b == args.precision_a:
            res = play(na, None, args.game, openings, cfg, args.sim_num_b, args.explore_factor_b, args.search_batch, args.search_batch_b)
        else:
            with CudaNetwork(model_b, net_game, device=args.device, batch_size=batch, n_streams=1, precision=args.precision_b) as nb:
                res = play(na, nb, args.game, openings, cfg, args.sim_num_b, args.explore_factor_b, args.search_batch, args.search_batch_b)
    out = args.out.open("w") if args.out else sys.stdout
    try:
        for k, st in enumerate(res.opening_status):
            if st:
                out.write(json.dumps({"opening": k, "status": STATUS_NAMES[st], "played": False}) + "\n")
        for g in res.games:
            out.write(json.dumps(game_row(g, openings, chess)) + "\n")
    finally:
        if args.out:
            out.close()
    if args.pgn:
        names = (f"A {args.model_a.name} {args.precision_a}", f"B {model_b.name} {args.precision_b}")
        with args.pgn.open("w") as f:
            for g in res.games:
                fen, opening = openings[g.opening]
                white, black = names if g.a_is_player1 else names[::-1]
                f.write(S.pgn_game(fen, opening, g.moves, g.winner, g.termination, white=white, black=black, event="cattus_b200 match",
                                   round_=f"{g.opening + 1}.{1 if g.a_is_player1 else 2}") + "\n")
    e = res.elo()
    summary = {"a_wins": res.a_wins, "draws": res.draws, "b_wins": res.b_wins, "games": len(res.games), "skipped_openings": res.skipped,
               "pentanomial": res.pairs, "score": None if e is None else round(e.score, 6),
               "elo": None if e is None else fmt_elo(e.elo), "elo_95": None if e is None else [fmt_elo(e.lo), fmt_elo(e.hi)],
               "seconds": round(res.seconds, 3), "games_per_s": round(len(res.games) / max(res.seconds, 1e-9), 3),
               "sims_per_s": round(res.simulations / max(res.seconds, 1e-9), 1), "minibatches": list(res.minibatches),
               "collisions": list(res.collisions)}
    print(json.dumps(summary), file=sys.stderr)
    return 0


if __name__ == "__main__":
    sys.exit(main())
