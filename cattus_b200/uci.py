"""UCI front-end with the B200 evaluator behind the search: the reference's `cattus` binary
(engine/src/bin/cattus.rs, engine/src/chess/uci.rs) with `CudaNetwork<ChessGame>` as the value function instead of
the `StockfishNet` placeholder it is built with today (cattus.rs:57-64; SURVEY.md section 8f-4).

    python -m cattus_b200.uci --config-file cfg.json

`cfg.json` is the reference's config (cattus.rs:16-42): {"model": {"model_path", "inference", "batch_size"},
"mcts": {"sim_num", "explore_factor", "temperature_policy", "prior_noise_alpha", "prior_noise_epsilon", "cache_size"},
"threads"}; `model.model_path` is a `.cb2` blob (cattus_b200.export) and `model.inference` may carry
{"engine": "cuda-b200", "device": 0, "precision": "bf16"} (precision "bf16", "fp32-check" or the opt-in "fp8" for 8x8 nets
with 64 / 128 / 256 filters).

`speculate` (top-level key, default 31; 0 = the reference's behaviour) lets up to that many likely next leaves ride along
with the leaf the search is waiting for; they only land in the value-function cache, so the moves played are unchanged
and a `go` needs about an eighth of the evaluator round trips.

`search_batch` (top-level key, default 1) L > 1 runs every `go` as a one-position analysis on the device-resident search
(cattus_b200.analysis) in minibatches of L descents under virtual loss (DESIGN.md section 15): the evaluator sees up to L
leaves of the tree at once instead of one.  Each `go` then starts from a FRESH tree with the position's history (no tree
is kept between `go`s), searches without root noise, and its result is that of the minibatched search, not the one-leaf
search's.  It prints `info depth <PV plies> nodes <sim_num> nps <n> score cp <cp> pv <moves>` before `bestmove`, where
cp = round(90 * tan(1.5637541897 * q)) of the side to move's mean score q in [-1, 1] (clamped to +-0.99), a monotone map.

Commands handled as in uci.rs:27-73: uci, isready, setoption, ucinewgame, position [fen <FEN> | startpos] [moves ...],
go (its arguments are parsed and ignored, as there), stop, quit.  One MctsPlayer per game: the tree of the previous
`go` is reused when the new position is in it; every search runs `mcts.sim_num` simulations with one leaf in flight.

`device_session` (top-level key, default false; needs `search_batch` >= 2) searches on one persistent device session
(cattus_b200.session, DESIGN.md section 17) instead: the tree of the previous `go` is kept when the new position is
within two plies of it, `go` is asynchronous (the input loop keeps answering `stop`, `isready` and `quit` during a
search), and `go`'s limits are honoured: `nodes`, `movetime`, `wtime` / `btime` / `winc` / `binc` / `movestogo` through
time_budget_ms (with the top-level `move_overhead_ms`, default 30), `infinite`, and `ponder` / `ponderhit` (the clock
starts at `ponderhit`).  After `infinite` or `ponder`, `bestmove` waits for `stop` (or `ponderhit`).  `depth`, `mate`
and `searchmoves` are parsed and ignored.  A bare `go` searches `mcts.sim_num` nodes.  It prints `info depth <PV plies>
nodes <this search's simulations> nps <n> time <ms> score cp <cp> pv <moves>` every `info_interval_ms` (default 500)
and once before `bestmove <move> ponder <reply>`.  `ucinewgame` drops the tree.  The model then has two evaluator
streams: the session holds one.
"""
from __future__ import annotations

import argparse
import json
import math
import sys
import threading
import time
from pathlib import Path
from typing import List, Optional, TextIO

from .network import CudaNetwork
from .selfplay import ChessSearch

GO_KEYS = ("searchmoves", "ponder", "wtime", "btime", "winc", "binc", "movestogo", "depth", "nodes", "mate", "movetime", "infinite")


def q_to_cp(q: float) -> int:
    """The side to move's mean score q in [-1, 1] as centipawns: round(90 * tan(1.5637541897 * q)), q clamped to +-0.99
    (monotone; 0 -> 0, +-0.5 -> +-90, +-0.99 -> +-2720)."""
    q = max(-0.99, min(0.99, float(q)))
    return int(round(90.0 * math.tan(1.5637541897 * q)))


def time_budget_ms(t: float, inc: float, movestogo: Optional[int], move_overhead_ms: float) -> float:
    """Milliseconds to search with `t` ms left on the clock and `inc` ms increment: min(t / 2, t / movestogo + 3/4 inc)
    - move_overhead_ms, movestogo 30 when not given, never below 0 (a search always completes one minibatch)."""
    mtg = movestogo if movestogo else 30
    return max(0.0, min(t / 2.0, t / mtg + 0.75 * inc) - move_overhead_ms)


def parse_args(args: List[str], keys) -> dict:
    """UCI::parse_args (uci.rs:177-192): words after a key belong to it; a repeated key or a word before any key is an error."""
    out: dict = {}
    key = None
    for a in args:
        if a in keys:
            if a in out:
                raise ValueError(f"arg '{a}' appears multiple times")
            out[a] = []
            key = a
        else:
            if key is None:
                raise ValueError(f"arg '{a}' has no key")
            out[key].append(a)
    return out


class UCI:
    def __init__(self, cfg: dict, model=None, eval_fn=None, out: TextIO = sys.stdout, session_factory=None):
        """session_factory (device_session only): (session cfg, search_batch) -> a cattus_b200.session.DeviceSearch; the
        default opens one on `model`."""
        cfg = dict(cfg)
        cfg.setdefault("speculate", 31 if (cfg.get("mcts") or {}).get("cache_size") else 0)
        self.cfg = cfg
        self.search_batch = int(cfg.get("search_batch", 1))
        if self.search_batch < 1:
            raise ValueError("search_batch must be >= 1")
        self.device_session = bool(cfg.get("device_session", False))
        if self.device_session and self.search_batch < 2:
            raise ValueError("device_session needs search_batch >= 2")
        self.session_factory = session_factory
        self.session = None
        self._search: Optional[dict] = None  # the running session search: release (Event), monitor (Thread), ponderhit timer, budget
        self._lock = threading.Lock()
        self.model = model
        self.eval_fn = eval_fn
        self.out = out
        self.options: dict = {}
        self.player: Optional[ChessSearch] = None
        self.fen: Optional[str] = None
        self.moves: Optional[List[str]] = None
        self.last_stats: Optional[dict] = None

    def send(self, s: str) -> None:
        if self.device_session:
            with self._lock:
                print(s, file=self.out, flush=True)
        else:
            print(s, file=self.out, flush=True)

    def handle(self, line: str) -> bool:
        """One command; False after `quit`."""
        words = line.split()
        if not words:
            return True
        command, args = words[0], words[1:]
        if self.device_session and command in ("go", "stop", "ponderhit", "ucinewgame", "position", "quit"):
            return self.handle_session(command, args)
        if command == "uci":
            self.send("id name cattus_b200 v1.0.0")
            self.send("id author cattus_b200")
            self.send("uciok")
        elif command == "isready":
            self.send("readyok")
        elif command == "setoption":
            a = parse_args(args, ("name", "value"))
            self.options[" ".join(a["name"])] = " ".join(a["value"])
        elif command == "ucinewgame":
            if self.player is not None:
                self.player.close()
            self.player = ChessSearch(self.cfg, self.model, self.eval_fn)
        elif command == "position":
            a = parse_args(args, ("fen", "startpos", "moves"))
            if ("fen" in a) == ("startpos" in a):
                raise ValueError("position cmd requires either fen or startpos")
            self.fen = " ".join(a["fen"]) if "fen" in a else None
            self.moves = list(a.get("moves", []))
        elif command == "go":
            parse_args(args, GO_KEYS)
            if self.search_batch > 1:
                if self.moves is None:
                    raise ValueError("go before position")
                self.go_batched()
                return True
            if self.player is None:  # the reference unwraps None here; a GUI that skips ucinewgame still gets a player
                self.player = ChessSearch(self.cfg, self.model, self.eval_fn)
            if self.moves is None:
                raise ValueError("go before position")
            best, stats = self.player.go(self.fen, self.moves)
            self.last_stats = stats
            self.send(f"info nodes {stats['simulations']} time {int(stats['seconds'] * 1000)} nps {int(stats['simulations'] / max(stats['seconds'], 1e-9))}")
            self.send(f"bestmove {best}")
        elif command in ("stop",):
            pass
        elif command in ("ponderhit", "start", "fen", "xyzzy"):
            self.send("uciok")
        elif command == "quit":
            return False
        else:
            print(f"unknown command {command}", file=sys.stderr)
        return True

    def go_batched(self) -> None:
        """One minibatched device analysis of the current position and history, from a fresh tree."""
        from .analysis import analyse
        from .selfplay import move_to_lan

        mc = dict(self.cfg.get("mcts") or {})
        mc["prior_noise_epsilon"] = 0.0  # an analysis has no root noise
        cfg = {"mcts": mc, "device_games": 1}
        for key in ("device_tree_kwords",):
            if key in self.cfg:
                cfg[key] = self.cfg[key]
        t0 = time.perf_counter()
        a = analyse(self.model, "chess", [(self.fen, list(self.moves))], cfg, search_batch=self.search_batch)[0]
        secs = time.perf_counter() - t0
        self.last_stats = {"simulations": a.simulations, "seconds": secs, "minibatches": a.minibatches, "collisions": a.collisions, "q": a.q,
                           "analysis": a}
        if a.status != 0:  # the game is over: there is no move to search
            self.send("bestmove 0000")
            return
        pv = " ".join(move_to_lan(m) for m in a.pv)
        self.send(f"info depth {len(a.pv)} nodes {a.simulations} nps {int(a.simulations / max(secs, 1e-9))} score cp {q_to_cp(a.q)} pv {pv}")
        self.send(f"bestmove {move_to_lan(a.best_move)}")

    # ------------------------------------------------------------------------------------------------ device session
    def handle_session(self, command: str, args: List[str]) -> bool:
        if command == "stop":
            self._release(stop=True)
        elif command == "ponderhit":
            srch = self._search
            if srch is not None and srch["ponder"] and not srch["release"].is_set():
                if srch["budget"] is None:  # pondering without a clock: the move is due now
                    self._release(stop=True)
                else:  # the clock starts now: a timer stops the search when the budget is spent
                    srch["timer"] = threading.Timer(srch["budget"] / 1000.0, self._deadline_stop, args=(srch,))
                    srch["timer"].start()
                    srch["release"].set()
        elif command == "quit":
            self.close()
            return False
        else:
            self._finish(stop=False)  # a search still running (a GUI waits for bestmove first) runs out, or ends if unbounded
            if command == "ucinewgame":
                if self.session is not None:
                    self.session.new_game()
            elif command == "position":
                a = parse_args(args, ("fen", "startpos", "moves"))
                if ("fen" in a) == ("startpos" in a):
                    raise ValueError("position cmd requires either fen or startpos")
                self.fen = " ".join(a["fen"]) if "fen" in a else None
                self.moves = list(a.get("moves", []))
            else:
                self.go_session(parse_args(args, GO_KEYS))
        return True

    def _open_session(self):
        if self.session is None:
            mc = dict(self.cfg.get("mcts") or {})
            mc["prior_noise_epsilon"] = 0.0  # a session's searches have no root noise
            cfg = {"mcts": mc}
            if "device_waves_in_flight" in self.cfg:
                cfg["device_waves_in_flight"] = self.cfg["device_waves_in_flight"]
            if self.session_factory is not None:
                self.session = self.session_factory(cfg, self.search_batch)
            else:
                from .session import DeviceSearch

                self.session = DeviceSearch(self.model, "chess", cfg, self.search_batch, int(self.cfg.get("device_tree_kwords", 0)))
        return self.session

    def go_session(self, a: dict) -> None:
        if self.moves is None:
            raise ValueError("go before position")
        s = self._open_session()
        s.set_position(self.fen, self.moves)
        white = (self.fen is None or self.fen.split()[1] == "w") == (len(self.moves) % 2 == 0)
        num = lambda k: float(a[k][0]) if a.get(k) else None  # noqa: E731
        clock = num("wtime" if white else "btime")
        budget = None
        if clock is not None:
            mtg = num("movestogo")
            budget = time_budget_ms(clock, num("winc" if white else "binc") or 0.0, int(mtg) if mtg else None,
                                    float(self.cfg.get("move_overhead_ms", 30)))
        nodes, movetime = None, None
        hold = "infinite" in a or "ponder" in a
        if not hold:
            if "nodes" in a:
                nodes = int(a["nodes"][0])
            if "movetime" in a:
                movetime = num("movetime")
            elif budget is not None:
                movetime = budget
            if nodes is None and movetime is None:
                nodes = int((self.cfg.get("mcts") or {}).get("sim_num", 800))
        srch = {"release": threading.Event(), "ponder": "ponder" in a, "budget": budget, "timer": None, "ended": False, "lock": threading.Lock()}
        if not hold:
            srch["release"].set()
        s.go(nodes=nodes, movetime_ms=movetime)
        srch["monitor"] = threading.Thread(target=self._monitor, args=(srch,), daemon=True)
        self._search = srch
        srch["monitor"].start()

    def _info_line(self, depth: int, nodes: int, secs: float, q: float, pv) -> str:
        from .selfplay import move_to_lan

        return (f"info depth {depth} nodes {nodes} nps {int(nodes / max(secs, 1e-9))} time {int(secs * 1000)} score cp {q_to_cp(q)} "
                f"pv {' '.join(move_to_lan(m) for m in pv)}")

    def _deadline_stop(self, srch: dict) -> None:
        """A ponderhit's budget is spent: stop the search, unless it has already ended (the session may be searching the
        next position by then)."""
        with srch["lock"]:
            if not srch["ended"]:
                self.session.stop()

    def _monitor(self, srch: dict) -> None:
        """Prints info lines while the search runs and sends bestmove once the search has ended and is released.  A search
        that fails is reported on stderr and answered with `bestmove 0000`."""
        from .selfplay import move_to_lan

        s = self.session
        interval = float(self.cfg.get("info_interval_ms", 500)) / 1000.0
        next_info = time.monotonic() + interval
        r, error = None, None
        try:
            while r is None:
                r = s.wait(timeout=max(0.0, next_info - time.monotonic()))
                if r is None:
                    snap = s.info()
                    if snap.valid:
                        self.send(self._info_line(len(snap.pv), snap.simulations, snap.seconds, snap.q, snap.pv))
                    next_info += interval
        except Exception as e:  # the GUI still needs its bestmove
            error = e
        with srch["lock"]:
            srch["ended"] = True
        if srch["timer"] is not None:
            srch["timer"].cancel()
        srch["release"].wait()
        if error is not None:
            print(f"error: search failed: {error}", file=sys.stderr)
            self.send("bestmove 0000")
            return
        self.last_stats = {"simulations": r.analysis.simulations, "seconds": r.seconds, "minibatches": r.analysis.minibatches,
                           "collisions": r.analysis.collisions, "q": r.analysis.q, "reused_visits": r.reused_visits, "stop_reason": r.stop_reason,
                           "analysis": r.analysis}
        a = r.analysis
        if a.status != 0:
            self.send("bestmove 0000")
            return
        self.send(self._info_line(len(a.pv), a.simulations, r.seconds, a.q, a.pv))
        self.send(f"bestmove {move_to_lan(a.best_move)}" + (f" ponder {move_to_lan(a.pv[1])}" if len(a.pv) > 1 else ""))

    def _release(self, stop: bool) -> None:
        srch = self._search
        if srch is None:
            return
        srch["release"].set()
        if stop:
            self.session.stop()

    def _finish(self, stop: bool) -> None:
        """Waits for the running search's bestmove; a held (infinite / ponder) search, or any with `stop`, is stopped."""
        srch = self._search
        if srch is None:
            return
        if stop or not srch["release"].is_set():
            self._release(stop=True)
        srch["monitor"].join()
        self._search = None

    def close(self) -> None:
        if self.device_session:
            self._finish(stop=True)
            if self.session is not None:
                self.session.close()
                self.session = None

    def run(self, inp: TextIO = sys.stdin) -> None:
        for line in inp:
            try:
                if not self.handle(line.strip()):
                    break
            except Exception as e:  # a malformed command must not take the engine down mid-game
                print(f"error: {e}", file=sys.stderr)
        if self.device_session:
            self._finish(stop=False)
            self.close()
        if self.player is not None:
            self.player.close()


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="cattus_b200.uci", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config-file", required=True, type=Path)
    args = ap.parse_args(argv)
    cfg = json.loads(args.config_file.read_text())
    model_cfg = cfg["model"]
    inference = model_cfg.get("inference") or {}
    if inference.get("engine", "cuda-b200") != "cuda-b200":
        raise SystemExit(f"this executable is the cuda-b200 engine; config.model.inference.engine is {inference.get('engine')!r} (there is no CPU fallback)")
    # room for the speculative rows: a device batch of up to 64 positions costs what one position costs; a minibatched
    # search writes up to search_batch rows per round
    batch = max(64, int(model_cfg.get("batch_size", 1)), int(cfg.get("search_batch", 1)))
    # a device session holds one evaluator stream for its lifetime
    with CudaNetwork(Path(model_cfg["model_path"]), "chess", device=int(inference.get("device", 0)), batch_size=batch,
                     n_streams=2 if cfg.get("device_session") else 1, precision=inference.get("precision", "bf16")) as nw:
        UCI(cfg, model=nw).run()
    return 0


if __name__ == "__main__":
    sys.exit(main())
