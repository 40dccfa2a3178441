"""Persistent device search sessions (include/cattus_b200_session.h, DESIGN.md section 17).

    with DeviceSearch(model, "chess", cfg, search_batch=256) as s:
        s.set_position(None, ["e2e4"])
        s.go(nodes=10000)
        r = s.wait()                  # SessionResult: r.analysis is a PositionAnalysis
        s.set_position(None, ["e2e4", "e7e5", "g1f3"])
        s.go(movetime_ms=500, on_info=print)   # keeps the subtree of the previous search
        r = s.wait()

A session owns one search tree on the device and searches it in minibatches of `search_batch` L >= 2 descents under
virtual loss.  The tree lives across searches: when the next position is the previous root, a child or a grandchild, its
subtree is kept; otherwise the search starts from a fresh root.  `go` returns at once; `stop` (from any thread) ends the
search at its next minibatch boundary; `wait` returns the result.  With fixed `nodes` and `minibatches` the results are
deterministic, and `minibatches` of a stopped search replays it.  `model` must be a CudaNetwork created with
n_streams >= 2: the session holds one evaluator lane for its lifetime and the handle's other entry points keep the rest.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence

from . import _lib
from .analysis import PositionAnalysis, collect
from .selfplay import SelfPlayRunner, move_from_lan, parse_game

STOP_REASONS = {1: "nodes", 2: "minibatches", 3: "stop", 4: "deadline", 5: "capacity", 6: "finished"}
FOREVER = 0xFFFFFFFF


@dataclass
class SessionResult:
    analysis: PositionAnalysis  # simulations: this search's new ones
    reused_visits: int          # the root's visits kept from the previous search (0: fresh root)
    stop_reason: str            # STOP_REASONS
    seconds: float              # from go to the end of the search


@dataclass
class Snapshot:
    valid: bool                 # False: no minibatch of this search reported yet
    searching: bool
    simulations: int
    minibatches: int
    collisions: int
    best_move: Optional[int]
    q: float
    seconds: float
    pv: List[int] = field(default_factory=list)


@dataclass
class _Api:
    """The calls a session goes through: the library's cattus_b200_session_* or the test emulation's of the same
    signatures, and the accessors of their one-entry results."""
    set_position: Callable
    new_game: Callable
    go: Callable
    stop: Callable
    info: Callable
    wait: Callable
    destroy: Callable
    count: Callable
    get: Callable
    children: Callable
    pv: Callable
    batches: Callable
    stats: Callable
    free: Callable
    error: Callable


def library_api() -> _Api:
    lib = _lib.load()
    return _Api(lib.cattus_b200_session_set_position, lib.cattus_b200_session_new_game, lib.cattus_b200_session_go, lib.cattus_b200_session_stop,
                lib.cattus_b200_session_info, lib.cattus_b200_session_wait, lib.cattus_b200_session_destroy, lib.cattus_b200_analysis_count,
                lib.cattus_b200_analysis_get, lib.cattus_b200_analysis_children, lib.cattus_b200_analysis_pv, lib.cattus_b200_analysis_batches,
                lib.cattus_b200_session_result_stats, lib.cattus_b200_analysis_free, lib.cattus_b200_last_error)


class DeviceSearch:
    def __init__(self, model, game: str, cfg: dict, search_batch: int, tree_kwords: int = 0):
        """model: a CudaNetwork of the game with n_streams >= 2.  cfg: the self-play JSON config ("mcts": explore_factor,
        cache_size; prior_noise_epsilon must be 0; "device_waves_in_flight").  tree_kwords: words of each tree buffer / 1024
        (0: the most the 2^26-word tree address space allows).  Raises CattusB200Error (EINVAL for L < 2, a model without a
        free evaluator lane, ...)."""
        lib = _lib.load()
        c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
        opts = _lib.SessionOpts(C.sizeof(_lib.SessionOpts), int(search_batch), int(tree_kwords))
        h = C.c_void_p()
        _lib.check(lib.cattus_b200_session_create(model._h, C.byref(c), C.byref(opts), C.byref(h)))
        self._init(library_api(), h, game)

    @classmethod
    def from_handle(cls, api: _Api, handle, game: str) -> "DeviceSearch":
        """A session created elsewhere (the test emulation), driven through `api`."""
        self = cls.__new__(cls)
        self._init(api, handle, game)
        return self

    def _init(self, api: _Api, handle, game: str) -> None:
        self._api = api
        self._h = handle
        self.chess = parse_game(game)[0] == _lib.GAME_CHESS
        self._poller: Optional[threading.Thread] = None
        self._poll_stop = threading.Event()

    def _check(self, rc: int) -> None:
        if rc != _lib.OK:
            raise _lib.CattusB200Error(rc, (self._api.error() or b"").decode(errors="replace"))

    def set_position(self, fen: Optional[str] = None, moves: Sequence = ()) -> None:
        """fen None: the game's initial position (the only choice for hex and tic-tac-toe); moves: chess LAN strings or
        integers as in cattus_b200.analysis."""
        flat = [move_from_lan(m) if (self.chess and isinstance(m, str)) else int(m) for m in moves]
        arr = (C.c_uint16 * max(1, len(flat)))(*flat)
        self._check(self._api.set_position(self._h, None if fen is None else fen.encode(), arr, len(flat)))

    def new_game(self) -> None:
        """The next search starts from a fresh root."""
        self._check(self._api.new_game(self._h))

    def go(self, nodes: Optional[int] = None, minibatches: Optional[int] = None, movetime_ms: Optional[float] = None,
           on_info: Optional[Callable[[Snapshot], None]] = None, info_interval_ms: float = 500.0) -> None:
        """Starts a search and returns at once.  None: no limit (the search then runs until stop() or the tree buffer is
        full).  on_info(Snapshot) is called from a helper thread every info_interval_ms while the search runs."""
        lim = _lib.SessionLimits(C.sizeof(_lib.SessionLimits), int(nodes or 0), int(minibatches or 0), 0,
                                 int(round(movetime_ms * 1000.0)) if movetime_ms else 0)
        if movetime_ms is not None and lim.deadline_us == 0:
            lim.deadline_us = 1  # movetime 0: one minibatch
        self._check(self._api.go(self._h, C.byref(lim)))
        if on_info is not None:
            self._poll_stop.clear()
            self._poller = threading.Thread(target=self._poll, args=(on_info, info_interval_ms / 1000.0), daemon=True)
            self._poller.start()

    def _poll(self, on_info, interval: float) -> None:
        while not self._poll_stop.wait(interval):
            snap = self.info()
            if snap.valid:
                on_info(snap)
            if not snap.searching:
                return

    def stop(self) -> None:
        self._check(self._api.stop(self._h))

    def info(self) -> Snapshot:
        s = _lib.SessionSnapshot()
        s.struct_size = C.sizeof(_lib.SessionSnapshot)
        self._check(self._api.info(self._h, C.byref(s)))
        return Snapshot(bool(s.valid), bool(s.searching), int(s.simulations), int(s.minibatches), int(s.collisions),
                        int(s.best_move) if s.valid else None, float(s.q), float(s.seconds), list(s.pv)[: s.pv_len])

    def wait(self, timeout: Optional[float] = None) -> Optional[SessionResult]:
        """The search's result, or None when it still runs after `timeout` seconds (None: wait for it)."""
        ms = FOREVER if timeout is None else max(0, min(FOREVER - 1, int(timeout * 1000.0)))
        r = C.c_void_p()
        rc = self._api.wait(self._h, ms, C.byref(r))
        if rc == _lib.SESSION_RUNNING:
            return None
        self._finish_poller()
        self._check(rc)
        try:
            a = collect(self._api.count, self._api.get, self._api.children, self._api.pv, r, self._api.batches)[0]
            st = _lib.SessionStats()
            st.struct_size = C.sizeof(_lib.SessionStats)
            self._check(self._api.stats(r, C.byref(st)))
            return SessionResult(a, int(st.reused_visits), STOP_REASONS.get(int(st.stop_reason), str(st.stop_reason)), float(st.seconds))
        finally:
            self._api.free(r)

    def search(self, **kw) -> SessionResult:
        """go(**kw) then wait()."""
        self.go(**kw)
        return self.wait()

    def _finish_poller(self) -> None:
        if self._poller is not None:
            self._poll_stop.set()
            if self._poller is not threading.current_thread():
                self._poller.join()
            self._poller = None

    def close(self) -> None:
        if self._h is not None:
            self._poll_stop.set()
            self._api.stop(self._h)
            self._finish_poller()
            self._api.destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
