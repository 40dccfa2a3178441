"""ctypes wrapper of tests/emul/libsession_emul.so (TEST INFRASTRUCTURE): persistent search sessions over the host
emulation of the device-resident search, with a Python evaluator callback, driven through cattus_b200.session."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

from cattus_b200 import _lib
from cattus_b200.selfplay import SelfPlayRunner, _eval_thunk, parse_game
from cattus_b200.session import DeviceSearch, _Api

HERE = Path(__file__).resolve().parent
SO = HERE / "libsession_emul.so"
SRC = HERE / "session_emul.cpp"
CSRC = HERE.parent.parent / "cattus_b200" / "csrc"


def build() -> Path:
    deps = [SRC, HERE / "search_batch_emul.cpp", HERE / "analysis_emul.cpp", HERE / "dsearch_emul.cpp"] + sorted(CSRC.glob("*.hpp")) + sorted(
        (HERE.parent.parent / "include").glob("*.h"))
    if SO.exists() and all(d.stat().st_mtime <= SO.stat().st_mtime for d in deps):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-fno-strict-aliasing", "-o", str(SO), str(SRC)],
                   check=True)
    return SO


_cached = None


def load():
    global _cached
    if _cached is None:
        lib = C.CDLL(str(build()))
        H, P = C.c_void_p, C.POINTER
        sig = {
            "session_emul_create": [H, H, H, C.c_uint32, C.c_uint32, C.c_uint32, P(H)],
            "session_emul_set_position": [H, C.c_char_p, P(C.c_uint16), C.c_uint32],
            "session_emul_new_game": [H],
            "session_emul_go": [H, P(_lib.SessionLimits)],
            "session_emul_stop": [H],
            "session_emul_info": [H, P(_lib.SessionSnapshot)],
            "session_emul_wait": [H, C.c_uint32, P(H)],
            "session_emul_batches": [H, C.c_uint32, P(C.c_uint32), P(C.c_uint32)],
            "session_emul_result_stats": [H, P(_lib.SessionStats)],
            "analysis_emul_count": [H, P(C.c_uint32)],
            "analysis_emul_get": [H, C.c_uint32, P(_lib.AnalysisPosition)],
            "analysis_emul_children": [H, C.c_uint32, P(C.c_uint16), P(C.c_uint32), P(C.c_float), P(C.c_float), C.c_uint32],
            "analysis_emul_pv": [H, C.c_uint32, P(C.c_uint16), C.c_uint32],
        }
        for name, args in sig.items():
            getattr(lib, name).argtypes = args
            getattr(lib, name).restype = C.c_int
        lib.session_emul_set_max_rows.argtypes = [H, C.c_uint32]
        lib.session_emul_set_max_rows.restype = None
        lib.session_emul_destroy.argtypes = [H]
        lib.session_emul_destroy.restype = None
        lib.analysis_emul_free.argtypes = [H]
        lib.analysis_emul_free.restype = None
        lib.session_emul_last_error.restype = C.c_char_p
        lib.session_emul_last_error.argtypes = []
        _cached = lib
    return _cached


def api() -> _Api:
    lib = load()
    return _Api(lib.session_emul_set_position, lib.session_emul_new_game, lib.session_emul_go, lib.session_emul_stop, lib.session_emul_info,
                lib.session_emul_wait, lib.session_emul_destroy, lib.analysis_emul_count, lib.analysis_emul_get, lib.analysis_emul_children,
                lib.analysis_emul_pv, lib.session_emul_batches, lib.session_emul_result_stats, lib.analysis_emul_free, lib.session_emul_last_error)


def create(game: str, cfg: dict, eval_fn, search_batch: int, *, tree_kwords: int = 256, max_batch: int = 4096, depth: int = 2,
           stop_after_waves: int = 0, opts_size: int = 0) -> DeviceSearch:
    """A DeviceSearch over the emulation.  tree_kwords: each tree buffer's kwords (small: the host allocates three of
    them); depth: waves in flight; stop_after_waves > 0: the stop word is written once that many waves have run.  Raises
    CattusB200Error."""
    lib = load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    g, s = parse_game(game)
    chess = g == _lib.GAME_CHESS
    words = 18 if chess else 3 * ((s * s + 63) // 64)
    errors: list = []
    thunk = _eval_thunk(eval_fn, words, chess, errors)
    opts = _lib.SessionOpts(opts_size or C.sizeof(_lib.SessionOpts), search_batch, tree_kwords)
    h = C.c_void_p()
    rc = lib.session_emul_create(C.cast(thunk, C.c_void_p), C.byref(c), C.byref(opts), max_batch, depth, stop_after_waves, C.byref(h))
    if rc != 0:
        raise _lib.CattusB200Error(rc, lib.session_emul_last_error().decode())
    ds = DeviceSearch.from_handle(api(), h, game)
    ds._keep = (thunk, c, errors)  # the callback must outlive the session
    return ds
