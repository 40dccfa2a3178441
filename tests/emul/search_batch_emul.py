"""ctypes wrapper of tests/emul/libsearch_batch_emul.so (TEST INFRASTRUCTURE): the batched analysis with minibatches under
virtual loss over the host emulation of the device-resident search, with a Python evaluator callback."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

from cattus_b200 import _lib
from cattus_b200.analysis import AnalysisOpts, collect, encode_positions
from cattus_b200.selfplay import SelfPlayRunner, _eval_thunk, parse_game

HERE = Path(__file__).resolve().parent
SO = HERE / "libsearch_batch_emul.so"
SRC = HERE / "search_batch_emul.cpp"
CSRC = HERE.parent.parent / "cattus_b200" / "csrc"


def build() -> Path:
    deps = [SRC, HERE / "analysis_emul.cpp", HERE / "dsearch_emul.cpp"] + sorted(CSRC.glob("*.hpp")) + sorted((HERE.parent.parent / "include").glob("*.h"))
    if SO.exists() and all(d.stat().st_mtime <= SO.stat().st_mtime for d in deps):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-fno-strict-aliasing", "-o", str(SO), str(SRC)],
                   check=True)
    return SO


_cached = None


def load():
    global _cached
    if _cached is None:
        lib = C.CDLL(str(build()))
        lib.search_batch_emul_run.restype = C.c_void_p
        lib.search_batch_emul_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_char_p),
                                              C.POINTER(C.c_uint16), C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32, C.c_uint32,
                                              C.POINTER(C.c_int)]
        lib.search_batch_emul_batches.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        lib.analysis_emul_error.restype = C.c_char_p
        lib.analysis_emul_error.argtypes = [C.c_void_p]
        lib.analysis_emul_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
        lib.analysis_emul_get.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(_lib.AnalysisPosition)]
        lib.analysis_emul_children.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16), C.POINTER(C.c_uint32), C.POINTER(C.c_float),
                                               C.POINTER(C.c_float), C.c_uint32]
        lib.analysis_emul_pv.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint16), C.c_uint32]
        lib.analysis_emul_free.argtypes = [C.c_void_p]
        _cached = lib
    return _cached


class EmulError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


def analyse(game: str, positions, cfg: dict, eval_fn, *, search_batch: int = 1, max_batch: int = 4096, pool_words: int = 1 << 16, depth: int = 2,
            roots_cap: int = 0, opts_size: int = 0):
    """-> [PositionAnalysis] with minibatches / collisions; raises EmulError(code, message).  search_batch 0 passes no
    options (NULL); opts_size overrides the options' struct_size.  depth: dsearch_emul_run's knobs (waves in flight | 256
    begin overlapped); the slots are cfg's device_games checked against max_batch."""
    lib = load()
    c = SelfPlayRunner(game, cfg)._fill(2, None, None, False, 0, 1)
    g, s = parse_game(game)
    chess = g == _lib.GAME_CHESS
    words = 18 if chess else 3 * ((s * s + 63) // 64)
    errors: list = []
    thunk = _eval_thunk(eval_fn, words, chess, errors)
    n, fa, ma, oa = encode_positions(game, positions)
    opts = None
    if search_batch:
        opts = AnalysisOpts()
        opts.struct_size = opts_size or C.sizeof(AnalysisOpts)
        opts.search_batch = search_batch
    code = C.c_int(0)
    h = lib.search_batch_emul_run(C.cast(thunk, C.c_void_p), C.byref(c), C.byref(opts) if opts is not None else None, max_batch, n, fa, ma, oa,
                                  pool_words, depth, roots_cap, C.byref(code))
    try:
        if errors:
            raise errors[0]
        err = lib.analysis_emul_error(h)
        if err:
            raise EmulError(code.value, err.decode())
        return collect(lib.analysis_emul_count, lib.analysis_emul_get, lib.analysis_emul_children, lib.analysis_emul_pv, h,
                       lib.search_batch_emul_batches)
    finally:
        lib.analysis_emul_free(h)
