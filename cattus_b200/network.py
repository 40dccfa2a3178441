"""Host-side mirror of the reference's `NNetwork` (engine/src/net/mod.rs:14-104) over the C ABI.

    NNetwork::new(model_path, inference_cfg, batch_size, cache)   ->  CudaNetwork(model, game, batch_size=..., cache=...)
    NNetwork::evaluate(position, to_planes)                       ->  CudaNetwork.evaluate(position)
    planes_to_tensor(samples, batch_size)                         ->  CudaNetwork.planes_to_tensor(words, batch_size)
    Model::run(input)                                             ->  CudaNetwork.run(nchw)
    metrics model.activation_count / model.run_duration           ->  CudaNetwork.metrics()

`evaluate` does what the Rust shim in INTEGRATION.md does around `cattus_b200_eval`: flip to the side-to-move view,
consult the position cache, build planes (+ legal bitmap for chess), call the blocking FFI, map the compact
probabilities back to `legal_moves()` order, un-flip.  Everything numeric happens on the GPU; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path
from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import Desc, Info, Metrics, check
from .cache import ValueFuncCache


def _ptr(a: np.ndarray, typ):
    return a.ctypes.data_as(typ)


class CudaNetwork:
    def __init__(self, model, game: str, *, device: int = 0, batch_size: int = 64, n_streams: int = 2,
                 precision: str = "bf16", cache: Optional[ValueFuncCache] = None, fused_trunk: bool = True, fault_inject: bool = False):
        """model: path to a .cb2 blob, or the blob bytes (cattus_b200.export.export_blob).

        precision: "bf16" (default), "fp32-check" (CUDA-core fp32, for parity checks) or "fp8" (opt-in: the conv trunk in
        e4m3 on the whole-trunk kernel; only 8x8 nets with 64 / 128 / 256 filters, anything else raises EINVAL -- see
        CATTUS_B200_PRECISION_FP8 in include/cattus_b200.h for its numerics)."""
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.cache = cache
        self.game = game
        desc = Desc()
        desc.struct_size = C.sizeof(Desc)
        desc.game = _lib.GAME_IDS[game]
        desc.device = device
        desc.max_batch = batch_size
        desc.n_streams = n_streams
        desc.flags = 0 if fused_trunk else 1  # bit 0: force the per-layer kernels (parity tests compare both paths)
        if fault_inject:
            desc.flags |= 2  # bit 1: tests only -- a head GEMM tile never publishes its accumulator (include/cattus_b200.h)
        desc.precision = _lib.PRECISION_IDS[precision]
        if isinstance(model, (bytes, bytearray, memoryview)):
            buf = bytes(model)
            check(self._lib.cattus_b200_create_from_memory(C.byref(desc), buf, len(buf), C.byref(self._h)))
        else:
            desc.weights_path = str(Path(model)).encode()
            check(self._lib.cattus_b200_create(C.byref(desc), C.byref(self._h)))
        info = Info()
        check(self._lib.cattus_b200_get_info(self._h, C.byref(info)))
        self.info = info
        self.board_size = info.board_size
        self.planes = info.planes
        self.moves = info.moves
        self.words_per_plane = info.words_per_plane
        self.words = info.planes * info.words_per_plane
        self.bitmap_bytes = info.legal_bitmap_bytes
        self.max_batch = info.max_batch
        self.needs_bitmap = game == "chess"
        self.trunk_path = _lib.TRUNK_PATH_NAMES[info.trunk_path]  # "fused" / "small" / "per-layer" / "fp32-check" (cattus_b200_info.trunk_path)
        self.fused_trunk = info.trunk_path == _lib.TRUNK_FUSED
        self.small_trunk = info.trunk_path == _lib.TRUNK_SMALL

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.cattus_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ the FFI calls
    def eval_planes(self, words: np.ndarray, bitmap: Optional[np.ndarray] = None) -> Tuple[np.ndarray, float]:
        """cattus_b200_eval: one leaf, blocking, thread-safe.  Returns (probs over legal moves in ascending nn index, value)."""
        w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1)
        assert w.size == self.words, f"expected {self.words} u64 words, got {w.size}"
        bm = None
        if bitmap is not None:
            bm = np.ascontiguousarray(bitmap, dtype=np.uint8).reshape(-1)
            assert bm.size == self.bitmap_bytes
        probs = np.empty(self.moves, dtype=np.float32)
        n = C.c_uint32(0)
        v = C.c_float(0)
        check(self._lib.cattus_b200_eval(self._h, _ptr(w, _lib._u64p), _ptr(bm, _lib._u8p) if bm is not None else None,
                                         _ptr(probs, _lib._f32p), self.moves, C.byref(n), C.byref(v)))
        return probs[: n.value].copy(), float(v.value)

    def eval_batch(self, words: np.ndarray, bitmaps: Optional[np.ndarray] = None, probs_cap: Optional[int] = None):
        """cattus_b200_eval_batch: n positions from host buffers.  Returns (probs flat, offsets[n+1], values[n])."""
        w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, self.words)
        n = w.shape[0]
        bm = None
        if bitmaps is not None:
            bm = np.ascontiguousarray(bitmaps, dtype=np.uint8).reshape(n, self.bitmap_bytes)
        cap = int(probs_cap if probs_cap is not None else n * min(self.moves, 256 if self.needs_bitmap else self.moves))
        probs = np.empty(max(cap, 1), dtype=np.float32)
        offsets = np.empty(n + 1, dtype=np.uint32)
        values = np.empty(max(n, 1), dtype=np.float32)
        check(self._lib.cattus_b200_eval_batch(self._h, _ptr(w, _lib._u64p), _ptr(bm, _lib._u8p) if bm is not None else None, n,
                                               _ptr(probs, _lib._f32p), cap, _ptr(offsets, _lib._u32p), _ptr(values, _lib._f32p)))
        return probs[: int(offsets[n])], offsets, values[:n]

    def planes_to_tensor(self, words: np.ndarray, batch_size: Optional[int] = None) -> np.ndarray:
        """planes_to_tensor (net/mod.rs:121-156) through the device encode kernel: [batch_size, C, S, S] f32."""
        w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, self.words)
        n = w.shape[0]
        bs = n if batch_size is None else batch_size
        out = np.empty((bs, self.planes, self.board_size, self.board_size), dtype=np.float32)
        check(self._lib.cattus_b200_encode(self._h, _ptr(w, _lib._u64p), n, bs, _ptr(out, _lib._f32p)))
        return out

    def run(self, nchw: np.ndarray):
        """Model::run (model.rs:146-218): dense f32 NCHW -> (policy logits [n, M], value [n, 1])."""
        x = np.ascontiguousarray(nchw, dtype=np.float32)
        n = x.shape[0]
        assert x.shape[1:] == (self.planes, self.board_size, self.board_size)
        logits = np.empty((n, self.moves), dtype=np.float32)
        values = np.empty((n, 1), dtype=np.float32)
        check(self._lib.cattus_b200_run_dense(self._h, _ptr(x, _lib._f32p), n, _ptr(logits, _lib._f32p), _ptr(values, _lib._f32p)))
        return logits, values

    def resident_upload(self, words: np.ndarray, bitmaps: Optional[np.ndarray] = None) -> int:
        w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, self.words)
        bm = None if bitmaps is None else np.ascontiguousarray(bitmaps, dtype=np.uint8).reshape(w.shape[0], self.bitmap_bytes)
        check(self._lib.cattus_b200_resident_upload(self._h, _ptr(w, _lib._u64p), _ptr(bm, _lib._u8p) if bm is not None else None, w.shape[0]))
        return w.shape[0]

    def eval_resident(self, n: int, stream: int = 0) -> None:
        check(self._lib.cattus_b200_eval_resident(self._h, n, C.c_void_p(stream) if stream else None))

    def resident_download(self, n: int):
        probs = np.empty(n * self.moves, dtype=np.float32)
        offsets = np.empty(n + 1, dtype=np.uint32)
        values = np.empty(n, dtype=np.float32)
        check(self._lib.cattus_b200_resident_download(self._h, n, _ptr(probs, _lib._f32p), probs.size, _ptr(offsets, _lib._u32p),
                                                      _ptr(values, _lib._f32p)))
        return probs[: int(offsets[n])], offsets, values

    def time_stage(self, stage: int, n: int, iters: int) -> np.ndarray:
        """Per-iteration device milliseconds (CUDA events on the evaluator stream, L2 flushed between iterations).
        stage 5 returns [iters, 3]: (encode + trunk, heads, tail) of the same pass, which add up to the pass."""
        ms = np.empty(iters * (3 if stage == 5 else 1), dtype=np.float32)
        check(self._lib.cattus_b200_time_stage(self._h, stage, n, iters, _ptr(ms, _lib._f32p)))
        return ms.reshape(iters, 3) if stage == 5 else ms

    def time_sustained(self, words: np.ndarray, bitmaps, n: int, n_batches: int, iters: int) -> float:
        """Milliseconds for `iters` back-to-back device batches rotating over n_batches distinct resident batches of n."""
        words = np.ascontiguousarray(words[: n * n_batches], dtype=np.uint64)
        assert len(words) == n * n_batches
        bm = None if bitmaps is None else np.ascontiguousarray(bitmaps[: n * n_batches], dtype=np.uint8)
        ms = C.c_float()
        check(self._lib.cattus_b200_time_sustained(self._h, _ptr(words, _lib._u64p), None if bm is None else _ptr(bm, _lib._u8p), n, n_batches, iters,
                                                   C.byref(ms)))
        return float(ms.value)

    def metrics(self) -> dict:
        """The keys the trainer reads from the self-play summary (train_process.py:176-186) + extras."""
        m = Metrics()
        check(self._lib.cattus_b200_get_metrics(self._h, C.byref(m)))
        return {"model.activation_count": int(m.activation_count), "model.run_duration": float(m.run_duration_ema),
                "model.run_duration_last": float(m.run_duration_last), "model.positions": int(m.positions),
                "model.mean_batch_fill": float(m.mean_batch_fill), "model.kernel_launches": int(m.kernel_launches)}

    # ------------------------------------------------------------------ ValueFunction::evaluate
    def evaluate(self, position):
        """`impl ValueFunction<Game> for NNetwork<Game>` (hex/net.rs:6-10, chess/net/mod.rs:11-15, ttt/net.rs:6-10)
        -> NNetwork::evaluate (net/mod.rs:74-87).  `position` is one of cattus_b200.games.{Hex,Ttt,Chess}Position.
        Returns ([(move, prob)] in legal_moves() order, value from Player1's perspective)."""
        pos, flipped = (position, False) if position.turn == 1 else (position.flipped(), True)

        def compute(p):
            words = p.to_planes_words()
            legal = p.legal_moves()
            idx = [p.move_to_nn_idx(m) for m in legal]
            bitmap = None
            if self.needs_bitmap:
                bitmap = np.zeros(self.bitmap_bytes, dtype=np.uint8)
                for i in idx:
                    bitmap[i >> 3] |= np.uint8(1 << (i & 7))
            probs, val = self.eval_planes(words, bitmap)
            assert len(probs) == len(legal), "device legal count differs from legal_moves()"
            # the device returns ascending nn index; hand them back in legal_moves() order
            rank = {i: k for k, i in enumerate(sorted(idx))}
            return [(m, float(probs[rank[i]])) for m, i in zip(legal, idx)], val

        res = self.cache.get_or_compute(pos.key(), lambda: compute(pos)) if self.cache is not None else compute(pos)
        if not flipped:
            return res
        moves_probs, val = res
        return [(position.flip_move(m), p) for m, p in moves_probs], -val
