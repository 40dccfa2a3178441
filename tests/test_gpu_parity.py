"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle on the same seeded inputs.

Bars (BASELINE.json north_star): feature planes and legal masks bit-exact; policy and value within max abs error
1e-4 in the fp32 check mode and 1e-2 at bf16.  The reference's own tolerance between its engines is rtol 1e-3 on the
policy and 1e-5 on the value (training/tests/test_net_output.py:28-33); the fp32 check mode is held to that shape too.
"""
import threading

import numpy as np
import pytest

from oracle import games, net
from tests.util import GOLDEN, make_network, oracle_eval, state_dict, synth_inputs

pytestmark = pytest.mark.gpu

TOL_FP32 = 1e-4  # max abs error on probabilities and value, fp32 check mode
TOL_BF16 = 1e-2  # max abs error on probabilities and value, bf16 tensor-core path

ALL = ["ttt", "hex4", "hex5", "hex7", "hex9", "hex11", "chess_dev", "chess_2x128", "chess10x128", "ttt_1x1", "hex11_1x1", "chess_1x1", "hex5_2x2",
       # widths / depths the reference's config recommends (chess_dev.yaml:30-37) outside the two whole-trunk kernels: per-layer path
       "chess_4x64", "chess_4x256", "hex7_4x32", "hex11_2x128",
       # the reference's second model type (net_utils.py:92-121)
       "ttt_simple", "hex5_simple", "hex11_simple", "chess_simple"]


# ----------------------------------------------------------------------------------------------- encode (bit-exact)
@pytest.mark.parametrize("tag,name", [("ttt", "ttt"), ("hex11", "hex11"), ("chess", "chess_dev"), ("rand3", "ttt"), ("rand4", "hex4"),
                                      ("rand5", "hex5"), ("rand7", "hex7"), ("rand9", "hex9"), ("rand11", "hex11"), ("rand8", "chess_dev")])
@pytest.mark.parametrize("precision", ["bf16", "fp32-check"])
def test_encode_bit_exact_vs_reference_fixtures(tag, name, precision):
    g = np.load(GOLDEN / "encode_ref.npz")
    words, ref = g[f"{tag}_words"], g[f"{tag}_tensor"].astype(np.float32)
    with make_network(name, precision=precision, batch_size=16) as nw:
        out = nw.planes_to_tensor(words, batch_size=len(words) + 3)
        assert out.dtype == np.float32 and out.shape == (len(words) + 3,) + ref.shape[1:]
        assert np.array_equal(out[: len(words)], ref)
        assert not out[len(words):].any()  # padding rows are zeros (net/mod.rs:144-152)


def test_encode_random_large_and_errors():
    from cattus_b200._lib import CattusB200Error, EINVAL, ERANGE

    for name, n in (("hex7", 4096), ("chess_dev", 2048), ("hex11", 1000)):
        cfg = net.CONFIGS[name]
        rng = np.random.default_rng(21)
        wpp = games.words_per_plane(cfg.board_size)
        words = rng.integers(0, 2 ** 64, size=(n, cfg.planes * wpp), dtype=np.uint64)
        with make_network(name, batch_size=4096) as nw:
            out = nw.planes_to_tensor(words)
            assert np.array_equal(out, games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes))
            with pytest.raises(CattusB200Error) as ei:  # the reference asserts 1..=batch_size (net/mod.rs:122-127)
                nw.planes_to_tensor(words[:5], batch_size=4)
            assert ei.value.code == EINVAL
            with pytest.raises(CattusB200Error) as ei:
                nw.planes_to_tensor(words[:5], batch_size=5000)
            assert ei.value.code == ERANGE


# ----------------------------------------------------------------------------------------------- Model::run parity
@pytest.mark.parametrize("name", ALL)
def test_run_dense_fp32_check_vs_reference_golden(name):
    """fp32 check mode against the outputs the reference's ConvNetV1 / SimpleTwoHeadedModel produced (tests/golden/net_ref_*.npz)."""
    g = np.load(GOLDEN / f"net_ref_{name}.npz")
    cfg = net.CONFIGS[name]
    x = games.planes_to_tensor_fast(g["words"], cfg.board_size, cfg.planes)
    with make_network(name, precision="fp32-check", batch_size=16) as nw:
        logits, values = nw.run(x)
    assert logits.shape == g["logits"].shape and values.shape == g["values"].shape
    err_l = np.abs(logits - g["logits"]).max()
    err_v = np.abs(values - g["values"]).max()
    print(f"{name}: fp32-check max|dlogit|={err_l:.3e} max|dvalue|={err_v:.3e}")
    assert err_l <= TOL_FP32 * max(1.0, np.abs(g["logits"]).max()) and err_v <= TOL_FP32
    np.testing.assert_allclose(logits, g["logits"], rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize("name", ALL)
def test_run_dense_bf16_vs_reference_golden(name):
    g = np.load(GOLDEN / f"net_ref_{name}.npz")
    cfg = net.CONFIGS[name]
    x = games.planes_to_tensor_fast(g["words"], cfg.board_size, cfg.planes)
    with make_network(name, precision="bf16", batch_size=16) as nw:
        logits, values = nw.run(x)
    err_l = np.abs(logits - g["logits"]).max()
    err_v = np.abs(values - g["values"]).max()
    print(f"{name}: bf16 max|dlogit|={err_l:.3e} (|logit|max {np.abs(g['logits']).max():.2f}) max|dvalue|={err_v:.3e}")
    assert err_v <= TOL_BF16
    # logits feed a softmax: what the contract bounds is the probability error, checked in test_eval_batch_*; here a
    # gross-error guard (a wrong tap, a permuted FC column or a missing ReLU moves logits by O(1))
    assert err_l <= 0.08 * max(1.0, np.abs(g["logits"]).max())


def test_info_says_which_trunk_path_a_handle_got():
    """cattus_b200_info.trunk_path: the whole-trunk kernels cover fixed shapes; everything else takes the per-layer kernel."""
    for name, want in (("chess10x128", "fused"), ("chess_2x128", "fused"), ("hex5", "small"), ("chess_dev", "small"), ("chess_4x64", "fused"),
                       ("chess_4x256", "fused"), ("hex7_4x32", "per-layer"), ("hex11_2x128", "per-layer"), ("hex5_simple", "dense")):
        with make_network(name, batch_size=16, n_streams=1) as nw:
            assert nw.trunk_path == want, (name, nw.trunk_path)
    with make_network("hex5", precision="fp32-check", batch_size=16, n_streams=1) as nw:
        assert nw.trunk_path == "fp32-check"
    with make_network("chess10x128", batch_size=16, n_streams=1, fused_trunk=False) as nw:
        assert nw.trunk_path == "per-layer"


# ----------------------------------------------------------------------------------------------- evaluate parity
def _check_eval(name, precision, n, seed, tol, batch_size=256, n_streams=2):
    words, bitmaps, legal = synth_inputs(name, n, seed)
    _, o_values, o_probs = oracle_eval(name, words, legal)
    with make_network(name, precision=precision, batch_size=batch_size, n_streams=n_streams) as nw:
        probs, offsets, values = nw.eval_batch(words, bitmaps)
        m = nw.metrics()
    counts = np.diff(offsets.astype(np.int64))
    assert counts.tolist() == [len(l) for l in legal]  # legal masks bit-exact (same count, same order by construction)
    assert offsets[0] == 0 and offsets[-1] == len(probs)
    worst_p = 0.0
    for i in range(n):
        p = probs[offsets[i]:offsets[i + 1]]
        if len(p):
            assert abs(float(p.sum()) - 1.0) < 1e-4
            worst_p = max(worst_p, float(np.abs(p - o_probs[i]).max()))
    worst_v = float(np.abs(values - o_values).max())
    print(f"{name}/{precision}: n={n} max|dprob|={worst_p:.3e} max|dvalue|={worst_v:.3e} batches={m['model.activation_count']}")
    assert worst_p <= tol and worst_v <= tol
    assert np.all(np.abs(values) <= 1.0)
    assert m["model.kernel_launches"] > 0 and m["model.positions"] >= n
    return probs, offsets, values


@pytest.mark.parametrize("name", ["ttt", "hex4", "hex5", "hex7", "hex9", "hex11", "chess_dev", "chess_2x128", "chess_4x64", "hex7_4x32", "hex11_2x128",
                                  "ttt_simple", "hex5_simple", "hex11_simple", "chess_simple"])
def test_eval_batch_fp32_check(name):
    _check_eval(name, "fp32-check", 48, 101, TOL_FP32, batch_size=32)


@pytest.mark.parametrize("name", ["ttt", "hex4", "hex5", "hex7", "hex9", "hex11", "chess_dev", "chess_2x128", "chess10x128", "chess_4x64", "chess_4x256",
                                  "hex7_4x32", "hex11_2x128", "ttt_simple", "hex5_simple", "hex11_simple", "chess_simple"])
def test_eval_batch_bf16(name):
    _check_eval(name, "bf16", 300, 202, TOL_BF16, batch_size=128)


def test_reference_fixture_positions_end_to_end():
    """The 14 positions of training/tests/test_net_output.py:138-204 through evaluate(), both precisions, tiny nets the
    reference's own parity test builds (1 block x 1 filter)."""
    from cattus_b200.games import HexPosition, TttPosition
    from oracle.gen_golden import HEX11_FIXTURES, TTT_FIXTURES

    for precision, tol in (("fp32-check", TOL_FP32), ("bf16", TOL_BF16)):
        with make_network("ttt_1x1", precision=precision, batch_size=8) as nw:
            for s in TTT_FIXTURES:
                x, o, turn = games.ttt_position_from_str(s)
                mp, val = nw.evaluate(TttPosition(x, o, turn))
                legal = [i for i in range(9) if not ((x | o) >> i) & 1]
                _, ov, op = oracle_eval("ttt_1x1", games.pack_planes([games.ttt_position_to_planes(x, o)], 3), [legal])
                assert [m for m, _ in mp] == legal
                assert np.abs(np.array([p for _, p in mp]) - op[0]).max() <= tol and abs(val - ov[0]) <= tol
        with make_network("hex11_1x1", precision=precision, batch_size=8) as nw:
            for s in HEX11_FIXTURES:
                red, blue, turn = games.hex_position_from_str(s, 11)
                mp, val = nw.evaluate(HexPosition(11, red, blue, turn))
                planes, legal, _ = games.hex_evaluate_inputs(red, blue, turn, 11)
                _, ov, op = oracle_eval("hex11_1x1", games.pack_planes([planes], 11), [legal])
                assert [m for m, _ in mp] == legal
                assert np.abs(np.array([p for _, p in mp]) - op[0]).max() <= tol and abs(val - ov[0]) <= tol


def test_reference_chess_fixture_positions_end_to_end():
    """The 5 chess positions of training/tests/test_net_output.py:198-204 from their FENs: the library's chess rules give
    planes, legal moves and policy indices (cattus_b200.games.ChessPosition.from_fen), evaluate() runs the net; checked
    against the oracle's rules (oracle/chess.py) + the oracle net, both precisions, the reference test's 1 x 1 net."""
    from cattus_b200.games import ChessPosition
    from oracle import chess as oc
    from oracle.gen_golden import CHESS_FIXTURES

    for precision, tol in (("fp32-check", TOL_FP32), ("bf16", TOL_BF16)):
        with make_network("chess_1x1", precision=precision, batch_size=8) as nw:
            for fen in CHESS_FIXTURES + ["rnbqkbnr/pppp1ppp/8/8/4pP2/8/PPPPP1PP/RNBQKBNR b KQkq f3 0 2"]:  # + black to move, en passant
                mp, val = nw.evaluate(ChessPosition.from_fen(fen))
                p = oc.ChessPosition.from_fen(fen)
                view = p if p.turn == oc.P1 else p.flipped()
                moves = view.legal_moves()
                nn = [oc.ChessPosition.to_nn_idx(m) for m in moves]
                _, ov, op = oracle_eval("chess_1x1", np.array([view.planes()], dtype=np.uint64), [sorted(nn)])
                rank = {idx: k for k, idx in enumerate(sorted(nn))}
                want = [op[0][rank[i]] for i in nn]
                real = moves if p.turn == oc.P1 else [oc.ChessPosition.flip_move(m) for m in moves]
                assert [m for m, _ in mp] == real
                assert np.abs(np.array([q for _, q in mp]) - np.array(want)).max() <= tol
                assert abs(val - (ov[0] if p.turn == oc.P1 else -ov[0])) <= tol


def test_flip_path_player2_to_move():
    """Not covered by any reference parity test (SURVEY.md section 4): blue to move -> planes [T(blue), T(red), ones],
    moves transposed back, value negated (hex/core.rs:324-334, :36-38; net/mod.rs:166-182)."""
    from cattus_b200.games import HexPosition

    rng = np.random.default_rng(77)
    with make_network("hex5", precision="fp32-check", batch_size=8) as nw:
        for _ in range(6):
            cells = rng.permutation(25)[: int(rng.integers(1, 20))]
            red = sum(1 << int(c) for c in cells[0::2])
            blue = sum(1 << int(c) for c in cells[1::2])
            mp, val = nw.evaluate(HexPosition(5, red, blue, 2))
            planes, legal, flipped = games.hex_evaluate_inputs(red, blue, 2, 5)
            assert flipped
            _, ov, op = oracle_eval("hex5", games.pack_planes([planes], 5), [legal])
            assert [m for m, _ in mp] == [games.hex_move_flipped(m, 5) for m in legal]
            assert np.abs(np.array([p for _, p in mp]) - op[0]).max() <= TOL_FP32 and abs(val - (-ov[0])) <= TOL_FP32
            assert sorted(m for m, _ in mp) == games.hex_legal_moves(red, blue, 5)


def test_non_finite_and_degenerate_policy_rows():
    """Clamp + masked softmax edge cases on the device tail (net/mod.rs:57-61, :106-119): a single legal move gets
    probability 1; no legal move gives an empty slice; a full board of legal moves sums to 1."""
    name = "hex4"
    full = (1 << 16) - 1
    samples = [games.hex_position_to_planes(full & ~(1 << 5), 0, 4), games.hex_position_to_planes(full, 0, 4), games.hex_position_to_planes(0, 0, 4)]
    words = games.pack_planes(samples, 4)
    with make_network(name, precision="bf16", batch_size=4) as nw:
        probs, offsets, values = nw.eval_batch(words)
    assert offsets.tolist() == [0, 1, 1, 17]
    assert probs[0] == 1.0 and abs(probs[1:].sum() - 1.0) < 1e-5 and np.isfinite(values).all()


# ----------------------------------------------------------------------------------------------- fused trunk
@pytest.mark.parametrize("name,n,batch", [("chess_0x128", 37, 64), ("chess_1x128", 37, 64), ("chess_2x128", 150, 64), ("chess10x128", 700, 512),
                                          # the other widths of the template (F = 64: two tiles per CTA at the larger batch; F = 256: 3-tap weight stages)
                                          ("chess_4x64", 37, 64), ("chess_4x64", 1500, 2048), ("chess_4x256", 37, 64), ("chess_4x256", 900, 1024)])
def test_fused_trunk_matches_per_layer_path_and_oracle(name, n, batch):
    """The whole-trunk kernel (trunk_fused.cuh: encode + stem + residual blocks, activations resident in shared memory,
    CTA pairs) against the per-layer tcgen05 GEMM path on the same handle parameters, and both against the oracle.
    Depth ladder (0, 1, 2, 10 blocks) localises a fault to the stem / conv1 / conv2+residual / steady state."""
    words, bitmaps, legal = synth_inputs(name, n, 313)
    _, o_values, o_probs = oracle_eval(name, words, legal)
    with make_network(name, batch_size=batch, fused_trunk=True) as a, make_network(name, batch_size=batch, fused_trunk=False) as b:
        assert a.fused_trunk and not b.fused_trunk
        assert a.info.kernels_per_batch < b.info.kernels_per_batch
        pa, oa, va = a.eval_batch(words, bitmaps)
        pb, ob, vb = b.eval_batch(words, bitmaps)
    assert np.array_equal(oa, ob)
    d_paths = max(float(np.abs(pa - pb).max()), float(np.abs(va - vb).max()))
    worst = max(float(np.abs(pa[oa[i]:oa[i + 1]] - o_probs[i]).max()) for i in range(n))
    worst_v = float(np.abs(va - o_values).max())
    print(f"{name}: fused vs per-layer {d_paths:.3e}; fused vs oracle prob {worst:.3e} value {worst_v:.3e}")
    assert d_paths <= TOL_BF16 and worst <= TOL_BF16 and worst_v <= TOL_BF16


@pytest.mark.parametrize("name", ["ttt", "hex4", "hex5", "hex7", "hex9", "hex11", "chess_dev"])
@pytest.mark.parametrize("n,batch", [(3, 4), (90, 128), (700, 1024), (5000, 4096)])
def test_small_trunk_matches_per_layer_path_and_oracle(name, n, batch):
    """The 16-filter whole-trunk kernel (trunk_small.cuh: encode + stem + residual blocks + both head convs, strip
    layout in shared memory) against the per-layer tcgen05 GEMM path and the oracle, at batch sizes that select every
    tiles-per-CTA variant (1, 2, 4, 8) and more than one round per CTA."""
    words, bitmaps, legal = synth_inputs(name, n, 515)
    with make_network(name, batch_size=batch, fused_trunk=True) as a, make_network(name, batch_size=batch, fused_trunk=False) as b:
        assert a.small_trunk and not b.small_trunk
        assert a.info.kernels_per_batch < b.info.kernels_per_batch
        pa, oa, va = a.eval_batch(words, bitmaps)
        pb, ob, vb = b.eval_batch(words, bitmaps)
        p1, _, v1 = a.eval_batch(words[:1], None if bitmaps is None else bitmaps[:1])
    assert np.array_equal(oa, ob)
    assert np.array_equal(p1, pa[oa[0]:oa[1]]) and v1[0] == va[0]  # batch invariant across tile variants
    d_paths = max(float(np.abs(pa - pb).max()), float(np.abs(va - vb).max()))
    idx = np.linspace(0, n - 1, min(n, 40)).astype(int)
    _, o_values, o_probs = oracle_eval(name, words[idx], [legal[i] for i in idx])
    worst = max([float(np.abs(pa[oa[i]:oa[i + 1]] - o_probs[k]).max()) for k, i in enumerate(idx) if len(legal[i])] + [0.0])
    worst_v = float(np.abs(va[idx] - o_values).max())
    print(f"{name} n={n}: small-trunk vs per-layer {d_paths:.3e}; vs oracle prob {worst:.3e} value {worst_v:.3e}")
    assert d_paths <= TOL_BF16 and worst <= TOL_BF16 and worst_v <= TOL_BF16


# ----------------------------------------------------------------------------------------------- batching semantics
def test_per_leaf_eval_is_thread_safe_and_batch_invariant():
    """cattus_b200_eval from many threads (the Batcher replacement, util/batch.rs:49-177) must return exactly what the
    bulk call returns for the same position, whatever batch it happened to ride in (ValueFuncCache relies on it)."""
    name = "hex7"
    n = 256
    words, _, legal = synth_inputs(name, n, 404)
    with make_network(name, precision="bf16", batch_size=32, n_streams=2) as nw:
        ref_probs, ref_off, ref_vals = nw.eval_batch(words)
        # 16 concurrent callers must share device batches.  How many leaves ride together depends on the host's thread
        # scheduling (a loaded box can serialise the Python threads), so the workload is repeated until one pass shows sharing;
        # the results are checked on every pass.
        shared = False
        for attempt in range(5):
            out = [None] * n
            start = threading.Barrier(16)
            before = nw.metrics()["model.activation_count"]

            def worker(k):
                start.wait()
                for i in range(k, n, 16):
                    out[i] = nw.eval_planes(words[i])

            threads = [threading.Thread(target=worker, args=(k,)) for k in range(16)]
            [t.start() for t in threads]
            [t.join() for t in threads]
            m = nw.metrics()
            for i in range(n):
                p, v = out[i]
                assert np.array_equal(p, ref_probs[ref_off[i]:ref_off[i + 1]]), f"position {i}: probabilities differ from the bulk call's"
                assert v == ref_vals[i], f"position {i}: value {v} differs from the bulk call's {ref_vals[i]}"
            leaf_batches = m["model.activation_count"] - before
            print("leaf batches:", leaf_batches, "fill:", m["model.mean_batch_fill"])
            if leaf_batches < n:
                shared = True
                break
        assert shared, "no two leaves shared a device batch in 5 passes of 16 concurrent callers"


@pytest.mark.parametrize("name", ["chess_dev", "hex5"])
def test_concurrent_bulk_batches_of_ragged_sizes(name):
    """Many host threads in cattus_b200_eval_batch at once with batch sizes that leave most of a bucket as padding (the
    self-play regime: all-padding rounds and tiles are skipped on the device) and chunks large enough for the shared
    packing helpers: every caller must get exactly the rows a single caller gets."""
    sizes = [1, 37, 129, 300, 650, 1100, 1290, 1500]
    words, bitmaps, _ = synth_inputs(name, 1500, 77)
    with make_network(name, precision="bf16", batch_size=2048, n_streams=8) as nw:
        ref_probs, ref_off, ref_vals = nw.eval_batch(words, bitmaps)
        errors = []

        def worker(k):
            try:
                for it in range(6):
                    b = sizes[(k + it) % len(sizes)]
                    p, o, v = nw.eval_batch(words[:b], None if bitmaps is None else bitmaps[:b])
                    assert np.array_equal(o, ref_off[: b + 1]) and np.array_equal(p, ref_probs[: ref_off[b]]) and np.array_equal(v, ref_vals[:b])
            except Exception as e:  # surfaced in the main thread below
                errors.append(e)

        threads = [threading.Thread(target=worker, args=(k,)) for k in range(12)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors[0]


def test_chess_per_leaf_with_bitmap_and_cache():
    from cattus_b200 import ValueFuncCache

    name = "chess_dev"
    words, bitmaps, legal = synth_inputs(name, 40, 55)
    with make_network(name, precision="bf16", batch_size=16, cache=ValueFuncCache(8)) as nw:
        ref_probs, ref_off, ref_vals = nw.eval_batch(words, bitmaps)
        for i in range(40):
            p, v = nw.eval_planes(words[i], bitmaps[i])
            assert np.array_equal(p, ref_probs[ref_off[i]:ref_off[i + 1]]) and v == ref_vals[i]
            assert len(p) == len(legal[i])


@pytest.mark.parametrize("name,n,batch", [("hex5", 20000, 4096), ("chess10x128", 3000, 1024)])
def test_full_size_properties(name, n, batch):
    """Sizes the oracle cannot finish quickly: size-independent properties.  (1) probabilities of every position sum
    to 1 and are non-negative; (2) |value| <= 1; (3) legal counts equal the popcount of the mask; (4) batch invariance:
    positions evaluated inside a large batch equal the same positions evaluated in a small one; (5) a sample is checked
    against the oracle."""
    words, bitmaps, legal = synth_inputs(name, n, 909)
    with make_network(name, precision="bf16", batch_size=batch, n_streams=2) as nw:
        probs, offsets, values = nw.eval_batch(words, bitmaps)
        sub = slice(100, 164)
        p2, o2, v2 = nw.eval_batch(words[sub], None if bitmaps is None else bitmaps[sub])
    counts = np.diff(offsets.astype(np.int64))
    assert counts.tolist() == [len(l) for l in legal]
    sums = np.add.reduceat(probs, offsets[:-1][counts > 0].astype(np.int64))
    assert np.abs(sums - 1.0).max() < 1e-4 and probs.min() >= 0.0
    assert np.abs(values).max() <= 1.0
    assert np.array_equal(p2, probs[offsets[100]:offsets[164]]) and np.array_equal(v2, values[sub])
    idx = np.linspace(0, n - 1, 24).astype(int)
    _, ov, op = oracle_eval(name, words[idx], [legal[i] for i in idx])
    worst = max(float(np.abs(probs[offsets[i]:offsets[i + 1]] - op[k]).max()) for k, i in enumerate(idx) if len(legal[i]))
    assert worst <= TOL_BF16 and np.abs(values[idx] - ov).max() <= TOL_BF16


@pytest.mark.parametrize("name", ["hex4", "chess_dev"])
@pytest.mark.parametrize("precision", ["bf16", "fp32-check"])
def test_non_finite_logits_are_clamped_like_the_reference(name, precision):
    """run_net replaces non-finite logits by f32::MIN before the softmax (net/mod.rs:57-61): a legal move whose logit
    overflowed gets probability 0, and a position whose legal moves ALL overflowed gets the uniform distribution
    (exp(MIN - MIN) = 1 each).  Forced here with two policy-FC rows of 3e38 (finite weights, infinite dot product)."""
    from cattus_b200 import CudaNetwork
    from cattus_b200.export import export_blob

    cfg = net.CONFIGS[name]
    sd = {k: np.array(v, copy=True) for k, v in state_dict(name).items()}
    hot = [3, 7]
    sd["_policy_head.2.weight"][hot, :] = 3.0e38
    n = 24
    words, bitmaps, legal = synth_inputs(name, n, 77)
    if bitmaps is not None:  # chess: make the hot moves legal everywhere, and ONLY them in the last two positions
        for i in range(n):
            keep = set(hot) if i >= n - 2 else set(legal[i]) | set(hot)
            legal[i] = sorted(keep)
            bitmaps[i] = games.bitmap_from_legal(legal[i], cfg.moves)
    x = games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    logits, o_values = net.convnet_forward(sd, cfg, x)
    assert not np.isfinite(logits[:, hot]).any(), "the construction did not overflow the hot logits"
    with CudaNetwork(export_blob(sd, cfg.game), cfg.game, batch_size=32, precision=precision) as nw:
        probs, offsets, values = nw.eval_batch(words, bitmaps)
    tol = TOL_BF16 if precision == "bf16" else TOL_FP32
    seen_partial = seen_all = 0
    for i in range(n):
        ref = games.calc_moves_probs(legal[i], games.clamp_non_finite(logits[i]))
        got = probs[offsets[i]:offsets[i + 1]]
        assert len(got) == len(ref)
        if not len(ref):
            continue
        assert np.abs(got - ref).max() <= tol
        is_hot = np.array([m in hot for m in legal[i]])
        if is_hot.all():
            assert np.allclose(got, 1.0 / len(got), atol=1e-6)
            seen_all += 1
        elif is_hot.any():
            assert (got[is_hot] == 0.0).all() and abs(float(got.sum()) - 1.0) < 1e-4
            seen_partial += 1
    assert seen_partial > 0 and (seen_all > 0 or bitmaps is None)
    assert np.abs(values - o_values.reshape(-1)).max() <= tol

