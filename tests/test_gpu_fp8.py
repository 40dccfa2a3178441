"""GPU (-m gpu): precision FP8 -- the e4m3 instantiations of the whole-trunk kernel -- against the FP8 emulation of the oracle
(oracle/fp8.py: convnet_forward_fp8) and against the fp32 goldens, plus the shapes it refuses.

Bars: kernel vs FP8 emulation within 1e-2 on probabilities and values (the bf16 path's tolerance against fp32; 2e-2 for the
10-block net, see TOL_DEEP); kernel vs the
fp32 goldens within value |delta| <= 0.05 and policy total variation <= 0.05 (tests/test_fp8_cpu.py holds the emulation to the
same bounds); outputs for a position are bit-identical whatever batch, lane or entry point it went through.
"""
import threading

import numpy as np
import pytest

from oracle import fp8, games, net
from tests.test_fp8_cpu import FP8_GOLDENS, TOL_TV, TOL_VALUE, _golden_inputs, _softmax
from tests.util import blob, make_network, state_dict, synth_inputs

pytestmark = pytest.mark.gpu

TOL = 1e-2
# Kernel and emulation are both exact to the contract, but their fp32 sums differ in the last bits, and where such a difference
# straddles an e4m3 rounding boundary one activation moves by a whole e4m3 step (2^-3 relative).  Depth amplifies those flips:
# measured on a B200, max |dprob| / |dvalue| was <= 1e-3 up to 4 blocks and 1.0e-2 / 1.3e-2 (B = 64) and 1.3e-2 / 1.4e-2 (B = 1500)
# for the 10-block net, whose random-init outputs are the most sensitive (DESIGN.md section 12).  That net gets 2e-2.
TOL_DEEP = {"chess10x128": 2e-2}


def _fp8_oracle(name, words, legal):
    cfg = net.CONFIGS[name]
    x = games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    logits, values = fp8.convnet_forward_fp8(state_dict(name), cfg, x)
    return values.reshape(-1), [games.calc_moves_probs(legal[i], games.clamp_non_finite(logits[i])) for i in range(len(legal))]


def test_fp8_handles_report_fused_trunk_and_precision():
    from cattus_b200._lib import PRECISION_FP8

    for name in ("chess_0x128", "chess_1x128", "chess_2x128", "chess10x128", "chess_4x64", "chess_4x256"):
        with make_network(name, precision="fp8", batch_size=16, n_streams=1) as nw:
            assert nw.trunk_path == "fused", (name, nw.trunk_path)
            assert nw.info.precision == PRECISION_FP8


# n = 1 and 7: one tile per CTA (split epilogue); 64: one tile, several pairs; >= 1024: two tiles per CTA (F <= 128), ragged buckets
@pytest.mark.parametrize("name,n,batch", [("chess_0x128", 7, 8), ("chess_1x128", 64, 64), ("chess_2x128", 1100, 2048),
                                          ("chess10x128", 1, 16), ("chess10x128", 7, 16), ("chess10x128", 64, 64), ("chess10x128", 1500, 2048),
                                          ("chess_4x64", 7, 16), ("chess_4x64", 1300, 2048), ("chess_4x256", 64, 64), ("chess_4x256", 1024, 1024)])
def test_fp8_kernel_matches_fp8_oracle(name, n, batch):
    words, bitmaps, legal = synth_inputs(name, n, 4242)
    with make_network(name, precision="fp8", batch_size=batch) as nw:
        probs, offsets, values = nw.eval_batch(words, bitmaps)
    assert np.diff(offsets.astype(np.int64)).tolist() == [len(l) for l in legal]
    idx = np.linspace(0, n - 1, min(n, 48)).astype(int)  # the CPU emulation of a large batch is slow: a spread sample
    o_values, o_probs = _fp8_oracle(name, words[idx], [legal[i] for i in idx])
    worst_p = max([float(np.abs(probs[offsets[i]:offsets[i + 1]] - o_probs[k]).max()) for k, i in enumerate(idx) if len(legal[i])] + [0.0])
    worst_v = float(np.abs(values[idx] - o_values).max())
    print(f"{name} n={n}: fp8 kernel vs fp8 oracle max|dprob|={worst_p:.3e} max|dvalue|={worst_v:.3e}")
    tol = TOL_DEEP.get(name, TOL)
    assert worst_p <= tol and worst_v <= tol


@pytest.mark.parametrize("name", FP8_GOLDENS)
def test_fp8_kernel_within_bounds_of_fp32_goldens(name):
    g, words, legal = _golden_inputs(name)
    _, bitmaps = games.synth_chess_positions(len(words), seed=11)
    with make_network(name, precision="fp8", batch_size=16) as nw:
        probs, offsets, values = nw.eval_batch(words, bitmaps)
    dv = float(np.abs(values - g["values"].reshape(-1)).max())
    tv = max(0.5 * float(np.abs(probs[offsets[i]:offsets[i + 1]] - _softmax(g["logits"][i], legal[i])).sum()) for i in range(len(words)))
    print(f"{name}: fp8 kernel vs fp32 golden max|dvalue|={dv:.4f} max policy TV={tv:.4f}")
    assert dv <= TOL_VALUE and tv <= TOL_TV


def test_fp8_batch_invariance_across_batches_lanes_and_entry_points():
    name = "chess10x128"
    n = 4096
    words, bitmaps, _ = synth_inputs(name, n, 515)
    with make_network(name, precision="fp8", batch_size=n, n_streams=4) as nw:
        ref_p, ref_o, ref_v = nw.eval_batch(words, bitmaps)
        for i in (0, 1, 777, n - 1):
            p1, o1, v1 = nw.eval_batch(words[i:i + 1], bitmaps[i:i + 1])
            assert np.array_equal(p1, ref_p[ref_o[i]:ref_o[i + 1]]) and v1[0] == ref_v[i], i
            p, v = nw.eval_planes(words[i], bitmaps[i])
            assert np.array_equal(p, ref_p[ref_o[i]:ref_o[i + 1]]) and v == ref_v[i], i
        # concurrent callers ride different evaluator lanes
        out, errors = [None] * 4, []

        def worker(k):
            try:
                out[k] = nw.eval_batch(words[k * 500:(k + 1) * 500 + 37], bitmaps[k * 500:(k + 1) * 500 + 37])
            except Exception as e:  # surfaced below
                errors.append(e)

        threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert not errors, errors[0]
        for k in range(4):
            p, o, v = out[k]
            lo, hi = k * 500, (k + 1) * 500 + 37
            assert np.array_equal(p, ref_p[ref_o[lo]:ref_o[hi]]) and np.array_equal(v, ref_v[lo:hi]), k
        # the device-resident path
        nw.resident_upload(words, bitmaps)
        nw.eval_resident(n)
        rp, ro, rv = nw.resident_download(n)
    assert np.array_equal(ro, ref_o) and np.array_equal(rp, ref_p) and np.array_equal(rv, ref_v)


def test_fp8_device_chess_games_equal_host_driver_games():
    from cattus_b200.selfplay import SelfPlayRunner
    from tests.test_gpu_dsearch import games_of
    from tests.test_selfplay_cpu import cfg_with

    base = dict(prior_noise_alpha=0.3, prior_noise_epsilon=0.25, temperature_policy=[[20, 1.0], [9999, 0.0]], seed=9, sim_num=16, max_moves=12)
    with make_network("chess10x128", precision="fp8", batch_size=64) as nw:
        assert nw.trunk_path == "fused"
        s_host, host = SelfPlayRunner("chess", cfg_with(cache_size=50000, threads=2, games_per_thread=2, **base)).generate_data(nw, None, 4, keep_records=True)
        s_dev, dev = SelfPlayRunner("chess", cfg_with(device_games=4, **base)).generate_data(nw, None, 4, keep_records=True)
    assert games_of(dev) == games_of(host)
    assert s_dev["metrics"]["selfplay.simulations"] == s_host["metrics"]["selfplay.simulations"]


@pytest.mark.parametrize("name,fused_trunk", [("hex5", True), ("chess_dev", True), ("chess_simple", True), ("chess10x128", False)])
def test_fp8_is_refused_outside_the_whole_trunk_kernel(name, fused_trunk):
    from cattus_b200 import CudaNetwork
    from cattus_b200._lib import EINVAL, CattusB200Error

    with pytest.raises(CattusB200Error) as ei:
        CudaNetwork(blob(name), net.CONFIGS[name].game, batch_size=16, precision="fp8", fused_trunk=fused_trunk)
    assert ei.value.code == EINVAL
    assert "FP8" in str(ei.value) and "64 / 128 / 256 filters" in str(ei.value)


def test_fp8_run_dense_is_refused():
    from cattus_b200._lib import EINVAL, CattusB200Error

    cfg = net.CONFIGS["chess_2x128"]
    words, bitmaps = games.synth_chess_positions(3, seed=1)
    x = games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    with make_network("chess_2x128", precision="fp8", batch_size=16) as nw:
        with pytest.raises(CattusB200Error) as ei:
            nw.run(x)
        assert ei.value.code == EINVAL and "FP8" in str(ei.value)
        probs, offsets, values = nw.eval_batch(words, bitmaps)  # the handle still works after the refusal
        assert np.isfinite(values).all()
