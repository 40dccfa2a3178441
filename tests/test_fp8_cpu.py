"""CPU: the FP8 (e4m3) numerics of CATTUS_B200_PRECISION_FP8, emulated by oracle/fp8.py: convnet_forward_fp8, and the FP8
instantiations of the whole-trunk kernel as the compiler builds them for sm_100a.

Bounds against the fp32 goldens (tests/golden/net_ref_*.npz, the reference ConvNetV1's outputs): value |delta| <= 0.05 and
total variation of the softmax over each position's legal moves <= 0.05.  About 10x the bf16 path's error; see DESIGN.md
section 12.
"""
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import fp8, games, net
from tests.util import GOLDEN, state_dict

FP8_GOLDENS = ["chess_4x64", "chess_2x128", "chess10x128", "chess_4x256"]  # every committed chess golden with 64 / 128 / 256 filters
TOL_VALUE = 0.05
TOL_TV = 0.05
CSRC = Path(__file__).resolve().parent.parent / "cattus_b200" / "csrc"


def _golden_inputs(name):
    g = np.load(GOLDEN / f"net_ref_{name}.npz")
    words, bitmaps = games.synth_chess_positions(len(g["words"]), seed=11)  # how oracle/gen_golden.py drew the golden positions
    assert np.array_equal(words, g["words"])
    legal = [games.legal_from_bitmap(bitmaps[i], net.CONFIGS[name].moves) for i in range(len(words))]
    return g, words, legal


def _softmax(logits, legal):
    z = logits[legal].astype(np.float64)
    z = np.exp(z - z.max())
    return z / z.sum()


def test_e4m3_round_is_rne_and_saturates():
    x = torch.tensor([1.0625, 1.1875, 3.125, -1.0625, 448.0, 449.0, 464.0, 1e6, -1e6, float("inf"), 2.0 ** -10, 3 * 2.0 ** -11, 0.0])
    got = fp8.e4m3_round(x)
    assert not torch.isnan(got).any()
    # 1.0625 is halfway between 1.0 and 1.125 -> even mantissa 1.0; 1.1875 between 1.125 and 1.25 -> 1.25; 3.125 between 3.0 and
    # 3.25 -> 3.0; 464 is halfway between 448 and the (non-finite in e4m3fn) 480 -> saturates; 2^-10 is half the smallest
    # subnormal 2^-9 -> 0; 1.5 * 2^-10 -> 2^-9
    want = [1.0, 1.25, 3.0, -1.0, 448.0, 448.0, 448.0, 448.0, -448.0, 448.0, 0.0, 2.0 ** -9, 0.0]
    assert got.tolist() == want
    # a value already on the e4m3 grid is kept
    grid = torch.arange(256, dtype=torch.uint8).view(torch.float8_e4m3fn).to(torch.float32)
    grid = grid[torch.isfinite(grid)]
    assert torch.equal(fp8.e4m3_round(grid), grid)


def test_per_channel_quantiser_maps_amax_to_448():
    w = torch.from_numpy(state_dict("chess_2x128")["_residual_blocks.0._conv1.weight"]).clone()
    w[5] = 0.0  # an all-zero channel
    q, d = fp8.quantize_per_channel(w)
    amax_q = q.abs().reshape(q.shape[0], -1).amax(dim=1)
    nz = torch.arange(w.shape[0]) != 5
    assert torch.all(amax_q[nz] == 448.0)
    assert torch.all(q[5] == 0.0) and d[5] == 1.0
    amax = w.abs().reshape(w.shape[0], -1).amax(dim=1)
    assert torch.equal(d[nz], (amax / 448.0)[nz])
    # dequantised weights are within half an e4m3 step (relative 2^-4) of the originals
    deq = q * d.reshape(-1, 1, 1, 1)
    assert torch.all((deq - w).abs() <= amax.reshape(-1, 1, 1, 1) * 2.0 ** -4 + 1e-12)


@pytest.mark.parametrize("name", ["chess_1x128", "chess_4x64"])
def test_emulation_without_quantisation_is_the_fp32_forward(name):
    cfg = net.CONFIGS[name]
    words, _ = games.synth_chess_positions(6, seed=3)
    x = games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    l0, v0 = fp8.convnet_forward_fp8(state_dict(name), cfg, x, quantize=False)
    lf, vf = net.convnet_forward(state_dict(name), cfg, x)
    np.testing.assert_allclose(l0, lf, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(v0, vf, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", FP8_GOLDENS)
def test_emulation_within_bounds_of_fp32_goldens(name):
    g, words, legal = _golden_inputs(name)
    cfg = net.CONFIGS[name]
    x = games.planes_to_tensor_fast(words, cfg.board_size, cfg.planes)
    logits, values = fp8.convnet_forward_fp8(state_dict(name), cfg, x)
    dv = float(np.abs(values - g["values"]).max())
    tv = max(0.5 * float(np.abs(_softmax(logits[i], legal[i]) - _softmax(g["logits"][i], legal[i])).sum()) for i in range(len(words)))
    print(f"{name}: fp8 emulation vs fp32 golden: max|dvalue|={dv:.4f} max policy TV={tv:.4f}")
    assert dv <= TOL_VALUE and tv <= TOL_TV
    assert dv > 0.0  # the emulation does quantise


def test_fp8_kernels_compile_without_spills_to_f8f6f4_mmas(tmp_path):
    """The FP8 instantiations of trunk_fused_kernel for sm_100a: no local-memory spills, and their MMAs are the kind::f8f6f4
    form (UTCQMMA in SASS), not the bf16 form (UTCHMMA)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cuobjdump = str(Path(nvcc).with_name("cuobjdump"))
    tu = tmp_path / "fp8_trunk.cu"
    tu.write_text('#include "trunk_fused.cuh"\n'
                  "void* fp8_kernels[] = {(void*)cb2::trunk_fused_kernel<64, __nv_fp8_e4m3>, (void*)cb2::trunk_fused_kernel<128, __nv_fp8_e4m3>,\n"
                  "                       (void*)cb2::trunk_fused_kernel<256, __nv_fp8_e4m3>};\n")
    cubin = tmp_path / "fp8_trunk.cubin"
    res = subprocess.run([nvcc, "-cubin", "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v", f"-I{CSRC}",
                          "-o", str(cubin), str(tu)], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    # ptxas prints, per entry function: "Compiling entry function '<mangled>'" ... "N bytes spill stores, M bytes spill loads"
    blocks = re.split(r"Compiling entry function '", res.stderr)[1:]
    fp8 = [b for b in blocks if b.startswith("_ZN3cb218trunk_fused_kernel") and "nv_fp8_e4m3" in b.split("'")[0]]
    assert len(fp8) == 3, res.stderr
    for b in fp8:
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", b)
        assert m and m.group(1) == "0" and m.group(2) == "0", b
    sass = subprocess.run([cuobjdump, "-sass", str(cubin)], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)[1:]
    seen = 0
    for f in funcs:
        if f.startswith("_ZN3cb218trunk_fused_kernel") and "nv_fp8_e4m3" in f.split("\n")[0]:
            seen += 1
            assert "UTCQMMA" in f and "UTCHMMA" not in f
    assert seen == 3
