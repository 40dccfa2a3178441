"""CPU oracle (TEST INFRASTRUCTURE ONLY) for the FP8 (e4m3) precision of the whole-trunk kernel
(CATTUS_B200_PRECISION_FP8): ConvNetV1's forward pass under the same numerics contract, in fp32 torch on the CPU.

Only `tests/` import this.
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np

from .net import BN_EPS, NetConfig

E4M3_MAX = 448.0  # largest finite e4m3 value


def e4m3_round(x):
    """fp32 torch tensor -> the nearest e4m3 value (round to nearest even), saturating to +-448, returned as fp32: what
    `cvt.rn.satfinite.e4m3x2.f32` computes.  torch's own cast returns NaN above 448, hence the clamp first."""
    import torch

    return x.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(torch.float32)


def fold_bn(sd: Dict[str, np.ndarray], conv_key: str, bn_prefix: str, affine: bool) -> Tuple[np.ndarray, np.ndarray]:
    """BatchNorm folded into the preceding bias-free conv exactly as cattus_b200.export writes it into the .cb2 blob
    (float64 arithmetic, stored as float32): w' = w * gamma / sqrt(var + eps), b' = beta - mean * gamma / sqrt(var + eps)."""
    w = np.asarray(sd[conv_key], dtype=np.float64)
    mean = np.asarray(sd[f"{bn_prefix}.running_mean"], dtype=np.float64)
    var = np.asarray(sd[f"{bn_prefix}.running_var"], dtype=np.float64)
    gamma = np.asarray(sd[f"{bn_prefix}.weight"], dtype=np.float64) if affine else np.ones_like(mean)
    beta = np.asarray(sd[f"{bn_prefix}.bias"], dtype=np.float64) if affine else np.zeros_like(mean)
    scale = gamma / np.sqrt(var + BN_EPS)
    return (w * scale[:, None, None, None]).astype(np.float32), (beta - mean * scale).astype(np.float32)


def quantize_per_channel(w):
    """Per-output-channel e4m3 weights (torch fp32 [OC, ...]): amax_oc = max |w_oc|, q = e4m3(w * (448 / amax_oc)), dequant
    factor d_oc = amax_oc / 448 (fp32); an all-zero channel gets d_oc = 1.  Returns (q as fp32 values, d [OC])."""
    import torch

    amax = w.abs().reshape(w.shape[0], -1).amax(dim=1)
    nz = amax > 0
    one = torch.ones_like(amax)
    qs = torch.where(nz, torch.tensor(E4M3_MAX, dtype=torch.float32) / torch.where(nz, amax, one), one)
    d = torch.where(nz, amax / torch.tensor(E4M3_MAX, dtype=torch.float32), one)
    return e4m3_round(w * qs.reshape(-1, *([1] * (w.dim() - 1)))), d


def convnet_forward_fp8(sd: Dict[str, np.ndarray], cfg: NetConfig, x: np.ndarray, quantize: bool = True) -> Tuple[np.ndarray, np.ndarray]:
    """ConvNetV1.forward under the FP8 numerics of the whole-trunk kernel (CATTUS_B200_PRECISION_FP8):
      1. the BN-folded weights of the stem, block convs and both 1x1 head convs are quantised per output channel
         (quantize_per_channel);
      2. every conv input (A operand) is cast to e4m3 without a scale (the 0/1 stem input is exact);
      3. products are accumulated in fp32;
      4. the epilogue computes relu(acc * d_oc + bias_oc (+ residual)) in fp32;
      5. the residual stream (the block input conv2 adds) is kept in bf16;
      6. the head convs' outputs are rounded to bf16 (the FC kernels' A operands); the head FCs, tanh and the policy logits
         are computed in fp32 here (the device runs them in bf16 as at precision BF16).
    quantize=False turns every cast and quantisation off: the result is then convnet_forward's to fp32 round-off.
    x [B,C,S,S] f32 -> (policy logits [B,M], value [B,1])."""
    import torch
    import torch.nn.functional as F

    assert cfg.arch == "convnet"
    t = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}
    ident = (lambda a: a)
    act8 = e4m3_round if quantize else ident
    res16 = (lambda a: a.to(torch.bfloat16).to(torch.float32)) if quantize else ident

    def conv(conv_key, bn_prefix, affine, a, pad):
        w, b = fold_bn(sd, conv_key, bn_prefix, affine)
        w = torch.from_numpy(w)
        if quantize:
            q, d = quantize_per_channel(w)
        else:
            q, d = w, torch.ones(w.shape[0], dtype=torch.float32)
        acc = F.conv2d(act8(a), q, padding=pad)
        return acc * d.reshape(1, -1, 1, 1) + torch.from_numpy(b).reshape(1, -1, 1, 1)

    with torch.no_grad():
        flow = torch.relu(conv("_conv1._conv.weight", "_conv1._bn", True, torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)), 1))
        for i in range(cfg.blocks):
            p = f"_residual_blocks.{i}"
            resid = res16(flow)
            h = torch.relu(conv(f"{p}._conv1.weight", f"{p}._bn1", False, flow, 1))
            flow = torch.relu(conv(f"{p}._conv2.weight", f"{p}._bn2", True, h, 1) + resid)
        v = res16(torch.relu(conv("_value_head.0._conv.weight", "_value_head.0._bn", False, flow, 0)))
        v = torch.relu(F.linear(v.flatten(1), t["_value_head.2.weight"], t["_value_head.2.bias"]))
        v = torch.tanh(F.linear(v, t["_value_head.4.weight"], t["_value_head.4.bias"]))
        p_ = res16(torch.relu(conv("_policy_head.0._conv.weight", "_policy_head.0._bn", False, flow, 0)))
        p_ = F.linear(p_.flatten(1), t["_policy_head.2.weight"], t["_policy_head.2.bias"])
    return p_.numpy(), v.numpy()
