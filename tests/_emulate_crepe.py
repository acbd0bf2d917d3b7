"""Float64 CPU emulation of the device CREPE network's data layout (comfy_rvc_b200/crepe.py, csrc/crepe_kernels.cu): the
polyphase conv1 operand, the tap matrices of `host_weights`, BatchNorm + pool into padded lines, and the packed classifier input.
It runs the same contractions the tcgen05 launches run, row for row, so it checks the layouts and the weight packing exactly."""
from __future__ import annotations

import torch

from comfy_rvc_b200 import crepe


def frames_operand(frames: torch.Tensor) -> torch.Tensor:
    """Normalised frames [B, 1024] -> conv1 operand [B][368][64]: row t, channel c = frame[4 t + c - 254] (0 outside)."""
    pad = torch.nn.functional.pad(frames, (254, 254 + 4 * 368 + 64 - 1532))
    idx = 4 * torch.arange(368)[:, None] + torch.arange(64)[None, :]
    return pad[:, idx]


def conv_rows(x: torch.Tensor, taps: torch.Tensor, bias: torch.Tensor, dil: int, g_off: int, lj: int) -> torch.Tensor:
    """One generic-kernel launch for one batch item: y[j] = relu(bias + sum_t x[j + g_off + t dil] @ taps[t]), rows outside x = 0."""
    L = x.shape[0]
    y = bias.double().expand(lj, -1).clone()
    for t in range(taps.shape[0]):
        r = torch.arange(lj) + g_off + t * dil
        ok = (r >= 0) & (r < L)
        xs = torch.zeros(lj, x.shape[1], dtype=torch.float64)
        xs[ok] = x[r[ok]]
        y += xs @ taps[t].double()
    return torch.relu(y)


def bn_pool(x: torch.Tensor, scale, shift, frames: int, L: int, p_in: int, in_off: int, p_out: int, out_off: int) -> torch.Tensor:
    C = x.shape[-1]
    x = x.reshape(frames, p_in, C)[:, in_off:in_off + L] * scale.double() + shift.double()
    pooled = torch.maximum(x[:, 0::2], x[:, 1::2])
    out = torch.zeros(frames, p_out, C, dtype=torch.float64)
    out[:, out_off:out_off + L // 2] = pooled
    return out


def network(frames: torch.Tensor, W: dict, model: str) -> torch.Tensor:
    """Normalised frames [B, 1024] -> classifier logits [B, 360], float64, through the device layouts."""
    cin, cout, nf = crepe.CHANNELS[model]
    L = crepe.LENGTHS
    B = frames.shape[0]
    x = frames_operand(frames.double())
    y = torch.stack([conv_rows(x[b], W["conv1.taps"], W["conv1.b"], 16, 0, 256) for b in range(B)])
    p = bn_pool(y, W["bn1.scale"], W["bn1.shift"], B, 256, 256, 0, 128, 0)
    y = torch.stack([conv_rows(p[b], W["conv2.taps"], W["conv2.b"], 1, -31, 128) for b in range(B)])
    p_prev = 128
    for i in range(2, 6):
        P = L[i] + 32
        p = bn_pool(y, W[f"bn{i}.scale"], W[f"bn{i}.shift"], B, L[i - 1], p_prev, 0, P, 31).reshape(B * P, -1)
        y = conv_rows(p, W[f"conv{i + 1}.taps"], W[f"conv{i + 1}.b"], 1, 0, B * P)
        p_prev = P
    feat = bn_pool(y, W["bn6.scale"], W["bn6.shift"], B, L[5], p_prev, 0, L[5] // 2, 0).reshape(B, nf)
    return (feat @ W["cls.taps"][0].double() + W["cls.b"].double())[:, :360]
