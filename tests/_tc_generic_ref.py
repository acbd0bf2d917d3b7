"""fp64 restatement of the generic epilogue of `rvcb200_op_conv_tc` (`generic = 1`, include/rvcb200.h) -- test
infrastructure for tests/test_tc_generic_gpu.py.

The kernel (csrc/conv_tc.cu, `epilogue_generic16` and its whole-tile form `epilogue_lean64`) applies the modes in this
order, and so does `generic_ref`:

   1. conv + bias + cond[b]
   2. + gather[gidx[b][t]], then * alpha
   3. gate on interleaved (tanh, sigmoid) column pairs: out[c] = tanh(v[2c]) * sigmoid(v[2c + 1])
   4. lrelu(pre_slope), then GELU (erf form)
   5. mask_pre: rows t >= out_len[b] -> 0
   6. residual: v + r (res_mode 1) or r - v (res_mode 2)
   7. relu
   8. + the running sum already in y32 (accum), then / div
   9. mask_post: rows t >= out_len[b] -> 0
  10. y16 = lrelu(v, out_slope), zeroed for rows t >= out_len[b] with mask16

Every argument is a tensor of the dtype / device the caller computes in (float64 for a reference).  `x` is the
activation COLUMN SLICE the launch reads ([B][L_in][Cin], i.e. what `ldx16` and the x16 pointer select); `w` is
[taps][Cin][Cout].  With `a_nt_stride` (grouped convolution) output tile nt (N columns) reads input channels
[nt * a_nt_stride, + Cin) of `x`, whose width is then a_nt_stride * (Cout / N - 1) + Cin.
"""
from __future__ import annotations

import torch

from tests._emulate import conv_cl


def _lrelu(v, slope):
    return torch.where(v > 0, v, v * slope) if slope != 1.0 else v


def row_mask(out_len, B, L, device):
    """[B][L][1] bool: True where t < out_len[b] (all True without out_len)."""
    if out_len is None:
        return torch.ones(B, L, 1, dtype=torch.bool, device=device)
    t = torch.arange(L, device=device)[None, :]
    return (t < out_len.to(device).long()[:, None])[:, :, None]


def generic_ref(x, w, bias, Lj, *, g_off=0, cond=None, gather=None, gidx=None, alpha=1.0, gate=False, pre_slope=1.0,
                gelu=False, mask_pre=False, res=None, res_mode=1, relu=False, acc=None, div=1.0, mask_post=False,
                out_len=None, out_slope=1.0, mask16=False, a_nt_stride=0, N=None):
    """Returns (v, y16) as `x.dtype` [B][Lj][Cout'] (Cout' = Cout / 2 with the gate): `v` is what y32 receives, `y16` the
    unrounded value the 16-bit output receives.  cond [B][Cout], gather [V][Cout], gidx [B][Lj] (int64), res / acc
    [B][Lj][Cout'], out_len [B] (int)."""
    B, L_in, _ = x.shape
    ntaps, Cin, Cout = w.shape
    if a_nt_stride:
        parts = []
        for nt in range(Cout // N):
            xs = x[:, :, nt * a_nt_stride:nt * a_nt_stride + Cin]
            parts.append(conv_cl(xs, w[None, :, :, nt * N:(nt + 1) * N], g_off=[g_off]))
        v = torch.cat(parts, dim=2)
    else:
        v = conv_cl(x, w[None], g_off=[g_off])
    v = v[:, :Lj] if L_in >= Lj else torch.nn.functional.pad(v, (0, 0, 0, Lj - L_in))
    v = v + bias
    if cond is not None:
        v = v + cond[:, None, :]
    if gather is not None:
        v = v + gather[gidx]
    v = v * alpha
    if gate:
        v = torch.tanh(v[..., 0::2]) * torch.sigmoid(v[..., 1::2])
    v = _lrelu(v, pre_slope)
    if gelu:
        v = 0.5 * v * (1.0 + torch.erf(v / 2 ** 0.5))
    valid = row_mask(out_len, B, Lj, v.device)
    zero = torch.zeros((), dtype=v.dtype, device=v.device)
    if mask_pre:
        v = torch.where(valid, v, zero)
    if res is not None:
        v = res - v if res_mode == 2 else v + res
    if relu:
        v = torch.clamp_min(v, 0.0)
    if acc is not None:
        v = v + acc
    v = v / div
    if mask_post:
        v = torch.where(valid, v, zero)
    y16 = _lrelu(v, out_slope)
    if mask16:
        y16 = torch.where(valid, y16, zero)
    return v, y16


def ulp16(v):
    """One fp16 ulp at |v| (2^-24 in the subnormal range), as float64."""
    a = v.abs().double()
    _, e = torch.frexp(a)                          # |v| = m 2^e, m in [0.5, 1); 0 -> e = 0
    u = torch.clamp(torch.ldexp(torch.ones_like(a), e - 11), min=2.0 ** -24)
    return torch.where(a == 0, torch.full_like(a, 2.0 ** -24), u)
