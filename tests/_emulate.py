"""CPU emulation of the channels-last convolution contract of `rvcb200_conv_desc`
(include/rvcb200.h) — test infrastructure for the host-side weight packing."""
from __future__ import annotations

import torch


def conv_cl(x, w, bias=None, g_off=(0,), dil=1, out_stride=1, in_slope=1.0, in_len=None):
    """x [B][L][Cin], w [G][taps][Cin][Cout] -> y [B][L*out_stride][Cout]   (Lj = L rows per group)."""
    B, L, Cin = x.shape
    G, ntaps, _, Cout = w.shape
    xa = torch.where(x > 0, x, x * in_slope)
    if in_len is not None:
        m = (torch.arange(L, device=x.device)[None, :] < in_len[:, None]).to(x.dtype)
        xa = xa * m[:, :, None]
    y = torch.zeros(B, L * out_stride, Cout, dtype=x.dtype, device=x.device)
    for g in range(G):
        acc = torch.zeros(B, L, Cout, dtype=x.dtype, device=x.device)
        for t in range(ntaps):
            off = g_off[g] + t * dil
            lo, hi = max(0, -off), min(L, L - off)
            if hi > lo:
                acc[:, lo:hi] += xa[:, lo + off:hi + off] @ w[g, t]
        if bias is not None:
            acc = acc + bias
        y[:, g::out_stride] = acc
    return y
