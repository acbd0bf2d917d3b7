"""GPU: the branch-closing epilogue of the specialised resblock kernel (rbconv_tc.cu) -- 16-bit lrelu-domain residual,
planar fp16 branch sum accumulated and divided by the branch count, 16-bit stream out, with and without the branch sum
written back (acc_nostore) -- at every divisor the host accepts, on ragged last tiles and with B > 1.  Each case is bit
for bit the generic tcgen05 kernel and matches the fp64 restatement."""
import ctypes as C
import math

import pytest
import torch

from comfy_rvc_b200 import _lib, weights
from tests._emulate import conv_cl
from tests.test_tc_gpu import PADF, from_pv, pitch, to_pv

pytestmark = pytest.mark.gpu

EPI_CASES = [
    # name, B, L, C, ntaps, dil   (C = 256: the stage-1 shapes of the 48k decoder; ragged last tiles; batch)
    ("c256_k3_d1", 1, 1000, 256, 3, 1),
    ("c256_k11_d5_b2", 2, 5001, 256, 11, 5),
    ("c256_k7_d3_b3", 3, 777, 256, 7, 3),
    ("c256_k11_d1_long", 1, 20003, 256, 11, 1),
    ("c128_k11_d5_b2", 2, 3001, 128, 11, 5),
    ("c64_k7_d1", 1, 2049, 64, 7, 1),
]


def _desc(x16, w16, bias, r16, y32, y16, L, Cc, ntaps, dil, div, nostore, bf16):
    d = _lib.TcConvDesc()
    d.x16, d.L_in, d.padf = x16.data_ptr(), L, PADF
    d.w16, d.bias = w16.data_ptr(), bias.data_ptr()
    d.Cin, d.ntaps, d.dil, d.G = Cc, ntaps, dil, 1
    d.g_off[0] = -((ntaps - 1) // 2) * dil
    d.N, d.Cout_total = Cc, Cc
    d.Lj, d.out_stride, d.Lp_out = L, 1, pitch(L)
    d.res16, d.res_neg_scale = r16.data_ptr(), 10.0
    d.y32, d.acc_f16, d.accum, d.div = y32.data_ptr(), 1, 1, div
    d.y16, d.out_slope = y16.data_ptr(), 0.1
    d.acc_nostore = int(nostore)
    d.in_bf16, d.out_bf16 = int(bf16), 0
    return d


@pytest.mark.parametrize("nostore", [False, True], ids=["store", "nostore"])
@pytest.mark.parametrize("div", [2.0, 3.0, 4.0])
@pytest.mark.parametrize("bf16", [False, True], ids=["fp16", "bf16"])
@pytest.mark.parametrize("case", EPI_CASES, ids=[c[0] for c in EPI_CASES])
def test_rbconv_branch_closer(case, bf16, div, nostore):
    name, B, L, Cc, ntaps, dil = case
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    dt = torch.bfloat16 if bf16 else torch.float16
    g = torch.Generator().manual_seed(len(name) * 13 + Cc + ntaps + int(div))
    x = torch.randn(B, L, Cc, generator=g).to(dt).float()
    w = (torch.randn(1, ntaps, Cc, Cc, generator=g) / math.sqrt(Cc * ntaps)).to(dt).float()
    bias = torch.randn(Cc, generator=g)
    s = torch.randn(B, L, Cc, generator=g)
    stream = torch.where(s > 0, s, s * 0.1).half()                  # the lrelu-domain stream the previous conv stored
    res = torch.where(stream > 0, stream.float(), stream.float() * 10.0)
    acc0 = torch.randn(B, L, Cc, generator=g).half().float()
    ref = conv_cl(x.double(), w.double(), bias.double(), g_off=[-((ntaps - 1) // 2) * dil], dil=dil, out_stride=1)
    ref = (ref + res.double() + acc0.double()) / div
    x16, r16 = x.to(dt).to(dev).contiguous(), stream.to(dev).contiguous()
    w16, bd = weights.pack_tc(w, dt).to(dev), bias.to(dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    outs = []
    for fn in (lib.rvcb200_op_rbconv_tc, lib.rvcb200_op_conv_tc):
        y32 = to_pv(acc0, 8, torch.float16).to(dev)
        y16 = torch.zeros(B, L, Cc, dtype=torch.float16, device=dev)
        # the generic kernel always writes the branch sum back: it is the reference for both outputs
        d = _desc(x16, w16, bd, r16, y32, y16, L, Cc, ntaps, dil, div, nostore and fn is lib.rvcb200_op_rbconv_tc, bf16)
        assert fn(C.byref(d), B, st) == 0
        torch.cuda.synchronize()
        outs.append((y32.cpu(), y16.cpu()))
    (y32, y16), (g32, g16) = outs
    assert torch.equal(y16.view(torch.int16), g16.view(torch.int16))
    want16 = torch.where(ref > 0, ref, ref * 0.1)
    assert (y16.double() - want16).abs().max().item() < 0.02
    got = from_pv(g32.float(), L).double()
    assert (got - ref).abs().max().item() < 6e-3
    if nostore:
        assert torch.equal(y32.view(torch.int16), to_pv(acc0, 8, torch.float16).view(torch.int16))   # untouched
    else:
        assert torch.equal(y32.view(torch.int16), g32.view(torch.int16))
        assert float(y32[:, :, :PADF].abs().max()) == 0.0 and float(y32[:, :, PADF + L:].abs().max()) == 0.0


def test_tc_convs_reject_inexact_divisors():
    """The divide-free mean is exact only for the divisors it was checked for: others are refused, not approximated."""
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    B, L, Cc, ntaps = 1, 300, 256, 3
    x16 = torch.zeros(B, L, Cc, dtype=torch.float16, device=dev)
    w16 = weights.pack_tc(torch.zeros(1, ntaps, Cc, Cc), torch.float16).to(dev)
    bd = torch.zeros(Cc, device=dev)
    y32 = torch.zeros(B, Cc // 8, pitch(L), 8, dtype=torch.float16, device=dev)
    y16 = torch.zeros(B, L, Cc, dtype=torch.float16, device=dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for div in (5.0, 2.5, 0.0):
        d = _desc(x16, w16, bd, x16, y32, y16, L, Cc, ntaps, 1, div, False, False)
        assert lib.rvcb200_op_rbconv_tc(C.byref(d), B, st) != 0
        assert lib.rvcb200_op_conv_tc(C.byref(d), B, st) != 0
