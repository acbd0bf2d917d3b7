"""CPU: the fp64 restatement of the generic tcgen05 epilogue (tests/_tc_generic_ref.py) on cases small enough to check by
hand -- the gate's column pairing, the sign of res_mode 2, the order of the masks, scale and slopes."""
import math

import torch

from tests._tc_generic_ref import generic_ref, ulp16


def _one(vals):
    """x = 1 at every row, one tap, Cin = 1: the convolution output of column c is w[c], i.e. `vals`."""
    w = torch.tensor(vals, dtype=torch.float64)[None, None, :]
    return torch.ones(1, 2, 1, dtype=torch.float64), w, torch.zeros(len(vals), dtype=torch.float64)


def test_gate_pairs_interleaved_columns():
    x, w, b = _one([0.5, -1.0, 2.0, 3.0])
    v, y16 = generic_ref(x, w, b, 2, gate=True)
    want = [math.tanh(0.5) / (1 + math.exp(1.0)), math.tanh(2.0) / (1 + math.exp(-3.0))]
    assert v.shape == (1, 2, 2)
    assert torch.allclose(v[0, 0], torch.tensor(want, dtype=torch.float64), rtol=0, atol=1e-15)
    assert torch.equal(v, y16)


def test_residual_modes_and_relu():
    x, w, b = _one([2.0, -4.0])
    r = torch.full((1, 2, 2), 5.0, dtype=torch.float64)
    assert torch.equal(generic_ref(x, w, b, 2, res=r, res_mode=1)[0][0, 0], torch.tensor([7.0, 1.0], dtype=torch.float64))
    assert torch.equal(generic_ref(x, w, b, 2, res=r, res_mode=2)[0][0, 0], torch.tensor([3.0, 9.0], dtype=torch.float64))
    r2 = torch.full((1, 2, 2), 1.0, dtype=torch.float64)
    assert torch.equal(generic_ref(x, w, b, 2, res=r2, relu=True)[0][0, 0], torch.tensor([3.0, 0.0], dtype=torch.float64))


def test_mask_order():
    """mask_pre zeroes the convolution before the residual (masked rows = residual), mask_post the result, mask16 only
    the 16-bit copy."""
    x, w, b = _one([2.0])
    r = torch.full((1, 2, 1), 5.0, dtype=torch.float64)
    ol = torch.tensor([1])
    v, _ = generic_ref(x, w, b, 2, res=r, mask_pre=True, out_len=ol)
    assert v[0, :, 0].tolist() == [7.0, 5.0]
    v, y16 = generic_ref(x, w, b, 2, res=r, mask_pre=True, mask_post=True, out_len=ol)
    assert v[0, :, 0].tolist() == [7.0, 0.0] and y16[0, :, 0].tolist() == [7.0, 0.0]
    v, y16 = generic_ref(x, w, b, 2, mask16=True, out_len=ol)
    assert v[0, :, 0].tolist() == [2.0, 2.0] and y16[0, :, 0].tolist() == [2.0, 0.0]


def test_scale_slopes_accum_div():
    x, w, b = _one([-1.0])
    g = torch.tensor([[0.5], [3.0]], dtype=torch.float64)
    gidx = torch.tensor([[1, 0]])
    v, _ = generic_ref(x, w, b + 0.25, 2, gather=g, gidx=gidx, alpha=2.0)     # (-1 + 0.25 + gather) * 2
    assert v[0, :, 0].tolist() == [4.5, -0.5]
    v, _ = generic_ref(x, w, b, 2, pre_slope=0.1, gelu=True)                  # lrelu before GELU
    assert abs(v[0, 0, 0].item() - 0.5 * -0.1 * (1 + math.erf(-0.1 / math.sqrt(2)))) < 1e-15
    acc = torch.full((1, 2, 1), 7.0, dtype=torch.float64)
    v, y16 = generic_ref(x, w, b, 2, acc=acc, div=3.0, out_slope=0.1)         # (v + acc) / div; out_slope on y16 only
    assert v[0, 0, 0].item() == 2.0 and y16[0, 0, 0].item() == 2.0
    v, y16 = generic_ref(x, w, b, 2, out_slope=0.1)
    assert v[0, 0, 0].item() == -1.0 and abs(y16[0, 0, 0].item() + 0.1) < 1e-15


def test_grouped_channel_slices():
    """a_nt_stride: output tile nt reads input channels [nt * stride, + Cin)."""
    x = torch.tensor([[[1.0, 10.0, 100.0]]], dtype=torch.float64)            # B 1, L 1, 3 channels
    w = torch.ones(1, 2, 2, dtype=torch.float64)                              # Cin 2, Cout 2, N 1
    v, _ = generic_ref(x, w, torch.zeros(2, dtype=torch.float64), 1, a_nt_stride=1, N=1)
    assert v[0, 0].tolist() == [11.0, 110.0]


def test_taps_and_offsets():
    x = torch.arange(1.0, 5.0, dtype=torch.float64)[None, :, None]            # rows 1 2 3 4
    w = torch.tensor([[[1.0]], [[10.0]]], dtype=torch.float64)                # tap 0 -> row t - 1, tap 1 -> row t
    v, _ = generic_ref(x, w, torch.zeros(1, dtype=torch.float64), 4, g_off=-1)
    assert v[0, :, 0].tolist() == [10.0, 21.0, 32.0, 43.0]


def test_ulp16():
    v = torch.tensor([1.0, 1.5, 2.0, 0.0, 1e-6, -65504.0, 2.0 ** -14])
    assert ulp16(v).tolist() == [2.0 ** -10, 2.0 ** -10, 2.0 ** -9, 2.0 ** -24, 2.0 ** -24, 32.0, 2.0 ** -24]
    h = torch.tensor([0.1, 3.3, 700.0]).half().double()
    assert bool(((h - torch.tensor([0.1, 3.3, 700.0], dtype=torch.float64)).abs() <= ulp16(h) / 2).all())
