"""GPU: the two HuBERT-only C ABI entries against fp64, and the front end at the lengths the benchmark runs.

* `rvcb200_op_hubert_conv0` (Conv1d 1 -> C, k 10, stride 5 -> GroupNorm -> GELU; statistics from the Gram matrix of the
  input windows, accumulated with double atomics over blocks of 256 frames);
* `rvcb200_op_layernorm16` (both `NV` instantiations of the row LayerNorm, with its fp16 copy);
* `HubertB200.extract_features` on 30 s and 60 s of audio, where the feature encoder runs at N = 256 and the projections
  at N = 128 / 256 (pass-by-pass epilogue, no residual prefetch) -- shapes the 10 s golden fixture never reaches."""
import ctypes as C
import types

import pytest
import torch
import torch.nn.functional as F

from comfy_rvc_b200 import _lib, synthetic
from comfy_rvc_b200.hubert import HubertB200
from tests._tc_generic_ref import ulp16

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
K0, S0, C0 = 10, 5, 512


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _conv0(x, w, gw, gb, stats, y16, B, n, Cn, K, S, y_bstride):
    return _lib.load().rvcb200_op_hubert_conv0(C.c_void_p(x.data_ptr()), C.c_void_p(w.data_ptr()), C.c_void_p(gw.data_ptr()),
                                               C.c_void_p(gb.data_ptr()), C.c_void_p(stats.data_ptr()),
                                               C.c_void_p(y16.data_ptr()), B, n, Cn, K, S, 1e-5, y_bstride, _stream())


@pytest.mark.parametrize("signal", ["speech", "dc", "zero"])
@pytest.mark.parametrize("L0", [1, 255, 256, 257, 191999])
def test_hubert_conv0_matches_fp64(L0, signal):
    dev = torch.device("cuda", 0)
    B = 2
    n = (L0 - 1) * S0 + K0 + 3                         # 3 trailing samples that make no further frame
    g = torch.Generator().manual_seed(L0 + len(signal))
    x = torch.randn(B, n, generator=g) * 0.3
    if signal == "dc":
        x = x * 0.1 + 10.0                             # |mean| >> std: the variance is a small difference of large moments
    elif signal == "zero":
        x = torch.zeros(B, n)
    w = torch.randn(C0, K0, generator=g) / K0 ** 0.5
    gw, gb = 1.0 + 0.1 * torch.randn(C0, generator=g), 0.3 * torch.randn(C0, generator=g)
    xd, wd, gwd, gbd = (t.to(dev).contiguous() for t in (x, w, gw, gb))
    y_bstride = L0 * C0 + 1000
    stats = torch.empty(B * 2 * C0, dtype=torch.float64, device=dev)
    outs = []
    for _ in range(2):
        y16 = torch.full((B * y_bstride,), float("nan"), dtype=torch.float16, device=dev)
        assert _conv0(xd, wd, gwd, gbd, stats, y16, B, n, C0, K0, S0, y_bstride) == 0
        torch.cuda.synchronize()
        outs.append(y16)
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), "two calls differ"
    yb = outs[0].view(B, y_bstride)
    assert bool(torch.isnan(yb[:, L0 * C0:]).all()), "wrote into the gap between batch items"
    got = yb[:, :L0 * C0].view(B, L0, C0).double()
    # fp64 reference on the device (checker only)
    win = xd.double().unfold(1, K0, S0)[:, :L0]                        # [B][L0][K]
    y = win @ wd.double().t()                                          # [B][L0][C]
    mean, var = y.mean(1, keepdim=True), y.var(1, unbiased=False, keepdim=True)
    scale = gwd.double() / torch.sqrt(var + 1e-5)
    v = (y - mean) * scale + gbd.double()
    ref = 0.5 * v * (1.0 + torch.erf(v / 2 ** 0.5))
    # the kernel recomputes the convolution and normalises in fp32: allow that arithmetic's rounding, scaled as it
    # propagates (|GELU'| <= 1.13), on top of one fp16 ulp
    mag = (win.abs() @ wd.double().abs().t()) + mean.abs()
    tol = ulp16(ref) + 1.13 * (2 * (K0 + 4) * EPS32 * mag * scale.abs() + 4 * EPS32 * v.abs())
    excess = ((got - ref).abs() - tol).max().item()
    print(f"conv0 L0={L0} {signal}: max|err| {(got - ref).abs().max().item():.3e}, "
          f"max err / ulp {((got - ref).abs() / ulp16(ref)).max().item():.2f}")
    assert excess <= 0
    if signal == "zero":                                              # y = 0, variance 0: GELU(gn_b) in every frame
        assert bool((got == got[:, :1]).all())
        gelu_b = 0.5 * gbd.double() * (1.0 + torch.erf(gbd.double() / 2 ** 0.5))
        assert bool(((got[:, 0] - gelu_b).abs() <= ulp16(gelu_b)).all())


def test_hubert_conv0_rejections():
    dev = torch.device("cuda", 0)
    x, w = torch.zeros(2000, device=dev), torch.zeros(C0 * 17, device=dev)
    gw, gb = torch.ones(C0, device=dev), torch.zeros(C0, device=dev)
    stats = torch.zeros(2 * C0, dtype=torch.float64, device=dev)
    y16 = torch.zeros(400 * C0, dtype=torch.float16, device=dev)
    assert _conv0(x, w, gw, gb, stats, y16, 1, 2000, C0, 10, 5, 399 * C0) == 0           # the base call is accepted
    torch.cuda.synchronize()
    assert _conv0(x, w, gw, gb, stats, y16, 1, 2000, C0, 17, 5, 399 * C0) == 1           # K > 16
    assert _conv0(x, w, gw, gb, stats, y16, 1, 9, C0, 10, 5, 399 * C0) == 1              # n < K
    assert _conv0(x, w, gw, gb, stats, y16, 1, 2000, 50, 10, 5, 399 * 50) == 1           # 2 C < K^2 + K (Gram scratch)


@pytest.mark.parametrize("Cn", [192, 256, 257, 512, 768, 1024])
def test_layernorm16_matches_fp64(Cn):
    dev = torch.device("cuda", 0)
    rows = 1003                                                        # not a multiple of the 8 rows per block
    g = torch.Generator().manual_seed(Cn)
    x = torch.randn(rows, Cn, generator=g)
    off = torch.zeros(rows, 1)
    off[::5] = 300.0 * torch.sign(torch.randn(len(range(0, rows, 5)), 1, generator=g))    # |mean| >> std rows
    x = x + off
    gamma, beta = 1.0 + 0.2 * torch.randn(Cn, generator=g), 0.5 * torch.randn(Cn, generator=g)
    xd, gd, bd = x.to(dev), gamma.to(dev), beta.to(dev)
    y = torch.full((rows + 8, Cn), float("nan"), device=dev)
    y16 = torch.full((rows + 8, Cn), float("nan"), dtype=torch.float16, device=dev)
    st = _lib.load().rvcb200_op_layernorm16(C.c_void_p(xd.data_ptr()), C.c_void_p(gd.data_ptr()), C.c_void_p(bd.data_ptr()),
                                            C.c_void_p(y.data_ptr()), C.c_void_p(y16.data_ptr()), rows, Cn, 1e-5, _stream())
    assert st == 0
    torch.cuda.synchronize()
    assert bool(torch.isnan(y[rows:]).all()) and bool(torch.isnan(y16[rows:]).all())
    got = y[:rows].double()
    ref = F.layer_norm(xd.double(), (Cn,), gd.double(), bd.double(), 1e-5)
    # fp32 single-warp sums: the mean carries ~(C/32 + 8) roundings of |x|, which the normalisation divides by std
    xs = xd.double()
    ratio = xs.mean(1, keepdim=True).abs() / xs.std(1, unbiased=False, keepdim=True)
    tol = 5e-5 + 1e-6 * (Cn / 32 + 8) * ratio * gd.double().abs().max()
    err = (got - ref).abs()
    plain = ratio[:, 0] < 10
    print(f"layernorm16 C={Cn}: max|err| {err[plain].max().item():.3e} (plain rows), {err[~plain].max().item():.3e} (offset rows)")
    assert bool((err <= tol).all())
    assert torch.equal(y16[:rows].view(torch.int16), y[:rows].half().view(torch.int16)), "y16 is not fp16(y)"


@pytest.mark.parametrize("seconds", [60.0, 30.0])
def test_hubert_long_input_matches_oracle(seconds):
    """The benchmark's utterance length: conv stack at N = 256, projections at N = 128 / 256, against the fp32 oracle run
    on the device (TF32 off) as a checker."""
    from oracle import hubert_oracle
    hsd = synthetic.make_hubert_state_dict(0)
    model = HubertB200(synthetic.HUBERT_BASE, hsd, "cuda:0")
    wav = synthetic.make_speech(seconds, seed=5).cuda()
    n = wav.shape[1]
    L1 = ((n - K0) // S0 + 1 - 3) // 2 + 1                           # rows of feature-encoder conv 1 (k 3, stride 2)
    assert (L1 + 127) // 128 >= 148                                   # hubert.py: conv 1 runs at N = 256
    flags = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
        sd_dev = {k: v.cuda() for k, v in hsd.items()}
        for version in ("v1", "v2"):
            f = model.extract_features(version=version, source=wav)
            ref = hubert_oracle.extract_features(sd_dev, types.SimpleNamespace(**synthetic.HUBERT_BASE), wav, version)
            torch.cuda.synchronize()
            assert f.shape == ref.shape
            snr = synthetic.snr_db(ref.cpu().numpy(), f.float().cpu().numpy())
            print(f"HuBERT {seconds:.0f} s {version}: SNR {snr:.1f} dB, {model.last_launches} launches")
            assert snr >= 45.0
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = flags
    if seconds == 60.0:                                               # 2 999 frames: the N = 128 / 256 images were used
        assert "fp.w@128" in model._w and "l0.ff1.w@256" in model._w
