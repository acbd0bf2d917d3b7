"""CREPE f0 estimator on the B200 kernels: a torchcrepe drop-in (`from comfy_rvc_b200 import crepe as torchcrepe`).

    pitch, periodicity = crepe.predict(audio [1, n] 16 kHz, 16000, hop_length, fmin, fmax, "full",
                                       decoder=crepe.decode.viterbi, return_periodicity=True, batch_size=..., device="cuda:0")

Weights: torchcrepe's state-dict layout (`conv{1..6}.weight [Co, Ci, k, 1]`, `conv{i}.bias`, `conv{i}_BN.*`,
`classifier.{weight, bias}`), loaded with `load_weights(model, path_or_state_dict)`; without that, `assets/{model}.pth` of an
installed torchcrepe is used.  Every FLOP of the network and the decoders runs in librvcb200.so (include/rvcb200.h):
  * `rvcb200_op_crepe_frames`: device audio -> normalised fp16 frames in conv1's operand layout (8 taps at dilation 16 over 64
    overlapping polyphase channels: K = 512, no im2col);
  * conv1..conv6 + ReLU and the classifier on the generic tcgen05 kernel (`rvcb200_op_conv_tc`).  conv1 / conv2 take one frame
    per batch item (the tensor map's zero fill is the padding); conv3..conv6 take the frames of a pass as ONE sequence of
    padded lines (L + 32 rows a frame, the 31 / 32 rows of zero padding shared between neighbours);
  * `rvcb200_op_crepe_bn_pool`: BatchNorm + max_pool (2, 1) into the next layer's layout (its padding rows written as 0);
  * `rvcb200_op_crepe_decode`: sigmoid, fmin / fmax masking, argmax / weighted_argmax / Viterbi (float64, one CTA per chunk)
    and the periodicity gather.
Frames go through the network in passes of `PASS_FRAMES`, so the network's scratch is fixed (~0.9 GB for `full`) whatever the
song length; the decoder's buffers are 5 KB per frame.  One host -> device copy of the audio, one device -> host copy of the
result (returned on `audio.device`, like torchcrepe).  The dither of `bins_to_cents` is drawn on the host with torchcrepe's own
call (numpy's global RNG, same order) and uploaded, so a seeded run gives torchcrepe's draws.
There is no PyTorch or CPU fallback: without the extension or a CUDA device every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import types
from typing import Dict, Optional, Union

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from .weights import pack_tc

CENTS_PER_BIN, MAX_FMAX, PITCH_BINS, SAMPLE_RATE, WINDOW_SIZE = 20, 2006.0, 360, 16000, 1024
UNVOICED = np.nan
CENTS_OFFSET = 1997.3794084376191
BN_EPS = 0.0010000000474974513
CHANNELS = {"full": ([1, 1024, 128, 128, 128, 256], [1024, 128, 128, 128, 256, 512], 2048),
            "tiny": ([1, 128, 16, 16, 16, 32], [128, 16, 16, 16, 32, 64], 256)}
LENGTHS = [256, 128, 64, 32, 16, 8]     # conv output rows per frame (before the pool)
FRAME_ROWS, FRAME_C, CONV1_TAPS, CONV1_DIL = 368, 64, 8, 16
PASS_FRAMES = 1024
N_PAD = 384                              # classifier outputs padded to a multiple of the N tile
BAND = 11
PADF = 32


# ---- convert ---------------------------------------------------------------------------------------------------------------
def _dither_noise(size) -> np.ndarray:
    import scipy.stats
    return scipy.stats.triang.rvs(c=0.5, loc=-20, scale=40, size=size)


def _bins_to_cents(bins):
    cents = CENTS_PER_BIN * bins + CENTS_OFFSET
    return cents + cents.new_tensor(_dither_noise(cents.size()))


def _bins_to_frequency(bins):
    return _cents_to_frequency(_bins_to_cents(bins))


def _cents_to_bins(cents, quantize_fn=torch.floor):
    return quantize_fn((cents - CENTS_OFFSET) / CENTS_PER_BIN).int()


def _cents_to_frequency(cents):
    return 10 * 2 ** (cents / 1200)


def _frequency_to_cents(frequency):
    return 1200 * torch.log2(frequency / 10.0)


def _frequency_to_bins(frequency, quantize_fn=torch.floor):
    return _cents_to_bins(_frequency_to_cents(frequency), quantize_fn)


convert = types.SimpleNamespace(bins_to_cents=_bins_to_cents, cents_to_bins=_cents_to_bins, bins_to_frequency=_bins_to_frequency,
                                frequency_to_bins=_frequency_to_bins, cents_to_frequency=_cents_to_frequency,
                                frequency_to_cents=_frequency_to_cents, dither=lambda c: c + c.new_tensor(_dither_noise(c.size())))


# ---- filter (torchcrepe >= 0.0.22: NaN-aware) ------------------------------------------------------------------------------
def _mean(signals: torch.Tensor, win_length: int = 9) -> torch.Tensor:
    """Average over a window, ignoring NaNs; a window with no valid value (or a zero mean) gives NaN."""
    assert signals.dim() == 2, "Input tensor must have 2 dimensions (batch_size, width)"
    signals = signals.unsqueeze(1)
    mask = ~torch.isnan(signals)
    masked_x = torch.where(mask, signals, torch.zeros_like(signals))
    ones = torch.ones(signals.size(1), 1, win_length, device=signals.device, dtype=signals.dtype)
    sum_pooled = F.conv1d(masked_x, ones, stride=1, padding=win_length // 2, groups=signals.size(1))
    valid = F.conv1d(mask.to(signals.dtype), ones, stride=1, padding=win_length // 2, groups=signals.size(1)).clamp(min=1)
    avg = sum_pooled / valid
    avg[avg == 0] = float("nan")
    return avg.squeeze(1)


def _median(signals: torch.Tensor, win_length: int) -> torch.Tensor:
    """Median over a window, ignoring NaNs (the lower median of the valid values); no valid value gives NaN."""
    assert signals.dim() == 2, "Input tensor must have 2 dimensions (batch_size, width)"
    signals = signals.unsqueeze(1)
    mask = ~torch.isnan(signals)
    masked_x = torch.where(mask, signals, torch.zeros_like(signals))
    padding = win_length // 2
    x = F.pad(masked_x, (padding, padding), mode="reflect")
    mask = F.pad(mask.float(), (padding, padding), mode="constant", value=0)
    x = x.unfold(2, win_length, 1)
    mask = mask.unfold(2, win_length, 1)
    x = x.contiguous().view(x.size()[:3] + (-1,))
    mask = mask.contiguous().view(mask.size()[:3] + (-1,))
    x_masked = torch.where(mask.bool(), x.double(), float("inf")).to(x)
    x_sorted, _ = torch.sort(x_masked, dim=-1)
    valid_count = mask.sum(dim=-1)
    median_idx = ((valid_count - 1) // 2).clamp(min=0)
    median_pooled = x_sorted.gather(-1, median_idx.unsqueeze(-1).long()).squeeze(-1)
    median_pooled[torch.isinf(median_pooled)] = float("nan")
    return median_pooled.squeeze(1)


filter = types.SimpleNamespace(mean=_mean, median=_median)  # noqa: A001  (torchcrepe's module name)


# ---- decode ------------------------------------------------------------------------------------------------------------------
# Called with masked probabilities [1, 360, T] (any device), like torchcrepe's decoders; the work runs on the device.
def _argmax(logits):
    return _decode_tensor(logits, 0)


def _weighted_argmax(logits):
    return _decode_tensor(logits, 1)


def _viterbi(logits):
    return _decode_tensor(logits, 2)


decode = types.SimpleNamespace(argmax=_argmax, weighted_argmax=_weighted_argmax, viterbi=_viterbi)
_MODES = {_argmax: 0, _weighted_argmax: 1, _viterbi: 2}


def viterbi_tables():
    """(log_trans band [360][23] float64, log of the out-of-band transition, log of the initial probability), exactly as
    librosa forms them from torchcrepe's transition matrix: log(max(12 - |i - j|, 0) / row sum + tiny)."""
    xx, yy = np.meshgrid(range(PITCH_BINS), range(PITCH_BINS))
    transition = np.maximum(12 - abs(xx - yy), 0)
    transition = transition / transition.sum(axis=1, keepdims=True)
    eps = np.finfo(np.float32).tiny
    log_trans = np.log(transition + eps)
    band = np.zeros((PITCH_BINS, 2 * BAND + 1))
    for k in range(PITCH_BINS):
        for d in range(-BAND, BAND + 1):
            if 0 <= k + d < PITCH_BINS:
                band[k, d + BAND] = log_trans[k, k + d]
    log_out = float(np.log(np.float64(0.0) + eps))
    log_init = float(np.log(np.full(PITCH_BINS, 1.0 / PITCH_BINS) + eps)[0])
    return band, log_out, log_init


_WCENTS: Optional[np.ndarray] = None


def _weighted_cents() -> np.ndarray:
    """torchcrepe caches `bins_to_cents(arange(360))` on the function at its first call: one dither draw per process."""
    global _WCENTS
    if _WCENTS is None:
        _WCENTS = CENTS_PER_BIN * np.arange(PITCH_BINS, dtype=np.float64) + CENTS_OFFSET + _dither_noise((PITCH_BINS,))
    return _WCENTS


def _device_of(device) -> torch.device:
    dev = torch.device(device) if device is not None else torch.device("cuda")
    if dev.type != "cuda":
        raise RuntimeError("comfy_rvc_b200.crepe runs on a CUDA (sm_100a) device; it has no CPU fallback")
    return torch.device("cuda", 0) if dev.index is None else dev


def _check(st: int, what: str):
    if st != 0:
        raise RuntimeError(f"{what} failed with status {st} ({_lib.STATUS.get(st, '?')})")


def decode_device(x: torch.Tensor, from_salience: bool, mode: int, lo: int, hi: int, chunk: int, dither: Optional[np.ndarray],
                  want_periodicity: bool = True, want_salience: bool = False):
    """Run `rvcb200_op_crepe_decode` on x [T][ld] fp32 (device): logits (from_salience False) or the sigmoid salience.
    Returns dict of device tensors: bins int32 [T], f0 float64 [T], periodicity fp32 [T] | None, salience | None, score | None."""
    lib, dev = _lib.load(), x.device
    T = int(x.shape[0])
    bins = torch.empty(T, dtype=torch.int32, device=dev)
    f0 = torch.empty(T, dtype=torch.float64, device=dev)
    per = torch.empty(T, dtype=torch.float32, device=dev) if want_periodicity else None
    sal = torch.empty(T, PITCH_BINS, dtype=torch.float32, device=dev) if (want_salience or mode == 2) else None
    dith = wc = lt = logp = ptr = score = None
    log_out = log_init = 0.0
    if mode != 1:
        dith = torch.as_tensor(np.ascontiguousarray(dither, dtype=np.float64)).to(dev)
    else:
        wc = torch.as_tensor(_weighted_cents()).to(dev)
    if mode == 2:
        band, log_out, log_init = viterbi_tables()
        lt = torch.as_tensor(band).to(dev)
        logp = torch.empty(T, PITCH_BINS, dtype=torch.float64, device=dev)
        ptr = torch.empty(T, PITCH_BINS, dtype=torch.int16, device=dev)
        score = torch.empty((T + chunk - 1) // chunk, dtype=torch.float64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    _check(lib.rvcb200_op_crepe_decode(p(x), int(x.stride(0)), int(from_salience), T, int(chunk), int(lo), int(hi), int(mode), p(dith),
                                       p(wc), p(lt), log_out, log_init, p(sal), p(logp), p(ptr), p(bins), p(f0), p(per), p(score),
                                       C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "rvcb200_op_crepe_decode")
    return {"bins": bins, "f0": f0, "periodicity": per, "salience": sal, "score": score}


def _decode_tensor(probabilities: torch.Tensor, mode: int):
    """torchcrepe's decoder call: masked probabilities [1, 360, T] -> (bins [1, T], pitch [1, T]) on the input's device."""
    if probabilities.dim() != 3 or probabilities.shape[0] != 1 or probabilities.shape[1] != PITCH_BINS:
        raise ValueError("probabilities must be [1, 360, frames]")
    dev = _device_of(probabilities.device if probabilities.is_cuda else None)
    s = probabilities[0].t().to(dev, torch.float32).contiguous()
    valid = torch.isfinite(s).all(dim=0).nonzero().flatten()
    lo, hi = (int(valid[0]), int(valid[-1]) + 1) if valid.numel() else (0, PITCH_BINS)
    T = int(s.shape[0])
    dither = _dither_noise((1, T)).reshape(-1) if mode != 1 else None
    with torch.cuda.device(dev):
        r = decode_device(torch.nan_to_num(s, neginf=0.0), True, mode, lo, hi, T, dither, want_periodicity=False)
    out_dev = probabilities.device
    return r["bins"].long()[None].to(out_dev), r["f0"].float()[None].to(out_dev)


# ---- the model ---------------------------------------------------------------------------------------------------------------
_ASSETS: Dict[str, Union[str, Dict[str, torch.Tensor]]] = {}


def load_weights(model: str, path_or_state_dict):
    """Register the weights `Crepe(model)` and `predict(..., model=model)` use (a path to torchcrepe's `{model}.pth` or a state dict)."""
    if model not in CHANNELS:
        raise ValueError(f"model must be 'full' or 'tiny', not {model!r}")
    _ASSETS[model] = path_or_state_dict
    _MODELS.pop(model, None)


def _default_weights(model: str):
    if model in _ASSETS:
        return _ASSETS[model]
    try:
        import torchcrepe as _tc  # noqa: F401
        path = os.path.join(os.path.dirname(_tc.__file__), "assets", f"{model}.pth")
        if os.path.exists(path):
            return path
    except ImportError:
        pass
    raise RuntimeError(f"no CREPE weights for model {model!r}: call comfy_rvc_b200.crepe.load_weights({model!r}, path_or_state_dict) "
                       "(torchcrepe's assets/{model}.pth) or install torchcrepe")


class Crepe:
    """torchcrepe's `Crepe(model)` on the B200 kernels; `weights`: path or state dict (default: see `load_weights`)."""

    def __init__(self, model: str = "full", weights=None, device=None):
        if model not in CHANNELS:
            raise ValueError(f"model must be 'full' or 'tiny', not {model!r}")
        self.model = model
        src = _default_weights(model) if weights is None else weights
        sd = torch.load(src, map_location="cpu") if isinstance(src, (str, bytes)) or hasattr(src, "__fspath__") else src
        self._sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items() if not k.endswith("num_batches_tracked")}
        cin, cout, nf = CHANNELS[model]
        for i in range(6):
            k = (512 if i == 0 else 64)
            want = {f"conv{i + 1}.weight": (cout[i], cin[i], k, 1), f"conv{i + 1}.bias": (cout[i],)}
            for s in ("weight", "bias", "running_mean", "running_var"):
                want[f"conv{i + 1}_BN.{s}"] = (cout[i],)
            for key, shape in want.items():
                if key not in self._sd or tuple(self._sd[key].shape) != shape:
                    raise ValueError(f"state dict is not torchcrepe's {model!r} layout: {key} "
                                     f"{tuple(self._sd[key].shape) if key in self._sd else 'missing'}, expected {shape}")
        if tuple(self._sd.get("classifier.weight", torch.empty(0)).shape) != (PITCH_BINS, nf):
            raise ValueError(f"state dict is not torchcrepe's {model!r} layout: classifier.weight")
        self.device = _device_of(device) if device is not None else None
        self._host = host_weights(self._sd, model)
        self._w: Optional[Dict[str, torch.Tensor]] = None
        self.last_launches = 0

    # ---- nn.Module-like protocol ------------------------------------------------------------------------------------------
    def eval(self):
        return self

    def half(self):
        return self

    def float(self):
        return self

    def to(self, device=None, *a, **k):
        if device is not None and not isinstance(device, torch.dtype):
            dev = _device_of(device)
            if dev != self.device:
                self.device, self._w = dev, None
        return self

    def _materialize(self, device=None):
        if device is not None:
            self.to(device)
        if self.device is None:
            self.device = _device_of(None)
        if not torch.cuda.is_available():
            raise RuntimeError("comfy_rvc_b200.crepe needs a CUDA (sm_100a) device; it has no CPU fallback")
        _lib.load()
        if self._w is None:
            w = {}
            for k, v in self._host.items():
                if k.endswith(".taps"):
                    w[k] = pack_tc(v, torch.float16, self._n_tile(k)).to(self.device)
                else:
                    w[k] = v.to(self.device).contiguous()
            self._w = w

    def _n_tile(self, key: str) -> int:
        cout = int(self._host[key].shape[-1])
        return 256 if cout % 256 == 0 else (128 if cout % 128 == 0 else cout)

    # ---- one pass of frames through the network ---------------------------------------------------------------------------
    def _conv(self, name: str, x16: int, rows: int, B: int, cin: int, cout: int, taps: int, dil: int, g_off: int, lj: int,
              y16: int = 0, y32: int = 0, relu: bool = True):
        w = self._w[name + ".taps"]
        d = _lib.TcConvDesc()
        d.x16, d.L_in, d.padf = x16, rows, PADF
        d.w16, d.bias = w.data_ptr(), self._w[name + ".b"].data_ptr()
        d.Cin, d.ntaps, d.dil, d.G = cin, taps, dil, 1
        d.g_off[0] = g_off
        d.N, d.Cout_total = self._n_tile(name + ".taps"), cout
        d.Lj, d.out_stride, d.Lp_out = lj, 1, ((lj + 127) // 128) * 128 + 128
        d.div, d.out_slope, d.alpha = 1.0, 1.0, 1.0
        d.pre_slope = 0.0 if relu else 1.0
        d.generic, d.f32_cl = 1, 1
        if y16:
            d.y16, d.ldy16 = y16, cout
        if y32:
            d.y32, d.ldy32 = y32, cout
        st = _lib.load().rvcb200_op_conv_tc(C.byref(d), B, self._stream)
        if st != 0:
            raise RuntimeError(f"rvcb200_op_conv_tc failed with status {st} ({name}: Cin={cin}, Cout={cout}, taps={taps}, rows={rows}, B={B})")
        self.last_launches += 1

    def _pool(self, i: int, x, frames: int, C_: int, L: int, p_in: int, in_off: int, p_out: int, out_off: int, out):
        lib = _lib.load()
        _check(lib.rvcb200_op_crepe_bn_pool(C.c_void_p(x.data_ptr()), C.c_void_p(self._w[f"bn{i}.scale"].data_ptr()),
                                            C.c_void_p(self._w[f"bn{i}.shift"].data_ptr()), C.c_void_p(out.data_ptr()), frames, C_, L,
                                            p_in, in_off, p_out, out_off, self._stream), "rvcb200_op_crepe_bn_pool")
        self.last_launches += 1

    def _scratch(self, nF: int):
        """Network scratch for passes of up to nF frames, kept between calls: conv outputs (a), pool outputs (b), logits."""
        cin, cout, nf = CHANNELS[self.model]
        cap = max(nF, getattr(self, "_scr_cap", 0))
        if getattr(self, "_scr_dev", None) != self.device or cap > getattr(self, "_scr_cap", 0):
            conv_rows = [LENGTHS[0], LENGTHS[1]] + [L + 32 for L in LENGTHS[2:]]
            pool_rows = [LENGTHS[1]] + [L + 32 for L in LENGTHS[2:]] + [LENGTHS[5] // 2]
            a = max(r * c for r, c in zip(conv_rows, cout))
            b = max(max(r * c for r, c in zip(pool_rows, cout)), nf)
            dev = self.device
            self._scr = {"frames": torch.empty(cap * FRAME_ROWS * FRAME_C, dtype=torch.float16, device=dev),
                         "a": torch.empty(cap * a, dtype=torch.float16, device=dev),
                         "b": torch.empty(cap * b, dtype=torch.float16, device=dev),
                         "logits": torch.empty(cap, N_PAD, dtype=torch.float32, device=dev)}
            self._scr_cap, self._scr_dev = cap, dev
        return self._scr

    def _network(self, audio, n: int, first: int, nF: int, hop: int, pad: bool, logits_out=None, taps=None):
        """Frames first .. first + nF - 1 of the device audio -> classifier logits fp32 [nF][384] (a view of the scratch)."""
        lib = _lib.load()
        cin, cout, nf = CHANNELS[self.model]
        s = self._scratch(nF)
        fr, A, Bf = s["frames"], s["a"], s["b"]
        _check(lib.rvcb200_op_crepe_frames(C.c_void_p(audio.data_ptr()), n, first, nF, hop, int(pad), C.c_void_p(fr.data_ptr()),
                                           self._stream), "rvcb200_op_crepe_frames")
        self.last_launches += 1
        if taps is not None:
            taps["frames16"] = fr[: nF * FRAME_ROWS * FRAME_C].view(nF, FRAME_ROWS, FRAME_C).clone()
        # conv1: one frame per batch item, 8 taps at dilation 16 over 368 rows x 64 polyphase channels -> 256 rows
        self._conv("conv1", fr.data_ptr(), FRAME_ROWS, nF, FRAME_C, cout[0], CONV1_TAPS, CONV1_DIL, 0, LENGTHS[0], y16=A.data_ptr())
        self._pool(1, A, nF, cout[0], LENGTHS[0], LENGTHS[0], 0, LENGTHS[1], 0, Bf)
        # conv2: one frame per batch item, the tensor map's zero fill supplies the (31, 32) padding
        self._conv("conv2", Bf.data_ptr(), LENGTHS[1], nF, cout[0], cout[1], 64, 1, -31, LENGTHS[1], y16=A.data_ptr())
        p_prev, off_prev, src, dst = LENGTHS[1], 0, A, Bf
        for i in range(2, 6):                       # conv3..conv6 over padded lines: frame f at rows f P + 31 .. f P + 31 + L - 1
            L = LENGTHS[i]
            P = L + 32
            self._pool(i, src, nF, cout[i - 1], LENGTHS[i - 1], p_prev, off_prev, P, 31, dst)
            if taps is not None:
                taps[f"in{i + 1}"] = dst[: nF * P * cout[i - 1]].view(nF, P, cout[i - 1]).clone()
            self._conv(f"conv{i + 1}", dst.data_ptr(), nF * P, 1, cout[i - 1], cout[i], 64, 1, 0, nF * P, y16=src.data_ptr())
            p_prev, off_prev = P, 0
        feat = dst                                  # [nF][4][C6] = the classifier's [nF][F], feature = time * C6 + channel
        self._pool(6, src, nF, cout[5], LENGTHS[5], p_prev, off_prev, LENGTHS[5] // 2, 0, feat)
        if taps is not None:
            taps["features"] = feat[: nF * nf].view(nF, nf).clone()
        logits = s["logits"] if logits_out is None else logits_out
        self._conv("cls", feat.data_ptr(), nF, 1, nf, N_PAD, 1, 1, 0, nF, y32=logits.data_ptr(), relu=False)
        return logits[:nF]

    @torch.no_grad()
    def forward_logits(self, frames_audio: torch.Tensor, hop: int, pad: bool, first: int, count: int, taps: Optional[dict] = None):
        """Classifier logits [count][360] fp32 (device) of frames first.. of `frames_audio` (device fp32 [n])."""
        self._materialize()
        with torch.cuda.device(self.device):
            self._begin()
            out = torch.empty(count, PITCH_BINS, dtype=torch.float32, device=self.device)
            for p0 in range(0, count, PASS_FRAMES):
                nF = min(PASS_FRAMES, count - p0)
                lg = self._network(frames_audio, int(frames_audio.numel()), first + p0, nF, hop, pad, taps=taps)
                out[p0:p0 + nF] = lg[:, :PITCH_BINS]
            return out

    def _begin(self):
        self.last_launches = 0
        self._stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __call__(self, frames: torch.Tensor, embed: bool = False) -> torch.Tensor:
        """torchcrepe's `Crepe.forward`: normalised frames [B, 1024] -> salience [B, 360] (sigmoid), on the device.
        The frames are treated as a signal at hop 1024 and normalised again by `rvcb200_op_crepe_frames` (a no-op up to
        rounding for frames `preprocess` produced)."""
        if embed:
            raise NotImplementedError("embed=True (the conv5 embedding) is not provided")
        self._materialize()
        x = frames.to(self.device, torch.float32).reshape(-1).contiguous()
        lg = self.forward_logits(x, WINDOW_SIZE, False, 0, int(frames.shape[0]))
        return torch.sigmoid(lg)

    forward = __call__


def host_weights(sd: Dict[str, torch.Tensor], model: str) -> Dict[str, torch.Tensor]:
    """torchcrepe's state dict -> the kernels' fp32 host images: `conv{i}.taps` [taps][Cin][Cout] (conv1: 8 taps over 64 polyphase
    channels, tap m channel c = kernel sample 64 m + c), `conv{i}.b`, `bn{i}.scale` / `bn{i}.shift` (y = x * scale + shift, the
    eval-mode BatchNorm of the ReLU output), `cls.taps` [1][F][384] / `cls.b` [384]."""
    cin, cout, nf = CHANNELS[model]
    W: Dict[str, torch.Tensor] = {}
    for i in range(1, 7):
        w = sd[f"conv{i}.weight"].double()[..., 0]                      # [Co][Ci][k]
        if i == 1:
            W["conv1.taps"] = w[:, 0, :].reshape(cout[0], CONV1_TAPS, FRAME_C).permute(1, 2, 0).float().contiguous()
        else:
            W[f"conv{i}.taps"] = w.permute(2, 1, 0).float().contiguous()
        W[f"conv{i}.b"] = sd[f"conv{i}.bias"].float().contiguous()
        p = f"conv{i}_BN."
        scale = sd[p + "weight"].double() / torch.sqrt(sd[p + "running_var"].double() + BN_EPS)
        W[f"bn{i}.scale"] = scale.float().contiguous()
        W[f"bn{i}.shift"] = (sd[p + "bias"].double() - sd[p + "running_mean"].double() * scale).float().contiguous()
    wc = torch.zeros(1, nf, N_PAD)
    wc[0, :, :PITCH_BINS] = sd["classifier.weight"].t()
    W["cls.taps"] = wc
    W["cls.b"] = torch.cat([sd["classifier.bias"].float(), torch.zeros(N_PAD - PITCH_BINS)])
    return W


_MODELS: Dict[str, Crepe] = {}


def _model(model: str, device) -> Crepe:
    m = _MODELS.get(model)
    if m is None:
        m = _MODELS[model] = Crepe(model)
    m.to(device)
    return m


# ---- torchcrepe's functional API -----------------------------------------------------------------------------------------------
def frame_count(n: int, hop: int, pad: bool) -> int:
    return 1 + n // hop if pad else 1 + (n - WINDOW_SIZE) // hop


def chunks(total: int, batch_size: Optional[int]):
    """Frame ranges [start, end) of torchcrepe's preprocess generator."""
    bs = total if batch_size is None else batch_size
    return [(i, min(total, i + bs)) for i in range(0, total, bs)]


def preprocess(audio, sample_rate, hop_length=None, batch_size=None, device="cpu", pad=True):
    """torchcrepe.preprocess: yields normalised frames [chunk, 1024] (float32, on `device`), computed on the host like torchcrepe
    (the device path of `predict` never materialises them)."""
    if sample_rate != SAMPLE_RATE:
        raise ValueError(f"comfy_rvc_b200.crepe takes {SAMPLE_RATE} Hz audio (torchcrepe resamples other rates; this path does not)")
    hop = sample_rate // 100 if hop_length is None else hop_length
    n = audio.size(1)
    total = frame_count(n, hop, pad)
    x = F.pad(audio, (WINDOW_SIZE // 2, WINDOW_SIZE // 2)) if pad else audio
    for s0, s1 in chunks(total, batch_size):
        frames = x[0, s0 * hop: (s1 - 1) * hop + WINDOW_SIZE].unfold(0, WINDOW_SIZE, hop).clone().to(device)
        frames -= frames.mean(dim=1, keepdim=True)
        frames /= torch.max(torch.tensor(1e-10, device=frames.device), frames.std(dim=1, keepdim=True))
        yield frames


def infer(frames, model="full", embed=False):
    """torchcrepe.infer: frames [B, 1024] -> salience [B, 360] on the device."""
    dev = frames.device if frames.is_cuda else None
    return _model(model, dev)(frames, embed=embed)


def postprocess(probabilities, fmin=0.0, fmax=MAX_FMAX, decoder=None, return_harmonicity=False, return_periodicity=False):
    """torchcrepe.postprocess on [1, 360, T] probabilities."""
    decoder = _viterbi if decoder is None else decoder
    probabilities = probabilities.detach().clone()
    lo = int(_frequency_to_bins(torch.tensor(fmin)))
    hi = int(_frequency_to_bins(torch.tensor(fmax), torch.ceil))
    probabilities[:, :lo] = -float("inf")
    probabilities[:, hi:] = -float("inf")
    bins, pitch = decoder(probabilities)
    if not (return_periodicity or return_harmonicity):
        return pitch
    per = probabilities.transpose(1, 2).reshape(-1, PITCH_BINS).gather(1, bins.reshape(-1, 1).to(torch.int64).to(probabilities.device))
    return pitch, per.reshape(probabilities.size(0), probabilities.size(2))


def _mask_range(fmin: float, fmax: float):
    lo = int(_frequency_to_bins(torch.tensor(fmin)))
    hi = int(_frequency_to_bins(torch.tensor(fmax), torch.ceil))
    return max(lo, 0), min(hi, PITCH_BINS)


@torch.no_grad()
def predict(audio, sample_rate, hop_length=None, fmin=50.0, fmax=MAX_FMAX, model="full", decoder=None, return_harmonicity=False,
            return_periodicity=False, batch_size=None, device="cpu", pad=True, crepe_model: Optional[Crepe] = None, taps=None):
    """torchcrepe.predict on the device.  audio [1, n] at 16 kHz; returns pitch [1, T] (and periodicity [1, T]) float32 on
    `audio.device`.  `device` names the CUDA device to run on ("cpu", torchcrepe's default, means the current CUDA device).
    `decoder` is one of `decode.argmax`, `decode.weighted_argmax`, `decode.viterbi` (default)."""
    decoder = _viterbi if decoder is None else decoder
    if decoder not in _MODES:
        raise ValueError("decoder must be comfy_rvc_b200.crepe.decode.argmax, .weighted_argmax or .viterbi")
    if sample_rate != SAMPLE_RATE:
        raise ValueError(f"comfy_rvc_b200.crepe takes {SAMPLE_RATE} Hz audio (torchcrepe resamples other rates; this path does not)")
    audio = torch.as_tensor(audio)
    if audio.dim() != 2 or audio.shape[0] != 1:
        raise ValueError("audio must be [1, n] (torchcrepe's batch of one)")
    want_per = return_periodicity or return_harmonicity
    hop = sample_rate // 100 if hop_length is None else int(hop_length)
    n = int(audio.shape[1])
    total = frame_count(n, hop, pad)
    if total <= 0:
        raise ValueError(f"audio of {n} samples holds no frame (pad={pad})")
    dev = _device_of(device if str(device) != "cpu" else (audio.device if audio.is_cuda else None))
    m = crepe_model if crepe_model is not None else _model(model, dev)
    m._materialize(dev)
    mode = _MODES[decoder]
    ch = chunks(total, batch_size)
    # torchcrepe's dither draws, in its call order: one per chunk (argmax / viterbi), or the cached weights (weighted_argmax)
    dither = np.concatenate([_dither_noise((1, e - s)).reshape(-1) for s, e in ch]) if mode != 1 else None
    if mode == 1:
        _weighted_cents()
    chunk = total if batch_size is None else int(batch_size)
    with torch.cuda.device(dev):
        x = audio[0].to(dev, torch.float32).contiguous()                       # the one host -> device copy
        logits = m.forward_logits(x, hop, pad, 0, total, taps=taps)
        lo, hi = _mask_range(fmin, fmax)
        r = decode_device(logits, False, mode, lo, hi, chunk, dither, want_periodicity=want_per, want_salience=taps is not None)
        if taps is not None:
            taps.update(logits=logits, **{k: v for k, v in r.items() if v is not None})
        pitch = r["f0"].float()
        out = torch.stack([pitch, r["periodicity"]]) if want_per else pitch[None]
        out = out.to(audio.device)                                             # the one device -> host copy
    if want_per:
        return out[0:1], out[1:2]
    return out
