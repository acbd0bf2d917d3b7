"""Torch-CPU restatement of torchcrepe (`Crepe`, `preprocess`, `postprocess`, `decode`, `convert`) and a float64 numpy restatement
of `librosa.sequence.viterbi` as torchcrepe calls it.

torchcrepe and librosa are not installed where this project is tested, so the distance between this file and the libraries
themselves is NOT measured; it restates their published code.  Two deliberate differences, both in the decoders:
  * f0 is evaluated in float64 (torchcrepe: float32 cents and float32 `10 * 2 ** (c / 1200)`, i.e. ~1e-7 relative);
  * the Viterbi observations are `log(softmax + tiny)` in float64 (torchcrepe: a float32 softmax handed to librosa, which
    takes the log in float32).  The recursion itself is librosa's: float64 values, first maximum on ties, backtrack from the
    first argmax of the last column.
The dither is drawn exactly like torchcrepe's `convert.dither` (numpy's global RNG, one call per chunk, one for the cached
weights of `weighted_argmax`).
"""
from __future__ import annotations

from typing import Dict, Iterator, Tuple

import numpy as np
import torch
import torch.nn.functional as F

CENTS_PER_BIN, MAX_FMAX, PITCH_BINS, SAMPLE_RATE, WINDOW_SIZE = 20, 2006.0, 360, 16000, 1024
CENTS_OFFSET = 1997.3794084376191
BN_EPS = 0.0010000000474974513
CHANNELS = {"full": ([1, 1024, 128, 128, 128, 256], [1024, 128, 128, 128, 256, 512], 2048),
            "tiny": ([1, 128, 16, 16, 16, 32], [128, 16, 16, 16, 32, 64], 256)}


# ---- the network -----------------------------------------------------------------------------------------------------------
def layer(x: torch.Tensor, sd: Dict[str, torch.Tensor], i: int, padding=(0, 0, 31, 32)) -> torch.Tensor:
    """`Crepe.layer`: pad -> conv -> ReLU -> BatchNorm (eval) -> max_pool (2, 1)."""
    x = F.pad(x, padding)
    x = F.conv2d(x, sd[f"conv{i}.weight"], sd[f"conv{i}.bias"], stride=(4, 1) if i == 1 else (1, 1))
    x = F.relu(x)
    p = f"conv{i}_BN."
    x = F.batch_norm(x, sd[p + "running_mean"], sd[p + "running_var"], sd[p + "weight"], sd[p + "bias"], False, 0.0, BN_EPS)
    return F.max_pool2d(x, (2, 1), (2, 1))


def crepe_forward(frames: torch.Tensor, sd: Dict[str, torch.Tensor], embed: bool = False) -> torch.Tensor:
    """`Crepe.forward`: frames [B, 1024] -> sigmoid salience [B, 360] (or the logits before the sigmoid with embed="logits")."""
    x = frames[:, None, :, None]
    x = layer(x, sd, 1, (0, 0, 254, 254))
    for i in range(2, 7):
        x = layer(x, sd, i)
    x = x.permute(0, 2, 1, 3).reshape(x.shape[0], -1)
    logits = F.linear(x, sd["classifier.weight"], sd["classifier.bias"])
    return logits if embed == "logits" else torch.sigmoid(logits)


def crepe_module(model: str = "full") -> torch.nn.Module:
    """torchcrepe's `Crepe` layer list as an nn.Module (the state-dict contract)."""
    cin, cout, nf = CHANNELS[model]

    class Crepe(torch.nn.Module):
        def __init__(self):
            super().__init__()
            for i in range(6):
                k, s = ((512, 1), (4, 1)) if i == 0 else ((64, 1), (1, 1))
                setattr(self, f"conv{i + 1}", torch.nn.Conv2d(cin[i], cout[i], k, s))
                setattr(self, f"conv{i + 1}_BN", torch.nn.BatchNorm2d(cout[i], eps=BN_EPS, momentum=0.0))
            self.in_features = nf
            self.classifier = torch.nn.Linear(nf, PITCH_BINS)

        def layer(self, x, conv, bn, padding=(0, 0, 31, 32)):
            return F.max_pool2d(bn(F.relu(conv(F.pad(x, padding)))), (2, 1), (2, 1))

        def forward(self, x):
            x = x[:, None, :, None]
            x = self.layer(x, self.conv1, self.conv1_BN, (0, 0, 254, 254))
            for i in range(2, 7):
                x = self.layer(x, getattr(self, f"conv{i}"), getattr(self, f"conv{i}_BN"))
            x = x.permute(0, 2, 1, 3).reshape(-1, self.in_features)
            return torch.sigmoid(self.classifier(x))

    return Crepe()


# ---- convert ---------------------------------------------------------------------------------------------------------------
def dither(cents: torch.Tensor) -> torch.Tensor:
    import scipy.stats
    noise = scipy.stats.triang.rvs(c=0.5, loc=-20, scale=40, size=cents.size())
    return cents + cents.new_tensor(noise)


def bins_to_cents(bins):
    return dither(CENTS_PER_BIN * bins + CENTS_OFFSET)


def cents_to_bins(cents, quantize_fn=torch.floor):
    return quantize_fn((cents - CENTS_OFFSET) / CENTS_PER_BIN).int()


def cents_to_frequency(cents):
    return 10 * 2 ** (cents / 1200)


def frequency_to_cents(frequency):
    return 1200 * torch.log2(frequency / 10.0)


def frequency_to_bins(frequency, quantize_fn=torch.floor):
    return cents_to_bins(frequency_to_cents(frequency), quantize_fn)


def bins_to_frequency(bins):
    return cents_to_frequency(bins_to_cents(bins))


# ---- preprocess ------------------------------------------------------------------------------------------------------------
def preprocess(audio: torch.Tensor, sample_rate: int, hop_length=None, batch_size=None, pad: bool = True) -> Iterator[torch.Tensor]:
    """torchcrepe.preprocess for 16 kHz audio [1, n]: yields normalised frames [chunk, 1024] per chunk of `batch_size`."""
    if sample_rate != SAMPLE_RATE:
        raise ValueError("the oracle covers 16 kHz input only")
    hop_length = sample_rate // 100 if hop_length is None else hop_length
    if pad:
        total_frames = 1 + int(audio.size(1) // hop_length)
        audio = F.pad(audio, (WINDOW_SIZE // 2, WINDOW_SIZE // 2))
    else:
        total_frames = 1 + int((audio.size(1) - WINDOW_SIZE) // hop_length)
    batch_size = total_frames if batch_size is None else batch_size
    for i in range(0, total_frames, batch_size):
        start = max(0, i * hop_length)
        end = min(audio.size(1), (i + batch_size - 1) * hop_length + WINDOW_SIZE)
        frames = F.unfold(audio[:, None, None, start:end], kernel_size=(1, WINDOW_SIZE), stride=(1, hop_length))
        frames = frames.transpose(1, 2).reshape(-1, WINDOW_SIZE).clone()
        frames -= frames.mean(dim=1, keepdim=True)
        frames /= torch.max(torch.tensor(1e-10), frames.std(dim=1, keepdim=True))
        yield frames


# ---- decoders (probabilities: [1, 360, T], masked with -inf) -------------------------------------------------------------
def _f0_from_bins(bins: torch.Tensor) -> torch.Tensor:
    """bins_to_frequency in float64 (same dither draw as torchcrepe)."""
    import scipy.stats
    noise = scipy.stats.triang.rvs(c=0.5, loc=-20, scale=40, size=bins.size())
    cents = CENTS_PER_BIN * bins.double() + CENTS_OFFSET + torch.as_tensor(noise, dtype=torch.float64)
    return 10 * 2 ** (cents / 1200)


def argmax(logits: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    bins = logits.argmax(dim=1)
    return bins, _f0_from_bins(bins)


def weighted_argmax(logits: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    bins = logits.argmax(dim=1)
    if not hasattr(weighted_argmax, "weights"):
        import scipy.stats
        noise = scipy.stats.triang.rvs(c=0.5, loc=-20, scale=40, size=(PITCH_BINS,))
        weighted_argmax.weights = (CENTS_PER_BIN * torch.arange(PITCH_BINS, dtype=torch.float64) + CENTS_OFFSET
                                   + torch.as_tensor(noise))[None, :, None]
    lg = logits.double().clone()
    start = torch.clamp(bins - 4, min=0)
    end = torch.clamp(bins + 5, max=PITCH_BINS)
    for b in range(lg.size(0)):
        for t in range(lg.size(2)):
            lg[b, :start[b, t], t] = -float("inf")
            lg[b, end[b, t]:, t] = -float("inf")
    probs = torch.sigmoid(lg)
    cents = (weighted_argmax.weights * probs).sum(dim=1) / probs.sum(dim=1)
    return bins, 10 * 2 ** (cents / 1200)


def viterbi_transition() -> np.ndarray:
    xx, yy = np.meshgrid(range(PITCH_BINS), range(PITCH_BINS))
    transition = np.maximum(12 - abs(xx - yy), 0)
    return transition / transition.sum(axis=1, keepdims=True)


def librosa_viterbi(prob: np.ndarray, transition: np.ndarray) -> Tuple[np.ndarray, float]:
    """`librosa.sequence.viterbi(prob [n_states, n_steps], transition)` with a uniform initial distribution, in float64.
    Returns (states [n_steps], log-probability of the path)."""
    prob = np.asarray(prob, dtype=np.float64)
    n_states, n_steps = prob.shape
    eps = np.finfo(np.float32).tiny
    log_trans = np.log(transition + eps)
    log_prob = np.log(prob + eps).T
    log_p_init = np.log(np.full(n_states, 1.0 / n_states) + eps)
    value = np.zeros((n_steps, n_states))
    ptr = np.zeros((n_steps, n_states), dtype=np.int64)
    value[0] = log_prob[0] + log_p_init
    for t in range(1, n_steps):
        trans_out = value[t - 1] + log_trans.T
        for j in range(n_states):
            ptr[t, j] = np.argmax(trans_out[j])
            value[t, j] = log_prob[t, j] + trans_out[j, ptr[t][j]]
    state = np.zeros(n_steps, dtype=np.int64)
    state[-1] = np.argmax(value[-1])
    for t in range(n_steps - 2, -1, -1):
        state[t] = ptr[t + 1, state[t + 1]]
    return state, float(value[-1, state[-1]])


def softmax64(logits: torch.Tensor) -> np.ndarray:
    """Softmax over the bins of [1, 360, T] in float64 (-inf -> 0)."""
    return torch.softmax(logits.double(), dim=1).numpy()


def viterbi(logits: torch.Tensor, return_score: bool = False):
    if not hasattr(viterbi, "transition"):
        viterbi.transition = viterbi_transition()
    seqs = softmax64(logits)
    res = [librosa_viterbi(s, viterbi.transition) for s in seqs]
    bins = torch.tensor(np.array([r[0] for r in res]))
    out = bins, _f0_from_bins(bins)
    return (out, [r[1] for r in res]) if return_score else out


# ---- postprocess / predict ---------------------------------------------------------------------------------------------------
def mask_range(fmin: float, fmax: float) -> Tuple[int, int]:
    return int(frequency_to_bins(torch.tensor(fmin))), int(frequency_to_bins(torch.tensor(fmax), torch.ceil))


def postprocess(probabilities: torch.Tensor, fmin=0.0, fmax=MAX_FMAX, decoder=viterbi, return_periodicity=False):
    probabilities = probabilities.detach().clone()
    lo, hi = mask_range(fmin, fmax)
    probabilities[:, :lo] = -float("inf")
    probabilities[:, hi:] = -float("inf")
    bins, pitch = decoder(probabilities)
    if not return_periodicity:
        return pitch
    per = probabilities.transpose(1, 2).reshape(-1, PITCH_BINS).gather(1, bins.reshape(-1, 1).to(torch.int64))
    return pitch, per.reshape(probabilities.size(0), probabilities.size(2))


def predict(audio: torch.Tensor, sample_rate: int, sd: Dict[str, torch.Tensor], hop_length=None, fmin=50.0, fmax=MAX_FMAX,
            decoder=viterbi, return_periodicity=False, batch_size=None, pad=True):
    """torchcrepe.predict on the CPU in float32 (f0 in float64, see the module docstring)."""
    results = []
    with torch.no_grad():
        for frames in preprocess(audio, sample_rate, hop_length, batch_size, pad):
            probabilities = crepe_forward(frames, sd).reshape(audio.size(0), -1, PITCH_BINS).transpose(1, 2)
            results.append(postprocess(probabilities, fmin, fmax, decoder, return_periodicity))
    if return_periodicity:
        pitch, per = zip(*results)
        return torch.cat(pitch, 1), torch.cat(per, 1)
    return torch.cat(results, 1)
