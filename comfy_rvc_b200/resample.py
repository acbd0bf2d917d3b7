"""Output resampling of `VC.pipeline` (`resample_sr`, vc_infer_pipeline.py:185-186): the filter design and the tables the
device kernel (`rvcb200_op_resample_poly`, csrc/pipeline_kernels.cu) reads.

The reference calls `librosa.resample(audio_opt, orig_sr=tgt_sr, target_sr=resample_sr)`, which with librosa >= 0.10 is
libsoxr's multi-stage "soxr_hq" resampler; that cannot be reproduced bit for bit.  This path instead computes exactly

    y = scipy.signal.resample_poly(x, up, down, window=h),   up / down = resample_sr / tgt_sr in lowest terms,
    y[j] = sum_m up * h[half_len + j * down - m * up] * x[m],  half_len = (len(h) - 1) / 2,  len(y) = ceil(len(x) * up / down)

(terms with an index outside h, or outside the song, are zero), with `h` a Kaiser-windowed sinc chosen to meet libsoxr's
published HQ spec: passband edge 0.913 x the lower Nyquist (soxr's default `passband_end`), stopband from 1.0 x the lower
Nyquist, 125 dB attenuation (`design`).  Its distance from soxr's output has not been measured.
"""
from __future__ import annotations

from math import gcd
from typing import Tuple

import numpy as np
from scipy import signal

PASSBAND_END = 0.913          # soxr's default passband edge, a fraction of the lower Nyquist
STOPBAND_DB = 125.0


def ratio(orig_sr: int, target_sr: int) -> Tuple[int, int]:
    """(up, down) = target_sr / orig_sr in lowest terms."""
    orig_sr, target_sr = int(orig_sr), int(target_sr)
    if orig_sr < 1 or target_sr < 1:
        raise ValueError(f"sample rates must be positive, got {orig_sr} -> {target_sr}")
    g = gcd(orig_sr, target_sr)
    return target_sr // g, orig_sr // g


def design(orig_sr: int, target_sr: int) -> Tuple[int, int, np.ndarray]:
    """(up, down, h): the float64 anti-aliasing filter of the orig_sr -> target_sr resampler, in scipy's `resample_poly`
    convention (cutoffs relative to the Nyquist of the up-sampled rate; odd length, symmetric)."""
    up, down = ratio(orig_sr, target_sr)
    m = max(up, down)
    numtaps, beta = signal.kaiserord(STOPBAND_DB, (1.0 - PASSBAND_END) / m)
    numtaps |= 1
    h = signal.firwin(numtaps, (PASSBAND_END + 1.0) / 2.0 / m, window=("kaiser", beta))
    return up, down, np.asarray(h, dtype=np.float64)


def taps_per_phase(n_taps: int, up: int) -> int:
    return -(-n_taps // up)


def phase_table(h: np.ndarray, up: int, dtype=np.float32) -> np.ndarray:
    """Phase-major table [up][stride]: row r holds up * h[r + k * up] for k < taps_per_phase, zeros after (stride = the tap
    count rounded up to 4, so rows start on 16 bytes).  Output j uses row (j * down + half_len) % up against
    x[(j * down + half_len) // up - k]."""
    h = np.asarray(h, dtype=np.float64)
    tpp = taps_per_phase(h.shape[0], up)
    stride = (tpp + 3) // 4 * 4
    hp = np.zeros(up * tpp)
    hp[: h.shape[0]] = h * up
    t = np.zeros((up, stride), dtype=np.float64)
    t[:, :tpp] = hp.reshape(tpp, up).T
    return np.ascontiguousarray(t.astype(dtype))


def out_len(n: int, up: int, down: int) -> int:
    """ceil(n * up / down): scipy's and librosa's output length."""
    return -(-int(n) * up // down)


def halo_len(n_taps: int, up: int) -> int:
    """Input samples a piece needs from each neighbour side: the left reach of an output is taps_per_phase - 1 samples, the
    right reach ceil(half_len / up)."""
    half_len = (n_taps - 1) // 2
    return max(taps_per_phase(n_taps, up), -(-half_len // up))
