"""ORACLE — TEST INFRASTRUCTURE ONLY.  `VC.pipeline` with the output resampling of vc_infer_pipeline.py:185-186, built on
`oracle.pipeline_oracle` and `tests._rms_oracle`.

The reference's `librosa.resample` (soxr_hq with librosa >= 0.10) cannot be pinned here; the resampler this path defines is
`scipy.signal.resample_poly(x, up, down, window=h)` with the filter of `comfy_rvc_b200.resample.design`, in float64."""
from __future__ import annotations

import numpy as np
from scipy import signal

from comfy_rvc_b200 import resample
from oracle import pipeline_oracle
from tests import _rms_oracle


def resample_song(audio_opt: np.ndarray, tgt_sr: int, resample_sr: int) -> np.ndarray:
    """:185-186 with the defined resampler; the input unchanged when the reference skips the step."""
    if resample_sr >= 16000 and tgt_sr != resample_sr:
        up, down, h = resample.design(tgt_sr, resample_sr)
        return signal.resample_poly(audio_opt, up, down, window=h)
    return audio_opt


def pipeline(*args, rms_mix_rate: float = 1.0, resample_sr: int = 0, **kw):
    """`pipeline_oracle.pipeline` (same arguments, same RNG draws) followed by :183 (`change_rms` when rms_mix_rate < 1),
    :185-186 (the resampling) and :188-189 (peak and int16) on the concatenated segment outputs."""
    _, parts, _ = pipeline_oracle.pipeline(*args, return_parts=True, **kw)
    audio = args[3] if len(args) > 3 else kw["audio"]
    c = args[4] if len(args) > 4 else kw["c"]
    audio_opt = np.concatenate(parts)
    if rms_mix_rate < 1:
        hp = signal.filtfilt(pipeline_oracle._BH, pipeline_oracle._AH, audio)                 # :122, the `audio` of :183
        audio_opt = _rms_oracle.change_rms(hp, 16000, audio_opt, c.tgt_sr, rms_mix_rate)
    return pipeline_oracle.to_int16(resample_song(audio_opt, c.tgt_sr, resample_sr))
