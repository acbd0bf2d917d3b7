"""ORACLE — TEST INFRASTRUCTURE ONLY.  The reference's volume-envelope mix, `change_rms` (/root/reference/lib/model_utils.py:39,
called at vc_infer_pipeline.py:183), on the CPU, and `VC.pipeline` with `rms_mix_rate < 1` built on `oracle.pipeline_oracle`.

librosa is unpinned in the reference's requirements and absent from this image, so `librosa.feature.rms` is restated
(`librosa_rms`) the way `oracle/rmvpe_oracle.py` restates the mel filterbank."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F
from scipy import signal

from oracle import pipeline_oracle


def librosa_rms(y: np.ndarray, frame_length: int, hop_length: int) -> np.ndarray:
    """`librosa.feature.rms(y=y, frame_length=frame_length, hop_length=hop_length)` with librosa >= 0.10 defaults, restated from
    librosa/feature/spectral.py `rms` and librosa/util/utils.py `frame` (0.10.x): `center=True` pads frame_length // 2 zeros on
    each side (`pad_mode="constant"`); frames are strided views hop_length apart with the within-frame axis at -2 (`util.frame`);
    `power = np.mean(np.power(x, 2, dtype=np.float32), axis=-2)` (float32 squares, numpy's float32 pairwise sum); then
    `np.sqrt`.  1-D y -> float32 of shape (1, 1 + len(y) // hop_length) when frame_length = 2 * hop_length."""
    y = np.asarray(y)
    pad = int(frame_length // 2)
    y = np.pad(y, (pad, pad), mode="constant")
    n_frames = 1 + (y.shape[-1] - frame_length) // hop_length
    xw = np.lib.stride_tricks.as_strided(y, shape=(n_frames, frame_length), strides=(y.strides[-1] * hop_length, y.strides[-1]),
                                         writeable=False)
    x = np.moveaxis(xw, -1, -2)                                     # (frame_length, n_frames), like util.frame
    power = np.mean(np.power(x, 2, dtype=np.float32), axis=-2, keepdims=True)
    return np.sqrt(power)


def change_rms(data1, sr1, data2, sr2, rate):
    """lib/model_utils.py:39-59, the reference's code with `librosa.feature.rms` -> `librosa_rms`; scales data2 in place."""
    rms1 = librosa_rms(y=data1, frame_length=sr1 // 2 * 2, hop_length=sr1 // 2)  # one point per half second
    rms2 = librosa_rms(y=data2, frame_length=sr2 // 2 * 2, hop_length=sr2 // 2)
    rms1 = torch.from_numpy(rms1)
    rms1 = F.interpolate(rms1.unsqueeze(0), size=data2.shape[0], mode="linear").squeeze()
    rms2 = torch.from_numpy(rms2)
    rms2 = F.interpolate(rms2.unsqueeze(0), size=data2.shape[0], mode="linear").squeeze()
    rms2 = torch.max(rms2, torch.zeros_like(rms2) + 1e-6)
    data2 *= (torch.pow(rms1, torch.tensor(1 - rate)) * torch.pow(rms2, torch.tensor(rate - 1))).numpy()
    return data2


def pipeline(*args, rms_mix_rate: float = 1.0, **kw):
    """`pipeline_oracle.pipeline` (same arguments, same RNG draws) with the mix of vc_infer_pipeline.py:183 applied to the
    concatenated segment outputs before the int16 conversion when rms_mix_rate < 1, like the reference."""
    return_parts = kw.pop("return_parts", False)
    res, parts, opt_ts = pipeline_oracle.pipeline(*args, return_parts=True, **kw)
    if rms_mix_rate < 1:
        audio = args[3] if len(args) > 3 else kw["audio"]
        c = args[4] if len(args) > 4 else kw["c"]
        hp = signal.filtfilt(pipeline_oracle._BH, pipeline_oracle._AH, audio)                 # :122, the `audio` of :183
        res = pipeline_oracle.to_int16(change_rms(hp, 16000, np.concatenate(parts), c.tgt_sr, rms_mix_rate))
    return (res, parts, opt_ts) if return_parts else res
