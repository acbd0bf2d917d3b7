"""Segmented conversion driver: drop-in for the reference's `VC` (FeatureExtractor constants + `vc` + `pipeline`).

Reference: /root/reference/vc_infer_pipeline.py:23-196 (`VC.vc`, `VC.pipeline`),
/root/reference/pitch_extraction.py:14-45 (constants), :252-304 (`get_f0` post-processing and the coarse
pitch quantiser), /root/reference/config.py:124-141 (the x_pad/x_query/x_center/x_max tiers).

Same names, arguments and results as the reference:

    vc = VC(tgt_sr, config)                       # config: anything with x_pad/x_query/x_center/x_max/is_half/device
    pcm_f32 = vc.vc(hubert, net_g, sid, audio0, pitch, pitchf, times, index, big_npy, index_rate, version, protect)
    pcm_i16 = vc.pipeline(hubert, net_g, sid, audio, times, f0_up_key, f0_method, merge_type, file_index, index_rate,
                          if_f0, filter_radius, tgt_sr, resample_sr, rms_mix_rate, version, protect, crepe_hop_length,
                          f0_autotune, rmvpe_onnx, f0_file, f0_min, f0_max)

What is different is where the work happens (B200-first, SURVEY.md §8e/§8f-1):
  * the reference loops over segments sequentially and, per segment, interpolates/blends with torch ops, copies the
    PCM to the host and `gc_collect()`s (a device sync + `empty_cache`).  Here a song is planned once on the host
    (the reference's own quiet-point search, bit-identical segmentation), every segment is enqueued on the stream
    without a host round trip (`rvcb200_op_prepare_feats` → `rvcb200_infer` → on-device trim), and the peak
    normalisation + int16 conversion run on the device (`rvcb200_op_absmax`, `rvcb200_op_to_int16`); one D2H of
    int16 PCM ends the call.
  * with `torch.distributed` initialised (one process per GPU) the segments are independent units: they are
    assigned longest-first to ranks, each rank converts its own, the only cross-segment reduction (`max|x|`, one
    float per rank) and the int16 pieces are gathered on the host; there is no collective on the data path.
  * segmentation is never changed for balance (it would change attention context and break parity).
  * the index blend (`index_rate > 0`, :59-75) runs on the device when the index is an `IndexIVFFlatB200` (comfy_rvc_b200/index.py:
    the same IVF-Flat nprobe-1 / flat-L2 top-1 search, gather and blend, enqueued with the segment), passed alone or as the first
    element of the `(index, big_npy)` tuple; each rank holds its own replica, so sharding needs nothing more.  Any other index
    (a faiss object, a file path, a test double) keeps the reference's host round trip per segment.
  * `rms_mix_rate < 1` (the volume-envelope mix `change_rms`, lib/model_utils.py:39, :183) runs on the device after the
    segment loop: both envelopes are built from half-second "half-block" sums, so each segment's output contributes its
    own rows to a [segments][half-blocks] table; under sharding one all-reduce of that table (each element has exactly one
    non-zero contributor) gives every rank the same envelope bits, and the sharded song stays bit-identical to the
    unsharded one.
  * `resample_sr` (`librosa.resample`, :185-186, when resample_sr >= 16000 and != tgt_sr) runs on the device after the mix and
    before the peak: `scipy.signal.resample_poly(x, up, down, window=h)` with the Kaiser-windowed sinc of
    `comfy_rvc_b200.resample.design` (libsoxr's HQ spec: passband to 0.913 of the lower Nyquist, >= 120 dB stopband from
    it), one fixed-order fp32 FMA chain per output (`rvcb200_op_resample_poly`).  The reference's soxr_hq resampler cannot
    be reproduced bit for bit and the distance to it has not been measured.  Segment i owns the outputs
    [ceil(O_i * up / down), ceil(O_{i+1} * up / down)); the filter's reach into neighbouring segments comes from a
    [segments][2][halo] table of every piece's first and last samples, all-reduced under sharding like the mix's table, so
    the sharded song stays bit-identical to the unsharded one.  `f0_autotune` is not supported.

HuBERT, the f0 estimators and faiss are upstream of this path (SURVEY.md §8f ranks 3-4): `model` is the caller's
HuBERT object, f0 estimators are looked up in `f0_method_dict` (register callables there) or passed as a
callable, and a preloaded `(index, big_npy)` tuple is honoured exactly like the reference does.
"""
from __future__ import annotations

import ctypes as C
import time
import traceback
from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
from scipy import signal

from . import _lib, resample
from .index import IndexIVFFlatB200

MAX_INT16 = 32768                                    # lib/audio.py:14
_BH, _AH = (np.ascontiguousarray(c, dtype=np.float64) for c in signal.butter(N=5, Wn=48, btype="high", fs=16000))   # :21
_ZI = np.ascontiguousarray(signal.lfilter_zi(_BH, _AH), dtype=np.float64)   # what filtfilt computes on every call (a strided view)


@dataclass
class PipelineConfig:
    """The attributes of the reference `config` object that `VC` reads (config.py:24-141)."""
    x_pad: int = 3
    x_query: int = 10
    x_center: int = 60
    x_max: int = 64
    is_half: bool = True
    device: str = "cuda:0"
    rmvpe_model_path: Optional[str] = None     # BASE_MODELS_DIR/rmvpe.pt in the reference (pitch_extraction.py:193)
    crepe_model_path: Optional[str] = None     # torchcrepe's assets/full.pth (f0_method "crepe")

    @classmethod
    def for_device(cls, is_half: bool = True, gpu_mem_gb: Optional[int] = None, device: str = "cuda:0") -> "PipelineConfig":
        """config.py:124-141: half tier (3,10,60,64); fp32 tier (1,6,38,41); <= 4 GB tier (1,5,30,32)."""
        t = (3, 10, 60, 64) if is_half else (1, 6, 38, 41)
        if gpu_mem_gb is not None and gpu_mem_gb <= 4:
            t = (1, 5, 30, 32)
        return cls(*t, is_half=is_half, device=device)


def hz_to_mel(hz):
    """lib/audio.py:302-304."""
    return 2595 * np.log10(1 + hz / 700)


# ------------------------------------------------------------------------------------------------------------
# host-side planning (pure integer / numpy work; shared by every rank, testable without a GPU)
# ------------------------------------------------------------------------------------------------------------
def filtfilt_pad(audio: np.ndarray, t_pad: int, out: Optional[np.ndarray] = None) -> np.ndarray:
    """`np.pad(signal.filtfilt(bh, ah, audio), (t_pad, t_pad), mode="reflect")` (vc_infer_pipeline.py:122 and :141) in C
    (csrc/host_plan.cu: scipy's own recursion with the order fixed at compile time, bit-identical to scipy / numpy, ~2.3x
    faster).  `out`: optional float64 buffer of n + 2 * t_pad elements (e.g. pinned staging memory)."""
    x = np.ascontiguousarray(audio, dtype=np.float64)
    n = x.shape[0]
    if x.ndim != 1 or n <= 18 or n <= t_pad:            # scipy raises for n <= padlen; short clips keep the numpy path
        return np.pad(signal.filtfilt(_BH, _AH, audio), (t_pad, t_pad), mode="reflect")
    if out is None:
        out = np.empty(n + 2 * t_pad, dtype=np.float64)
    scratch = np.empty(n + 36, dtype=np.float64)
    st = _lib.load().rvcb200_host_filtfilt_pad(x.ctypes.data, n, _BH.ctypes.data, _AH.ctypes.data, _ZI.ctypes.data,
                                               len(_BH) - 1, t_pad, out.ctypes.data, scratch.ctypes.data)
    if st != 0:
        raise RuntimeError("rvcb200_host_filtfilt_pad: bad argument")
    return out[: n + 2 * t_pad]


def split_points(audio: np.ndarray, window: int, t_query: int, t_center: int, t_max: int,
                 padded: Optional[np.ndarray] = None) -> List[int]:
    """Quiet-point search of vc_infer_pipeline.py:123-135 on the high-passed audio.  `padded`: `audio` already
    reflect-padded by window // 2 on both sides (a view of the song's t_pad-padded buffer: the inner window // 2 samples
    of a longer reflect padding are the same values)."""
    audio_pad = padded if padded is not None else np.pad(audio, (window // 2, window // 2), mode="reflect")
    opt_ts: List[int] = []
    if audio_pad.shape[0] > t_max:
        # sliding |sum| over `window` samples: a cumulative-sum form of the reference's 160 shifted adds would round
        # differently, so keep the reference's accumulation order (float64, one add per shift) -- but only over the
        # 2*t_query samples around each centre that are ever looked at (each element's sum is independent of the others,
        # so this is bit-identical to summing the whole song: 3x less host work for a 10 min song)
        n = audio.shape[0]
        # float64 (what filtfilt returns): the same sums in the same order, in C over all host threads (csrc/host_plan.cu;
        # _lib.load() raises if the library is not built).  Other dtypes keep the reference's numpy loop.
        native = _lib.load().rvcb200_host_quiet_point if audio_pad.dtype == np.float64 and audio_pad.flags.c_contiguous else None
        for t in range(t_center, n, t_center):
            lo, hi = t - t_query, min(t + t_query, n)
            if native is not None:
                j = int(native(audio_pad.ctypes.data, lo, hi, window, 0))
                if j >= 0:
                    opt_ts.append(lo + j)
                    continue
            seg = np.zeros(hi - lo, dtype=audio.dtype)
            for i in range(window):
                seg += audio_pad[lo + i: hi + i]
            seg = np.abs(seg)
            opt_ts.append(lo + int(np.where(seg == seg.min())[0][0]))
    return opt_ts


@dataclass(frozen=True)
class Segment:
    index: int
    start: int                 # sample range [start, end) in the t_pad-padded 16 kHz audio
    end: int
    f0_start: int              # frame range in the song-level pitch arrays
    f0_end: int

    @property
    def n_samples(self) -> int:
        return self.end - self.start


def plan_segments(n_padded: int, opt_ts: Sequence[int], window: int, t_pad2: int) -> List[Segment]:
    """The (start, end) slices of vc_infer_pipeline.py:167-180 as an explicit list."""
    segs: List[Segment] = []
    s = 0
    t = None
    for i, t in enumerate(opt_ts):
        t = t // window * window
        end = t + t_pad2 + window
        segs.append(Segment(i, s, end, s // window, end // window))
        s = t
    start = t if t is not None else 0
    segs.append(Segment(len(segs), start, n_padded, start // window, 1 << 62))
    return segs


def hubert_frames(n_samples: int) -> int:
    """Frames a HuBERT/ContentVec front end emits for n 16 kHz samples (receptive field 400, hop 320)."""
    return (n_samples - 400) // 320 + 1


def assign_segments(lengths: Sequence[int], world: int) -> List[List[int]]:
    """Longest-processing-time-first assignment of segments to ranks (deterministic; ties by index)."""
    order = sorted(range(len(lengths)), key=lambda i: (-lengths[i], i))
    load = [0] * world
    out: List[List[int]] = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda k: (load[k], k))
        out[r].append(i)
        load[r] += lengths[i]
    return [sorted(x) for x in out]


def makespan_bound(lengths: Sequence[int], world: int) -> float:
    """Best possible speed-up of this segment list on `world` ranks = Σlen / max rank load under LPT."""
    loads = [sum(lengths[i] for i in idx) for idx in assign_segments(lengths, world)]
    return sum(lengths) / max(max(loads), 1)


# ------------------------------------------------------------------------------------------------------------
class FeatureExtractor:
    """Constants and f0 post-processing of /root/reference/pitch_extraction.py:13-45, :252-304."""

    def __init__(self, tgt_sr, config, onnx: bool = False):
        self.x_pad, self.x_query, self.x_center, self.x_max, self.is_half = (
            config.x_pad, config.x_query, config.x_center, config.x_max, config.is_half)
        self.sr = 16000
        self.window = 160
        self.f0_bins = 256
        self.t_pad = self.sr * self.x_pad
        self.t_pad_tgt = tgt_sr * self.x_pad
        self.t_pad2 = self.t_pad * 2
        self.t_query = self.sr * self.x_query
        self.t_center = self.sr * self.x_center
        self.t_max = self.sr * self.x_max
        self.device = config.device
        self.onnx = onnx
        # the reference registers pm/harvest/dio/rmvpe/crepe here (pitch_extraction.py:28-45).  RMVPE -- the nodes' default
        # (custom_nodes/rvc_nodes.py:49) -- runs on the B200 kernels (comfy_rvc_b200/rmvpe.py); the CPU estimators (parselmouth,
        # pyworld) are upstream of this path: register any callable `fn(x=, f0_up_key=, f0_min=, f0_max=, ...) -> f0[frames]`.
        # CREPE runs on the B200 kernels too (comfy_rvc_b200/crepe.py).
        self.f0_method_dict = {"rmvpe": self.get_rmvpe, "rmvpe+": self.get_pitch_dependant_rmvpe, "crepe": self.get_crepe}
        self.rmvpe_model_path = getattr(config, "rmvpe_model_path", None)
        self.crepe_model_path = getattr(config, "crepe_model_path", None)

    def _rmvpe(self):
        """pitch_extraction.py:192-193: built on first use and kept; attach a ready model as `self.model_rmvpe` to share it."""
        if not hasattr(self, "model_rmvpe"):
            if not self.rmvpe_model_path:
                raise RuntimeError("f0_method 'rmvpe' needs `model_rmvpe` (a comfy_rvc_b200.RMVPE) or `config.rmvpe_model_path` (rmvpe.pt)")
            from .rmvpe import RMVPE
            self.model_rmvpe = RMVPE(self.rmvpe_model_path, is_half=self.is_half, device=self.device, onnx=self.onnx)
        return self.model_rmvpe

    def get_rmvpe(self, x, *args, **kwargs):
        """pitch_extraction.py:191-195."""
        return self._rmvpe().infer_from_audio(x, thred=0.03)

    def get_pitch_dependant_rmvpe(self, x, f0_min=0, f0_max=40000, *args, **kwargs):
        """pitch_extraction.py:197-201."""
        return self._rmvpe().infer_from_audio_with_pitch(x, thred=0.03, f0_min=f0_min, f0_max=f0_max)

    def _crepe(self):
        """Built on first use and kept, like `_rmvpe`; attach a ready `comfy_rvc_b200.crepe.Crepe("full")` as `self.model_crepe`
        to share it.  Without either, the weights registered with `crepe.load_weights("full", ...)` (or an installed
        torchcrepe's) are used."""
        if not hasattr(self, "model_crepe"):
            from . import crepe
            self.model_crepe = crepe.Crepe("full", weights=self.crepe_model_path, device=self.device)
        return self.model_crepe

    def get_crepe(self, x, f0_min=50, f0_max=1100, crepe_hop_length=160, model="full", **kwargs):
        """f0 by CREPE on the device.  The assumed recipe (the RVC-lineage `get_f0_crepe_computation`; the reference's own
        wrapper was not available when this was written) -- change it here and nowhere else:
          1. x = float32(x) / quantile(|x|, 0.999);
          2. predict(x, 16000, crepe_hop_length, f0_min, f0_max, "full", batch_size = 2 * crepe_hop_length, pad=True)
             (Viterbi decode);
          3. values < 0.001 -> NaN;  4. np.interp onto p_len = len(x) // 160 frames;  5. nan_to_num."""
        from . import crepe
        x = x.astype(np.float32)
        x /= np.quantile(np.abs(x), 0.999)
        audio = torch.from_numpy(x)[None]
        pitch = crepe.predict(audio, self.sr, crepe_hop_length, f0_min, f0_max, model, batch_size=crepe_hop_length * 2,
                              device=self.device, pad=True, crepe_model=self._crepe())
        source = np.array(pitch.squeeze(0).cpu().float().numpy())
        source[source < 0.001] = np.nan
        p_len = x.shape[0] // self.window
        target = np.interp(np.arange(0, len(source) * p_len, len(source)) / p_len, np.arange(0, len(source)), source)
        return np.nan_to_num(target)

    def load_index(self, file_index):
        """pitch_extraction.py:49-73: a preloaded `(index, big_npy)` tuple, an `IndexIVFFlatB200` (device blend), "" for none, or a
        faiss file path."""
        index = big_npy = None
        try:
            if isinstance(file_index, tuple):
                index, big_npy = file_index
            elif isinstance(file_index, IndexIVFFlatB200):                                     # the device index alone
                index = file_index
            elif file_index == "" or file_index is None:
                index = None
            else:
                import faiss  # not part of this image; same failure behaviour as the reference (prints, continues)
                index = faiss.read_index(file_index)
                big_npy = index.reconstruct_n(0, index.ntotal)
        except Exception as e:  # noqa: BLE001
            print(f"Could not open Faiss index file for reading. {e}")
        return index, big_npy

    def get_f0(self, x, f0_up_key, f0_method, merge_type="median", filter_radius=3, crepe_hop_length=160,
               f0_autotune=False, rmvpe_onnx=False, inp_f0=None, f0_min=50, f0_max=1100, **kwargs):
        """pitch_extraction.py:252-304 → (f0_coarse int16 [frames], f0 float [frames])."""
        time_step = self.window / self.sr * 1000
        f0_mel_min = hz_to_mel(f0_min)
        f0_mel_max = hz_to_mel(f0_max)
        params = {"x": x, "f0_up_key": f0_up_key, "f0_min": f0_min, "f0_max": f0_max, "time_step": time_step,
                  "filter_radius": filter_radius, "crepe_hop_length": crepe_hop_length, "model": "full", "onnx": rmvpe_onnx}
        if hasattr(f0_method, "pop") and len(f0_method) == 1:
            f0_method = f0_method.pop()
        if isinstance(f0_method, list):
            stack = [np.asarray(self._f0_fn(m)(**params), dtype=np.float64) for m in f0_method]
            n = max(len(s) for s in stack)
            stack = np.stack([np.pad(s, (0, n - len(s))) for s in stack])                 # lib/audio.py:257-262
            merge = {"min": np.nanmin, "max": np.nanmax, "median": np.nanmedian}.get(merge_type, np.nanmean)
            f0 = merge(stack, axis=0)                                                      # lib/utils.py:104-108
        else:
            f0 = self._f0_fn(f0_method)(**params)
        if f0_autotune:
            raise NotImplementedError("f0_autotune (lib/audio.py:274) is outside the synthesis hot path")
        f0 = np.array(f0, copy=True)
        f0 *= pow(2, f0_up_key / 12)
        tf0 = self.sr // self.window
        if inp_f0 is not None:                                                             # :282-292
            delta_t = np.round((inp_f0[:, 0].max() - inp_f0[:, 0].min()) * tf0 + 1).astype("int16")
            replace_f0 = np.interp(list(range(delta_t)), inp_f0[:, 0] * 100, inp_f0[:, 1])
            shape = f0[self.x_pad * tf0: self.x_pad * tf0 + len(replace_f0)].shape[0]
            f0[self.x_pad * tf0: self.x_pad * tf0 + len(replace_f0)] = replace_f0[:shape]
        f0_mel = hz_to_mel(f0)
        f0_mel = (f0_mel - f0_mel_min) * (self.f0_bins - 2) / (f0_mel_max - f0_mel_min) + 1
        f0_mel = np.clip(f0_mel, a_min=1, a_max=self.f0_bins - 1)
        f0_coarse = np.rint(f0_mel).astype(np.int16)
        return f0_coarse, f0

    def _f0_fn(self, method) -> Callable:
        if callable(method):
            return method
        if method not in self.f0_method_dict:
            raise Exception(f"Method {method} not found.")      # same message as pitch_extraction.py:229
        return self.f0_method_dict[method]


# ------------------------------------------------------------------------------------------------------------
class VC(FeatureExtractor):
    """Drop-in for /root/reference/vc_infer_pipeline.py:23 `class VC(FeatureExtractor)`.

    Extra keyword arguments (all optional, the reference call `VC(tgt_sr, config)` keeps working):
      noise : "device" (default) — per-segment CUDA generator seeded by (seed, segment index): results do not depend
              on how segments are sharded;  "reference" — the three draws of every segment come from the global
              torch CPU RNG in the reference's order (parity tests).
      group : torch.distributed process group to shard segments over (default: the world group when initialised).
    """

    def __init__(self, tgt_sr, config, onnx: bool = False, noise: str = "device", seed: int = 0, group=None):
        super().__init__(tgt_sr, config, onnx)
        if noise not in ("device", "reference"):
            raise ValueError(noise)
        self.noise_mode, self.seed, self.group = noise, int(seed), group
        self._host_group = None
        self._stage_buf: Optional[torch.Tensor] = None
        self._out_buf: Optional[torch.Tensor] = None
        self._resample_tables: dict = {}                 # (tgt_sr, resample_sr, device) -> `_resample_table` result
        self.last_plan: Optional[dict] = None

    # ---- one segment ------------------------------------------------------------------------------------
    def _torch_device(self) -> torch.device:
        dev = torch.device(self.device)
        if dev.type != "cuda":
            raise RuntimeError("comfy_rvc_b200.VC needs a CUDA device; the product path has no CPU fallback")
        return torch.device("cuda", dev.index if dev.index is not None else 0)

    def _segment_noise(self, net_g, i: int, T: int, staged):
        cfg = net_g.cfg
        dev = staged["dev"]
        if self.noise_mode == "reference":
            nz = torch.randn(1, cfg.inter_channels, T)          # models.py:685/801 (:908 for the no-f0 classes)
            if not cfg.f0:
                return (nz,)
            ri = torch.rand(1, 1)                               # models.py:378
            ns = torch.randn(1, T * cfg.upp, 1)                 # models.py:409
            return nz, ri, ns
        g = torch.Generator(device=dev).manual_seed(self.seed * 1000003 + i)
        nz = torch.randn(1, cfg.inter_channels, T, device=dev, generator=g)
        if not cfg.f0:
            return (nz,)
        ri = torch.rand(1, 1, device=dev, generator=g)
        ns = torch.randn(1, T * cfg.upp, 1, device=dev, generator=g)
        return nz, ri, ns

    def _vc_device(self, model, net_g, sid, audio0, n_samples: int, pitch, pitchf, index, big_npy, index_rate, version,
                   protect, noise=None) -> torch.Tensor:
        """`VC.vc` up to (not including) the D2H copy: returns the segment's PCM as a device tensor [L] fp32.
        `audio0` is a device tensor [n] (fp32 or fp16)."""
        dev = audio0.device
        lib = _lib.load()
        feats = audio0.view(1, -1)
        padding_mask = torch.zeros(feats.shape, dtype=torch.bool, device=dev)
        inputs = {"source": feats, "padding_mask": padding_mask, "output_layer": 9 if version == "v1" else 12}
        feats = model.extract_features(version=version, **inputs)                              # :48-55
        if callable(noise):      # "reference" noise: drawn AFTER the feature extractor, like models.py:801 after :48-55 -- HuggingFace's
            noise = noise()      # HuBERT consumes the global generator itself (one torch.rand([]) per encoder layer and forward)
        use_f0 = pitch is not None and pitchf is not None
        feats0 = feats if (protect < 0.5 and use_f0) else None                                 # :57-58 (no clone needed)
        if isinstance(index, IndexIVFFlatB200) and index_rate > 0:                             # :59-75 on the device
            feats = index.blend(feats, index_rate, self.is_half)
        elif index is not None and big_npy is not None and index_rate > 0:                     # :59-75, host like the reference
            npy = feats[0].float().cpu().numpy()
            score, ix = index.search(npy, k=1)
            weight = np.square(1 / score)
            weight /= weight.sum(axis=1, keepdims=True)
            npy = np.sum(big_npy[ix] * np.expand_dims(weight, axis=2), axis=1)
            if self.is_half:
                npy = npy.astype("float16")
            feats = torch.from_numpy(npy).unsqueeze(0).to(dev) * index_rate + (1 - index_rate) * feats
        if feats.dtype not in (torch.float32, torch.float16):
            feats = feats.float()
            feats0 = feats0.float() if feats0 is not None else None
        feats = feats.contiguous()
        F_, Cf = int(feats.shape[1]), int(feats.shape[2])
        p_len = min(n_samples // self.window, 2 * F_)                                          # :83
        if use_f0:
            pitch = pitch[:, :p_len].contiguous()                                              # :86-87
            pitchf = pitchf[:, :p_len].contiguous()
            if pitch.shape[1] < p_len:
                raise ValueError(f"pitch has {pitch.shape[1]} frames, segment needs {p_len}")
        phone = torch.empty(1, p_len, Cf, device=dev, dtype=torch.float32)
        use_protect = 1 if feats0 is not None else 0
        f0p = feats0.contiguous() if feats0 is not None else feats
        if f0p.dtype != feats.dtype:
            f0p = f0p.to(feats.dtype)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.rvcb200_op_prepare_feats(                                               # :77-95 in one kernel
            C.c_void_p(feats.data_ptr()), C.c_void_p(f0p.data_ptr()), 0 if feats.dtype == torch.float32 else 1,
            C.c_void_p(pitchf.data_ptr() if use_f0 else None), C.c_void_p(phone.data_ptr()), F_, p_len, Cf, float(protect),
            use_protect,
            C.c_void_p(stream)), None, "prepare_feats")
        p_len_t = torch.full((1,), p_len, device=dev, dtype=torch.int64)                       # :96 (no H2D copy)
        kw = {"noise": noise} if noise is not None else {}
        if use_f0:
            return net_g.infer(phone, p_len_t, pitch, pitchf, sid, **kw)[0][0, 0]              # :97-101
        return net_g.infer(phone, p_len_t, sid, **kw)[0][0, 0]                                 # :102-105

    def vc(self, model, net_g, sid, audio0, pitch, pitchf, times, index, big_npy, index_rate, version, protect):
        """Same contract as the reference `VC.vc` (vc_infer_pipeline.py:25-114): numpy in, float32 numpy PCM out."""
        dev = self._torch_device()
        feats = torch.from_numpy(np.ascontiguousarray(audio0))
        feats = feats.half() if self.is_half else feats.float()
        if feats.dim() == 2:
            feats = feats.mean(-1)
        assert feats.dim() == 1, feats.dim()
        with torch.cuda.device(dev):
            o = self._vc_device(model, net_g, sid, feats.to(dev), int(audio0.shape[0]), pitch, pitchf, index, big_npy,
                                index_rate, version, protect)
            return o.data.cpu().float().numpy()

    # ---- sharding helpers -----------------------------------------------------------------------------
    def _dist(self):
        import torch.distributed as dist
        if self.group is None and not (dist.is_available() and dist.is_initialized()):
            return None, 0, 1
        return dist, dist.get_rank(self.group), dist.get_world_size(self.group)

    def _gloo_group(self, dist):
        """Host-side gathers go through a gloo group (created once, collectively) when the data group is NCCL."""
        if self._host_group is None:
            if dist.get_backend(self.group) == "gloo":
                self._host_group = self.group if self.group is not None else dist.group.WORLD
            else:
                ranks = dist.get_process_group_ranks(self.group) if self.group is not None else None
                self._host_group = dist.new_group(ranks=ranks, backend="gloo")
        return self._host_group

    # ---- the song-level driver ---------------------------------------------------------------------------
    def plan(self, audio: np.ndarray):
        """Host-side planning shared by all ranks: high-pass, quiet points, padded audio, segment list."""
        audio = np.asarray(audio)
        n, h = audio.shape[0], self.window // 2
        if audio.ndim == 1 and n > max(self.t_pad, 18) and self.t_pad >= h:
            audio_pad = filtfilt_pad(audio, self.t_pad, out=self._staging(n + 2 * self.t_pad))  # :122 + :141, one pass
            audio = audio_pad[self.t_pad: self.t_pad + n]
            padded = audio_pad[self.t_pad - h: self.t_pad + n + h]
        else:
            audio = signal.filtfilt(_BH, _AH, audio)                                           # :122
            audio_pad = np.pad(audio, (self.t_pad, self.t_pad), mode="reflect")                # :141
            padded = None
        opt_ts = split_points(audio, self.window, self.t_query, self.t_center, self.t_max, padded)   # :123-135
        segs = plan_segments(audio_pad.shape[0], opt_ts, self.window, self.t_pad2)
        return audio, audio_pad, opt_ts, segs

    def _pinned_out(self, n: int) -> torch.Tensor:
        """Reusable pinned int16 buffer for the song's single D2H copy (cudaHostAlloc of ~60 MB costs ~10 ms per call)."""
        if self._out_buf is None or self._out_buf.numel() < n:
            self._out_buf = torch.empty(max(n, 1), dtype=torch.int16).pin_memory()
        return self._out_buf[:n]

    def _staging(self, n: int) -> np.ndarray:
        """Reusable float64 host buffer the filtered, padded song is written into: pinned when a CUDA device is present
        (it is the source of the song's one H2D copy), plain memory otherwise (host-only planning)."""
        if self._stage_buf is None or self._stage_buf.numel() < n:
            t = torch.empty(n, dtype=torch.float64)
            self._stage_buf = t.pin_memory() if torch.cuda.is_available() else t
        return self._stage_buf.numpy()[:n]

    def pipeline(self, model, net_g, sid, audio, times, f0_up_key, f0_method, merge_type, file_index, index_rate, if_f0,
                 filter_radius, tgt_sr, resample_sr, rms_mix_rate, version, protect, crepe_hop_length, f0_autotune,
                 rmvpe_onnx, f0_file=None, f0_min=50, f0_max=1600, all_ranks: bool = False):
        """Same contract as the reference `VC.pipeline` (vc_infer_pipeline.py:116-196) → int16 PCM at `tgt_sr`.

        Under `torch.distributed` every rank must call it with the same arguments; rank 0 (or every rank with
        `all_ranks=True`) returns the song, the others return None."""
        if rms_mix_rate < 1:
            self._require_device_mix()
        resampling = resample_sr >= 16000 and tgt_sr != resample_sr                            # :185
        if resampling:
            self._require_device_resample()
        dist, rank, world = self._dist()
        t0 = time.time()
        index, big_npy = self.load_index(file_index)
        audio, audio_pad, opt_ts, segs, staged_audio = self._plan_song(np.asarray(audio))
        t_plan = time.time()
        inp_f0 = None
        if f0_file is not None:                                                                # :144-149
            try:
                with open(f0_file.name, "r") as f:
                    inp_f0 = np.array([list(map(float, line.split(","))) for line in f.read().strip("\n").split("\n")],
                                      dtype="float32")
            except Exception:  # noqa: BLE001
                traceback.print_exc()
        pitch = pitchf = None
        if if_f0 == 1:                                                                         # :153-162
            pitch, pitchf = self.get_f0(audio_pad, f0_up_key, f0_method, merge_type, filter_radius, crepe_hop_length,
                                        f0_autotune, rmvpe_onnx, inp_f0, f0_min, f0_max)
            p_len = min(pitch.shape[0], pitchf.shape[0])
            pitch = pitch[:p_len].astype(np.int64)
            pitchf = pitchf[:p_len].astype(np.float32)
        if (pitch is None) != (not getattr(getattr(net_g, "cfg", None), "f0", True)):
            raise ValueError("if_f0 does not match the synthesizer class (f0 vs `_nono`)")
        lengths = [s.n_samples for s in segs]
        assignment = assign_segments(lengths, world)
        mine = assignment[rank]
        self.last_plan = {"opt_ts": list(opt_ts), "segments": segs, "assignment": assignment,
                          "makespan_bound": makespan_bound(lengths, world)}
        staged = self._stage(audio_pad, pitch, pitchf, sid, net_g, staged_audio)               # H2D once per song
        if rms_mix_rate >= 1:
            staged.pop("audio64", None)                                                        # only the mix reads it
        t1 = time.time()
        times[1] += t1 - t0                                                                    # :164-165
        ev0 = self._record_event(staged)
        parts = []
        for s in segs:
            T_formula = min(s.n_samples // self.window, 2 * hubert_frames(s.n_samples))
            run = s.index in mine
            noise = None
            if self.noise_mode == "reference":          # every rank advances the global stream past every segment, in the
                if run:                                 # reference's order: the front end's own draws, then the synthesizer's
                    noise = (lambda s=s, T=T_formula: self._segment_noise(net_g, s.index, T, staged))
                else:
                    for _ in range(int(getattr(model, "rng_draws_per_call", 0))):
                        torch.rand([])
                    self._segment_noise(net_g, s.index, T_formula, staged)
            elif run:
                noise = self._segment_noise(net_g, s.index, T_formula, staged)
            if run:
                parts.append((s.index, self._convert(staged, model, net_g, s, T_formula, index, big_npy, index_rate,
                                                     version, protect, noise)))
        sizes = None
        if world > 1:            # every rank derives all piece sizes from the plan (400 / 320 frame formula of the front end)
            sizes = [min(s.n_samples // self.window, 2 * hubert_frames(s.n_samples)) * net_g.cfg.upp - 2 * self.t_pad_tgt for s in segs]
        if rms_mix_rate < 1:                                                                   # :183, before the peak
            mix_sizes = sizes if sizes is not None else [len(p) for _, p in parts]             # world 1: every part, in order
            self._rms_mix(staged, parts, mix_sizes, audio.shape[0], tgt_sr, rms_mix_rate, dist, world)
        if resampling:                                                                         # :185-186, before the peak
            parts, out_sizes = self._resample(staged, parts, sizes if sizes is not None else [len(p) for _, p in parts],
                                              tgt_sr, resample_sr, dist, world)
            sizes = out_sizes if sizes is not None else None
        t_enq = time.time()
        if world > 1 and self._device_collectives(dist, staged):
            # NCCL group: the peak is one 4-byte all-reduce and the int16 pieces travel GPU to GPU (NVLink); rank 0 orders
            # them on the device and does the song's single D2H -- no pickling, no host round trip per rank
            out = self._finalize_gather_device(staged, parts, sizes, assignment, dist, rank, world, all_ranks)
            self._timing(staged, ev0, t0, t_plan, t1, t_enq)
            times[2] += time.time() - t1
            return out

        def exchange_peak(local_peak: float) -> float:                                         # the only reduction
            if world == 1:
                return local_peak
            peaks = [None] * world
            dist.all_gather_object(peaks, float(local_peak), group=self._gloo_group(dist))
            return max(peaks)

        mine_np = self._finalize(staged, parts, exchange_peak if world > 1 else None)          # :182-189
        self._timing(staged, ev0, t0, t_plan, t1, t_enq)
        if world > 1:
            gathered = [None] * world
            hg = self._gloo_group(dist)
            if all_ranks:
                dist.all_gather_object(gathered, mine_np, group=hg)
            else:
                dist.gather_object(mine_np, gathered if rank == 0 else None, dst=dist.get_global_rank(hg, 0), group=hg)
            if rank != 0 and not all_ranks:
                times[2] += time.time() - t1
                return None
            mine_np = {}
            for d in gathered:
                mine_np.update(d)
        out = np.concatenate([mine_np[i] for i in range(len(segs))])
        times[2] += time.time() - t1
        return out

    # ---- volume-envelope mix (change_rms, lib/model_utils.py:39, vc_infer_pipeline.py:183): host logic ---------------
    def _rms_mix(self, staged, parts, sizes, n_in: int, tgt_sr: int, rate: float, dist=None, world: int = 1):
        """Scale this rank's trimmed segment outputs `parts` [(segment index, samples)] in place by
        rms1 ** (1 - rate) * max(rms2, 1e-6) ** (rate - 1), the reference's `change_rms(audio, 16000, audio_opt, tgt_sr, rate)`.

        librosa.feature.rms with frame_length = 2 * hop (sr // 2 * 2 and sr // 2 for every sr) and centre padding makes frame f
        the sum of half-blocks f - 1 and f (half-block b = samples [b * hop, (b + 1) * hop)).  rms1 comes from the staged
        float64 input song (one piece, every rank).  For rms2, segment i (global offset = sum of sizes[:i]) writes its
        half-block sums into row i of a [segments][half-blocks] float64 table; under sharding the table is all-reduced
        (each element has one non-zero contributor, so the sum is exact in any order) and the rows are folded in segment
        order: the same bits on every rank and for every world size.  `sizes`: every segment's output length."""
        hop1, hop2 = self.sr // 2, int(tgt_sr) // 2
        offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        N = int(offs[-1])
        if N == 0:
            return
        for i, p in parts:
            if len(p) != sizes[i]:
                raise RuntimeError("HuBERT front end does not follow the 400/320 frame formula; segment sizes cannot be "
                                   "derived from the plan for the device-side gather")
        dev = staged["dev"]
        t1 = torch.zeros(1, 1 + n_in // hop1, dtype=torch.float64, device=dev)
        x1 = staged["audio64"][self.t_pad: self.t_pad + n_in]                              # the high-passed, unpadded song
        self._mix_power(staged, x1, 0, hop1, t1[0, : (n_in - 1) // hop1 + 1])
        rms1 = self._mix_fold(staged, t1, 2 * hop1)
        t2 = torch.zeros(len(sizes), 1 + N // hop2, dtype=torch.float64, device=dev)
        for i, p in parts:
            o, n = int(offs[i]), int(sizes[i])
            if n:
                self._mix_power(staged, p, o, hop2, t2[i, o // hop2: (o + n - 1) // hop2 + 1])
        if world > 1:
            if self._device_collectives(dist, staged):
                dist.all_reduce(t2, op=dist.ReduceOp.SUM, group=self.group)
            else:
                h = t2.cpu()
                dist.all_reduce(h, op=dist.ReduceOp.SUM, group=self._gloo_group(dist))
                if h is not t2:
                    t2.copy_(h)
        rms2 = self._mix_fold(staged, t2, 2 * hop2)
        for i, p in parts:
            self._mix_gain(staged, p, int(offs[i]), N, rms1, rms2, rate)

    # ---- output resampling (librosa.resample, vc_infer_pipeline.py:185-186): host logic ----------------------------------
    def _resample(self, staged, parts, sizes, tgt_sr: int, resample_sr: int, dist=None, world: int = 1):
        """Resample this rank's segment outputs `parts` [(segment index, samples)] from tgt_sr to resample_sr
        (`resample.design`, scipy's resample_poly).  Returns (resampled parts, every segment's resampled size).

        Segment i starts at input sample O_i = sum(sizes[:i]) and owns the outputs [ceil(O_i * up / down),
        ceil(O_{i+1} * up / down)), an exact partition of the resampled song.  An output's filter reaches up to H samples
        into the neighbouring segments, which may live on other ranks: each rank writes the first and last H samples of its
        pieces into their rows of a [segments][2][H] float32 table, zero elsewhere; under sharding the table is all-reduced
        (one non-zero contributor per element, so the sum is exact) and every segment's halos are assembled from the rows
        around it.  The same path runs at world size 1, and every output is one fixed-order sum, so the sharded song is
        bit-identical to the unsharded one.  `sizes`: every segment's input length."""
        up, down, half_len, tpp, table = self._resample_table(staged, tgt_sr, resample_sr)
        H = resample.halo_len(2 * half_len + 1, up)
        offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        N = int(offs[-1])
        bounds = [resample.out_len(int(o), up, down) for o in offs]
        out_sizes = [bounds[i + 1] - bounds[i] for i in range(len(sizes))]
        for i, p in parts:
            if len(p) != sizes[i]:
                raise RuntimeError("HuBERT front end does not follow the 400/320 frame formula; segment sizes cannot be "
                                   "derived from the plan for the device-side gather")
        dev = staged["dev"]
        edges = torch.zeros(len(sizes), 2, H, dtype=torch.float32, device=dev)
        for i, p in parts:
            n = min(H, len(p))
            if n:
                p_t = torch.as_tensor(p, device=dev)
                edges[i, 0, :n] = p_t[:n]
                edges[i, 1, H - n:] = p_t[len(p) - n:]
        if world > 1:
            if self._device_collectives(dist, staged):
                dist.all_reduce(edges, op=dist.ReduceOp.SUM, group=self.group)
            else:
                h = edges.cpu()
                dist.all_reduce(h, op=dist.ReduceOp.SUM, group=self._gloo_group(dist))
                if h is not edges:
                    edges.copy_(h)
        out = []
        for i, p in parts:
            left, need, k = [], H, i - 1                                   # the last H samples before segment i
            while need > 0 and k >= 0:
                n = min(need, int(sizes[k]))
                if n:
                    left.insert(0, edges[k, 1, H - n:])
                need -= n
                k -= 1
            right, need, k = [], H, i + 1                                  # the first H samples after it
            while need > 0 and k < len(sizes):
                n = min(need, int(sizes[k]))
                if n:
                    right.append(edges[k, 0, :n])
                need -= n
                k += 1
            cat = lambda xs: torch.cat(xs) if xs else edges.new_zeros(0)
            out.append((i, self._resample_span(staged, table, up, down, tpp, half_len, cat(left), p, cat(right), int(offs[i]), N,
                                               bounds[i], bounds[i + 1])))
        return out, out_sizes

    # ---- hooks with a host default (the CPU test double overrides the device ones below) ------------------------
    def _plan_song(self, audio: np.ndarray):
        """Planning for `pipeline`: like `plan`, but with a CUDA device the quiet-point search runs there on the staged
        float64 song (same sums in the same order, `rvcb200_op_quiet_point`), so the song crosses PCIe once, as float64,
        straight from the pinned buffer the filter wrote.  Returns (..., staged float64 device tensor or None)."""
        dev = torch.device(self.device)
        n, h = audio.shape[0], self.window // 2
        if (dev.type != "cuda" or not torch.cuda.is_available() or type(self)._stage is not VC._stage
                or not (audio.ndim == 1 and n > max(self.t_pad, 18) and self.t_pad >= h)):
            return (*self.plan(audio), None)
        dev = self._torch_device()
        lib = _lib.load()
        with torch.cuda.device(dev):
            audio_pad = filtfilt_pad(audio, self.t_pad, out=self._staging(n + 2 * self.t_pad))  # :122 + :141
            audio_d = torch.from_numpy(audio_pad).to(dev, non_blocking=True)
            opt_ts: List[int] = []
            if n + 2 * h > self.t_max:                                                         # :127
                centres = list(range(self.t_center, n, self.t_center))
                nb = 64
                bv = torch.empty(len(centres), nb, dtype=torch.float64, device=dev)
                bj = torch.empty(len(centres), nb, dtype=torch.int64, device=dev)
                stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                base = audio_d.data_ptr() + (self.t_pad - h) * 8                               # audio reflect-padded by window // 2
                for k, t in enumerate(centres):
                    lo, hi = t - self.t_query, min(t + self.t_query, n)
                    _lib.check(lib.rvcb200_op_quiet_point(C.c_void_p(base), lo, hi, self.window, C.c_void_p(bv[k].data_ptr()),
                                                          C.c_void_p(bj[k].data_ptr()), nb, stream), None, "quiet_point")
                bv_h, bj_h = bv.cpu().numpy(), bj.cpu().numpy()                                # one small D2H (sync)
                for k in range(len(centres)):
                    best_v, best_j = np.inf, -1
                    for b in range(nb):                                                        # ascending ranges: first minimum
                        if bj_h[k, b] >= 0 and bv_h[k, b] < best_v:
                            best_v, best_j = bv_h[k, b], int(bj_h[k, b])
                    if best_j < 0:                                                             # every sum NaN: numpy's argmin rule
                        best_j = centres[k] - self.t_query
                    opt_ts.append(best_j)
        segs = plan_segments(audio_pad.shape[0], opt_ts, self.window, self.t_pad2)
        return audio_pad[self.t_pad: self.t_pad + n], audio_pad, opt_ts, segs, audio_d

    # ---- device side of the song-level driver (everything below touches the GPU) -----------------------------
    def _require_device_mix(self):
        """Checked before planning: the volume-envelope mix has no host implementation."""
        if torch.device(self.device).type != "cuda":
            raise NotImplementedError("rms_mix_rate < 1 (change_rms, lib/model_utils.py:39) runs on the device only; "
                                      "no CPU fallback")

    def _mix_power(self, staged, x, offset: int, hop: int, out):
        """Half-block sums of float32(x)^2 for the piece x (float32 / float64) at global sample `offset` into `out` (float64,
        one value per half-block the piece touches), `rvcb200_op_rms_halfblock`."""
        if x.dtype not in (torch.float32, torch.float64) or not x.is_contiguous() or not out.is_contiguous():
            raise ValueError("rms mix: contiguous float32 / float64 pieces only")
        with torch.cuda.device(staged["dev"]):
            stream = C.c_void_p(torch.cuda.current_stream(staged["dev"]).cuda_stream)
            _lib.check(_lib.load().rvcb200_op_rms_halfblock(C.c_void_p(x.data_ptr()), 1 if x.dtype == torch.float64 else 0, x.numel(),
                                                            offset, hop, C.c_void_p(out.data_ptr()), stream), None, "rms_halfblock")

    def _mix_fold(self, staged, table, frame_length: int):
        """Frame RMS (float32, one per column) of a [rows][half-blocks] table, rows folded in order (`rvcb200_op_rms_fold`)."""
        rms = torch.empty(table.shape[1], dtype=torch.float32, device=table.device)
        with torch.cuda.device(staged["dev"]):
            stream = C.c_void_p(torch.cuda.current_stream(staged["dev"]).cuda_stream)
            _lib.check(_lib.load().rvcb200_op_rms_fold(C.c_void_p(table.data_ptr()), table.shape[0], table.shape[1], frame_length,
                                                       C.c_void_p(rms.data_ptr()), stream), None, "rms_fold")
        return rms

    def _mix_gain(self, staged, x, offset: int, n_total: int, rms1, rms2, rate: float):
        """x (float32 samples [offset, offset + len) of the n_total-sample song) *= the mix gain, in place (`rvcb200_op_rms_gain`)."""
        if x.dtype != torch.float32 or not x.is_contiguous():
            raise ValueError("rms mix: contiguous float32 output pieces only")
        with torch.cuda.device(staged["dev"]):
            stream = C.c_void_p(torch.cuda.current_stream(staged["dev"]).cuda_stream)
            _lib.check(_lib.load().rvcb200_op_rms_gain(C.c_void_p(x.data_ptr()), x.numel(), offset, n_total, C.c_void_p(rms1.data_ptr()),
                                                       rms1.numel(), C.c_void_p(rms2.data_ptr()), rms2.numel(), float(rate), stream),
                       None, "rms_gain")

    def _require_device_resample(self):
        """Checked before planning: the output resampling has no host implementation."""
        if torch.device(self.device).type != "cuda":
            raise NotImplementedError("resample_sr (librosa.resample, vc_infer_pipeline.py:185-186) runs on the device only; "
                                      "no CPU fallback")

    def _resample_table(self, staged, tgt_sr: int, resample_sr: int):
        """(up, down, half_len, taps per phase, device phase table) of tgt_sr -> resample_sr, designed once per rate pair and
        device and kept on this object."""
        key = (int(tgt_sr), int(resample_sr), staged["dev"])
        cache = self._resample_tables
        if key not in cache:
            up, down, h = resample.design(tgt_sr, resample_sr)
            tab = torch.from_numpy(resample.phase_table(h, up)).to(staged["dev"])
            cache[key] = (up, down, (h.shape[0] - 1) // 2, resample.taps_per_phase(h.shape[0], up), tab)
        return cache[key]

    def _resample_span(self, staged, table, up, down, tpp, half_len, left, piece, right, piece_off: int, n_song: int,
                       out_lo: int, out_hi: int):
        """Outputs [out_lo, out_hi) of the resampled song from [left | piece | right] (`rvcb200_op_resample_poly`)."""
        if any(t.dtype != torch.float32 or not t.is_contiguous() for t in (left, piece, right)):
            raise ValueError("resample: contiguous float32 pieces only")
        out = torch.empty(out_hi - out_lo, dtype=torch.float32, device=staged["dev"])
        ptr = lambda t: C.c_void_p(t.data_ptr() if t.numel() else None)
        with torch.cuda.device(staged["dev"]):
            stream = C.c_void_p(torch.cuda.current_stream(staged["dev"]).cuda_stream)
            _lib.check(_lib.load().rvcb200_op_resample_poly(
                ptr(table), up, down, tpp, half_len, ptr(left), left.numel(), ptr(piece), piece.numel(), ptr(right), right.numel(),
                piece_off, n_song, out_lo, out_hi, ptr(out), stream), None, "resample_poly")
        return out

    def _record_event(self, staged):
        if staged["dev"].type != "cuda":
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(staged["dev"]))
        return ev

    def _timing(self, staged, ev0, t0, t_plan, t_stage, t_enq):
        """Where the call's time went: host phases by wall clock, the enqueued device work by CUDA events."""
        ev1 = self._record_event(staged)
        if ev1 is not None:
            ev1.synchronize()
        self.last_plan["host_s"] = {"plan": t_plan - t0, "f0_and_stage": t_stage - t_plan, "enqueue": t_enq - t_stage,
                                    "total": time.time() - t0}
        self.last_plan["device_ms"] = ev0.elapsed_time(ev1) if ev0 is not None else None

    def _device_collectives(self, dist, staged) -> bool:
        return staged["dev"].type == "cuda" and dist.get_backend(self.group) == "nccl"

    def _stage(self, audio_pad, pitch, pitchf, sid, net_g, staged_audio=None) -> dict:
        dev = self._torch_device()
        with torch.cuda.device(dev):
            # the whole song, once: float64 from the (pinned) staging buffer, rounded to the model dtype on the device --
            # the same single rounding as the reference's `torch.from_numpy(audio0).half() / .float()` (:40-44)
            audio_d = staged_audio if staged_audio is not None else torch.from_numpy(audio_pad).to(dev, non_blocking=True)
            return {
                "dev": dev,
                "audio": audio_d.half() if self.is_half else audio_d.float(),
                "audio64": audio_d,                                                            # the input envelope of the rms mix
                "sid": torch.as_tensor(sid).reshape(1).to(dev).long(),                         # :151
                "pitch": torch.from_numpy(pitch).to(dev).unsqueeze(0) if pitch is not None else None,
                "pitchf": torch.from_numpy(pitchf).to(dev).unsqueeze(0) if pitchf is not None else None,
            }

    def _convert(self, staged, model, net_g, s: Segment, T_formula: int, index, big_npy, index_rate, version, protect, noise):
        """One segment, enqueued without a host round trip; returns the trimmed PCM as a device tensor."""
        dev = staged["dev"]
        with torch.cuda.device(dev):
            o = self._vc_device(model, net_g, staged["sid"], staged["audio"][s.start:s.end], s.n_samples,
                                staged["pitch"][:, s.f0_start:s.f0_end] if staged["pitch"] is not None else None,
                                staged["pitchf"][:, s.f0_start:s.f0_end] if staged["pitchf"] is not None else None,
                                index, big_npy, index_rate, version, protect, noise=noise)
            if self.noise_mode == "reference" and o.shape[0] != T_formula * net_g.cfg.upp:
                raise RuntimeError("HuBERT front end does not follow the 400/320 frame formula; reference-order noise "
                                   "cannot be pre-drawn")
            return o[self.t_pad_tgt: o.shape[0] - self.t_pad_tgt]                              # :174/:180 trim, on device

    def _finalize_gather_device(self, staged, parts, sizes_h, assignment, dist, rank, world, all_ranks):
        """`_finalize` + the gather for an NCCL group, all on the device: peak = all-reduce(max) of one float; every rank
        converts its segments to int16 against the song-wide peak; the pieces go to rank 0 (to every rank with
        `all_ranks`) as bytes over NVLink; the destination orders them by segment index and copies the song to the host
        once.  No collective touches the synthesis itself (SURVEY.md §8e)."""
        dev = staged["dev"]
        lib = _lib.load()
        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            local = torch.cat([p for _, p in parts]) if parts else torch.empty(0, device=dev)
            peak = torch.zeros(1, device=dev, dtype=torch.float32)
            _lib.check(lib.rvcb200_op_absmax(C.c_void_p(local.data_ptr()), local.numel(), C.c_void_p(peak.data_ptr()), 1,
                                             stream), None, "absmax")
            dist.all_reduce(peak, op=dist.ReduceOp.MAX, group=self.group)                      # :188, the only reduction
            for i, p in parts:           # every rank derives all piece sizes from the plan (400 / 320 frame formula of the front end)
                if int(p.numel()) != sizes_h[i]:
                    raise RuntimeError("HuBERT front end does not follow the 400/320 frame formula; segment sizes cannot be "
                                       "derived from the plan for the device-side gather")
            pcm = torch.empty(local.numel(), device=dev, dtype=torch.int16)
            _lib.check(lib.rvcb200_op_to_int16(C.c_void_p(local.data_ptr()), local.numel(), C.c_void_p(peak.data_ptr()),
                                               C.c_void_p(pcm.data_ptr()), stream), None, "to_int16")
            per_rank = [sum(sizes_h[i] for i in assignment[r]) for r in range(world)]
            dst_ranks = list(range(world)) if all_ranks else [0]
            bufs = {}
            ops = []
            grp = self.group
            g = (lambda r: dist.get_global_rank(grp, r)) if grp is not None else (lambda r: r)
            mine = pcm.view(torch.uint8)
            if rank in dst_ranks:
                for r in range(world):
                    if r == rank:
                        bufs[r] = mine
                    elif per_rank[r]:
                        bufs[r] = torch.empty(2 * per_rank[r], device=dev, dtype=torch.uint8)
                        ops.append(dist.P2POp(dist.irecv, bufs[r], g(r), group=grp))
            if mine.numel():
                for d in dst_ranks:
                    if d != rank:
                        ops.append(dist.P2POp(dist.isend, mine, g(d), group=grp))
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            if rank not in dst_ranks:
                torch.cuda.current_stream(dev).synchronize()
                return None
            offs = np.concatenate([[0], np.cumsum(sizes_h)]).astype(np.int64)
            song = torch.empty(int(offs[-1]), device=dev, dtype=torch.int16)
            for r in range(world):
                o = 0
                for i in assignment[r]:
                    n = sizes_h[i]
                    song[offs[i]: offs[i] + n] = bufs[r].view(torch.int16)[o: o + n]
                    o += n
            out_h = self._pinned_out(song.numel())
            out_h.copy_(song, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        return out_h.numpy().copy()              # the caller owns the result; the pinned buffer is reused by the next song

    def _finalize(self, staged, parts, exchange_peak) -> dict:
        """Concatenate this rank's trimmed segments, peak-normalise against the song-wide max and convert to int16 on the
        device (vc_infer_pipeline.py:182-189); one D2H.  Returns {segment index: int16 array}."""
        dev = staged["dev"]
        lib = _lib.load()
        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            local = torch.cat([p for _, p in parts]) if parts else torch.empty(0, device=dev)
            peak = torch.zeros(1, device=dev, dtype=torch.float32)
            _lib.check(lib.rvcb200_op_absmax(C.c_void_p(local.data_ptr()), local.numel(), C.c_void_p(peak.data_ptr()), 1,
                                             stream), None, "absmax")
            if exchange_peak is not None:
                peak.fill_(exchange_peak(float(peak.item())))
            pcm = torch.empty(local.numel(), device=dev, dtype=torch.int16)
            _lib.check(lib.rvcb200_op_to_int16(C.c_void_p(local.data_ptr()), local.numel(), C.c_void_p(peak.data_ptr()),
                                               C.c_void_p(pcm.data_ptr()), stream), None, "to_int16")
            out_h = self._pinned_out(pcm.numel())
            out_h.copy_(pcm, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        out = out_h.numpy()
        res, off = {}, 0
        for i, p in parts:
            n = int(p.numel())
            res[i] = out[off:off + n].copy()
            off += n
        return res


def get_vc(model_path, file_index=None, config=None, device=None):
    """Reference `get_vc` (vc_infer_pipeline.py:198-249) on the B200 classes: checkpoint → {vc, cpt, net_g, ...}."""
    import os
    from .synthesizer import (SynthesizerTrnMs256NSFsid, SynthesizerTrnMs768NSFsid, SynthesizerTrnMs256NSFsid_nono,
                              SynthesizerTrnMs768NSFsid_nono)
    config = config or PipelineConfig()
    cpt = torch.load(model_path, map_location="cpu")
    tgt_sr = cpt["config"][-1]
    cpt["config"][-3] = cpt["weight"]["emb_g.weight"].shape[0]       # n_spk
    if_f0 = cpt.get("f0", 1)
    version = cpt.get("version", "v1")
    if if_f0 == 1:                                                     # the 4-way dispatch of vc_infer_pipeline.py:205-218
        cls = SynthesizerTrnMs256NSFsid if version == "v1" else SynthesizerTrnMs768NSFsid
    else:
        cls = SynthesizerTrnMs256NSFsid_nono if version == "v1" else SynthesizerTrnMs768NSFsid_nono
    net_g = cls(*cpt["config"], is_half=config.is_half)
    del net_g.enc_q
    net_g.load_state_dict(cpt["weight"], strict=False)
    net_g.eval().to(device if device else config.device)
    net_g = net_g.half() if config.is_half else net_g.float()
    vc = VC(tgt_sr, config)
    model_name = os.path.basename(model_path).split(".")[0]
    if isinstance(file_index, str) and file_index and os.path.exists(file_index):
        file_index = vc.load_index(file_index)
        if file_index[0] is None:
            file_index = ""
    elif not isinstance(file_index, (tuple, IndexIVFFlatB200)):
        file_index = ""
    return {"vc": vc, "cpt": cpt, "net_g": net_g, "model_name": model_name, "file_index": file_index, "sr": cpt["config"][-1]}
