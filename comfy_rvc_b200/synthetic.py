"""Deterministic synthetic checkpoints, inputs and noise (no network, no real checkpoints).

Recipe follows SURVEY.md §8(d): seeded weights stored through fp16 exactly like real RVC
"small model" files (/root/reference/training_cli.py:41-45), non-zero
`flow.flows.*.post` (the reference zero-initialises it, modules.py:432-434, which would make
the flow an identity and hide bugs), `phone ~ N(0,1)`, a smooth voiced f0 contour with
unvoiced gaps, `pitch` from the reference's mel quantiser
(/root/reference/pitch_extraction.py:266-267,296-302; lib/audio.py:302-304), and the three noise tensors drawn in the
reference's call order (models.py:685/801 `randn_like[B,192,T]`, :378 `rand(B,1)`,
:409 `randn_like[B,L,1]`).

Everything is generated on the CPU with `torch.Generator` so the same seeds give the same
tensors in the build container and on the GPU box (same image, same torch build).
"""
from __future__ import annotations

import math
import zlib
from typing import Dict, Tuple

import numpy as np
import torch

from .config import SynthConfig, state_dict_shapes


def _fan_in(shape) -> int:
    n = 1
    for d in shape[1:]:
        n *= d
    return max(n, 1)


def make_state_dict(cfg: SynthConfig, seed: int = 0, fp16_roundtrip: bool = True) -> Dict[str, torch.Tensor]:
    """Random but well-conditioned weights in the reference state_dict layout.

    Weight-normed layers get independent `weight_v` and a `weight_g` that is the row norm of v
    perturbed by ±10 % so the fold `g*v/||v||` is actually exercised.  Gains are chosen so that
    activations stay O(1) through the 72 residual convs, LeakyReLU sees both signs and the
    final tanh is neither saturated nor tiny.
    """
    shapes = state_dict_shapes(cfg)
    sd: Dict[str, torch.Tensor] = {}
    for key in sorted(shapes):
        shape = shapes[key]
        g = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
        if key.endswith("weight_g"):
            continue  # derived from weight_v below
        r = torch.randn(shape, generator=g, dtype=torch.float32)
        if key.endswith(".gamma"):
            t = 1.0 + 0.1 * r
        elif key.endswith(".beta"):
            t = 0.1 * r
        elif key.endswith(".bias"):
            t = 0.05 * r
        elif key == "emb_g.weight":
            t = r
        elif key == "enc_p.emb_pitch.weight":
            t = 0.05 * r
        elif "emb_rel_" in key:
            t = r * (shape[-1] ** -0.5)
        elif key == "dec.m_source.l_linear.weight":
            t = 0.8 + 0.1 * r
        elif key.startswith("dec.ups.") and key.endswith("weight_v"):
            # ConvTranspose1d [C_in, C_out, k]; each output sample sees k/u taps of C_in inputs
            i = int(key.split(".")[2])
            taps = max(shape[2] // cfg.upsample_rates[i], 1)
            t = r * (1.4 / math.sqrt(shape[0] * taps))
        elif key.startswith("dec.noise_convs."):
            t = r * (8.0 / math.sqrt(shape[2]))
        elif key.startswith("dec.resblocks."):
            t = r * (0.9 / math.sqrt(_fan_in(shape)))
        elif key == "dec.conv_post.weight":
            t = r * (0.3 / math.sqrt(_fan_in(shape)))
        elif key.endswith(".post.weight"):
            t = r * (0.5 / math.sqrt(_fan_in(shape)))
        elif key == "enc_p.proj.weight":
            t = r * (0.45 / math.sqrt(_fan_in(shape)))
        else:
            t = r * (1.0 / math.sqrt(_fan_in(shape)))
        sd[key] = t
    for key in sorted(shapes):
        if key.endswith("weight_g"):
            v = sd[key[:-1] + "v"]
            gk = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
            norm = v.reshape(v.shape[0], -1).norm(dim=1).reshape(shapes[key])
            sd[key] = norm * (1.0 + 0.1 * torch.randn(shapes[key], generator=gk))
    if fp16_roundtrip:
        sd = {k: v.half().float() for k, v in sd.items()}
    return sd


def coarse_pitch(f0: np.ndarray, f0_min: float = 50.0, f0_max: float = 1100.0, bins: int = 256) -> np.ndarray:
    """Mel quantiser of /root/reference/pitch_extraction.py:266-267,296-302 (hz_to_mel = 2595 log10(1+f/700),
    lib/audio.py:302-304; the constant cancels in the ratio)."""
    mel = lambda f: 1127.0 * np.log(1.0 + np.asarray(f, dtype=np.float64) / 700.0)
    m_min, m_max = mel(f0_min), mel(f0_max)
    m = mel(f0)
    m = (m - m_min) * (bins - 2) / (m_max - m_min) + 1
    m = np.clip(m, 1, bins - 1)
    return np.rint(m).astype(np.int64)


def make_f0(T: int, frame_rate: float = 100.0, variant: str = "contour", seed: int = 1) -> np.ndarray:
    """Synthetic f0 [T] in Hz: 220·2^(0.5 sin(2π 0.3 t)) with 0.7 s unvoiced gaps every 5 s."""
    t = np.arange(T, dtype=np.float64) / frame_rate
    if variant == "contour":
        f0 = 220.0 * np.power(2.0, 0.5 * np.sin(2 * np.pi * 0.3 * t))
    elif variant == "uniform":
        rng = np.random.default_rng(seed)
        f0 = rng.uniform(100.0, 400.0, size=T)
    elif variant == "unvoiced":
        f0 = np.zeros(T)
    else:
        raise ValueError(variant)
    if variant != "unvoiced":
        gap = (np.mod(t, 5.0) >= 2.0) & (np.mod(t, 5.0) < 2.7)
        f0 = np.where(gap, 0.0, f0)
    return f0.astype(np.float32)


def make_inputs(cfg: SynthConfig, B: int, T: int, seed: int = 1, lengths=None, f0_variant: str = "contour"):
    """(phone[B,T,C_f] f32, lengths[B] i64, pitch[B,T] i64, pitchf[B,T] f32, sid[B] i64) on CPU."""
    g = torch.Generator().manual_seed(seed)
    phone = torch.randn(B, T, cfg.feat_dim, generator=g, dtype=torch.float32)
    f0 = np.stack([np.roll(make_f0(T, variant=f0_variant, seed=seed + b), 37 * b) for b in range(B)])
    pitchf = torch.from_numpy(f0.astype(np.float32))
    pitch = torch.from_numpy(coarse_pitch(f0))
    if lengths is None:
        lengths = [T] * B
    lengths = torch.tensor(list(lengths), dtype=torch.int64)
    sid = torch.zeros(B, dtype=torch.int64)
    return phone, lengths, pitch, pitchf, sid


def draw_noise(cfg: SynthConfig, B: int, T: int, seed: int = 7) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The three RNG draws of one `infer()` in the reference's order and shapes (CPU mt19937).

    Returns (noise_zp[B,192,T], rand_ini[B,1], noise_sine[B,L,1]).  `rand_ini` is zeroed by the
    reference for the fundamental (models.py:378-381) but still advances the stream.
    """
    st = torch.random.get_rng_state()
    try:
        torch.manual_seed(seed)
        nz = torch.randn(B, cfg.inter_channels, T)
        ri = torch.rand(B, 1)
        ns = torch.randn(B, T * cfg.upp, 1)
    finally:
        torch.random.set_rng_state(st)
    return nz, ri, ns


def to_int16(audio: np.ndarray) -> np.ndarray:
    """Peak-normalise and truncate exactly like /root/reference/vc_infer_pipeline.py:188-189."""
    audio = np.asarray(audio)
    audio_max = np.abs(audio).max() / 0.99
    return (audio * 32768 / audio_max).astype(np.int16)


def snr_db(ref: np.ndarray, est: np.ndarray) -> float:
    """SDR formula of /root/reference/lib/karafan/compare.py:21-35: 10 log10(Σref² / Σ(ref−est)²)."""
    ref = np.asarray(ref, dtype=np.float64)
    est = np.asarray(est, dtype=np.float64)
    num = np.sum(ref ** 2)
    den = np.sum((ref - est) ** 2)
    return float(10.0 * np.log10(num / max(den, 1e-300)))


# ---------------------------------------------------------------------------------------------
# Pipeline-level synthetic stand-ins (VC.pipeline / VC.vc, /root/reference/vc_infer_pipeline.py:25-196).
# HuBERT, the f0 estimators and faiss sit upstream of the synthesis path (SURVEY.md §8f) and are not
# available offline; these deterministic doubles have the same call signatures and output shapes.
# ---------------------------------------------------------------------------------------------
def make_song(seconds: float, seed: int = 0, sr: int = 16000) -> np.ndarray:
    """Band-limited noise with a slow amplitude modulation so that quiet points exist (float64, 16 kHz)."""
    n = int(round(seconds * sr))
    rng = np.random.default_rng(seed)
    white = rng.standard_normal(n + 15)
    x = np.convolve(white, np.ones(16) / 16.0, mode="valid")[:n]
    t = np.arange(n, dtype=np.float64) / sr
    am = 0.05 + 0.95 * np.sin(2 * np.pi * 0.37 * t + 0.3 * seed) ** 2
    return 0.4 * x * am


def pipeline_f0(x, **_unused) -> np.ndarray:
    """Synthetic f0 "method" with the reference's estimator signature (pitch_extraction.py:252-268 passes
    x=, f0_up_key=, f0_min=, ... as keywords): one value per 160-sample hop of the padded audio."""
    n = int(np.asarray(x).shape[0]) // 160
    t = np.arange(n, dtype=np.float64) / 100.0
    f0 = 180.0 * np.power(2.0, 0.6 * np.sin(2 * np.pi * 0.45 * t))
    gap = np.mod(t, 1.7) < 0.4
    return np.where(gap, 0.0, f0)


class FakeHubert:
    """Deterministic stand-in for `HubertModelWithFinalProj.extract_features`
    (/root/reference/lib/infer_pack/loaders.py:43-61): 20 ms hop, receptive field 400 samples, so
    `source[1, n]` → `[1, (n - 400)//320 + 1, C_f]`; values are N(0,1) seeded by n."""

    def __init__(self, feat_dim: int, seed: int = 100, device_rng: bool = False):
        # device_rng: draw the features on `source`'s device (throughput measurements: a real front end produces its
        # features there; the CPU generator is what the reference-minted pipeline fixtures were made with)
        self.feat_dim, self.seed, self.device_rng = feat_dim, seed, device_rng

    def extract_features(self, version=None, source=None, padding_mask=None, output_layer=None, **_):
        n = int(source.shape[-1])
        frames = (n - 400) // 320 + 1
        if self.device_rng and source.device.type == "cuda":
            g = torch.Generator(device=source.device).manual_seed(self.seed + n)
            return torch.randn(1, frames, self.feat_dim, generator=g, device=source.device, dtype=torch.float32).to(source.dtype)
        g = torch.Generator().manual_seed(self.seed + n)
        feats = torch.randn(1, frames, self.feat_dim, generator=g, dtype=torch.float32)
        return feats.to(device=source.device, dtype=source.dtype)


class FakeIndex:
    """Brute-force stand-in for a faiss `IndexFlatL2` over `big_npy` (vc_infer_pipeline.py:60-74 only calls
    `.search(npy, k=1)`; squared-L2 scores like faiss)."""

    def __init__(self, feat_dim: int, n: int = 48, seed: int = 5):
        g = torch.Generator().manual_seed(seed)
        self.big_npy = torch.randn(n, feat_dim, generator=g, dtype=torch.float32).numpy()

    def search(self, npy: np.ndarray, k: int = 1):
        a = np.asarray(npy, dtype=np.float64)
        b = self.big_npy.astype(np.float64)
        d = (a * a).sum(1, keepdims=True) - 2.0 * a @ b.T + (b * b).sum(1)[None, :]
        ix = np.argsort(d, axis=1, kind="stable")[:, :k]
        return np.take_along_axis(d, ix, axis=1).astype(np.float32), ix.astype(np.int64)


# ---------------------------------------------------------------------------------------------
# HuBERT / ContentVec front end (SURVEY.md §8f rank 3): seeded weights in the HuggingFace `HubertModel` key layout the
# reference loads (/root/reference/lib/infer_pack/loaders.py:21-32, + `final_proj`), base architecture.
# ---------------------------------------------------------------------------------------------
HUBERT_BASE = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                   conv_dim=(512,) * 7, conv_stride=(5, 2, 2, 2, 2, 2, 2), conv_kernel=(10, 3, 3, 3, 3, 2, 2), conv_bias=False,
                   feat_extract_norm="group", feat_extract_activation="gelu", hidden_act="gelu", num_conv_pos_embeddings=128,
                   num_conv_pos_embedding_groups=16, do_stable_layer_norm=False, layer_norm_eps=1e-5,
                   classifier_proj_size=256, feat_proj_layer_norm=True)


def hubert_state_dict_shapes(h: dict = HUBERT_BASE) -> Dict[str, Tuple[int, ...]]:
    H, I = h["hidden_size"], h["intermediate_size"]
    s: Dict[str, Tuple[int, ...]] = {"masked_spec_embed": (H,)}
    cin = 1
    for i, (c, k) in enumerate(zip(h["conv_dim"], h["conv_kernel"])):
        s[f"feature_extractor.conv_layers.{i}.conv.weight"] = (c, cin, k)
        cin = c
    s["feature_extractor.conv_layers.0.layer_norm.weight"] = (h["conv_dim"][0],)
    s["feature_extractor.conv_layers.0.layer_norm.bias"] = (h["conv_dim"][0],)
    s["feature_projection.layer_norm.weight"] = (cin,)
    s["feature_projection.layer_norm.bias"] = (cin,)
    s["feature_projection.projection.weight"] = (H, cin)
    s["feature_projection.projection.bias"] = (H,)
    kp, g = h["num_conv_pos_embeddings"], h["num_conv_pos_embedding_groups"]
    s["encoder.pos_conv_embed.conv.bias"] = (H,)
    s["encoder.pos_conv_embed.conv.parametrizations.weight.original0"] = (1, 1, kp)
    s["encoder.pos_conv_embed.conv.parametrizations.weight.original1"] = (H, H // g, kp)
    s["encoder.layer_norm.weight"] = (H,)
    s["encoder.layer_norm.bias"] = (H,)
    for l in range(h["num_hidden_layers"]):
        p = f"encoder.layers.{l}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            s[p + f"attention.{n}.weight"] = (H, H)
            s[p + f"attention.{n}.bias"] = (H,)
        for n in ("layer_norm", "final_layer_norm"):
            s[p + n + ".weight"] = (H,)
            s[p + n + ".bias"] = (H,)
        s[p + "feed_forward.intermediate_dense.weight"] = (I, H)
        s[p + "feed_forward.intermediate_dense.bias"] = (I,)
        s[p + "feed_forward.output_dense.weight"] = (H, I)
        s[p + "feed_forward.output_dense.bias"] = (H,)
    s["final_proj.weight"] = (h["classifier_proj_size"], H)
    s["final_proj.bias"] = (h["classifier_proj_size"],)
    return s


def make_hubert_state_dict(seed: int = 0, h: dict = HUBERT_BASE, fp16_roundtrip: bool = True) -> Dict[str, torch.Tensor]:
    """Seeded, well-conditioned weights (fan-in scaled; LayerNorm / GroupNorm gains near 1) stored through fp16 like the
    shipped `content-vec-best.safetensors`."""
    sd: Dict[str, torch.Tensor] = {}
    for key, shape in sorted(hubert_state_dict_shapes(h).items()):
        g = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
        r = torch.randn(shape, generator=g, dtype=torch.float32)
        if key.endswith("layer_norm.weight") or key.endswith("original0"):
            t = 1.0 + 0.1 * r
        elif key.endswith(".bias"):
            t = 0.05 * r
        elif key == "masked_spec_embed":
            t = r
        elif key.endswith("original1"):
            t = r * (1.0 / math.sqrt(shape[1] * shape[2]))
        elif "feature_extractor" in key:
            t = r * (1.6 / math.sqrt(_fan_in(shape)))          # GELU roughly halves the variance
        else:
            t = r * (1.0 / math.sqrt(_fan_in(shape)))
        sd[key] = t
    if fp16_roundtrip:
        sd = {k: v.half().float() for k, v in sd.items()}
    return sd


def make_speech(seconds: float, seed: int = 0, sr: int = 16000) -> torch.Tensor:
    """Synthetic 16 kHz 'speech' [1, n] for the front end: harmonic tone with vibrato + noise bursts, peak ~0.5."""
    n = int(round(seconds * sr))
    t = torch.arange(n, dtype=torch.float64) / sr
    g = torch.Generator().manual_seed(seed + 77)
    f0 = 140.0 + 40.0 * torch.sin(2 * math.pi * 0.7 * t + seed)
    ph = 2 * math.pi * torch.cumsum(f0, 0) / sr
    x = sum(torch.sin(k * ph) / k for k in range(1, 6)) * 0.2
    env = 0.55 + 0.45 * torch.sin(2 * math.pi * 1.3 * t)
    x = x * env + 0.05 * torch.randn(n, generator=g, dtype=torch.float64) * (torch.sin(2 * math.pi * 0.4 * t) > 0.3)
    return x.float()[None, :]


# ---- RMVPE (SURVEY §8f rank 4) --------------------------------------------------------------------------------------------
def rmvpe_state_dict_shapes(n_blocks: int = 4, en_de_layers: int = 5, inter_layers: int = 4, en_out: int = 16,
                            n_mels: int = 128, hidden: int = 256, n_class: int = 360) -> Dict[str, Tuple[int, ...]]:
    """Key -> shape of `E2E(4, 1, (2, 2))` (/root/reference/lib/rmvpe.py:431-472, built at :578), in module order."""
    s: Dict[str, Tuple[int, ...]] = {}

    def bn(p, c):
        s[p + "weight"], s[p + "bias"], s[p + "running_mean"], s[p + "running_var"] = (c,), (c,), (c,), (c,)
        s[p + "num_batches_tracked"] = ()

    def block(p, cin, cout):                                  # ConvBlockRes, rmvpe.py:232-267
        s[p + "conv.0.weight"] = (cout, cin, 3, 3)
        bn(p + "conv.1.", cout)
        s[p + "conv.3.weight"] = (cout, cout, 3, 3)
        bn(p + "conv.4.", cout)
        if cin != cout:
            s[p + "shortcut.weight"], s[p + "shortcut.bias"] = (cout, cin, 1, 1), (cout,)

    bn("unet.encoder.bn.", 1)
    cin, cout = 1, en_out
    for i in range(en_de_layers):
        for j in range(n_blocks):
            block(f"unet.encoder.layers.{i}.conv.{j}.", cin if j == 0 else cout, cout)
        cin, cout = cout, cout * 2
    for i in range(inter_layers):
        for j in range(n_blocks):
            block(f"unet.intermediate.layers.{i}.conv.{j}.", cin if (i == 0 and j == 0) else cout, cout)
    cin = cout
    for i in range(en_de_layers):
        cout = cin // 2
        p = f"unet.decoder.layers.{i}."
        s[p + "conv1.0.weight"] = (cin, cout, 3, 3)           # ConvTranspose2d: [C_in][C_out][3][3]
        bn(p + "conv1.1.", cout)
        for j in range(n_blocks):
            block(p + f"conv2.{j}.", cout * 2 if j == 0 else cout, cout)
        cin = cout
    s["cnn.weight"], s["cnn.bias"] = (3, en_out, 3, 3), (3,)
    for sfx in ("", "_reverse"):
        s["fc.0.gru.weight_ih_l0" + sfx] = (3 * hidden, 3 * n_mels)
        s["fc.0.gru.weight_hh_l0" + sfx] = (3 * hidden, hidden)
        s["fc.0.gru.bias_ih_l0" + sfx] = (3 * hidden,)
        s["fc.0.gru.bias_hh_l0" + sfx] = (3 * hidden,)
    s["fc.1.weight"], s["fc.1.bias"] = (n_class, 2 * hidden), (n_class,)
    return s


def make_rmvpe_state_dict(seed: int = 0, **arch) -> Dict[str, torch.Tensor]:
    """Seeded RMVPE weights in the reference's state_dict layout (the real `rmvpe.pt` is 181 MB and not available offline).
    He-scaled convolutions, non-trivial BatchNorm statistics, and small BatchNorm gains so that the 56 residual blocks keep the
    activations O(1)-O(10); the final Linear is scaled up so the salience is not flat."""
    g = torch.Generator().manual_seed(1000 + seed)
    rn = lambda *shape: torch.randn(*shape, generator=g)
    ru = lambda *shape: torch.rand(*shape, generator=g)
    sd: Dict[str, torch.Tensor] = {}
    for k, shape in rmvpe_state_dict_shapes(**arch).items():
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(100, dtype=torch.long)
        elif k.endswith("running_mean"):
            sd[k] = 0.1 * rn(*shape)
        elif k.endswith("running_var"):
            sd[k] = 0.5 + ru(*shape)
        elif k.rsplit(".", 1)[0].endswith(("conv.1", "conv.4", "conv1.1")) or k.startswith("unet.encoder.bn."):
            first_bn = k.startswith("unet.encoder.bn.")
            if k.endswith("weight"):
                sd[k] = (0.25 + 0.3 * ru(*shape)) if not first_bn else torch.full(shape, 0.35)
            else:
                sd[k] = 0.1 * rn(*shape) if not first_bn else torch.full(shape, 1.2)
        elif "gru" in k:
            sd[k] = (ru(*shape) * 2 - 1) / 16.0
        elif k == "fc.1.weight":
            sd[k] = rn(*shape) * 0.15
        elif k == "fc.1.bias":
            sd[k] = -2.0 + 0.1 * rn(*shape)
        elif k == "cnn.weight":
            sd[k] = rn(*shape) * 0.25 * math.sqrt(2.0 / _fan_in(shape))
        elif k.endswith("bias"):
            sd[k] = 0.1 * rn(*shape)
        elif k.endswith("conv1.0.weight"):                                 # transposed conv: fan-in = C_in * 9 / 4 on average
            sd[k] = rn(*shape) * math.sqrt(2.0 / (shape[0] * 9 / 4))
        else:
            sd[k] = rn(*shape) * math.sqrt(2.0 / _fan_in(shape))
    return sd


# ---- CREPE (torchcrepe's `full` / `tiny`) ------------------------------------------------------------------------------------
def crepe_state_dict_shapes(model: str = "full") -> Dict[str, Tuple[int, ...]]:
    """Key -> shape of torchcrepe's `Crepe(model)` state dict, in module order."""
    cin, cout, nf = {"full": ([1, 1024, 128, 128, 128, 256], [1024, 128, 128, 128, 256, 512], 2048),
                     "tiny": ([1, 128, 16, 16, 16, 32], [128, 16, 16, 16, 32, 64], 256)}[model]
    s: Dict[str, Tuple[int, ...]] = {}
    for i in range(6):
        s[f"conv{i + 1}.weight"] = (cout[i], cin[i], 512 if i == 0 else 64, 1)
        s[f"conv{i + 1}.bias"] = (cout[i],)
        for k in ("weight", "bias", "running_mean", "running_var"):
            s[f"conv{i + 1}_BN.{k}"] = (cout[i],)
        s[f"conv{i + 1}_BN.num_batches_tracked"] = ()
    s["classifier.weight"], s["classifier.bias"] = (360, nf), (360,)
    return s


def make_crepe_state_dict(seed: int = 0, model: str = "full") -> Dict[str, torch.Tensor]:
    """Seeded CREPE weights in torchcrepe's layout (the real `full.pth` is not available offline).  He-scaled convolutions,
    BatchNorm statistics near what a ReLU output of that scale has (so every layer's output stays O(1)), BatchNorm gains of
    both signs on a few channels (exercising the sign of the scale), and a classifier scaled so that the logits spread over
    several units: the median gap between the two largest in-range logits is far above the fp16 path's error."""
    g = torch.Generator().manual_seed(2000 + seed)
    rn = lambda *shape: torch.randn(*shape, generator=g)
    ru = lambda *shape: torch.rand(*shape, generator=g)
    sd: Dict[str, torch.Tensor] = {}
    for k, shape in crepe_state_dict_shapes(model).items():
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(0, dtype=torch.long)
        elif k.endswith("running_mean"):
            sd[k] = 0.4 + 0.1 * rn(*shape)
        elif k.endswith("running_var"):
            sd[k] = 0.3 + 0.2 * ru(*shape)
        elif "_BN.weight" in k:
            w = 0.8 + 0.4 * ru(*shape)
            sd[k] = torch.where(ru(*shape) < 0.05, -w, w)
        elif "_BN.bias" in k:
            sd[k] = 0.1 * rn(*shape)
        elif k == "classifier.weight":
            sd[k] = rn(*shape) * 1.5 / math.sqrt(shape[1])
        elif k == "classifier.bias":
            sd[k] = -1.0 + 0.5 * rn(*shape)
        elif k.endswith("bias"):
            sd[k] = 0.05 * rn(*shape)
        else:
            sd[k] = rn(*shape) * math.sqrt(2.0 / _fan_in(shape))
    return sd
