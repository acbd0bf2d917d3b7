"""GPU: the CREPE f0 estimator on the B200 kernels (comfy_rvc_b200/crepe.py) against the torch-CPU oracle (oracle/crepe_oracle.py),
seeded weights (synthetic.make_crepe_state_dict), `full` and `tiny`.

Tolerances (the contractions run on fp16 operands with fp32 accumulation, the decoders in float64):
  * network: logit SNR >= 40 dB and sigmoid max |err| <= 0.02 against the fp32 oracle;
  * decoders on the SAME salience: argmax / weighted_argmax bins identical and f0 within 1e-12 relative; Viterbi bins identical
    on >= 99.9 % of the frames and the path's log-probability equal to the oracle's optimum to 1e-12 relative (so any
    difference is a tie between equally likely paths);
  * end to end with the dither seeded: >= 97 % of the frames within 5 cents, periodicity max |err| <= 0.02.
"""
import numpy as np
import pytest
import torch

from comfy_rvc_b200 import crepe, synthetic
from oracle import crepe_oracle as O

pytestmark = pytest.mark.gpu

_MODELS = {}


def model_for(name, seed=0):
    key = (name, seed)
    if key not in _MODELS:
        _MODELS[key] = (crepe.Crepe(name, weights=synthetic.make_crepe_state_dict(seed, name), device="cuda:0"),
                        synthetic.make_crepe_state_dict(seed, name))
    return _MODELS[key]


def snr_db(ref, est):
    ref, est = np.asarray(ref, np.float64), np.asarray(est, np.float64)
    return 10 * np.log10(np.sum(ref ** 2) / max(np.sum((ref - est) ** 2), 1e-300))


def cents_err(a, b):
    return np.abs(1200 * np.log2(np.asarray(a, np.float64) / np.asarray(b, np.float64)))


@pytest.mark.parametrize("name", ["full", "tiny"])
@pytest.mark.parametrize("seconds", [3.0, 12.37])         # 301 frames; 1238 frames = one full pass + a partial one
def test_network_vs_oracle(name, seconds):
    m, sd = model_for(name)
    audio = synthetic.make_speech(seconds, seed=3)
    frames = next(O.preprocess(audio, 16000, 160, None, True))
    ref = O.crepe_forward(frames, sd, embed="logits").numpy()
    x = audio[0].cuda()
    got = m.forward_logits(x, 160, True, 0, frames.shape[0]).cpu().numpy()
    assert got.shape == ref.shape
    assert snr_db(ref, got) >= 40.0
    assert np.abs(1 / (1 + np.exp(-ref)) - 1 / (1 + np.exp(-got))).max() <= 0.02


def _salience(name, seconds=4.0, seed=5):
    m, sd = model_for(name)
    audio = synthetic.make_speech(seconds, seed=seed)
    frames = next(O.preprocess(audio, 16000, 160, None, True))
    return torch.sigmoid(O.crepe_forward(frames, sd, embed="logits"))           # [T, 360] fp32, the oracle's salience


@pytest.mark.parametrize("mode", [0, 1])
def test_argmax_decoders_same_salience(mode):
    s = _salience("tiny")
    lo, hi = O.mask_range(50.0, 1100.0)
    T = s.shape[0]
    np.random.seed(11)
    if hasattr(O.weighted_argmax, "weights"):
        del O.weighted_argmax.weights
    crepe._WCENTS = None
    probs = s.t()[None].clone()
    probs[:, :lo], probs[:, hi:] = -float("inf"), -float("inf")
    st = np.random.get_state()
    bins_ref, f0_ref = (O.argmax if mode == 0 else O.weighted_argmax)(probs)
    np.random.set_state(st)
    dither = crepe._dither_noise((1, T)).reshape(-1) if mode == 0 else None
    r = crepe.decode_device(s.cuda(), True, mode, lo, hi, T, dither)
    assert np.array_equal(r["bins"].cpu().numpy(), bins_ref[0].numpy())
    np.testing.assert_allclose(r["f0"].cpu().numpy(), f0_ref[0].double().numpy(), rtol=1e-12, atol=0)
    per_ref = s[torch.arange(T), bins_ref[0]].numpy()
    assert np.array_equal(r["periodicity"].cpu().numpy(), per_ref)


@pytest.mark.parametrize("chunk", [None, 37])
def test_viterbi_same_salience(chunk):
    s = _salience("tiny", seconds=6.0)
    lo, hi = O.mask_range(50.0, 1100.0)
    T = s.shape[0]
    ch = T if chunk is None else chunk
    probs = s.t()[None].clone()
    probs[:, :lo], probs[:, hi:] = -float("inf"), -float("inf")
    trans = O.viterbi_transition()
    ref_bins, ref_scores = [], []
    for c0 in range(0, T, ch):
        st, sc = O.librosa_viterbi(O.softmax64(probs[:, :, c0:c0 + ch])[0], trans)
        ref_bins.append(st)
        ref_scores.append(sc)
    ref_bins = np.concatenate(ref_bins)
    dither = np.zeros(T)
    r = crepe.decode_device(s.cuda(), True, 2, lo, hi, ch, dither)
    got = r["bins"].cpu().numpy()
    assert np.mean(got == ref_bins) >= 0.999
    np.testing.assert_allclose(r["score"].cpu().numpy(), np.array(ref_scores), rtol=1e-12, atol=0)
    f0_ref = 10 * 2 ** ((20.0 * got + O.CENTS_OFFSET) / 1200)
    np.testing.assert_allclose(r["f0"].cpu().numpy(), f0_ref, rtol=1e-12, atol=0)
    np.testing.assert_array_equal(r["periodicity"].cpu().numpy(), s[torch.arange(T), torch.as_tensor(got).long()].numpy())


@pytest.mark.parametrize("name", ["full", "tiny"])
@pytest.mark.parametrize("decoder", ["viterbi", "weighted_argmax", "argmax"])
@pytest.mark.parametrize("batch_size", [None, 320])
def test_predict_end_to_end(name, decoder, batch_size):
    m, sd = model_for(name)
    crepe.load_weights(name, sd)
    audio = synthetic.make_speech(5.0, seed=7)
    if hasattr(O.weighted_argmax, "weights"):
        del O.weighted_argmax.weights
    crepe._WCENTS = None
    np.random.seed(123)
    p_ref, per_ref = O.predict(audio, 16000, sd, 160, 50.0, 1100.0, getattr(O, decoder), True, batch_size, True)
    np.random.seed(123)
    p, per = crepe.predict(audio, 16000, 160, 50.0, 1100.0, name, getattr(crepe.decode, decoder), return_periodicity=True,
                           batch_size=batch_size, device="cuda:0")
    assert p.device == audio.device and p.dtype == torch.float32 and p.shape == p_ref.shape
    assert np.mean(cents_err(p_ref[0].numpy(), p[0].numpy()) <= 5.0) >= 0.97
    assert np.abs(per_ref[0].numpy() - per[0].numpy()).max() <= 0.02


def test_predict_pad_false_and_hop():
    m, sd = model_for("tiny")
    crepe.load_weights("tiny", sd)
    audio = synthetic.make_speech(2.0, seed=9)[:, :31111]
    np.random.seed(5)
    p_ref = O.predict(audio, 16000, sd, 97, 50.0, 2006.0, O.argmax, False, 64, False)
    np.random.seed(5)
    p = crepe.predict(audio, 16000, 97, 50.0, 2006.0, "tiny", crepe.decode.argmax, batch_size=64, device="cuda:0", pad=False)
    assert p.shape == p_ref.shape == (1, 1 + (31111 - 1024) // 97)
    assert np.mean(cents_err(p_ref[0].numpy(), p[0].numpy()) <= 5.0) >= 0.97


def test_ten_minute_song_bounded_scratch():
    m, sd = model_for("full")
    audio = synthetic.make_song(600.0, seed=2)
    audio = torch.as_tensor(audio, dtype=torch.float32)[None]
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    p = crepe.predict(audio, 16000, 160, 50.0, 1100.0, "full", crepe.decode.viterbi, batch_size=320, device="cuda:0",
                      crepe_model=m)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    T = 1 + audio.shape[1] // 160
    assert p.shape == (1, T) and torch.isfinite(p).all()
    assert peak <= 2 * 1024 ** 3, peak


def _recipe_f0(x, f0_min, f0_max, hop, pitch_fn):
    """The RVC-lineage crepe recipe `FeatureExtractor.get_crepe` implements, around any `predict`-like pitch_fn."""
    x = x.astype(np.float32)
    x /= np.quantile(np.abs(x), 0.999)
    source = np.array(pitch_fn(torch.from_numpy(x)[None]).squeeze(0).cpu().float().numpy())
    source[source < 0.001] = np.nan
    p_len = x.shape[0] // 160
    target = np.interp(np.arange(0, len(source) * p_len, len(source)) / p_len, np.arange(0, len(source)), source)
    return np.nan_to_num(target)


def test_pipeline_crepe_method():
    from comfy_rvc_b200 import pipeline as pl
    from comfy_rvc_b200.config import NAMED_CONFIGS
    from tests.test_parity_gpu import build_net
    cfg = NAMED_CONFIGS["40k"]
    net = build_net(cfg, synthetic.make_state_dict(cfg, seed=2), "fp16")
    hub = synthetic.FakeHubert(cfg.feat_dim)
    m, sd = model_for("full")
    audio = synthetic.make_speech(50.0, seed=8)[0].double().numpy()
    seen = {}

    def device_f0(x, f0_min=50, f0_max=1100, crepe_hop_length=160, **_):
        seen["x"] = np.array(x)
        return _recipe_f0(x, f0_min, f0_max, crepe_hop_length,
                          lambda a: crepe.predict(a, 16000, crepe_hop_length, f0_min, f0_max, "full", batch_size=2 * crepe_hop_length,
                                                  device="cuda:0", crepe_model=m))

    outs = []
    for method in ("crepe", "device_crepe"):
        vc = pl.VC(cfg.sr, pl.PipelineConfig(1, 5, 30, 32, is_half=False, device="cuda:0"))
        vc.model_crepe = m
        vc.f0_method_dict["device_crepe"] = device_f0
        np.random.seed(99)
        torch.manual_seed(3)
        outs.append(vc.pipeline(hub, net, 0, audio.copy(), [0, 0, 0], 0, method, "median", "", 0.0, 1, 3, cfg.sr, 0, 1.0, "v1",
                                0.33, 160, False, False, None, 50, 1100))
        assert len(vc.last_plan["segments"]) == 2
    assert outs[0].dtype == np.int16 and np.array_equal(outs[0], outs[1])
    # the recipe's f0 against the oracle's (network on cuDNN in fp32, TF32 off), same dither draws
    torch.backends.cudnn.allow_tf32 = False
    sd_dev = {k: v.cuda() for k, v in sd.items()}

    def oracle_pitch(a):
        ps = []
        for frames in O.preprocess(a, 16000, 160, 320, True):
            probs = O.crepe_forward(frames.cuda(), sd_dev).cpu().reshape(1, -1, 360).transpose(1, 2)
            ps.append(O.postprocess(probs, 50.0, 1100.0, O.viterbi))
        return torch.cat(ps, 1)

    np.random.seed(99)
    f_dev = device_f0(seen["x"])
    np.random.seed(99)
    f_ref = _recipe_f0(seen["x"], 50, 1100, 160, oracle_pitch)
    both = (f_dev > 0) & (f_ref > 0)
    assert np.mean(both) >= 0.9
    assert np.mean(cents_err(f_ref[both], f_dev[both]) <= 5.0) >= 0.97
