"""CPU: the CREPE oracle (oracle/crepe_oracle.py) against torchcrepe's layer list, the framing of `preprocess`, the float64
Viterbi against brute-force path enumeration, and the device layouts / weight packing of comfy_rvc_b200/crepe.py emulated in
float64 (tests/_emulate_crepe.py)."""
import itertools

import numpy as np
import pytest
import torch

from comfy_rvc_b200 import crepe, synthetic
from oracle import crepe_oracle as O
from tests import _emulate_crepe as E


@pytest.mark.parametrize("model", ["full", "tiny"])
def test_oracle_equals_module(model):
    sd = synthetic.make_crepe_state_dict(1, model)
    m = O.crepe_module(model)
    m.load_state_dict(sd)                       # strict: the state-dict contract, num_batches_tracked included
    m.eval()
    frames = next(O.preprocess(synthetic.make_speech(0.1, seed=2), 16000, 160, None, True))
    with torch.no_grad():
        np.testing.assert_array_equal(O.crepe_forward(frames, sd).numpy(), m(frames).numpy())
    assert set(sd) == set(m.state_dict())


@pytest.mark.parametrize("pad", [True, False])
@pytest.mark.parametrize("n", [16000, 16000 + 77, 2048 + 159])
@pytest.mark.parametrize("batch_size", [None, 1, 512])
def test_preprocess_frames_and_chunks(pad, n, batch_size):
    audio = synthetic.make_speech(n / 16000 + 0.01, seed=4)[:, :n]
    hop = 160
    total = 1 + n // hop if pad else 1 + (n - 1024) // hop
    assert crepe.frame_count(n, hop, pad) == total
    got = list(O.preprocess(audio, 16000, hop, batch_size, pad))
    bounds = crepe.chunks(total, batch_size)
    assert [g.shape[0] for g in got] == [e - s for s, e in bounds]
    assert sum(g.shape[0] for g in got) == total
    ours = list(crepe.preprocess(audio, 16000, hop, batch_size, "cpu", pad))
    for a, b in zip(got, ours):
        np.testing.assert_allclose(a.numpy(), b.numpy(), rtol=0, atol=1e-5)
    # frame f is samples [f hop, f hop + 1024) of the (padded) audio, normalised
    x = torch.nn.functional.pad(audio, (512, 512)) if pad else audio
    f = total - 1
    raw = x[0, f * hop: f * hop + 1024]
    ref = (raw - raw.mean()) / torch.clamp(raw.std(), min=1e-10)
    np.testing.assert_allclose(torch.cat(got)[f].numpy(), ref.numpy(), rtol=0, atol=1e-5)


def _brute_force(prob, trans):
    eps = np.finfo(np.float32).tiny
    lp, lt = np.log(prob + eps), np.log(trans + eps)
    li = np.log(np.full(prob.shape[0], 1.0 / prob.shape[0]) + eps)
    best, arg = -np.inf, None
    for path in itertools.product(range(prob.shape[0]), repeat=prob.shape[1]):      # lexicographic: first = lowest
        v = li[path[0]] + lp[path[0], 0]
        for t in range(1, len(path)):
            v = v + lt[path[t - 1], path[t]] + lp[path[t], t]
        if v > best:
            best, arg = v, path
    return np.array(arg), best


@pytest.mark.parametrize("seed", range(6))
def test_viterbi_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    S, T = 4, 5
    prob = rng.random((S, T))
    if seed % 2:
        prob = np.round(prob * 2) / 2 + 0.1          # many exact ties
    prob /= prob.sum(axis=0, keepdims=True)
    trans = np.maximum(3 - np.abs(np.subtract.outer(np.arange(S), np.arange(S))), 0).astype(np.float64)
    if seed % 3 == 0:
        trans = np.ones((S, S))                       # every path ties on transitions
    trans /= trans.sum(axis=1, keepdims=True)
    states, score = O.librosa_viterbi(prob, trans)
    ref_states, ref_score = _brute_force(prob, trans)
    assert np.isclose(score, ref_score, rtol=1e-12, atol=0)
    # on exact ties the two may pick different optimal paths; the path found must itself score the optimum
    eps = np.finfo(np.float32).tiny
    lp, lt = np.log(prob + eps), np.log(trans + eps)
    v = np.log(np.float64(1.0 / S) + eps) + lp[states[0], 0] + sum(lt[states[t - 1], states[t]] + lp[states[t], t] for t in range(1, T))
    assert np.isclose(v, ref_score, rtol=1e-12, atol=0)
    if seed % 2 == 0 and seed % 3:
        np.testing.assert_array_equal(states, ref_states)


def test_viterbi_band_tables():
    band, log_out, log_init = crepe.viterbi_tables()
    trans = O.viterbi_transition()
    lt = np.log(trans + np.finfo(np.float32).tiny)
    for k in (0, 5, 180, 359):
        for d in range(-11, 12):
            if 0 <= k + d < 360:
                assert band[k, d + 11] == lt[k, k + d]
    assert (lt[np.abs(np.subtract.outer(np.arange(360), np.arange(360))) > 11] == log_out).all()
    # an in-band step always beats any out-of-band one (the kernel's shortcut for out-of-band predecessors)
    assert band[band != 0].min() > log_out


@pytest.mark.parametrize("model", ["full", "tiny"])
def test_host_packing_reproduces_oracle(model):
    sd = synthetic.make_crepe_state_dict(0, model)
    frames = next(O.preprocess(synthetic.make_speech(0.05, seed=6), 16000, 160, None, True))[:3]
    ref = O.crepe_forward(frames.double(), {k: v.double() for k, v in sd.items()}, embed="logits")
    assert (sd["conv2_BN.weight"] < 0).any()             # channels with a negative BatchNorm scale take the same path
    got = E.network(frames.double(), crepe.host_weights(sd, model), model)
    # the host images are fp32 (the fold itself is float64): ~1e-7 relative
    assert (got - ref).abs().max() <= 1e-5 * ref.abs().max()


def test_postprocess_mask_and_convert():
    lo, hi = O.mask_range(50.0, 2006.0)
    assert (lo, hi) == crepe._mask_range(50.0, 2006.0)
    f = torch.tensor([55.0, 440.0, 1000.0])
    np.testing.assert_array_equal(crepe.convert.frequency_to_bins(f).numpy(), O.frequency_to_bins(f).numpy())
    np.testing.assert_allclose(crepe.convert.cents_to_frequency(crepe.convert.frequency_to_cents(f)).numpy(), f.numpy(), rtol=1e-6)
    np.random.seed(0)
    a = crepe.convert.bins_to_cents(torch.arange(5))
    np.random.seed(0)
    b = O.bins_to_cents(torch.arange(5))
    np.testing.assert_array_equal(a.numpy(), b.numpy())


def test_filters_nan_aware():
    x = torch.tensor([[1.0, float("nan"), 3.0, 4.0, float("nan"), float("nan"), float("nan"), 8.0, 9.0]])
    m = crepe.filter.median(x, 3)
    assert m.shape == x.shape
    assert m[0, 0] == 1.0 and m[0, 2] == 3.0 and torch.isnan(m[0, 5])
    a = crepe.filter.mean(x, 3)
    assert a[0, 1] == 2.0 and torch.isnan(a[0, 5])


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(RuntimeError):
        crepe.predict(torch.zeros(1, 4000), 16000, model="tiny", device="cpu",
                      crepe_model=crepe.Crepe("tiny", weights=synthetic.make_crepe_state_dict(0, "tiny")))


def test_rejects_other_sample_rates():
    with pytest.raises(ValueError):
        crepe.predict(torch.zeros(1, 4000), 44100)


def test_pipeline_registers_crepe():
    from comfy_rvc_b200.pipeline import FeatureExtractor, PipelineConfig
    fe = FeatureExtractor(40000, PipelineConfig())
    assert fe.f0_method_dict["crepe"] == fe.get_crepe
    with pytest.raises(Exception, match="Method pm not found"):
        fe._f0_fn("pm")
