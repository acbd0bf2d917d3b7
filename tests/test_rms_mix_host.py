"""CPU: the volume-envelope mix of `VC.pipeline` (`rms_mix_rate < 1`, change_rms of lib/model_utils.py:39, called at
vc_infer_pipeline.py:183) -- the interpolation formula the device kernel follows, the librosa restatement, and the driver's
host logic (half-block ranges, table, exchange, fold order) with numpy compute hooks, single-process and over world_size-2
gloo."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from comfy_rvc_b200 import pipeline as pl
from comfy_rvc_b200 import synthetic
from oracle import pipeline_oracle, rvc_oracle
from tests import _rms_oracle
from tests._host_vc import HostVC, OracleNet
from tests._util import load_pipeline_golden


def interp_linear(env: np.ndarray, N: int, d: np.ndarray) -> np.ndarray:
    """float32 emulation of csrc/pipeline_kernels.cu `interp_linear` (torch's CPU F.interpolate, mode="linear",
    align_corners=False): t = float32(d) + 0.5f, src = fma(t, scale, -0.5f), y = fma(x0, 1 - lam, x1 * lam).  Each fused
    operation is evaluated exactly in float64 (float32 * float32 fits in 53 bits) and rounded once to float32."""
    env = np.asarray(env, np.float32).reshape(-1)
    n_in = env.shape[0]
    scale = np.float32(n_in) / np.float32(N)
    t = d.astype(np.float32) + np.float32(0.5)
    src = np.maximum((t.astype(np.float64) * np.float64(scale) - 0.5).astype(np.float32), np.float32(0))
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = np.minimum(i0 + 1, n_in - 1)
    lam = np.clip(src - i0.astype(np.float32), np.float32(0), np.float32(1))
    r = env[i1] * lam
    return (env[i0].astype(np.float64) * (np.float32(1) - lam).astype(np.float64) + r.astype(np.float64)).astype(np.float32)


@pytest.mark.parametrize("n_in,N", [(1, 7), (2, 7), (21, 1000), (21, 160_000), (1201, 9_600_000), (1201, 28_800_000),
                                    (3601, 16_777_217), (3601, 86_400_000)])
def test_interpolation_formula_is_torch_bit_for_bit(n_in, N):
    """The index rounding the gain kernel copies: with N > 2^24, float32(d) + 0.5 already rounds, and a "more accurate" index
    is up to 9 % off at N = 86.4 M.  A change of torch's CPU kernel shows up here first."""
    x = np.random.default_rng(n_in + N).random(n_in).astype(np.float32)
    want = F.interpolate(torch.from_numpy(x)[None, None], size=N, mode="linear").reshape(-1).numpy()
    step = 1 << 23
    for lo in range(0, N, step):
        d = np.arange(lo, min(N, lo + step), dtype=np.int64)
        got = interp_linear(x, N, d)
        assert np.array_equal(got, want[lo: lo + d.shape[0]]), (n_in, N, lo)


@pytest.mark.parametrize("sr,n,dtype", [(16000, 16000 * 7 + 123, np.float64), (16000, 8000, np.float64), (40000, 20000 * 5, np.float32),
                                        (48000, 48000 * 3 + 1, np.float32), (32000, 17, np.float32), (22050, 22050 * 2 + 5, np.float32)])
def test_librosa_rms_restatement(sr, n, dtype):
    """`librosa_rms` against an independent float64 direct sum over zero-padded frames of float32-rounded squares; frame count
    1 + len // hop; change_rms with rate 1 is the identity."""
    rng = np.random.default_rng(n)
    y = (rng.standard_normal(n) * 0.3).astype(dtype)
    y[: n // 5] = 0.0                                                           # silent frames too
    hop, fl = sr // 2, sr // 2 * 2
    r = _rms_oracle.librosa_rms(y, fl, hop)
    assert r.dtype == np.float32 and r.shape == (1, 1 + n // hop)
    sq = np.pad(np.square(y.astype(np.float32)).astype(np.float64), (hop, hop))
    want = np.array([np.sqrt(sq[f * hop: f * hop + fl].sum() / fl) for f in range(1 + n // hop)])
    np.testing.assert_allclose(r[0], want, rtol=2e-7, atol=0)
    out = (rng.standard_normal(n * 2) * 0.1).astype(np.float32)
    assert np.array_equal(_rms_oracle.change_rms(y.astype(np.float64), 16000, out.copy(), 32000, 1.0), out)


class NumpyMixHooks:
    """The three compute hooks of the mix (`_mix_power`, `_mix_fold`, `_mix_gain`) in numpy, with the kernels' definitions."""

    def _require_device_mix(self):
        pass

    def _stage(self, audio_pad, pitch, pitchf, sid, net_g, staged_audio=None):
        staged = super()._stage(audio_pad, pitch, pitchf, sid, net_g, staged_audio)
        staged["audio64"] = audio_pad
        return staged

    def _mix_power(self, staged, x, offset, hop, out):
        x = np.asarray(x)
        sq = np.square(x.astype(np.float32)).astype(np.float64)
        first = offset // hop
        cuts = np.arange(first + 1, (offset + len(x) - 1) // hop + 1) * hop - offset
        sums = np.add.reduceat(sq, np.concatenate([[0], cuts]).astype(np.int64))
        assert out.shape[0] == sums.shape[0]
        self.power_calls.append((offset, len(x), hop, out.shape[0]))
        out.copy_(torch.from_numpy(sums))

    def _mix_fold(self, staged, table, frame_length):
        t = table.numpy()
        hb = np.zeros(t.shape[1])
        for row in t:                                                           # segment order
            hb = hb + row
        fr = hb.copy()
        fr[1:] += hb[:-1]
        rms = np.sqrt((fr / frame_length).astype(np.float32))
        self.folded.append(rms)
        return rms

    def _mix_gain(self, staged, x, offset, n_total, rms1, rms2, rate):
        d = np.arange(offset, offset + len(x), dtype=np.int64)
        e1 = interp_linear(rms1, n_total, d)
        e2 = np.maximum(interp_linear(rms2, n_total, d), np.float32(1e-6))
        gain = np.power(e1, np.float32(1 - rate)) * np.power(e2, np.float32(rate - 1))
        x *= gain.astype(np.float32)


class MixHostVC(NumpyMixHooks, HostVC):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.power_calls, self.folded = [], []


def test_host_logic_ranges_table_and_fold():
    """A 48 kHz song cut into pieces with frames straddling two and three segments (a 5000-sample segment inside one
    48000-sample frame) and a last segment shorter than one frame: every piece writes exactly the half-blocks it touches,
    the folded envelope is librosa's RMS of the concatenation, and the mixed pieces are change_rms of the concatenation."""
    vc = MixHostVC(48000, pl.PipelineConfig(1, 1, 2, 3, is_half=False, device="cpu"))
    rng = np.random.default_rng(4)
    sizes = [30000, 5000, 71000, 24000, 3000]
    n_in = 16000 * 3 + 777
    hp = rng.standard_normal(n_in) * 0.2
    hp[: 9000] = 0.0                                                             # a silent input frame (gain 0)
    song = (rng.standard_normal(sum(sizes)) * 0.3).astype(np.float32)
    song[24000:96000] = 0.0                                                     # a silent output frame (the 1e-6 clamp)
    staged = {"dev": torch.device("cpu"), "audio64": np.pad(hp, (vc.t_pad, vc.t_pad))}
    offs = np.concatenate([[0], np.cumsum(sizes)])
    parts = [(i, song[offs[i]: offs[i + 1]].copy()) for i in range(len(sizes))]
    vc._rms_mix(staged, parts, sizes, n_in, 48000, 0.25)
    hop = 24000
    assert vc.power_calls[0] == (0, n_in, 8000, (n_in - 1) // 8000 + 1)
    for (o, n, h, k), s, off in zip(vc.power_calls[1:], sizes, offs):
        assert (o, n, h) == (off, s, hop) and k == (off + s - 1) // hop - off // hop + 1
    rms1, rms2 = vc.folded
    np.testing.assert_allclose(rms1, _rms_oracle.librosa_rms(hp, 16000, 8000)[0], rtol=2e-7, atol=0)
    np.testing.assert_allclose(rms2, _rms_oracle.librosa_rms(song, 48000, hop)[0], rtol=2e-7, atol=1e-30)
    want = _rms_oracle.change_rms(hp, 16000, song.copy(), 48000, 0.25)
    got = np.concatenate([p for _, p in parts])
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-12)
    assert np.all(got[:9000] == 0) and np.all(np.isfinite(got))


def _run(case, rate):
    cfg = case["cfg"]
    vc = MixHostVC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device="cpu"), noise="reference")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    net = OracleNet(cfg, case["sd"])
    torch.manual_seed(case["rseed"])
    out = vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                      case["file_index"], case["index_rate"], 1, 3, cfg.sr, 0, rate, case["version"], case["protect"], 160,
                      False, False, None, 50, 1100)
    return out, vc.last_plan


@pytest.mark.parametrize("rate", [0.0, 0.25])
def test_song_with_mix_matches_oracle(rate):
    case = load_pipeline_golden("p1_40k_v1_4seg")
    torch.set_num_threads(1)
    out, plan = _run(case, rate)
    cfg = case["cfg"]
    torch.manual_seed(case["rseed"])
    c = pipeline_oracle.Constants(*case["tiers"], tgt_sr=cfg.sr)
    want = _rms_oracle.pipeline(rvc_oracle.fold_weight_norm(case["sd"]), cfg, case["hubert"], case["audio"].copy(), c,
                                synthetic.pipeline_f0, f0_up_key=case["f0_up_key"], file_index=case["file_index"],
                                index_rate=case["index_rate"], version=case["version"], protect=case["protect"],
                                rms_mix_rate=rate)
    assert len(plan["segments"]) > 1
    assert out.dtype == np.int16 and out.shape == want.shape and np.abs(out).max() == 32440
    assert np.abs(out.astype(np.int32) - want.astype(np.int32)).max() <= 1
    base = _run(case, 1.0)[0]
    assert np.abs(out.astype(np.int32) - base.astype(np.int32)).max() > 100      # the mix did something


def _worker(rank, world, port, name, rate, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out, plan = _run(load_pipeline_golden(name), rate)
        q.put((rank, None if out is None else out.copy(), plan["assignment"]))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_sharded_mix_world2_gloo_is_bit_identical():
    """Segments sharded over 2 ranks: the output envelope table is exchanged with one all-reduce and folded in segment
    order, so rank 0's song equals the single-process song bit for bit."""
    torch.set_num_threads(1)
    name, rate = "p1_40k_v1_4seg", 0.25
    single, _ = _run(load_pipeline_golden(name), rate)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, name, rate, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {}
    for _ in procs:
        r, out, assignment = q.get(timeout=600)
        res[r] = (out, assignment)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[1][0] is None and all(len(r) > 0 for r in res[0][1])
    assert np.array_equal(res[0][0], single)


def test_product_vc_refuses_the_mix_without_a_device():
    """No CPU fallback: with a CPU device `rms_mix_rate < 1` is refused before planning (audio=None is never touched)."""
    vc = pl.VC(40000, pl.PipelineConfig(1, 1, 2, 3, is_half=False, device="cpu"))
    with pytest.raises(NotImplementedError, match="no CPU fallback"):
        vc.pipeline(None, None, 0, None, [0, 0, 0], 0, "synthetic", "median", "", 0.0, 1, 3, 40000, 0, 0.25, "v1", 0.5, 160,
                    False, False)
