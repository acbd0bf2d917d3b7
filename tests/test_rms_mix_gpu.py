"""GPU: the volume-envelope mix of `VC.pipeline` (`rms_mix_rate < 1`, change_rms of lib/model_utils.py:39, called at
vc_infer_pipeline.py:183) -- the three kernels through the C ABI, the driver's mix on a 10-minute 48 kHz song, the whole
song against the pipeline oracle, and the sharded song over NCCL."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import comfy_rvc_b200 as rvc
from comfy_rvc_b200 import _lib, synthetic
from comfy_rvc_b200 import pipeline as pl
from oracle import pipeline_oracle, rvc_oracle
from tests import _rms_oracle
from tests._util import load_pipeline_golden

pytestmark = pytest.mark.gpu


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr())


def halfblock_ref(x: np.ndarray, offset: int, hop: int) -> np.ndarray:
    sq = np.square(x.astype(np.float32)).astype(np.float64)
    cuts = np.arange(offset // hop + 1, (offset + len(x) - 1) // hop + 1) * hop - offset
    return np.add.reduceat(sq, np.concatenate([[0], cuts]).astype(np.int64))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_halfblock_power_kernel(dtype):
    lib = _lib.load()
    rng = np.random.default_rng(7)
    song = (rng.standard_normal(1_000_003) * 0.3).astype(dtype)
    hop = 8000 if dtype == np.float64 else 24000
    n = song.shape[0]
    pieces = [(0, n), (0, 5000), (n - 777, 777), (123, hop // 3), (hop - 10, 20), (31_337, 250_001), (hop * 7, hop * 3),
              (n - hop * 2 - 5, hop * 2 + 5), (0, 1)]
    dev = torch.from_numpy(song).cuda()
    for off, ln in pieces:
        nb = (off + ln - 1) // hop - off // hop + 1
        out = torch.full((nb,), np.nan, dtype=torch.float64, device="cuda")
        assert lib.rvcb200_op_rms_halfblock(_p(dev[off:]), 1 if dtype == np.float64 else 0, ln, off, hop, _p(out), _st()) == 0
        got = out.cpu().numpy()
        want = halfblock_ref(song[off: off + ln], off, hop)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, err_msg=str((off, ln)))
        # the same piece at another global offset with the same half-block alignment: the same bits
        out2 = torch.full((nb,), np.nan, dtype=torch.float64, device="cuda")
        assert lib.rvcb200_op_rms_halfblock(_p(dev[off:]), 1 if dtype == np.float64 else 0, ln, off + 5 * hop, hop, _p(out2), _st()) == 0
        assert torch.equal(out, out2)
    out = torch.zeros(4, dtype=torch.float64, device="cuda")
    for args in ((None, 0, 10, 0, hop), (_p(dev), 2, 10, 0, hop), (_p(dev), 0, -1, 0, hop), (_p(dev), 0, 10, -1, hop),
                 (_p(dev), 0, 10, 0, 0)):
        assert lib.rvcb200_op_rms_halfblock(*args, _p(out), _st()) == 1
    assert lib.rvcb200_op_rms_halfblock(_p(dev), 0, 10, 0, hop, None, _st()) == 1
    assert lib.rvcb200_op_rms_fold(None, 1, 4, 16000, _p(out), _st()) == 1
    assert lib.rvcb200_op_rms_fold(_p(out), 0, 4, 16000, _p(out), _st()) == 1
    torch.cuda.synchronize()


def test_fold_kernel():
    lib = _lib.load()
    rng = np.random.default_rng(3)
    t = rng.random((5, 301)) * (rng.random((5, 301)) < 0.4)
    t[:, 17] = 0.0
    td = torch.from_numpy(t).cuda()
    rms = torch.empty(301, dtype=torch.float32, device="cuda")
    assert lib.rvcb200_op_rms_fold(_p(td), 5, 301, 48000, _p(rms), _st()) == 0
    hb = np.zeros(301)
    for row in t:
        hb = hb + row
    fr = hb.copy()
    fr[1:] += hb[:-1]
    assert np.array_equal(rms.cpu().numpy(), np.sqrt((fr / 48000).astype(np.float32)))


def gain_ref(rms1: np.ndarray, rms2: np.ndarray, N: int, rate: float) -> torch.Tensor:
    """The torch lines of change_rms (lib/model_utils.py:45-51) on given float32 envelopes."""
    r1 = F.interpolate(torch.from_numpy(rms1)[None, None], size=N, mode="linear").squeeze()
    r2 = F.interpolate(torch.from_numpy(rms2)[None, None], size=N, mode="linear").squeeze()
    r2 = torch.max(r2, torch.zeros_like(r2) + 1e-6)
    return (torch.pow(r1, torch.tensor(1 - rate)) * torch.pow(r2, torch.tensor(rate - 1))).reshape(-1)


@pytest.mark.parametrize("N", [7, 1_000_003, 28_800_000, 86_400_000])
def test_gain_kernel(N):
    lib = _lib.load()
    rng = np.random.default_rng(N)
    n1, n2 = 1 + (N // 3) // 8000, 1 + N // 24000
    rms1 = (rng.random(n1) * 0.3).astype(np.float32)
    rms2 = (rng.random(n2) * 0.5).astype(np.float32)
    if n1 > 2 and n2 > 4:
        rms1[n1 // 2] = 0.0                                                # a silent input frame: gain 0
        rms2[n2 // 3] = 0.0                                                # a silent output frame: the 1e-6 clamp
        rms2[n2 // 3 + 1] = 3e-7
    e1, e2 = torch.from_numpy(rms1).cuda(), torch.from_numpy(rms2).cuda()
    x = (rng.standard_normal(N) * 0.2).astype(np.float32)
    xd = torch.from_numpy(x).cuda()
    ones = torch.empty(N, dtype=torch.float32, device="cuda")
    peak = torch.zeros(1, dtype=torch.float32, device="cuda")
    pcm = torch.empty(N, dtype=torch.int16, device="cuda")
    for rate in (0.0, 0.25, 0.5, 0.99):
        want = gain_ref(rms1, rms2, N, rate).numpy()
        ones.fill_(1.0)
        # in two pieces at their global offsets, the second starting at an odd (unaligned) sample
        cut = N // 2 + 1
        for off, ln in ((0, cut), (cut, N - cut)):
            assert lib.rvcb200_op_rms_gain(_p(ones[off:]), ln, off, N, _p(e1), n1, _p(e2), n2, rate, _st()) == 0
        got = ones.cpu().numpy()
        ulp = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
        print(f"N {N} rate {rate}: gain max {ulp.max()} ulp, {np.mean(ulp > 0) * 100:.3f} % differ")
        assert ulp.max() <= 4 and np.array_equal(got == 0, want == 0)
        y = xd.clone()
        assert lib.rvcb200_op_rms_gain(_p(y), N, 0, N, _p(e1), n1, _p(e2), n2, rate, _st()) == 0
        assert lib.rvcb200_op_absmax(_p(y), N, _p(peak), 1, _st()) == 0
        assert lib.rvcb200_op_to_int16(_p(y), N, _p(peak), _p(pcm), _st()) == 0
        ref = synthetic.to_int16(x * want)
        d = np.abs(pcm.cpu().numpy().astype(np.int32) - ref.astype(np.int32)).max()
        assert d <= 1, (rate, d)
    for args in ((None, N, 0, N, _p(e1), n1, _p(e2), n2, 0.5), (_p(ones), N, 1, N, _p(e1), n1, _p(e2), n2, 0.5),
                 (_p(ones), N, 0, N, None, n1, _p(e2), n2, 0.5), (_p(ones), N, 0, N, _p(e1), 0, _p(e2), n2, 0.5),
                 (_p(ones), N, 0, N, _p(e1), n1, _p(e2), n2, float("nan")), (_p(ones), -1, 0, N, _p(e1), n1, _p(e2), n2, 0.5)):
        assert lib.rvcb200_op_rms_gain(*args, _st()) == 1
    torch.cuda.synchronize()


def test_ten_minute_mix_through_the_driver():
    """600 s at 48 kHz in 10 pieces of uneven length (frames straddle pieces), the filtered 16 kHz song as the input envelope,
    through `VC._rms_mix` directly: within +-1 LSB of the reference's change_rms + int16 conversion.  N = 28.8 M > 2^24."""
    vc = pl.VC(48000, pl.PipelineConfig.for_device(is_half=True))
    audio = synthetic.make_song(600.0, seed=12)
    audio_pad = pl.filtfilt_pad(audio, vc.t_pad)
    hp = audio_pad[vc.t_pad: vc.t_pad + audio.shape[0]].copy()
    N = 600 * 48000
    rng = np.random.default_rng(5)
    t = np.arange(N) / 48000.0
    song = (np.sin(2 * np.pi * 220 * t) * (0.2 + 0.15 * np.sin(2 * np.pi * 0.05 * t)) + rng.standard_normal(N) * 0.02).astype(np.float32)
    song[48000 * 100: 48000 * 102] = 0.0                                        # a silent output stretch
    cuts = np.sort(rng.choice(np.arange(1, N), 9, replace=False))
    sizes = np.diff(np.concatenate([[0], cuts, [N]])).tolist()
    dev = torch.device("cuda:0")
    staged = {"dev": dev, "audio64": torch.from_numpy(audio_pad).to(dev)}
    song_d = torch.from_numpy(song).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    # pieces are views of separate buffers (like the trimmed infer outputs), at unaligned starts
    bufs = [torch.zeros(s + 3, dtype=torch.float32, device=dev) for s in sizes]
    parts = []
    for i, b in enumerate(bufs):
        b[3:].copy_(song_d[offs[i]: offs[i + 1]])
        parts.append((i, b[3:]))
    for rate in (0.0, 0.5):
        work = [(i, p.clone()) for i, p in parts]
        vc._rms_mix(staged, work, sizes, hp.shape[0], 48000, rate)
        y = torch.cat([p for _, p in work]).cpu().numpy()
        want = pipeline_oracle.to_int16(_rms_oracle.change_rms(hp, 16000, song.copy(), 48000, rate))
        d = np.abs(synthetic.to_int16(y).astype(np.int32) - want.astype(np.int32))
        print(f"10 min, rate {rate}: max {d.max()} LSB, {np.mean(d > 0) * 100:.4f} % differ")
        assert d.max() <= 1


def _product(case, rate, precision="fp32", mix_spy=None):
    from tests.test_parity_gpu import build_net
    cfg = case["cfg"]
    net = build_net(cfg, case["sd"], precision)
    vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device="cuda:0"), noise="reference")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    if mix_spy is not None:
        vc._rms_mix = mix_spy
    torch.manual_seed(case["rseed"])
    return vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                       case["file_index"], case["index_rate"], 1, 3, cfg.sr, 0, rate, case["version"], case["protect"], 160,
                       False, False, None, 50, 1100)


def _oracle_parts(case):
    torch.manual_seed(case["rseed"])
    c = pipeline_oracle.Constants(*case["tiers"], tgt_sr=case["cfg"].sr)
    _, parts, _ = pipeline_oracle.pipeline(rvc_oracle.fold_weight_norm(case["sd"]), case["cfg"], case["hubert"], case["audio"].copy(),
                                           c, synthetic.pipeline_f0, f0_up_key=case["f0_up_key"], file_index=case["file_index"],
                                           index_rate=case["index_rate"], version=case["version"], protect=case["protect"],
                                           return_parts=True)
    from scipy import signal
    hp = signal.filtfilt(pipeline_oracle._BH, pipeline_oracle._AH, case["audio"])
    return np.concatenate(parts), hp


@pytest.mark.parametrize("name", ["p1_40k_v1_4seg", "p3_48k_v2_single"])
def test_song_with_mix_matches_oracle(name):
    """fp32 path, reference-order noise: the song with rms_mix_rate 0 / 0.25 / 0.5 within +-1 LSB of the oracle (the reference's
    change_rms on the oracle's concatenated segments), peak 32440; rms_mix_rate = 1 never enters the mix."""
    case = load_pipeline_golden(name)
    opt, hp = _oracle_parts(case)
    sr = case["cfg"].sr
    for rate in (0.0, 0.25, 0.5):
        out = _product(case, rate)
        want = pipeline_oracle.to_int16(_rms_oracle.change_rms(hp, 16000, opt.copy(), sr, rate))
        d = np.abs(out.astype(np.int32) - want.astype(np.int32))
        print(f"{name} rate {rate}: max {d.max()} LSB, {np.mean(d > 0) * 100:.3f} % differ")
        assert out.dtype == np.int16 and out.shape == want.shape
        assert d.max() <= 1 and np.abs(out).max() == 32440

    def no_mix(*a, **k):
        raise AssertionError("rms_mix_rate = 1 entered the mix")
    base = _product(case, 1.0, mix_spy=no_mix)
    assert np.abs(base.astype(np.int32) - case["gold"]["out_i16"].astype(np.int32)).max() <= 1
    if name == "p1_40k_v1_4seg":
        out16 = _product(case, 0.25, precision="fp16")
        want = pipeline_oracle.to_int16(_rms_oracle.change_rms(hp, 16000, opt.copy(), sr, 0.25))
        snr = synthetic.snr_db(want.astype(np.float64), out16.astype(np.float64))
        print(f"{name} fp16, rate 0.25: song SNR {snr:.1f} dB")
        assert snr >= 45.0


def _nccl_worker(rank, world, port, name, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        case = load_pipeline_golden(name)
        cfg = case["cfg"]
        net = rvc.SynthesizerTrnMs256NSFsid(*cfg.to_positional(), is_half=False) if cfg.feat_dim == 256 else \
            rvc.SynthesizerTrnMs768NSFsid(*cfg.to_positional(), is_half=False)
        del net.enc_q
        net.load_state_dict({k: v.half() for k, v in case["sd"].items()}, strict=False)
        net.eval().to(f"cuda:{rank}")
        net = net.float().set_precision("fp32")
        vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device=f"cuda:{rank}"), noise="reference")
        vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
        torch.manual_seed(case["rseed"])
        out = vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                          case["file_index"], case["index_rate"], 1, 3, cfg.sr, 0, 0.25, case["version"], case["protect"], 160,
                          False, False, None, 50, 1100, all_ranks=True)
        q.put((rank, out.copy(), vc.last_plan["assignment"]))
    finally:
        dist.destroy_process_group()


def test_sharded_mix_nccl_is_bit_identical():
    """Two GPUs: the output envelope table is all-reduced over NCCL; every rank's song equals the unsharded one bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    name = "p1_40k_v1_4seg"
    single = _product(load_pipeline_golden(name), 0.25)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, name, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = {}
        for _ in procs:
            r, out, assignment = q.get(timeout=900)
            res[r] = (out, assignment)
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
    assert all(len(r) > 0 for r in res[0][1])
    assert np.array_equal(res[0][0], single) and np.array_equal(res[1][0], single)
