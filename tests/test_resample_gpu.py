"""GPU: the output resampling of `VC.pipeline` (`resample_sr`, vc_infer_pipeline.py:185-186) -- the kernel through the C ABI
against the float64 closed form (scipy's resample_poly with `comfy_rvc_b200.resample.design`), split invariance, whole songs
against the pipeline oracle, and the sharded song over NCCL."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
from scipy import signal

import comfy_rvc_b200 as rvc
from comfy_rvc_b200 import _lib, resample, synthetic
from comfy_rvc_b200 import pipeline as pl
from oracle import pipeline_oracle, rvc_oracle
from tests import _rms_oracle, _resample_oracle
from tests._util import load_pipeline_golden

pytestmark = pytest.mark.gpu

PAIRS = [(48000, 44100), (40000, 44100), (32000, 44100), (40000, 48000), (48000, 16000), (32000, 22050)]


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr() if t is not None and t.numel() else None)


class Filter:
    def __init__(self, orig, target):
        self.up, self.down, self.h = resample.design(orig, target)
        self.tpp = resample.taps_per_phase(self.h.shape[0], self.up)
        self.half_len = (self.h.shape[0] - 1) // 2
        self.H = resample.halo_len(self.h.shape[0], self.up)
        self.tab = torch.from_numpy(resample.phase_table(self.h, self.up)).cuda()

    def launch(self, left, piece, right, piece_off, n_song, out_lo, out_hi, out):
        return _lib.load().rvcb200_op_resample_poly(_p(self.tab), self.up, self.down, self.tpp, self.half_len, _p(left), left.numel(),
                                                    _p(piece), piece.numel(), _p(right), right.numel(), piece_off, n_song, out_lo,
                                                    out_hi, _p(out), _st())

    def whole(self, x_d):
        n = x_d.numel()
        out = torch.full((resample.out_len(n, self.up, self.down),), np.nan, dtype=torch.float32, device="cuda")
        empty = x_d[:0]
        assert self.launch(empty, x_d, empty, 0, n, 0, out.numel(), out) == 0
        return out


def _song_like(n, sr, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    x = np.sin(2 * np.pi * 220 * t) * (0.3 + 0.2 * np.sin(2 * np.pi * 0.3 * t)) + 0.2 * np.sin(2 * np.pi * (sr * 0.45) * t)
    return (x + rng.standard_normal(n) * 0.02).astype(np.float32)


@pytest.mark.parametrize("orig,target", PAIRS)
def test_kernel_matches_float64_closed_form(orig, target):
    """1 sample to 10 minutes (10 min for the two 44.1 kHz / 48 kHz pairs users ask for most; 30 s for the others, which
    keeps the float64 reference on the host short): max |y - y64| <= 1e-5 max |x|."""
    f = Filter(orig, target)
    long_n = orig * (600 if (orig, target) in ((48000, 44100), (40000, 48000)) else 30)
    rng = np.random.default_rng(orig + target)
    for n in (1, 7, f.h.shape[0] // f.up + 5, 10_007, long_n):
        for kind in ("random", "song"):
            x = (rng.standard_normal(n) * 0.3).astype(np.float32) if kind == "random" else _song_like(n, orig, n)
            got = f.whole(torch.from_numpy(x).cuda()).cpu().numpy()
            want = signal.resample_poly(x.astype(np.float64), f.up, f.down, window=f.h)
            assert got.shape == want.shape
            err = np.abs(got - want).max() / np.abs(x).max()
            print(f"{orig} -> {target}, n {n} {kind}: max |err| / max |x| = {err:.2e}")
            assert err <= 1e-5


@pytest.mark.parametrize("orig,target", [(48000, 44100), (40000, 44100), (48000, 16000), (32000, 22050)])
def test_any_split_is_bit_identical(orig, target):
    """Pieces of an input partition (some shorter than the halo) with H-sample halos, and arbitrary output ranges over the
    whole song: every launch gives exactly the bits of a single launch."""
    f = Filter(orig, target)
    rng = np.random.default_rng(1)
    n = orig * 20 + 17
    x_d = torch.from_numpy((rng.standard_normal(n) * 0.3).astype(np.float32)).cuda()
    ref = f.whole(x_d)
    cuts = np.sort(np.concatenate([rng.choice(np.arange(1, n), 6, replace=False), [1000, 1003, 1003 + f.H // 2]]))
    offs = np.concatenate([[0], np.unique(cuts), [n]])
    pieces = []
    for a, b in zip(offs[:-1], offs[1:]):
        a, b = int(a), int(b)
        lo, hi = resample.out_len(a, f.up, f.down), resample.out_len(b, f.up, f.down)
        out = torch.full((hi - lo,), np.nan, dtype=torch.float32, device="cuda")
        # halos as separate buffers, like the driver's table slices
        left, right = x_d[max(a - f.H, 0): a].clone(), x_d[b: b + f.H].clone()
        assert f.launch(left, x_d[a:b].clone(), right, a, n, lo, hi, out) == 0
        pieces.append(out)
    assert torch.equal(torch.cat(pieces), ref)
    for lo, hi in ((0, 1), (1, 2), (5, 4000), (12_345, 12_345 + 3 * f.up + 7), (ref.numel() - 9, ref.numel())):
        out = torch.full((hi - lo,), np.nan, dtype=torch.float32, device="cuda")
        assert f.launch(x_d[:0], x_d, x_d[:0], 0, n, lo, hi, out) == 0
        assert torch.equal(out, ref[lo:hi]), (lo, hi)


def test_abi_refuses_bad_arguments():
    f = Filter(48000, 44100)
    x = torch.zeros(100_000, dtype=torch.float32, device="cuda")
    out = torch.zeros(200_000, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    e = x[:0]
    ok = (_p(f.tab), f.up, f.down, f.tpp, f.half_len, _p(e), 0, _p(x[1000:2000]), 1000, _p(x[2000:2000 + f.H]), f.H, 1000, 100_000,
          resample.out_len(1000, f.up, f.down) + 300, resample.out_len(2000, f.up, f.down), _p(out))
    assert lib.rvcb200_op_resample_poly(*ok[:5], _p(x[1000 - f.H:1000]), f.H, *ok[7:], _st()) == 0
    bad = [
        (0, None),                      # no table
        (1, 0), (2, 0), (3, 0),         # up, down, tpp
        (4, f.tpp * f.up),              # half_len beyond the filter
        (11, 50),                       # the piece placed elsewhere in the song: the window misses the outputs' reach
        (12, 1500),                     # song shorter than piece + halo
        (13, -1), (14, 0),              # out_lo < 0, out_hi < out_lo
        (15, None),                     # no output buffer
    ]
    for i, v in bad:
        args = list(ok)
        args[i] = v
        assert lib.rvcb200_op_resample_poly(*args, _st()) == 1, (i, v)
    # the outputs near the piece's left edge reach into the song before it: refused without a left halo
    assert lib.rvcb200_op_resample_poly(*ok[:13], resample.out_len(1000, f.up, f.down), ok[14], ok[15], _st()) == 1
    # a misaligned table
    tab_odd = torch.zeros(f.tab.numel() + 1, dtype=torch.float32, device="cuda")[1:]
    assert lib.rvcb200_op_resample_poly(_p(tab_odd), *ok[1:], _st()) == 1
    torch.cuda.synchronize()


def _product(case, rate, resample_sr, precision="fp32", span_spy=None):
    from tests.test_parity_gpu import build_net
    cfg = case["cfg"]
    net = build_net(cfg, case["sd"], precision)
    vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device="cuda:0"), noise="reference")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    if span_spy is not None:
        vc._resample_span = span_spy
    torch.manual_seed(case["rseed"])
    return vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                       case["file_index"], case["index_rate"], 1, 3, cfg.sr, resample_sr, rate, case["version"], case["protect"], 160,
                       False, False, None, 50, 1100)


def _oracle_parts(case):
    torch.manual_seed(case["rseed"])
    c = pipeline_oracle.Constants(*case["tiers"], tgt_sr=case["cfg"].sr)
    _, parts, _ = pipeline_oracle.pipeline(rvc_oracle.fold_weight_norm(case["sd"]), case["cfg"], case["hubert"], case["audio"].copy(),
                                           c, synthetic.pipeline_f0, f0_up_key=case["f0_up_key"], file_index=case["file_index"],
                                           index_rate=case["index_rate"], version=case["version"], protect=case["protect"],
                                           return_parts=True)
    hp = signal.filtfilt(pipeline_oracle._BH, pipeline_oracle._AH, case["audio"])
    return np.concatenate(parts), hp


def _want(opt, hp, sr, rate, resample_sr):
    y = opt.copy()
    if rate < 1:
        y = _rms_oracle.change_rms(hp, 16000, y, sr, rate)
    return pipeline_oracle.to_int16(_resample_oracle.resample_song(y, sr, resample_sr))


@pytest.mark.parametrize("name", ["p1_40k_v1_4seg", "p3_48k_v2_single"])
def test_song_with_resampling_matches_oracle(name):
    """fp32 path, reference-order noise: every resample_sr x rms_mix_rate within +-1 LSB of the oracle, peak 32440; fp16
    synthesis SNR >= 45 dB; resample_sr 0, 8000 and the model's rate never enter the step."""
    case = load_pipeline_golden(name)
    opt, hp = _oracle_parts(case)
    sr = case["cfg"].sr
    for resample_sr in (44100, 48000 if sr != 48000 else 32000, 16000):
        for rate in (1.0, 0.25):
            out = _product(case, rate, resample_sr)
            want = _want(opt, hp, sr, rate, resample_sr)
            d = np.abs(out.astype(np.int32) - want.astype(np.int32))
            print(f"{name} resample_sr {resample_sr} rate {rate}: max {d.max()} LSB, {np.mean(d > 0) * 100:.3f} % differ")
            assert out.dtype == np.int16 and out.shape == want.shape
            assert d.max() <= 1 and np.abs(out).max() == 32440

    def no_span(*a, **k):
        raise AssertionError("resampling ran although the reference skips it")
    base = _product(case, 1.0, 0)
    assert np.abs(base.astype(np.int32) - case["gold"]["out_i16"].astype(np.int32)).max() <= 1
    for resample_sr in (0, 8000, sr):
        assert np.array_equal(_product(case, 1.0, resample_sr, span_spy=no_span), base)
    out16 = _product(case, 0.25, 44100, precision="fp16")
    want = _want(opt, hp, sr, 0.25, 44100)
    snr = synthetic.snr_db(want.astype(np.float64), out16.astype(np.float64))
    print(f"{name} fp16, resample_sr 44100, rate 0.25: song SNR {snr:.1f} dB")
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
                          case["file_index"], case["index_rate"], 1, 3, cfg.sr, 44100, 0.25, case["version"], case["protect"], 160,
                          False, False, None, 50, 1100, all_ranks=True)
        q.put((rank, out.copy(), vc.last_plan["assignment"]))
    finally:
        dist.destroy_process_group()


def test_sharded_resampling_nccl_is_bit_identical():
    """Two GPUs: the halo table is all-reduced over NCCL; every rank's song equals the unsharded one bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    name = "p1_40k_v1_4seg"
    single = _product(load_pipeline_golden(name), 0.25, 44100)
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
