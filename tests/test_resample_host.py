"""CPU: the output resampling of `VC.pipeline` (`resample_sr`, vc_infer_pipeline.py:185-186) -- the filter design against
its spec, the phase-major table through the kernel's indexing against scipy's resample_poly, the output partition with
halos, and the driver's host logic (halo table, exchange) with a numpy compute hook, single-process and over world_size-2
gloo."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy import signal

from comfy_rvc_b200 import pipeline as pl
from comfy_rvc_b200 import resample, synthetic
from oracle import pipeline_oracle, rvc_oracle
from tests import _resample_oracle
from tests._host_vc import HostVC, OracleNet
from tests._util import load_pipeline_golden
from tests.test_rms_mix_host import NumpyMixHooks

PAIRS = [(48000, 44100), (40000, 44100), (32000, 44100), (40000, 48000), (48000, 16000), (32000, 22050)]
EXTRA_PAIRS = [(48000, 22050), (40000, 16000)]


def kernel_ref(tab, up, down, tpp, half_len, x, x_first, n_song, out_lo, out_hi):
    """numpy restatement of `resample_poly_kernel`'s indexing: y[j] = sum_k tab[r][k] * x[m0 - k], k ascending, with
    t = j * down + half_len, r = t % up, m0 = t // up.  `x` holds the global samples [x_first, x_first + len(x)); samples
    outside the song are zero, and every sample inside it that an output reaches must be in `x`.  Accumulates in the
    table's dtype, one output's sum independent of the others."""
    j = np.arange(out_lo, out_hi, dtype=np.int64)
    t = j * down + half_len
    r, m0 = t % up, t // up
    acc = np.zeros(j.shape[0], dtype=tab.dtype)
    for k in range(tpp):
        m = m0 - k
        inside = (m >= 0) & (m < n_song)
        loc = m - x_first
        assert np.all((loc[inside] >= 0) & (loc[inside] < len(x))), "input window does not cover the outputs"
        v = np.where(inside, x[np.clip(loc, 0, max(len(x) - 1, 0))] if len(x) else 0, 0).astype(tab.dtype)
        acc = acc + tab[r, k] * v
    return acc


def _spec(orig, target):
    up, down, h = resample.design(orig, target)
    w, H = signal.freqz(h, worN=1 << 20)
    f = w / np.pi
    m = max(up, down)
    return up, down, h, np.abs(np.abs(H[f <= resample.PASSBAND_END / m]) - 1).max(), \
        20 * np.log10(np.abs(H[f >= 1.0 / m]).max())


@pytest.mark.parametrize("orig,target", PAIRS + EXTRA_PAIRS)
def test_design_meets_spec(orig, target):
    up, down, h, dev, stop_db = _spec(orig, target)
    print(f"{orig} -> {target}: {up}/{down}, {h.shape[0]} taps, passband deviation {dev:.2e}, stopband {stop_db:.1f} dB")
    assert h.dtype == np.float64 and h.shape[0] % 2 == 1 and np.array_equal(h, h[::-1])
    assert dev <= 1e-6 and stop_db <= -120.0
    assert resample.ratio(orig, target) == (up, down) and np.gcd(up, down) == 1


@pytest.mark.parametrize("orig,target", PAIRS)
def test_phase_table_through_kernel_indexing_is_resample_poly(orig, target):
    up, down, h = resample.design(orig, target)
    tab = resample.phase_table(h, up, dtype=np.float64)
    tpp, half_len = resample.taps_per_phase(h.shape[0], up), (h.shape[0] - 1) // 2
    assert tab.shape == (up, (tpp + 3) // 4 * 4) and np.all(tab[:, tpp:] == 0)
    assert np.array_equal(resample.phase_table(h, up), tab.astype(np.float32))
    for n in (1, 7, h.shape[0] // up // 2 + 3, 5 * down + 3, 40_000 + down - 1):   # shorter than the filter, not a multiple of down
        x = np.random.default_rng(n).standard_normal(n)
        want = signal.resample_poly(x, up, down, window=h)
        assert want.shape[0] == resample.out_len(n, up, down)
        got = kernel_ref(tab, up, down, tpp, half_len, x, 0, n, 0, want.shape[0])
        assert np.abs(got - want).max() <= 1e-12 * max(np.abs(want).max(), 1e-300), (n, np.abs(got - want).max())


class NumpyResampleHooks:
    """The compute hooks of the resampling (`_resample_table`, `_resample_span`) in float64 numpy, with the kernel's indexing."""

    def _require_device_resample(self):
        pass

    def _resample_table(self, staged, tgt_sr, resample_sr):
        up, down, h = resample.design(tgt_sr, resample_sr)
        return up, down, (h.shape[0] - 1) // 2, resample.taps_per_phase(h.shape[0], up), resample.phase_table(h, up, np.float64)

    def _resample_span(self, staged, table, up, down, tpp, half_len, left, piece, right, piece_off, n_song, out_lo, out_hi):
        left, right = np.asarray(left), np.asarray(right)
        self.span_calls.append((piece_off, len(piece), len(left), len(right), out_lo, out_hi))
        x = np.concatenate([left, np.asarray(piece), right]).astype(np.float64)
        return kernel_ref(table, up, down, tpp, half_len, x, piece_off - len(left), n_song, out_lo, out_hi).astype(np.float32)


class ResampleHostVC(NumpyResampleHooks, NumpyMixHooks, HostVC):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.power_calls, self.folded, self.span_calls = [], [], []


@pytest.mark.parametrize("orig,target", [(48000, 44100), (40000, 16000), (32000, 22050)])
def test_partition_and_halos(orig, target):
    """Pieces shorter than the halo (50 and 3 samples) resampled one by one through the halo table and concatenated equal
    resample_poly of the concatenation; the per-piece sizes partition ceil(N * up / down)."""
    vc = ResampleHostVC(orig, pl.PipelineConfig(1, 1, 2, 3, is_half=False, device="cpu"))
    sizes = [30000, 50, 71000, 3, 2000]
    rng = np.random.default_rng(11)
    song = (rng.standard_normal(sum(sizes)) * 0.3).astype(np.float32)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    parts = [(i, song[offs[i]: offs[i + 1]].copy()) for i in range(len(sizes))]
    out, out_sizes = vc._resample({"dev": torch.device("cpu")}, parts, sizes, orig, target)
    up, down, h = resample.design(orig, target)
    H = resample.halo_len(h.shape[0], up)
    assert sizes[1] < H and sizes[3] < H
    assert sum(out_sizes) == resample.out_len(sum(sizes), up, down)
    assert [len(p) for _, p in out] == out_sizes and [i for i, _ in out] == list(range(len(sizes)))
    want = signal.resample_poly(song.astype(np.float64), up, down, window=h)
    got = np.concatenate([p for _, p in out])
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-6 * np.abs(want).max()
    for (o, n, nl, nr, lo, hi), s, off in zip(vc.span_calls, sizes, offs):           # halos clipped at the song's ends only
        assert (o, n) == (off, s) and nl == min(H, off) and nr == min(H, sum(sizes) - off - s)


def _run(case, rate, resample_sr):
    cfg = case["cfg"]
    vc = ResampleHostVC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device="cpu"), noise="reference")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    net = OracleNet(cfg, case["sd"])
    torch.manual_seed(case["rseed"])
    out = vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                      case["file_index"], case["index_rate"], 1, 3, cfg.sr, resample_sr, rate, case["version"], case["protect"], 160,
                      False, False, None, 50, 1100)
    return out, vc.last_plan, vc


def _oracle(case, rate, resample_sr):
    cfg = case["cfg"]
    torch.manual_seed(case["rseed"])
    c = pipeline_oracle.Constants(*case["tiers"], tgt_sr=cfg.sr)
    return _resample_oracle.pipeline(rvc_oracle.fold_weight_norm(case["sd"]), cfg, case["hubert"], case["audio"].copy(), c,
                                     synthetic.pipeline_f0, f0_up_key=case["f0_up_key"], file_index=case["file_index"],
                                     index_rate=case["index_rate"], version=case["version"], protect=case["protect"],
                                     rms_mix_rate=rate, resample_sr=resample_sr)


@pytest.mark.parametrize("rate", [1.0, 0.25])
def test_song_with_resampling_matches_oracle(rate):
    case = load_pipeline_golden("p1_40k_v1_4seg")
    torch.set_num_threads(1)
    out, plan, vc = _run(case, rate, 44100)
    want = _oracle(case, rate, 44100)
    assert len(plan["segments"]) > 1 and len(vc.span_calls) == len(plan["segments"])
    assert out.dtype == np.int16 and out.shape == want.shape and np.abs(out).max() == 32440
    assert np.abs(out.astype(np.int32) - want.astype(np.int32)).max() <= 1


def test_no_resampling_below_16k_or_at_the_model_rate():
    """resample_sr 0, 8000 and == tgt_sr: the step is skipped (no span call), the song is unchanged."""
    case = load_pipeline_golden("p1_40k_v1_4seg")
    torch.set_num_threads(1)
    base = None
    for rs in (0, 8000, case["cfg"].sr):
        out, _, vc = _run(case, 1.0, rs)
        assert vc.span_calls == []
        if base is None:
            base = out
        assert np.array_equal(out, base)


def _worker(rank, world, port, name, rate, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out, plan, _ = _run(load_pipeline_golden(name), rate, 44100)
        q.put((rank, None if out is None else out.copy(), plan["assignment"]))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("rate", [1.0, 0.25])
def test_sharded_resampling_world2_gloo_is_bit_identical(rate):
    """Segments sharded over 2 ranks: the halo table is exchanged with one all-reduce, so rank 0's song equals the
    single-process song bit for bit and stays within +-1 LSB of the oracle."""
    torch.set_num_threads(1)
    name = "p1_40k_v1_4seg"
    single, _, _ = _run(load_pipeline_golden(name), rate, 44100)
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
    want = _oracle(load_pipeline_golden(name), rate, 44100)
    assert np.abs(res[0][0].astype(np.int32) - want.astype(np.int32)).max() <= 1


def test_product_vc_refuses_resampling_without_a_device():
    """No CPU fallback: with a CPU device a resample_sr that needs the step is refused before planning."""
    vc = pl.VC(40000, pl.PipelineConfig(1, 1, 2, 3, is_half=False, device="cpu"))
    with pytest.raises(NotImplementedError, match="no CPU fallback"):
        vc.pipeline(None, None, 0, None, [0, 0, 0], 0, "synthetic", "median", "", 0.0, 1, 3, 40000, 44100, 1.0, "v1", 0.5, 160,
                    False, False)
