"""CPU: bench.py's contract pieces that need no GPU -- the reference arm prints exactly one JSON line with the agreed
keys, `--dump-outputs` writes the same arrays on every run, and the algorithmic FLOP / byte models reproduce the figures of
SURVEY.md §8(d) / DESIGN.md §4."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from comfy_rvc_b200.config import NAMED_CONFIGS  # noqa: E402


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-frames", "20"], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["unit"] == "audio-s/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # under torchrun every rank but 0 exits 0 without work and without output
    env["RANK"], env["WORLD_SIZE"] = "1", "2"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_dumps_its_last_timed_step(tmp_path):
    """Two runs write the same arrays, and they are the oracle's outputs for the LAST timed step (the second of two: noise
    seed 8), each under its own name."""
    from oracle import rvc_oracle
    from comfy_rvc_b200 import synthetic
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
            "--cpu-frames", "20", "--dump-outputs"]
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    for d in ("a", "b"):
        out = subprocess.run(args + [str(tmp_path / d)], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
    cfg = NAMED_CONFIGS["48k_v2"]
    w = rvc_oracle.fold_weight_norm(synthetic.make_state_dict(cfg))
    inputs = synthetic.make_inputs(cfg, 1, 20)
    step = lambda seed: rvc_oracle.infer(w, cfg, *inputs, *synthetic.draw_noise(cfg, 1, 20, seed=seed))
    # the oracle's CPU reductions depend on the thread count: recompute the step with the reference arm's (bench.py: one
    # thread per host core), not with whatever this process was started with or an earlier test left behind
    prev = torch.get_num_threads()
    torch.set_num_threads(os.cpu_count() or 1)
    try:
        o, x_mask, (z, z_p, m_p, logs_p) = step(8)
        first = step(7)[0].numpy()                   # the first timed step's waveform is a different one
    finally:
        torch.set_num_threads(prev)
    want = {"audio": o, "x_mask": x_mask, "z": z, "z_p": z_p, "m_p": m_p, "logs_p": logs_p}
    for name, ref in want.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == tuple(ref.shape) and np.array_equal(a, b), name
        np.testing.assert_allclose(a, ref.numpy(), rtol=1e-5, atol=1e-5, err_msg=name)
    assert np.abs(np.load(tmp_path / "a" / "audio.npy") - first).max() > 1e-3
    out = subprocess.run(args[:4] + ["--steps", "0"], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_dump_outputs_samples_above_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 4 * 1000)
    outs = (torch.arange(3000.0).reshape(1, 1, 3000), torch.ones(1, 1, 10), tuple(torch.zeros(1, 4, 10) for _ in range(4)))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    a = np.load(tmp_path / "a" / "audio.npy")
    total = sum(np.load(tmp_path / "a" / f"{n}.npy").nbytes for n in ("audio", "x_mask", "z", "z_p", "m_p", "logs_p"))
    assert total <= 4 * 1000 and a.dtype == np.float32 and a.size > 900
    assert np.all(np.diff(a) > 0) and np.array_equal(a, np.load(tmp_path / "b" / "audio.npy"))


def test_algorithmic_flop_model_matches_survey():
    cfg = NAMED_CONFIGS["48k_v2"]
    macs = bench.algorithmic_macs(cfg, 6000)
    gflop_per_audio_s = 2.0 * sum(macs.values()) / 1e9 / 60.0
    assert gflop_per_audio_s == pytest.approx(115.271, abs=2e-3)             # SURVEY.md §8(d)
    assert 2.0 * macs["resblocks"] / 1e9 / 60.0 == pytest.approx(106.52, abs=1e-2)
    cfg = NAMED_CONFIGS["40k"]
    macs = bench.algorithmic_macs(cfg, 1000)
    assert 2.0 * sum(macs.values()) / 1e9 / 10.0 == pytest.approx(94.245, abs=2e-3)


def test_resblock_byte_model(monkeypatch):
    """DESIGN.md §4: 28.1 GB per 60 s step as two launches per pair, 19.8 GB with the C <= 64, k <= 7 and C = 32, k = 11
    pairs fused."""
    cfg = NAMED_CONFIGS["48k_v2"]
    monkeypatch.setenv("RVCB200_FUSE_PAIRS", "0")
    rd, wr = bench.resblock_bytes(cfg, 6000)
    assert (rd + wr) / 1e9 == pytest.approx(28.13, abs=0.01)
    monkeypatch.setenv("RVCB200_FUSE_PAIRS", "1")
    rd, wr = bench.resblock_bytes(cfg, 6000)
    assert (rd + wr) / 1e9 == pytest.approx(19.83, abs=0.01)
    E = 6000 * 480 * 32                                                      # a fused 's' pair moves 4 B per element
    assert bench.pair_is_fused(32, 3) and bench.pair_is_fused(64, 7) and not bench.pair_is_fused(128, 3) and not bench.pair_is_fused(64, 11) and bench.pair_is_fused(32, 11)
    assert E == 92160000
