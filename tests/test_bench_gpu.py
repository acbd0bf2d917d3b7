"""GPU: `bench.py --dump-outputs` on the product arm writes what the last timed `infer()` returned, under its own names,
and two runs with the same arguments write the same arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_product_arm_dump_is_repeatable(tmp_path):
    sys.path.insert(0, ROOT)
    from comfy_rvc_b200.config import NAMED_CONFIGS
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--seconds", "1", "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
            "--no-gpu-incumbent", "--no-front-end", "--no-extra-precision", "--no-parity", "--dump-outputs"]
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    for d in ("a", "b"):
        out = subprocess.run(args + [str(tmp_path / d)], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip())
        assert line["steps"] == 2
    cfg = NAMED_CONFIGS["48k_v2"]
    T, Ci = 100, cfg.inter_channels
    shapes = {"audio": (1, 1, T * cfg.upp), "x_mask": (1, 1, T), "z": (1, Ci, T), "z_p": (1, Ci, T), "m_p": (1, Ci, T),
              "logs_p": (1, Ci, T)}
    for name, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), name
        assert np.array_equal(a, b), name
    assert np.abs(np.load(tmp_path / "a" / "audio.npy")).max() > 0
    assert (np.load(tmp_path / "a" / "x_mask.npy") == 1).all()
