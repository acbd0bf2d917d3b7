#!/usr/bin/env python
"""Cost of the volume-envelope mix (`rms_mix_rate < 1`, change_rms of lib/model_utils.py:39) in `VC.pipeline`.

A 10 min synthetic 16 kHz song through VC.pipeline at 48k_v2 (fake HuBERT, synthetic f0, fp16 tensor-core synthesis, the
half-precision tier x_pad/x_query/x_center/x_max = 3/10/60/64), rms_mix_rate = 1 and 0.25 alternated in one process:
    * mix_ms      device time of the mix's launches (CUDA events around the driver's `_rms_mix`)
    * device_ms   the song's device time (`last_plan["device_ms"]`), wall_s the call's wall time
    * host_change_rms_s  the reference's change_rms (librosa restatement + torch CPU) on this machine's cores, same N
Prints the card name and power limit with the numbers; one JSON line per measurement, also written to --out.

    python tools/bench_rms_mix.py [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import comfy_rvc_b200 as rvc  # noqa: E402
from comfy_rvc_b200 import pipeline as pl, synthetic  # noqa: E402
from comfy_rvc_b200.config import NAMED_CONFIGS  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.strip().split(",")[:2]]
        info.update(name=name, power_limit_w=float(power))
    except Exception as e:  # noqa: BLE001 -- the number is still reported, without the limit
        info["power_limit_error"] = repr(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    gpu = card()
    emit({"card": gpu})
    cfg = NAMED_CONFIGS["48k_v2"]
    sd = synthetic.make_state_dict(cfg)
    net = rvc.SynthesizerTrnMs768NSFsid(*cfg.to_positional(), is_half=True)
    del net.enc_q
    net.load_state_dict({k: v.half() for k, v in sd.items()}, strict=False)
    net = net.eval().to(dev).set_precision("fp16")
    hubert = synthetic.FakeHubert(cfg.feat_dim, device_rng=True)
    audio = synthetic.make_song(args.seconds, seed=0)
    vc = pl.VC(cfg.sr, pl.PipelineConfig(3, 10, 60, 64, is_half=False, device=str(dev)), noise="device")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    mix_events = []
    inner = vc._rms_mix

    def timed_mix(staged, *a, **k):
        s = torch.cuda.current_stream(staged["dev"])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        inner(staged, *a, **k)
        e1.record(s)
        mix_events.append((e0, e1))
    vc._rms_mix = timed_mix

    def run(rate):
        torch.cuda.synchronize(dev)
        mix_events.clear()
        t0 = time.perf_counter()
        out = vc.pipeline(hubert, net, 0, audio.copy(), [0, 0, 0], 0, "synthetic", "median", "", 0.0, 1, 3, cfg.sr, 0, rate,
                          "v2", 0.5, 160, False, False, None, 50, 1100)
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        mix_ms = mix_events[0][0].elapsed_time(mix_events[0][1]) if mix_events else None
        return out, wall, vc.last_plan["device_ms"], mix_ms

    rates = (1.0, 0.25)
    for r in rates:                                                            # warm-up: every shape once
        run(r)
    res = {r: [] for r in rates}
    for _ in range(args.reps):
        for r in rates:
            out, wall, dms, mms = run(r)
            res[r].append((wall, dms, mms))
            emit({"rms_mix_rate": r, "wall_s": round(wall, 4), "device_ms": round(dms, 3),
                  "mix_ms": None if mms is None else round(mms, 4), "segments": len(vc.last_plan["segments"]),
                  "samples": int(out.shape[0])})
    n_out = int(out.shape[0])
    summary = {"config": f"48k_v2 VC.pipeline, {args.seconds:.0f} s song, fp16 synthesis, tier (3, 10, 60, 64)", "card": gpu,
               "reps": args.reps}
    for r in rates:
        w, d, m = zip(*res[r])
        summary[f"rate_{r}"] = {"wall_s_median": round(float(np.median(w)), 4), "wall_s": [round(x, 4) for x in w],
                                "device_ms_median": round(float(np.median(d)), 3), "device_ms": [round(x, 3) for x in d],
                                "mix_ms_median": None if m[0] is None else round(float(np.median(m)), 4),
                                "mix_ms": None if m[0] is None else [round(x, 4) for x in m]}
    # the reference's change_rms on the host (librosa restatement + torch CPU), same N, same cores
    from scipy import signal
    from oracle import pipeline_oracle
    from tests import _rms_oracle
    hp = signal.filtfilt(pipeline_oracle._BH, pipeline_oracle._AH, audio)
    y = (np.random.default_rng(0).standard_normal(n_out) * 0.1).astype(np.float32)
    host = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        _rms_oracle.change_rms(hp, 16000, y.copy(), cfg.sr, 0.25)
        host.append(time.perf_counter() - t0)
    summary["host_change_rms_s"] = {"median": round(float(np.median(host)), 4), "runs": [round(x, 4) for x in host],
                                    "cpu_threads": torch.get_num_threads(), "cpus": os.cpu_count()}
    emit(summary)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
