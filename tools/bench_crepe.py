"""CREPE on the B200: `crepe.predict` wall time per call, per-convolution kernel time and achieved TFLOP/s, and the eager-PyTorch
incumbent (torchcrepe's network as the oracle's functional form on cuDNN, fp32 with TF32 off and fp16) in the same process.

    python tools/bench_crepe.py [--out profiles/r3_crepe_b200.jsonl] [--seconds 10 60 600] [--reps 5]

Writes one JSON line per measurement (card name and power limit in every line).  Useful MACs per frame are the `full` model's
(conv1 134 M, conv2 1074 M, conv3..6 201 M, classifier 0.7 M); executed MACs count the padded rows of the line layout of
conv3..conv6 (L + 32 rows a frame) and the 24 padded classifier columns.
"""
from __future__ import annotations

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

from comfy_rvc_b200 import crepe, synthetic  # noqa: E402
from oracle import crepe_oracle as O  # noqa: E402

PEAK_TFLOPS = 2250.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def conv_macs(model="full"):
    """(name, useful MACs per frame, executed MACs per frame) of each contraction."""
    cin, cout, nf = crepe.CHANNELS[model]
    L = crepe.LENGTHS
    out = [("conv1", 512 * cout[0] * L[0], 512 * cout[0] * L[0]),
           ("conv2", 64 * cin[1] * cout[1] * L[1], 64 * cin[1] * cout[1] * L[1])]
    for i in range(2, 6):
        kc = 64 * max(cin[i], 64) * cout[i]
        out.append((f"conv{i + 1}", 64 * cin[i] * cout[i] * L[i], kc * (L[i] + 32)))
    out.append(("classifier", nf * 360, nf * crepe.N_PAD))
    return out


def time_call(fn, reps):
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), float(np.min(ts))


def per_conv(m: crepe.Crepe, nF: int, reps: int):
    """Kernel time of each launch of one pass of nF frames (CUDA events around `reps` back-to-back launches)."""
    audio = synthetic.make_speech(nF * 160 / 16000 + 0.1, seed=1)[0].cuda()
    m._materialize()
    m._begin()
    launches = []
    orig_conv = m._conv
    m._conv = lambda name, *a, **k: (launches.append(("conv", name, a, k)), orig_conv(name, *a, **k))[1]
    m._network(audio, int(audio.numel()), 0, nF, 160, True)
    m._conv = orig_conv
    res = {}
    for _, name, a, k in launches:
        orig_conv(name, *a, **k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            orig_conv(name, *a, **k)
        e1.record()
        torch.cuda.synchronize()
        res[name] = e0.elapsed_time(e1) / reps
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_crepe_b200.jsonl"))
    ap.add_argument("--seconds", type=float, nargs="+", default=[10.0, 60.0, 600.0])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    sd = synthetic.make_crepe_state_dict(0, "full")
    m = crepe.Crepe("full", weights=sd, device="cuda:0")
    gflop_frame = 2 * sum(u for _, u, _ in conv_macs()) / 1e9
    for sec in args.seconds:
        audio = torch.as_tensor(synthetic.make_song(sec, seed=4), dtype=torch.float32)[None]
        T = 1 + audio.shape[1] // 160
        for bs in (None, 320):
            fn = lambda: crepe.predict(audio, 16000, 160, 50.0, 1100.0, "full", crepe.decode.viterbi, batch_size=bs, device="cuda:0",
                                       crepe_model=m)
            fn()
            med, best = time_call(fn, args.reps if sec < 600 else max(2, args.reps // 2))
            emit({"what": "predict", "seconds": sec, "frames": T, "hop": 160, "model": "full", "decoder": "viterbi",
                  "batch_size": bs, "ms_median": med * 1e3, "ms_min": best * 1e3, "audio_s_per_s": sec / med,
                  "useful_tflops": gflop_frame * T / med / 1e3})
        # the network alone (no decode), same frames
        x = audio[0].cuda()
        fn = lambda: m.forward_logits(x, 160, True, 0, T)
        fn()
        med, best = time_call(fn, args.reps)
        emit({"what": "network", "seconds": sec, "frames": T, "ms_median": med * 1e3, "useful_tflops": gflop_frame * T / med / 1e3})
    # per-contraction kernel time on one full pass
    nF = crepe.PASS_FRAMES
    t = per_conv(m, nF, 20)
    for name, useful, executed in conv_macs():
        ms = t["cls" if name == "classifier" else name]
        emit({"what": "kernel", "conv": name, "frames": nF, "ms": ms, "useful_gmac": useful * nF / 1e9,
              "executed_gmac": executed * nF / 1e9, "useful_tflops": 2 * useful * nF / ms / 1e9,
              "executed_tflops": 2 * executed * nF / ms / 1e9, "frac_of_2250": 2 * useful * nF / ms / 1e9 / PEAK_TFLOPS})
    # the eager incumbent: the oracle's functional network on cuDNN, 60 s of frames in passes of 1024
    audio = synthetic.make_song(60.0, seed=4)
    frames = next(O.preprocess(torch.as_tensor(audio, dtype=torch.float32)[None], 16000, 160, None, True)).cuda()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    for dt in (torch.float32, torch.float16):
        sdd = {k: (v.cuda().to(dt) if v.is_floating_point() else v.cuda()) for k, v in sd.items()}
        fr = frames.to(dt)

        def inc():
            with torch.no_grad():
                for p0 in range(0, fr.shape[0], 1024):
                    O.crepe_forward(fr[p0:p0 + 1024], sdd)
        inc()
        med, _ = time_call(inc, 3)
        emit({"what": "incumbent_network", "dtype": str(dt), "seconds": 60.0, "frames": int(fr.shape[0]), "ms_median": med * 1e3,
              "useful_tflops": gflop_frame * fr.shape[0] / med / 1e3})
    x = torch.as_tensor(audio, dtype=torch.float32).cuda()
    fn = lambda: m.forward_logits(x, 160, True, 0, int(frames.shape[0]))
    fn()
    med, _ = time_call(fn, 3)
    emit({"what": "network_same_call", "seconds": 60.0, "frames": int(frames.shape[0]), "ms_median": med * 1e3,
          "useful_tflops": gflop_frame * frames.shape[0] / med / 1e3})
    with open(args.out, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
