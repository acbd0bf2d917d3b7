#!/usr/bin/env python
"""Cost of the output resampling (`resample_sr`, vc_infer_pipeline.py:185-186) in `VC.pipeline`.

    * kernel: `rvcb200_op_resample_poly` on a 10 min song for each rate pair below, one launch over the whole song, CUDA events
      around --launches back-to-back launches after a warm-up; achieved MAC/s (outputs x taps per phase, the work the kernel
      does) against the fp32 CUDA-core rate of DESIGN.md §6 (148 SMs x 128 lanes x 2 x 1965 MHz = 74.4 TFLOP/s).  Input and
      output (up to 0.23 GB) are read and written once per launch, so they come mostly from HBM; the tap table stays in L2.
    * song: a 10 min synthetic 16 kHz song through VC.pipeline at 48k_v2 (fake HuBERT, synthetic f0, fp16 tensor-core synthesis,
      tier 3/10/60/64), resample_sr = 0 and 44100 alternated in one process: device_ms (`last_plan["device_ms"]`), wall_s, and
      resample_ms (CUDA events around the driver's `_resample`).
Prints the card name and power limit with the numbers; one JSON line per measurement, also written to --out.

    python tools/bench_resample.py [--reps 3] [--launches 20] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import comfy_rvc_b200 as rvc  # noqa: E402
from comfy_rvc_b200 import _lib, resample, synthetic  # noqa: E402
from comfy_rvc_b200 import pipeline as pl  # noqa: E402
from comfy_rvc_b200.config import NAMED_CONFIGS  # noqa: E402
from tools.bench_rms_mix import card  # noqa: E402

PAIRS = [(48000, 44100), (40000, 44100), (32000, 44100), (40000, 48000), (48000, 16000), (32000, 22050)]
FP32_FLOPS = 148 * 128 * 2 * 1965e6


def kernel_pass(seconds, launches, emit):
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = []
    for orig, target in PAIRS:
        up, down, h = resample.design(orig, target)
        tpp, half_len = resample.taps_per_phase(h.shape[0], up), (h.shape[0] - 1) // 2
        tab = torch.from_numpy(resample.phase_table(h, up)).cuda()
        n = int(seconds * orig)
        x = torch.randn(n, device="cuda") * 0.3
        n_out = resample.out_len(n, up, down)
        out = torch.empty(n_out, device="cuda")

        def go():
            _lib.check(lib.rvcb200_op_resample_poly(C.c_void_p(tab.data_ptr()), up, down, tpp, half_len, None, 0, C.c_void_p(x.data_ptr()),
                                                    n, None, 0, 0, n, 0, n_out, C.c_void_p(out.data_ptr()), st), None, "resample_poly")
        for _ in range(3):
            go()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            go()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / launches
        macs = n_out * tpp
        d = {"kernel": "resample_poly", "pair": f"{orig}->{target}", "up_down": [up, down], "taps": int(h.shape[0]),
             "taps_per_phase": tpp, "seconds": seconds, "outputs": n_out, "ms": round(ms, 4),
             "gmac_per_s": round(macs / ms / 1e6, 1), "fp32_share": round(2 * macs / (ms * 1e-3) / FP32_FLOPS, 3)}
        emit(d)
        rows.append(d)
    return rows


def song_pass(seconds, reps, emit):
    dev = torch.device("cuda:0")
    cfg = NAMED_CONFIGS["48k_v2"]
    sd = synthetic.make_state_dict(cfg)
    net = rvc.SynthesizerTrnMs768NSFsid(*cfg.to_positional(), is_half=True)
    del net.enc_q
    net.load_state_dict({k: v.half() for k, v in sd.items()}, strict=False)
    net = net.eval().to(dev).set_precision("fp16")
    hubert = synthetic.FakeHubert(cfg.feat_dim, device_rng=True)
    audio = synthetic.make_song(seconds, seed=0)
    vc = pl.VC(cfg.sr, pl.PipelineConfig(3, 10, 60, 64, is_half=False, device=str(dev)), noise="device")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    events = []
    inner = vc._resample

    def timed(staged, *a, **k):
        s = torch.cuda.current_stream(staged["dev"])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        r = inner(staged, *a, **k)
        e1.record(s)
        events.append((e0, e1))
        return r
    vc._resample = timed

    def run(rs):
        torch.cuda.synchronize(dev)
        events.clear()
        t0 = time.perf_counter()
        out = vc.pipeline(hubert, net, 0, audio.copy(), [0, 0, 0], 0, "synthetic", "median", "", 0.0, 1, 3, cfg.sr, rs, 1.0,
                          "v2", 0.5, 160, False, False, None, 50, 1100)
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        span = events[0][0].elapsed_time(events[0][1]) if events else None
        return out, wall, vc.last_plan["device_ms"], span

    settings = (0, 44100)
    for rs in settings:
        run(rs)
    res = {rs: [] for rs in settings}
    for _ in range(reps):
        for rs in settings:
            out, wall, dms, rsm = run(rs)
            res[rs].append((wall, dms, rsm))
            emit({"resample_sr": rs, "wall_s": round(wall, 4), "device_ms": round(dms, 3),
                  "resample_ms": None if rsm is None else round(rsm, 4), "segments": len(vc.last_plan["segments"]),
                  "samples": int(out.shape[0])})
    summary = {"config": f"48k_v2 VC.pipeline, {seconds:.0f} s song, fp16 synthesis, tier (3, 10, 60, 64), rms_mix_rate 1",
               "reps": reps}
    for rs in settings:
        w, d, r = zip(*res[rs])
        summary[f"resample_sr_{rs}"] = {"wall_s_median": round(float(np.median(w)), 4), "wall_s": [round(x, 4) for x in w],
                                        "device_ms_median": round(float(np.median(d)), 3), "device_ms": [round(x, 3) for x in d],
                                        "resample_ms_median": None if r[0] is None else round(float(np.median(r)), 4)}
    return summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    gpu = card()
    emit({"card": gpu})
    kernel_pass(args.seconds, args.launches, emit)
    summary = song_pass(args.seconds, args.reps, emit)
    summary["card"] = gpu
    emit(summary)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
