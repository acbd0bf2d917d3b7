#!/usr/bin/env python
"""Cost of the device index blend (`index_rate > 0` with an `IndexIVFFlatB200`, vc_infer_pipeline.py:59-75).

1. Kernels, one 60 s v2 segment: F = 3000 HuBERT frames of d = 768 (fp16, as with fp16 synthesis) against seeded clustered
   indices at RVC's own sizes (nlist = min(16 sqrt(N), N // 39)): N = 50 000 (nlist 1282), N = 200 000 (nlist 5128), and
   N = 200 000 with power-law list sizes and empty lists.  CUDA events around 20 back-to-back calls, `--reps` times:
       coarse_ms   rvcb200_op_ivf_assign alone; its arithmetic 2 F nlist d is computed here and reported as achieved
                   TFLOP/s against the fp32 CUDA-core rate SMs x 128 lanes x 2 x max SM clock (nvidia-smi)
       blend_ms    assign + scan + blend (`IndexIVFFlatB200.blend`), the whole per-segment cost, event span of back-to-back calls
       kernel_ms   the same calls' device time from a torch.profiler pass of its own: the sum of the durations of their kernels
                   and memsets per call (per kernel in kernels_us), so a host that cannot keep ahead of the device does not
                   inflate it; blend_ms close to kernel_ms shows that the host kept up
   The vectors (154 MB / 614 MB) do not fit the 126 MB L2; the centroids (4 / 16 MB) do, as they do in a song.
2. Song: a 10 min synthetic 16 kHz song through VC.pipeline at 48k_v2 (fake HuBERT, synthetic f0, fp16 tensor-core synthesis,
   tier 3/10/60/64), the N = 200 000 index, index_rate 0 and 0.75 alternated: device_ms (`last_plan["device_ms"]`) and wall_s.
Prints the card name and power limit with the numbers; one JSON line per measurement, also written to --out.  faiss is timed
only if it is importable (it is recorded as not measured otherwise).

    python tools/bench_index_blend.py [--reps 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import comfy_rvc_b200 as rvc  # noqa: E402
from comfy_rvc_b200 import IndexIVFFlatB200, _lib, pipeline as pl, synthetic  # noqa: E402
from comfy_rvc_b200.config import NAMED_CONFIGS  # noqa: E402


def card():
    p = torch.cuda.get_device_properties(0)
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sms": p.multi_processor_count, "max_sm_clock_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in q.stdout.strip().split(",")[:3]]
        info.update(name=name, power_limit_w=float(power), max_sm_clock_mhz=float(clk))
    except Exception as e:  # noqa: BLE001 -- the number is still reported, without the limit
        info["power_limit_error"] = repr(e)
    return info


def rvc_nlist(N):
    """RVC's train-index rule: n_ivf = min(int(16 * sqrt(N)), N // 39)."""
    return min(int(16 * math.sqrt(N)), N // 39)


def make_index(N, d, skew, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    nlist = rvc_nlist(N)
    cent = torch.randn(nlist, d, generator=g, device=dev)
    if skew:
        w = 1.0 / torch.arange(1, nlist + 1, device=dev, dtype=torch.float64) ** 1.1
        w[torch.randperm(nlist, generator=g, device=dev)[: nlist // 10]] = 0.0
        owner = torch.multinomial(w.float(), N, replacement=True, generator=g)
    else:
        owner = torch.randint(0, nlist, (N,), generator=g, device=dev)
    owner = owner.sort().values
    sizes = torch.bincount(owner, minlength=nlist)
    offs = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), sizes.cumsum(0)])
    vec = cent[owner] + 0.35 * torch.randn(N, d, generator=g, device=dev)
    labels = torch.randperm(N, generator=g, device=dev)
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device=dev)
    return idx, vec, {"N": N, "nlist": nlist, "skewed": skew, "max_list": int(sizes.max()), "empty_lists": int((sizes == 0).sum())}


def timed(fn, n, reps, dev):
    fn()
    torch.cuda.synchronize(dev)
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / n)
    return out


def profiled(fn, n, dev):
    """Device time per call (kernels + memsets, ms) and per-kernel microseconds per call, from a profiler pass."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize(dev)
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            key = e.name.replace("void ", "").replace("rvc::(anonymous namespace)::", "").split("<")[0].split("(")[0].strip()
            per[key] = per.get(key, 0.0) + e.time_range.elapsed_us()
    return sum(per.values()) / n / 1e3, {k: round(v / n, 2) for k, v in sorted(per.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=3000)
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    lines = []

    def emit(dct):
        print(json.dumps(dct), flush=True)
        lines.append(dct)

    gpu = card()
    emit({"card": gpu})
    peak = None
    if gpu["max_sm_clock_mhz"]:
        peak = gpu["sms"] * 128 * 2 * gpu["max_sm_clock_mhz"] * 1e6 / 1e12
    F, d = args.frames, 768
    lib = _lib.load()
    song_index = None
    for N, skew in ((50_000, False), (200_000, False), (200_000, True)):
        idx, vec, meta = make_index(N, d, skew, seed=N + skew, dev=dev)
        g = torch.Generator(device=dev).manual_seed(1)
        feats = (vec[torch.randint(0, N, (F,), generator=g, device=dev)] + 0.3 * torch.randn(F, d, generator=g, device=dev)).half()
        feats = feats.unsqueeze(0)
        coarse = torch.empty(F, dtype=torch.int64, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        x = feats[0]

        def assign():
            _lib.check(lib.rvcb200_op_ivf_assign(C.c_void_p(x.data_ptr()), 1, d, F, d, C.c_void_p(idx.centroids.data_ptr()),
                                                 C.c_void_p(idx.cnorm.data_ptr()), idx.nlist, C.c_void_p(coarse.data_ptr()), st),
                       None, "ivf_assign")
        c_ms = timed(assign, 20, args.reps, dev)
        b_ms = timed(lambda: idx.blend(feats, 0.75, True), 20, args.reps, dev)
        k_ms, per_kernel = profiled(lambda: idx.blend(feats, 0.75, True), 20, dev)
        flop = 2.0 * F * idx.nlist * d
        cm = float(np.median(c_ms))
        row = {"kernels": f"F {F}, d {d}, fp16 queries", **meta, "coarse_ms": [round(t, 4) for t in c_ms],
               "blend_ms": [round(t, 4) for t in b_ms], "coarse_ms_median": round(cm, 4),
               "blend_ms_median": round(float(np.median(b_ms)), 4), "kernel_ms": round(k_ms, 4), "kernels_us": per_kernel,
               "coarse_gflop": round(flop / 1e9, 3),
               "coarse_tflops": round(flop / (cm * 1e-3) / 1e12, 2), "fp32_core_peak_tflops": None if peak is None else round(peak, 1)}
        if peak:
            row["coarse_share_of_fp32_peak"] = round(row["coarse_tflops"] / peak, 3)
        emit(row)
        if N == 200_000 and not skew:
            song_index = idx
        else:
            del idx
        del vec, feats
        torch.cuda.empty_cache()

    cfg = NAMED_CONFIGS["48k_v2"]
    sd = synthetic.make_state_dict(cfg)
    net = rvc.SynthesizerTrnMs768NSFsid(*cfg.to_positional(), is_half=True)
    del net.enc_q
    net.load_state_dict({k: v.half() for k, v in sd.items()}, strict=False)
    net = net.eval().to(dev).set_precision("fp16")
    hubert = synthetic.FakeHubert(cfg.feat_dim, device_rng=True)
    audio = synthetic.make_song(args.seconds, seed=0)
    vc = pl.VC(cfg.sr, pl.PipelineConfig(3, 10, 60, 64, is_half=True, device=str(dev)), noise="device")
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0

    def run(rate):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        vc.pipeline(hubert, net, 0, audio.copy(), [0, 0, 0], 0, "synthetic", "median", song_index, rate, 1, 3, cfg.sr, 0, 1.0,
                    "v2", 0.5, 160, False, False, None, 50, 1100)
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t0, vc.last_plan["device_ms"]

    rates = (0.0, 0.75)
    for r in rates:
        run(r)
    res = {r: [] for r in rates}
    for _ in range(args.reps):
        for r in rates:
            wall, dms = run(r)
            res[r].append((wall, dms))
            emit({"index_rate": r, "wall_s": round(wall, 4), "device_ms": round(dms, 3), "segments": len(vc.last_plan["segments"])})
    summary = {"config": f"48k_v2 VC.pipeline, {args.seconds:.0f} s song, fp16 synthesis, tier (3, 10, 60, 64), IndexIVFFlatB200 "
                         f"N 200000 nlist {rvc_nlist(200_000)}", "card": gpu, "reps": args.reps}
    for r in rates:
        w, dm = zip(*res[r])
        summary[f"index_rate_{r}"] = {"wall_s_median": round(float(np.median(w)), 4), "wall_s": [round(x, 4) for x in w],
                                      "device_ms_median": round(float(np.median(dm)), 3), "device_ms": [round(x, 3) for x in dm]}
    summary["device_ms_difference_median"] = round(summary["index_rate_0.75"]["device_ms_median"]
                                                   - summary["index_rate_0.0"]["device_ms_median"], 3)
    try:
        import faiss  # noqa: F401
        summary["faiss"] = "importable, not timed by this tool"
    except ImportError:
        summary["faiss"] = "not installed on this machine: no faiss timing was taken"
    emit(summary)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for dct in lines:
                f.write(json.dumps(dct) + "\n")


if __name__ == "__main__":
    main()
