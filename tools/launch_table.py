#!/usr/bin/env python
"""Per-launch kernel times of the bench workload (48k_v2, B = 1, 60 s) from torch.profiler, in launch order.

    python tools/launch_table.py --out out/launches_head.json                 # the library in the tree
    RVCB200_LIB=build_variants/librvcb200_base.so python tools/launch_table.py --out out/launches_base.json
    python tools/launch_table.py --compare out/launches_base.json out/launches_head.json \
        --filter rbconv_tc_kernel > table.md

Eager launches (no graph replay), warm-ups first, then --steps profiled steps: each launch's time is the median over
those steps of its CUDA activity duration.  Two captures of libraries with the same launch sequence compare row by row.
"""
import argparse
import json
import os
import re
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def capture(args):
    import torch
    import comfy_rvc_b200 as rvc
    from comfy_rvc_b200 import _lib, synthetic
    from comfy_rvc_b200.config import NAMED_CONFIGS
    cfg = NAMED_CONFIGS[args.config]
    T = int(round(args.seconds * 100))
    sd = synthetic.make_state_dict(cfg)
    cls = rvc.SynthesizerTrnMs256NSFsid if cfg.feat_dim == 256 else rvc.SynthesizerTrnMs768NSFsid
    net = cls(*cfg.to_positional(), is_half=args.precision != "fp32")
    del net.enc_q
    net.load_state_dict({k: v.half() for k, v in sd.items()}, strict=False)
    net.eval().to("cuda:0").set_precision(args.precision)
    net.graph_max_frames = 0
    ins = [t.cuda() for t in synthetic.make_inputs(cfg, 1, T)]
    noise = net.draw_noise(1, T)
    for _ in range(3):
        net.infer(*ins, noise=noise)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            net.infer(*ins, noise=noise)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and "Memcpy" not in e.name and "Memset" not in e.name),
                key=lambda e: e.time_range.start)
    n = len(ev) // args.steps
    assert n * args.steps == len(ev), f"{len(ev)} kernels over {args.steps} steps"
    rows = []
    for i in range(n):
        names = {ev[s * n + i].name for s in range(args.steps)}
        assert len(names) == 1, names
        rows.append({"i": i, "kernel": ev[i].name,
                     "us": statistics.median(ev[s * n + i].time_range.elapsed_us() for s in range(args.steps))})
    props = torch.cuda.get_device_properties(0)
    out = {"lib": _lib.LIB_PATH, "gpu": props.name, "config": args.config, "precision": args.precision, "T": T,
           "steps": args.steps, "kernels_per_step": n, "launches": rows}
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(f"{n} kernels per step, {sum(r['us'] for r in rows) / 1e3:.3f} ms summed -> {args.out}")


def compare(args):
    a, b = (json.load(open(p)) for p in args.compare)
    ra, rb = a["launches"], b["launches"]
    assert [r["kernel"] for r in ra] == [r["kernel"] for r in rb], "the two captures launch different kernel sequences"
    print(f"| # | kernel | base us | head us | head / base |\n|---|---|---|---|---|")
    sa = sb = 0.0
    for x, y in zip(ra, rb):
        if args.filter not in x["kernel"]:
            continue
        sa += x["us"]; sb += y["us"]
        name = re.sub(r"^void |\w+::|\(anonymous namespace\)::", "", x["kernel"]).split("(")[0]
        print(f"| {x['i']} | `{name}` | {x['us']:.1f} | {y['us']:.1f} | {y['us'] / x['us']:.3f} |")
    print(f"| | **sum** | {sa:.1f} | {sb:.1f} | {sb / max(sa, 1e-9):.3f} |")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--config", default="48k_v2")
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", help="JSON file the capture is written to")
    ap.add_argument("--compare", nargs=2, metavar=("BASE", "HEAD"))
    ap.add_argument("--filter", default="", help="only rows whose kernel name contains this")
    args = ap.parse_args()
    if not args.compare and not args.out:
        ap.error("--out is required for a capture")
    compare(args) if args.compare else capture(args)


if __name__ == "__main__":
    main()
