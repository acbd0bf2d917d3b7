#!/usr/bin/env python
"""Headline benchmark: seconds of output audio synthesised per second (RTF^-1).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp32|fp16|bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference        # the reference algorithm's CPU path (oracle port) on the SAME step, rank 0 only

A "step" is one `net_g.infer()` of the BASELINE.json workload `configs[1]`: 48k_v2
(SynthesizerTrnMs768NSFsid), one 60 s segment of synthetic 768-d features + f0 (T = 6000 frames,
2 880 000 output samples) with seeded random weights, per GPU.  Segments are independent
(SURVEY.md §8e), so N GPUs run N segments with no collective on the data path: weak scaling,
value = N * 60 s / max-over-ranks device time.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from comfy_rvc_b200 import synthetic  # noqa: E402
from comfy_rvc_b200.config import NAMED_CONFIGS  # noqa: E402


def algorithmic_macs(cfg, T: int) -> dict:
    """MACs per batch item by component — the formula of SURVEY.md §8(d) (banded rel-pos, 1 MAC = 2 FLOP)."""
    H, F, Ci = cfg.hidden_channels, cfg.filter_channels, cfg.inter_channels
    U0 = cfg.upsample_initial_channel
    R = sum(len(ds) * 2 * k for k, ds in zip(cfg.resblock_kernel_sizes, cfg.resblock_dilation_sizes)) \
        if cfg.resblock == "1" else sum(len(ds) * k for k, ds in zip(cfg.resblock_kernel_sizes, cfg.resblock_dilation_sizes))
    pre = T * Ci * U0 * 7
    ups = noise = res = 0
    L, C = T, U0
    for i, (u, k) in enumerate(zip(cfg.upsample_rates, cfg.upsample_kernel_sizes)):
        Cn, Ln = C // 2, L * u
        ups += L * C * Cn * k
        noise += Ln * Cn * cfg.noise_conv_geometry(i)[0]
        res += Ln * Cn * Cn * R
        L, C = Ln, Cn
    post = L * C * 7
    half = Ci // 2
    flow = cfg.n_flows * T * (half * H + cfg.flow_wn_layers * H * 2 * H * cfg.flow_kernel + 2 * H * 2 * H + H * H + H * half)
    W = 2 * cfg.window_size + 1
    enc_lin = T * cfg.feat_dim * H + cfg.n_layers * (4 * T * H * H + 2 * T * H * F * cfg.kernel_size) + T * H * 2 * Ci
    attn = cfg.n_layers * (2 * T * T * H + 2 * 2 * T * W * (H // cfg.n_heads))
    return {"conv_pre": pre, "ups": ups, "noise": noise, "resblocks": res, "conv_post": post, "flow": flow,
            "enc_linear": enc_lin, "attention": attn}


def pair_is_fused(C: int, k: int) -> bool:
    """ResBlock1 pairs that run as ONE kernel with h in shared memory (csrc/rbpair_tc.cu: rbpair_tc_supported)."""
    return os.environ.get("RVCB200_FUSE_PAIRS", "1") != "0" and C in (32, 64) and (k in (3, 7) or (k == 11 and C == 32))


def resblock_bytes(cfg, T: int):
    """Algorithmic HBM bytes (read, write) of the decoder resblock convolutions of one item on the tensor path
    (DESIGN.md §3: one fp16 stream copy, h as one 16-bit tensor -- or not at all where the pair is fused --, planar fp16
    branch sum)."""
    rd = wr = 0
    L, C = T, cfg.upsample_initial_channel
    nk = len(cfg.resblock_kernel_sizes)
    for i, u in enumerate(cfg.upsample_rates):
        L, C = L * u, C // 2
        E = L * C
        last_stage = i == len(cfg.upsample_rates) - 1
        for j, ds in enumerate(cfg.resblock_dilation_sizes):
            for d_i in range(len(ds)):
                if cfg.resblock == "1" and pair_is_fused(C, cfg.resblock_kernel_sizes[j]):
                    rd += 2 * E                                   # fused pair: stream in (h and the residual stay on the SM)
                elif cfg.resblock == "1":
                    rd += 2 * E; wr += 2 * E                      # conv1: stream in, h out
                    rd += 4 * E                                   # conv2: h + residual from the stream
                else:
                    rd += 2 * E
                if d_i < len(ds) - 1:
                    wr += 2 * E                                   # stream out
                else:
                    rd += 2 * E if j > 0 else 0                   # branch sum in
                    wr += 2 * E                                   # branch sum out
                    if j == nk - 1 and not last_stage:
                        wr += 2 * E                               # operand of the next transposed conv
    return rd, wr


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "burst": d["bf16_tflops"],
                "src": "measured (MEASURED_PEAKS.json, sustained: the class is timed inside a long step)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "burst": 1590.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_rate(cfg, T: int, reps: int, warmup: int, threads: int, warmup_T: int = 0, check=None):
    """RTF^-1 of the reference algorithm on the host cores (oracle port, fp32 PyTorch CPU).  `warmup` untimed steps at
    `warmup_T` frames (default: the timed size), then `reps` timed steps at T frames."""
    from oracle import rvc_oracle
    prev = torch.get_num_threads()
    torch.set_num_threads(threads)
    try:
        sd = synthetic.make_state_dict(cfg)
        w = rvc_oracle.fold_weight_norm(sd)
        times = []
        for i in range(warmup + reps):
            Ti = T if i >= warmup or not warmup_T else warmup_T
            phone, lens, pitch, pitchf, sid = synthetic.make_inputs(cfg, 1, Ti)
            noise = synthetic.draw_noise(cfg, 1, Ti, seed=7 + max(i - warmup, 0))     # first timed step = the g2 fixture's draw
            t0 = time.perf_counter()
            outs = rvc_oracle.infer(w, cfg, phone, lens, pitch, pitchf, sid, *noise)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            if i == warmup and check is not None:
                check["first_timed_output"] = outs[0][0, 0].numpy()
            if check is not None:
                check["last_timed"] = outs
    finally:
        torch.set_num_threads(prev)
    audio_s = T * cfg.upp / cfg.sr
    return audio_s / float(np.median(times)), audio_s, times


def oracle_vs_fixture(o, config_name: str, T: int):
    """The CPU leg's first timed step is the g2 fixture's step: how far the oracle port is from the waveform the unmodified
    reference produced (the oracle's pin at BASELINE size, re-checked on the machine that runs the bench)."""
    path = os.path.join(ROOT, "tests", "golden", "g2_48k_v2_T6000.npz")
    if o is None or config_name != "48k_v2" or T != 6000 or not os.path.exists(path):
        return None
    gold = np.load(path, allow_pickle=True)
    d = np.abs(synthetic.to_int16(o).astype(np.int32) - gold["o_i16"][0].astype(np.int32))
    return {"int16_max_lsb_diff": int(d.max()), "int16_frac_differing": float((d > 0).mean()),
            "against": "tests/golden/g2_48k_v2_T6000.npz (unmodified reference, 1 CPU thread)"}


def gpu_incumbent_rate(cfg, T: int, dev, half: bool, reps: int = 3):
    """The eager-PyTorch incumbent on the same GPU (SURVEY.md §8d, §2.2): the oracle port -- pure torch.nn.functional, the
    reference's own op sequence -- on CUDA tensors, cuDNN / cuBLAS kernels, fp16 as the reference ships it on CUDA
    (`is_half`, /root/reference/vc_infer_pipeline.py:223-226) or fp32 with TF32 off.  Same step as the product arm
    (noise drawn on the device inside the step).  The port's attention is the banded form, i.e. it does LESS work than
    the reference's zero-padded relative-position matmuls: the incumbent figure errs on the fast side."""
    from oracle import rvc_oracle
    tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dt = torch.float16 if half else torch.float32
        sd = synthetic.make_state_dict(cfg)
        w = {k: v.to(dev, dtype=dt) for k, v in rvc_oracle.fold_weight_norm(sd).items()}
        phone, lens, pitch, pitchf, sid = [t.to(dev) for t in synthetic.make_inputs(cfg, 1, T)]
        L = T * cfg.upp

        def step():
            nz = torch.randn(1, cfg.inter_channels, T, device=dev, dtype=dt)
            ri = torch.rand(1, 1, device=dev)
            ns = torch.randn(1, L, 1, device=dev)
            return rvc_oracle.infer(w, cfg, phone.to(dt), lens, pitch, pitchf, sid, nz, ri, ns)[0]

        for _ in range(2):
            step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            o = step()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / reps
        del w, o
        torch.cuda.empty_cache()
        return T * cfg.upp / cfg.sr / (ms / 1e3), ms
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf


def rmvpe_incumbent(wav, dev, half: bool, reps: int = 3):
    """The eager-PyTorch incumbent of the f0 estimator on the same GPU: the oracle's functional form of lib/rmvpe.py (cuDNN
    convolutions) with a `torch.nn.GRU` holding the same weights (cuDNN GRU, what the reference's `nn.GRU` runs), fp16 (`is_half`)
    or fp32 with TF32 off.  Returns (ms per call, salience [frames, 360] fp32 on the host).  Measurement context only."""
    from oracle import rmvpe_oracle as ro
    tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dt = torch.float16 if half else torch.float32
        sd = synthetic.make_rmvpe_state_dict(0)
        gru = torch.nn.GRU(384, 256, num_layers=1, batch_first=True, bidirectional=True)
        gru.load_state_dict({k[len("fc.0.gru."):]: v for k, v in sd.items() if k.startswith("fc.0.gru.")})
        gru = gru.to(dev, dt).eval()
        sd_dev = {k: v.to(dev) for k, v in sd.items()}
        ro._BASIS_CACHE["basis"] = ro.stft_forward_basis().to(dev)
        ro._BASIS_CACHE["mel"] = torch.from_numpy(ro.mel_filterbank()).float().to(dev)

        def call():
            with torch.no_grad():
                mel = ro.log_mel(torch.from_numpy(wav).float().to(dev)[None])
                n = mel.shape[-1]
                mel = torch.nn.functional.pad(mel, (0, min(32 * ((n - 1) // 32 + 1) - n, n)), mode="reflect")
                return ro.e2e_forward(sd_dev, mel.to(dt), gru=lambda x: gru(x)[0], dtype=dt)[0, :n].float().cpu().numpy()

        for _ in range(2):
            call()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            hid = call()
        e1.record()
        torch.cuda.synchronize(dev)
        ro._BASIS_CACHE.clear()
        del gru, sd_dev
        torch.cuda.empty_cache()
        return e0.elapsed_time(e1) / reps, hid
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf


def parity_block(net, cfg, T: int, precision: str, config_name: str):
    """One more step of the timed workload with the fixture's seeded noise injected (the timed steps draw theirs on the
    device like the reference, so their waveforms are not comparable sample by sample), checked OUTSIDE the timed region
    against the waveform the unmodified reference produced for this step in the build container
    (tests/golden/g2_48k_v2_T6000.npz, minted by tests/golden/make_golden_big.py)."""
    path = os.path.join(ROOT, "tests", "golden", "g2_48k_v2_T6000.npz")
    if config_name != "48k_v2" or T != 6000 or not os.path.exists(path):
        return {"checked": False, "why": "the reference-minted fixture covers the default workload only (48k_v2, T=6000)"}
    gold = np.load(path, allow_pickle=True)
    inputs = synthetic.make_inputs(cfg, 1, T, seed=int(gold["meta"][6]))
    noise = synthetic.draw_noise(cfg, 1, T, seed=int(gold["meta"][7]))
    dev = net._device
    o = net.infer(*[t.to(dev) for t in inputs], noise=noise)[0][0, 0].cpu().numpy()
    i16 = gold["o_i16"][0].astype(np.float64)
    ref = (i16 + 0.5 * np.sign(i16)) * float(gold["audio_max"][0]) / 32768.0       # mid-point of the truncation step
    d = np.abs(synthetic.to_int16(o).astype(np.int32) - gold["o_i16"][0].astype(np.int32))
    gate = "int16 within +-1 LSB" if precision == "fp32" else "SNR >= 45 dB"
    snr = synthetic.snr_db(ref, o)
    ok = bool(d.max() <= 1) if precision == "fp32" else bool(snr >= 45.0)
    return {"checked": True, "against": "tests/golden/g2_48k_v2_T6000.npz (unmodified reference, fp32 CPU, same weights / inputs / noise)",
            "snr_db": snr, "int16_max_lsb_diff": int(d.max()), "int16_frac_differing": float((d > 0).mean()),
            "gate": gate, "pass": ok, "samples": int(o.shape[0])}


def measured_traffic(precision: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel class from the committed ncu capture of this
    build (profiles/r2_dram_traffic.json, written by tools/ncu_traffic.py from `ncu --metrics dram__bytes_*` over one
    step of this command); None if no capture exists for the precision."""
    p = os.path.join(ROOT, "profiles", "r2_dram_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p)).get(precision)
    return d


_REAL_STDOUT = None


DUMP_BUDGET_BYTES = 64_000_000


def dump_outputs(out_dir: str, outs):
    """Writes what one `infer()` returned -- `(o, x_mask, (z, z_p, m_p, logs_p))` -- as `out_dir/<name>.npy` in float32, so
    two builds run with the same arguments can be compared array for array.  Above 64 MB in all, every array keeps the same
    fixed, seeded sample of its flattened elements."""
    o, x_mask, (z, z_p, m_p, logs_p) = outs
    arrays = {"audio": o, "x_mask": x_mask, "z": z, "z_p": z_p, "m_p": m_p, "logs_p": logs_p}
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    keep = min(1.0, DUMP_BUDGET_BYTES / sum(a.size * 4 for a in arrays.values()))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def claim_stdout():
    """stdout carries exactly ONE JSON line: everything libraries print there (NCCL's version banner under
    NCCL_DEBUG=VERSION, warnings of child tools) is sent to stderr for the lifetime of the process."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["fp32", "fp16", "bf16"],
                    help="bf16 (default; BASELINE north_star's tensor path, SNR >= 45 dB gate), fp16 (the reference's own GPU "
                         "dtype, same speed, ~61 dB) or fp32 (CUDA-core path, +-1 LSB gate)")
    ap.add_argument("--config", default="48k_v2")
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--cpu-frames", type=int, default=0,
                    help="frames per step of the CPU arms (default 0 = the full step, same T as the product arm)")
    ap.add_argument("--cpu-1thread-frames", type=int, default=500, help="frames of the bounded 1-thread CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-incumbent", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-front-end", action="store_true")
    ap.add_argument("--no-extra-precision", action="store_true", help="skip the fp16 leg beside the bf16 headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step's infer() returned as DIR/<name>.npy (float32, at most 64 MB in all; "
                         "under torchrun, rank 0's outputs only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    cfg = NAMED_CONFIGS[args.config]
    T = int(round(args.seconds * 100))
    audio_s = T * cfg.upp / cfg.sr
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = f"{args.config} SynthesizerTrnMs{cfg.feat_dim}NSFsid.infer, B=1, T={T} frames ({audio_s:.0f} s segment) per GPU"
    metric = "seconds of output audio synthesised per second (RTF^-1)"
    # the SAME dict in both arms (the driver compares them): it names the workload only
    config = {"workload": workload, "parallelism": f"segments x{world}, no collective",
              "l2": "no flush needed: each step streams >1 GB of stage activations (>> 126 MB L2)"}
    cpu_T = args.cpu_frames if args.cpu_frames > 0 else T

    # ------------------------------------------------------------------ reference arm (CPU) -------
    if args.impl == "reference":
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        steps, warm = args.steps, max(0, args.warmup)
        # every step is the product arm's step: one full infer() of T frames on all host cores (oracle port, fp32).
        # EXACTLY `steps` timed steps after `warm` untimed ones; value = audio produced / total time of the K steps
        chk = {}
        _, sample_s, times = cpu_oracle_rate(cfg, cpu_T, steps, warm, threads, check=chk)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, chk["last_timed"])
        rate = steps * sample_s / float(np.sum(times))
        sample = (f"oracle/rvc_oracle.py (fp32 PyTorch CPU restatement of the reference infer), {cpu_T} frames = {sample_s:.1f} s "
                  f"audio per step" + (" = the full step" if cpu_T == T else " (bounded sample of the step)"))
        line = {
            "impl": "reference", "metric": metric, "value": rate, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": float(np.mean(times)) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "timed_sample": sample,
            "cpu_baseline": {"value": rate, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        pin = oracle_vs_fixture(chk.get("first_timed_output"), args.config, cpu_T)
        if pin:
            line["oracle_vs_reference_fixture"] = pin
        emit(line)
        return

    # ------------------------------------------------------------------ product arm (CUDA) --------
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    import comfy_rvc_b200 as rvc
    from comfy_rvc_b200 import _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    sd = synthetic.make_state_dict(cfg)
    cls = rvc.SynthesizerTrnMs256NSFsid if cfg.feat_dim == 256 else rvc.SynthesizerTrnMs768NSFsid
    net = cls(*cfg.to_positional(), is_half=args.precision != "fp32")
    del net.enc_q
    net.load_state_dict({k: v.half() for k, v in sd.items()}, strict=False)
    net.eval().to(dev).set_precision(args.precision)

    phone, lens, pitch, pitchf, sid = synthetic.make_inputs(cfg, 1, T, seed=1 + rank)
    host = [t.pin_memory() for t in (phone, lens, pitch, pitchf, sid)]
    devin = [t.to(dev) for t in host]
    torch.manual_seed(1234 + rank)
    lib = _lib.load()

    def step_resident():
        return net.infer(*devin)             # draws its noise with torch on the device, like the reference

    # the warm-up holds each step's outputs until the next step returns, as the timed loop does, so the allocator
    # already has blocks for both when the timed region starts
    for _ in range(max(3, args.warmup)):
        outs = step_resident()
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        for _ in range(8):                   # keep the GPU under load until nvidia-smi has delivered its first samples
            step_resident()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        outs = step_resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    del outs
    launches = net.last_launches * args.steps
    graph_replay = bool(getattr(net, "last_graph_replay", False))   # the timed steps ran as replays of the captured step
    # per-class kernel times: a second pass of the same K steps with a CUDA-event pair around every launch (the event
    # records sit between kernels and serialise their programmatic dependent launches, so they stay out of `value`)
    lib.rvcb200_profile_enable(net._ctx, 1)
    keep_graph, net.graph_max_frames = net.graph_max_frames, 0     # a replayed graph has no per-launch events
    for _ in range(args.steps):
        step_resident()
    torch.cuda.synchronize()
    net.graph_max_frames = keep_graph
    cls_ms = (C.c_double * 8)()
    cls_n = (C.c_int64 * 8)()
    lib.rvcb200_profile_collect(net._ctx, cls_ms, cls_n)
    lib.rvcb200_profile_enable(net._ctx, 0)

    # end-to-end through the public API with host buffers: every step copies its inputs from pinned host memory and its PCM
    # back.  The driver is pipelined the way a serving loop would be: inputs of step i+1 travel on a copy stream while step i
    # computes, the PCM of step i-1 leaves on another; the synthesizer itself runs on the current stream.
    out_host = torch.empty(1, 1, T * cfg.upp, dtype=torch.float32).pin_memory()
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    cur = torch.cuda.current_stream(dev)

    # two preallocated sets of device input buffers (no allocator traffic in the loop): set k is refilled on the copy
    # stream as soon as the step that last read it has finished
    dev_in = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host] for _ in range(2)]
    read_done = [None, None]

    def fetch(i):
        k = i % 2
        with torch.cuda.stream(s_in):
            if read_done[k] is not None:
                s_in.wait_event(read_done[k])
            for d, h in zip(dev_in[k], host):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(s_in)
        return dev_in[k], ev

    def run_e2e(n, stamps=None):
        nxt = fetch(0)
        for i in range(n):
            ins, ev = nxt
            cur.wait_event(ev)
            nxt = fetch(i + 1)                         # H2D of the next step's inputs overlaps this step's kernels
            o = net.infer(*ins)[0]
            done = torch.cuda.Event(enable_timing=stamps is not None)
            done.record(cur)
            if stamps is not None:
                stamps.append(done)
            read_done[i % 2] = done
            s_out.wait_event(done)
            with torch.cuda.stream(s_out):
                out_host.copy_(o, non_blocking=True)   # D2H of this step's PCM overlaps the next step's kernels
            o.record_stream(s_out)
        cur.wait_stream(s_out)
        cur.wait_stream(s_in)
        read_done[0] = read_done[1] = None

    # warm-up: lets the caching allocator reach its steady set of blocks.  At least as many iterations as the timed region: since the
    # step replays from a CUDA graph the host runs the whole region ahead of the GPU, every step's output tensors are live at once
    # (record_stream), and a shorter warm-up left cudaMalloc calls inside the timed region (seen as one ~50 ms stall in 2 of 12 runs)
    run_e2e(max(max(3, args.warmup) + 3, args.steps + 2))
    barrier()
    f0_, f1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0_.record()
    e2e_stamps = []
    run_e2e(args.steps, e2e_stamps)
    f1_.record()
    barrier()
    ms_e2e = f0_.elapsed_time(f1_)
    # per-step completion times of the same K steps (diagnostic: a single stalled step shows up as max >> median)
    e2e_step_ms = [f0_.elapsed_time(e2e_stamps[0])] + [e2e_stamps[i - 1].elapsed_time(e2e_stamps[i]) for i in range(1, len(e2e_stamps))]
    clocks = sampler.stop() if sampler else None

    if dist is not None:
        print(f"rank {rank}: {ms / args.steps:.3f} ms/step resident, {ms_e2e / args.steps:.3f} ms/step end to end", file=sys.stderr)
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    value = world * args.steps * audio_s / (ms / 1e3)
    e2e_value = world * args.steps * audio_s / (ms_e2e / 1e3)
    macs = algorithmic_macs(cfg, T)
    conv_flops = 2.0 * macs["resblocks"]                      # class 0: the dominant kernel (decoder resblock convs)
    conv_ms_per_launch = cls_ms[0] / max(cls_n[0], 1)
    conv_launches_per_step = cls_n[0] / args.steps
    peaks = load_peaks()
    achieved = conv_flops / conv_launches_per_step / (conv_ms_per_launch * 1e-3) / 1e12
    rb_rd, rb_wr = resblock_bytes(cfg, T)
    rb_bytes = (rb_rd + rb_wr) / max(conv_launches_per_step, 1)
    tr = measured_traffic(args.precision)
    h2d = sum(t.numel() * t.element_size() for t in host)
    line = {
        "metric": metric, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "fp16": "f16 operands, f32 accumulate", "bf16": "bf16 operands (resblocks) / f16 operands (ladder, encoder, flow), f32 accumulate"}[args.precision],
        "data": "synthetic (seeded random-init weights stored as fp16, N(0,1) features, contour f0)",
        "config": config, "precision": args.precision,
        "roofline_pass": "per-launch CUDA events in a second pass of the same K steps (kept out of `value`)",
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": T * cfg.upp * 4,
                "ms_per_step": ms_e2e / args.steps,
                "step_ms_median": sorted(e2e_step_ms)[len(e2e_step_ms) // 2], "step_ms_max": max(e2e_step_ms)},
        "gpu_launches": int(launches),
        "launch_mode": ("CUDA graph replay of the step captured during warm-up (synthesizer.py: shapes seen before); gpu_launches = its kernel nodes"
                        if graph_replay else "stream launches"),
        "roofline": {"bound": "tensor", "kernel": "decoder resblock convolutions (rbconv_tc_kernel + fused-pair rbpair_tc_kernel on tcgen05; conv_f32_kernel in fp32 mode)",
                     "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                     "traffic": (tr["bytes_per_step"] / tr["launches_per_step"]) if tr else None,
                     "traffic_source": (tr["source"] if tr else "no ncu capture committed for this precision"),
                     "peak_burst": peaks["burst"], "frac_of_burst": achieved / peaks["burst"],
                     "algorithmic_bytes_per_launch": rb_bytes, "achieved_hbm_gbs": rb_bytes / (conv_ms_per_launch * 1e-3) / 1e9,
                     "hbm_peak_gbs": peaks["hbm_gbs"], "hbm_frac": rb_bytes / (conv_ms_per_launch * 1e-3) / 1e9 / peaks["hbm_gbs"],
                     "peak_source": peaks["src"],
                     "launches_per_step": conv_launches_per_step, "avg_launch_ms": conv_ms_per_launch,
                     "algorithmic_gflop_per_step": conv_flops / 1e9,
                     "share_of_step": cls_ms[0] / max(sum(cls_ms), 1e-9)},
        "time_by_class_ms_per_step": {"dec_resblocks": cls_ms[0] / args.steps, "attention": cls_ms[1] / args.steps,
                                      "sine_source": cls_ms[2] / args.steps, "glue": cls_ms[3] / args.steps,
                                      "dec_pre_ups": cls_ms[4] / args.steps, "flow": cls_ms[5] / args.steps,
                                      "enc_linear": cls_ms[6] / args.steps},
        "algorithmic_gflop_per_step": {k: 2.0 * v / 1e9 for k, v in macs.items()},
        "clocks": clocks,
    }
    if not args.no_parity:
        line["parity"] = parity_block(net, cfg, T, args.precision, args.config)
    if world == 1 and args.precision == "bf16" and not args.no_extra_precision:
        # the drop-in's own default for `is_half` checkpoints is fp16 operands (the reference's GPU dtype): same K steps
        net.set_precision("fp16")
        for _ in range(max(3, args.warmup)):
            step_resident()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            step_resident()
        g1.record()
        torch.cuda.synchronize()
        ms16 = g0.elapsed_time(g1)
        line["fp16"] = {"value": args.steps * audio_s / (ms16 / 1e3), "unit": "audio-s/s", "ms_per_step": ms16 / args.steps,
                        "note": "set_precision('fp16'): what get_vc(is_half=True) selects; device-resident inputs like `value`"}
        if not args.no_parity:
            line["fp16"]["parity"] = parity_block(net, cfg, T, "fp16", args.config)
        net.set_precision(args.precision)
    if world == 1 and not args.no_front_end:
        # the step in front of the synthesizer in the real node (SURVEY.md §8f rank 3): HuBERT / ContentVec features of the
        # same 60 s of 16 kHz audio on the same kernels (comfy_rvc_b200.HubertB200), device-resident input; context for how
        # a whole VC.vc segment divides between front end and synthesis -- not part of `value`
        try:
            from comfy_rvc_b200.hubert import HubertB200
            hub = HubertB200(synthetic.HUBERT_BASE, synthetic.make_hubert_state_dict(0), dev)
            src = synthetic.make_speech(audio_s, seed=1).to(dev)
            for _ in range(3):
                hub.extract_features(version="v2", source=src)
            torch.cuda.synchronize()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(args.steps):
                hub.extract_features(version="v2", source=src)
            h1.record()
            torch.cuda.synchronize()
            hms = h0.elapsed_time(h1) / args.steps
            line["front_end"] = {"what": "HubertB200.extract_features(v2) on the segment's 16 kHz audio", "ms_per_segment": hms,
                                 "audio_s_per_s": audio_s / (hms / 1e3), "launches": hub.last_launches,
                                 "segment_ms_front_end_plus_synthesis": hms + ms / args.steps}
            del hub, src
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            line["front_end"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        # ... and the other model in front of it (SURVEY.md §8f rank 4): RMVPE f0 of the same audio (comfy_rvc_b200.RMVPE),
        # host audio in, host f0 out like the reference's `infer_from_audio`
        try:
            from comfy_rvc_b200.rmvpe import RMVPE
            rm = RMVPE(synthetic.make_rmvpe_state_dict(0), is_half=True, device=dev)
            wav = synthetic.make_speech(audio_s, seed=1)[0].numpy()
            for _ in range(3):
                rm.infer_from_audio(wav)
            torch.cuda.synchronize()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(args.steps):
                rm.infer_from_audio(wav)
            h1.record()
            torch.cuda.synchronize()
            rms = h0.elapsed_time(h1) / args.steps
            line["f0_front_end"] = {"what": "RMVPE.infer_from_audio on the segment's 16 kHz audio (host in, host out)",
                                    "ms_per_segment": rms, "audio_s_per_s": audio_s / (rms / 1e3), "launches": rm.last_launches}
            if not args.no_gpu_incumbent:
                taps = {}
                rm.infer_from_audio(wav, taps=taps)
                ours = taps["hidden"].cpu().numpy().astype(np.float64)
                lg = lambda q: np.log(np.clip(q, 1e-7, 1 - 1e-7)) - np.log1p(-np.clip(q, 1e-7, 1 - 1e-7))
                ms32, ref = rmvpe_incumbent(wav, dev, False)
                ms16, h16 = rmvpe_incumbent(wav, dev, True)
                line["f0_front_end"]["gpu_incumbent"] = {
                    "fp32_tf32_off_ms": ms32, "fp16_ms": ms16, "logit_snr_db_vs_incumbent_fp32": synthetic.snr_db(lg(ref), lg(ours)),
                    "incumbent_fp16_logit_snr_db": synthetic.snr_db(lg(ref), lg(h16)),
                    "what": "the same network in eager PyTorch on this GPU (oracle/rmvpe_oracle.py's functional form + torch.nn.GRU)"}
            del rm
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            line["f0_front_end"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    if world == 1 and not args.no_gpu_incumbent:
        inc = {}
        for name, half in (("fp16", True), ("fp32_tf32_off", False)):
            try:
                v, ms_i = gpu_incumbent_rate(cfg, T, dev, half)
                inc[name] = {"value": v, "unit": "audio-s/s", "ms_per_step": ms_i}
            except Exception as e:                      # e.g. out of memory on a smaller part: report, do not fail the line
                inc[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        inc["what"] = ("eager PyTorch (cuDNN/cuBLAS) on this GPU: oracle/rvc_oracle.py, the reference's op sequence, on CUDA "
                       "tensors, same step, 3 timed reps after 2 warm-ups; measurement context only, never on the product path")
        line["gpu_incumbent"] = inc
    if world == 1 and not args.no_cpu_baseline:        # the CPU leg is timed at N = 1 only (rank 0's host cores)
        threads = os.cpu_count() or 1
        # all host cores on the FULL step (one timed step after a short warm-up step), and one thread on a bounded sample
        chk = {}
        rate, sample_s, _ = cpu_oracle_rate(cfg, cpu_T, 1, 1, threads, warmup_T=min(200, cpu_T), check=chk)
        n1 = min(args.cpu_1thread_frames, cpu_T)
        rate1, sample1_s, _ = cpu_oracle_rate(cfg, n1, 1, 1, 1, warmup_T=min(100, n1))
        line["cpu_baseline"] = {"value": rate, "unit": "audio-s/s", "cores": threads, "kind": "port",
                                "sample": f"oracle/rvc_oracle.py fp32 PyTorch CPU, {cpu_T} frames = {sample_s:.1f} s audio"
                                          + (" (the full step)" if cpu_T == T else "") + ", one timed step",
                                "one_thread": {"value": rate1, "unit": "audio-s/s", "cores": 1,
                                               "sample": f"{n1} frames = {sample1_s:.1f} s audio, one timed step"}}
        pin = oracle_vs_fixture(chk.get("first_timed_output"), args.config, cpu_T)
        if pin:
            line["cpu_baseline"]["oracle_vs_reference_fixture"] = pin
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
