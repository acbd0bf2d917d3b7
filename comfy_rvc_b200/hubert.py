"""HuBERT / ContentVec feature extractor on the B200 kernels (SURVEY.md §8f rank 3: the step in front of the synthesis path).

Drop-in for the reference's `HubertModelWithFinalProj` (/root/reference/lib/infer_pack/loaders.py:10-61), which is
HuggingFace `transformers.HubertModel` (base architecture) + a `final_proj` Linear:

    model = HubertB200.from_safetensors(path, device)          # or HubertB200(config_dict, state_dict, device)
    feats = model.extract_features(version=version, source=audio16k[1, n], padding_mask=..., output_layer=...)

as called by `VC.vc` (/root/reference/vc_infer_pipeline.py:48-55): v1 -> 9th hidden state + final_proj (256-d), v2 -> 12th
hidden state (768-d); the reference indexes `hidden_states[output_layer - 1]` (loaders.py:56), so 8 / 11 encoder layers
run.  State-dict keys are HuggingFace's (what `content-vec-best.safetensors` holds).

Host code is Python like the reference's; every FLOP runs in librvcb200.so through the C ABI (include/rvcb200.h):
  * feature encoder layer 0 (1 -> 512, k 10, stride 5) + GroupNorm + GELU: `rvcb200_op_hubert_conv0` (hubert_kernels.cu);
  * layers 1-6 (512 -> 512, k 3 / 2, stride 2): a stride-2 convolution over [L][512] is a stride-1 convolution over the
    same memory viewed as [L/2][1024] -- two taps for k = 3 (the second tap's upper half is zero), one for k = 2 -- so they
    run on the generic tcgen05 implicit-GEMM kernel (`rvcb200_op_conv_tc`, GELU in the epilogue);
  * LayerNorms: `rvcb200_op_layernorm16`; projections / feed-forward / q|k|v / out: `rvcb200_op_conv_tc` (1 tap);
  * positional convolution (k 128, 16 groups of 48 channels): one 128-tap launch, an N tile per group that reads its own 48
    input channels (`a_nt_stride`; K = 48 meets the zero K padding of the weight image), GELU + residual in the epilogue;
  * attention: `rvcb200_op_attention_tc` (flash-style tcgen05 kernel of the text encoder) with 12 heads of 64 channels
    laid out in its 128-channel-per-head operand format, relative-position tables zero.
There is no PyTorch or CPU fallback: without the extension or a CUDA device `extract_features` raises.
"""
from __future__ import annotations

import ctypes as C
import json
import math
from typing import Dict, Optional

import torch

from . import _lib
from .weights import pack_tc

PADF = 32            # conv_tc.cuh kPadF (unused by the channels-last generic path, but part of the descriptor)
HEAD_PAD = 128       # channels per head in the attention operand layout (attention_tc.cu DKP)
HEAD_OUT = 96        # channels per head in the attention output (attention_tc.cu DKV)


def _cfg_get(cfg, key, default=None):
    return cfg.get(key, default) if isinstance(cfg, dict) else getattr(cfg, key, default)


class HubertB200:
    """See module docstring.  `config`: dict or object with HuggingFace HubertConfig fields."""

    def __init__(self, config, state_dict: Dict[str, torch.Tensor], device="cuda:0"):
        g = lambda k, d=None: _cfg_get(config, k, d)
        self.hidden, self.n_layers, self.n_heads = int(g("hidden_size")), int(g("num_hidden_layers")), int(g("num_attention_heads"))
        self.inter = int(g("intermediate_size"))
        self.conv_dim, self.conv_kernel, self.conv_stride = tuple(g("conv_dim")), tuple(g("conv_kernel")), tuple(g("conv_stride"))
        self.kpos, self.gpos = int(g("num_conv_pos_embeddings")), int(g("num_conv_pos_embedding_groups"))
        self.eps = float(g("layer_norm_eps", 1e-5))
        self.proj_size = int(g("classifier_proj_size", 256))
        dk = self.hidden // self.n_heads
        ok = (g("feat_extract_norm", "group") == "group" and not g("do_stable_layer_norm", False) and not g("conv_bias", False)
              and g("feat_extract_activation", "gelu") == "gelu" and g("hidden_act", "gelu") == "gelu"
              and g("feat_proj_layer_norm", True) and not g("conv_pos_batch_norm", False)
              and len(set(self.conv_dim)) == 1 and self.conv_dim[0] % 64 == 0 and self.conv_kernel[0] <= 16
              and all(s == 2 and k in (2, 3) for k, s in zip(self.conv_kernel[1:], self.conv_stride[1:]))
              and dk <= HEAD_OUT and dk % 8 == 0 and self.kpos == 128 and self.hidden % self.gpos == 0
              and (self.hidden // self.gpos) % 16 == 0 and self.hidden <= 1024)
        if not ok:
            raise ValueError("HubertB200 is built for the HuBERT-base / ContentVec architecture (group-norm feature encoder, "
                             "post-norm encoder, 128-tap grouped positional convolution)")
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", 0)
        self._sd = {k: v.detach().to("cpu", torch.float32) for k, v in state_dict.items()}
        need = ["feature_projection.projection.weight", "encoder.layer_norm.weight", "final_proj.weight"]
        missing = [k for k in need if k not in self._sd]
        if missing:
            raise RuntimeError(f"missing keys in state_dict: {missing}")
        self._w: Optional[Dict[str, torch.Tensor]] = None
        self.last_launches = 0
        self.rng_draws_per_call = self.n_layers       # global-generator draws of one reference forward (see extract_features)

    # ---- reference loader protocol (loaders.py:21-32) ------------------------------------------------------------
    @staticmethod
    def from_safetensors(path: str, device="cuda:0", framework="pt") -> "HubertB200":
        from safetensors import safe_open
        assert path.endswith(".safetensors"), f"{path} must end with '.safetensors'"
        with safe_open(path, framework=framework, device="cpu") as f:
            metadata = f.metadata()
            sd = {key: f.get_tensor(key) for key in f.keys()}
        return HubertB200(json.loads(metadata["config"]), sd, device)

    def eval(self):
        return self

    def to(self, device=None, *a, **k):
        if device is not None and not isinstance(device, torch.dtype):
            dev = torch.device(device)
            if dev.type == "cuda" and dev.index is None:
                dev = torch.device("cuda", 0)
            if dev != self.device:
                self.device, self._w = dev, None
        return self

    def half(self):
        return self

    def float(self):
        return self

    # ---- weights -> device images ------------------------------------------------------------------------------------
    def _materialize(self):
        if self._w is not None:
            return
        if not torch.cuda.is_available() or self.device.type != "cuda":
            raise RuntimeError("comfy_rvc_b200.HubertB200 needs a CUDA (sm_100a) device; it has no CPU fallback")
        _lib.load()
        sd, dev, H = self._sd, self.device, self.hidden
        W: Dict[str, torch.Tensor] = {}
        f32 = lambda t: t.to(dev, torch.float32).contiguous()
        img = lambda w, n: pack_tc(w, torch.float16, n).to(dev)          # [taps][C_in][C_out] -> tcgen05 weight image
        self._src: Dict[str, torch.Tensor] = {}                          # fp32 sources of the re-tileable projections

        def proj(name, w):                                               # image for the default N = 64; others on demand
            self._src[name] = w.contiguous()
            return img(w, 64)
        C0 = self.conv_dim[0]
        W["conv0.w"] = f32(sd["feature_extractor.conv_layers.0.conv.weight"][:, 0, :])               # [C][K]
        W["conv0.gn_w"] = f32(sd["feature_extractor.conv_layers.0.layer_norm.weight"])
        W["conv0.gn_b"] = f32(sd["feature_extractor.conv_layers.0.layer_norm.bias"])
        W["zeros"] = torch.zeros(max(4 * H, self.inter, 3 * self.n_heads * HEAD_PAD), device=dev)
        for i in range(1, len(self.conv_kernel)):
            w = sd[f"feature_extractor.conv_layers.{i}.conv.weight"]                                  # [C_out][C_in][k]
            k = w.shape[2]
            taps = torch.zeros(2 if k == 3 else 1, 2 * C0, C0)
            taps[0, :C0], taps[0, C0:] = w[:, :, 0].t(), w[:, :, 1].t()                               # rows 2t, 2t+1
            if k == 3:
                taps[1, :C0] = w[:, :, 2].t()                                                         # row 2t+2
            W[f"conv{i}.w"] = img(taps, 256)
        W["fp.ln_w"], W["fp.ln_b"] = f32(sd["feature_projection.layer_norm.weight"]), f32(sd["feature_projection.layer_norm.bias"])
        W["fp.w"] = proj("fp.w", sd["feature_projection.projection.weight"].t()[None])
        W["fp.b"] = f32(sd["feature_projection.projection.bias"])
        p = "encoder.pos_conv_embed.conv."
        if p + "parametrizations.weight.original0" in sd:
            wpos = torch._weight_norm(sd[p + "parametrizations.weight.original1"], sd[p + "parametrizations.weight.original0"], 2)
        elif p + "weight_g" in sd:
            wpos = torch._weight_norm(sd[p + "weight_v"], sd[p + "weight_g"], 2)
        else:
            wpos = sd[p + "weight"]
        cg = H // self.gpos
        # grouped convolution as ONE launch: N tile gi = group gi (its cg output channels), which reads input channels
        # [gi * cg, + cg) (`a_nt_stride`): the image is [128 taps][cg in][H out] with N = cg
        W["pos.w"] = img(wpos.permute(2, 1, 0).contiguous(), cg)
        W["pos.b"] = f32(sd[p + "bias"])
        W["enc.ln_w"], W["enc.ln_b"] = f32(sd["encoder.layer_norm.weight"]), f32(sd["encoder.layer_norm.bias"])
        nh, dk = self.n_heads, H // self.n_heads
        for l in range(self.n_layers):
            q = f"encoder.layers.{l}."
            wq = torch.zeros(H, 3 * nh * HEAD_PAD)
            bq = torch.zeros(3 * nh * HEAD_PAD)
            for pi, n in enumerate(("q_proj", "k_proj", "v_proj")):
                wn, bn = sd[q + f"attention.{n}.weight"].t(), sd[q + f"attention.{n}.bias"]          # [in][out]
                sc = dk ** -0.5 if pi == 0 else 1.0                                                    # HubertAttention scaling
                for h in range(nh):
                    c0 = (pi * nh + h) * HEAD_PAD
                    wq[:, c0:c0 + dk] = wn[:, h * dk:(h + 1) * dk] * sc
                    bq[c0:c0 + dk] = bn[h * dk:(h + 1) * dk] * sc
            W[f"l{l}.qkv.w"], W[f"l{l}.qkv.b"] = proj(f"l{l}.qkv.w", wq[None]), f32(bq)
            wo = torch.zeros(nh * HEAD_OUT, H)
            wt = sd[q + "attention.out_proj.weight"].t()                                               # [in][out]
            for h in range(nh):
                wo[h * HEAD_OUT:h * HEAD_OUT + dk] = wt[h * dk:(h + 1) * dk]
            W[f"l{l}.o.w"], W[f"l{l}.o.b"] = proj(f"l{l}.o.w", wo[None]), f32(sd[q + "attention.out_proj.bias"])
            W[f"l{l}.ln1_w"], W[f"l{l}.ln1_b"] = f32(sd[q + "layer_norm.weight"]), f32(sd[q + "layer_norm.bias"])
            W[f"l{l}.ff1.w"] = proj(f"l{l}.ff1.w", sd[q + "feed_forward.intermediate_dense.weight"].t()[None])
            W[f"l{l}.ff1.b"] = f32(sd[q + "feed_forward.intermediate_dense.bias"])
            W[f"l{l}.ff2.w"] = proj(f"l{l}.ff2.w", sd[q + "feed_forward.output_dense.weight"].t()[None])
            W[f"l{l}.ff2.b"] = f32(sd[q + "feed_forward.output_dense.bias"])
            W[f"l{l}.ln2_w"], W[f"l{l}.ln2_b"] = f32(sd[q + "final_layer_norm.weight"]), f32(sd[q + "final_layer_norm.bias"])
        W["final.w"] = img(sd["final_proj.weight"].t()[None], 64)
        W["final.b"] = f32(sd["final_proj.bias"])
        W["ek0"] = torch.zeros(32, 128, dtype=torch.float16, device=dev)     # no relative-position terms in HuBERT
        W["evt0"] = torch.zeros(128, 64, dtype=torch.float16, device=dev)
        self._w = W

    # ---- one generic tcgen05 contraction -----------------------------------------------------------------------------
    def _gemm(self, x16, L_in, Cin, w16, bias, Cout, Lj, *, ntaps=1, g_off=0, n_tile=64, ldx16=0, gelu=False, y16=None,
              ldy16=0, y32=None, ldy32=0, res32=None, ldr32=0, a_nt_stride=0):
        d = _lib.TcConvDesc()
        d.x16, d.L_in, d.padf = x16, L_in, PADF
        d.w16, d.bias = w16.data_ptr(), bias.data_ptr()
        d.Cin, d.ntaps, d.dil, d.G = Cin, ntaps, 1, 1
        d.g_off[0] = g_off
        d.N, d.Cout_total = n_tile, Cout
        d.Lj, d.out_stride, d.Lp_out = Lj, 1, ((Lj + 127) // 128) * 128 + 128
        d.div, d.out_slope, d.alpha, d.pre_slope = 1.0, 1.0, 1.0, 1.0
        d.generic, d.f32_cl, d.ldx16 = 1, 1, ldx16
        d.gelu = 1 if gelu else 0
        d.a_nt_stride = a_nt_stride
        if y16 is not None:
            d.y16, d.ldy16 = y16, ldy16
        if y32 is not None:
            d.y32, d.ldy32 = y32, ldy32
        if res32 is not None:
            d.res32, d.ldr32, d.res_mode = res32, ldr32, 1
        st = _lib.load().rvcb200_op_conv_tc(C.byref(d), 1, self._stream)
        if st != 0:
            raise RuntimeError(f"rvcb200_op_conv_tc failed with status {st} (Cin={Cin}, Cout={Cout}, taps={ntaps}, rows={Lj})")
        self.last_launches += 1

    def _tiled(self, name, rows, Cout):
        """(weight image, N tile) for a projection of `rows` x `Cout` outputs: the widest N in {256, 128, 64} that still
        yields a full wave of 128-row tiles (>= 132 CTAs) -- a wide tile re-reads the activation rows from L2 fewer times
        (N = 64: every 128 x K block is fetched C_out / 64 times); short inputs keep N = 64 to occupy more SMs."""
        mt = (rows + 127) // 128
        n = 64
        for cand in (256, 128):
            if Cout % cand == 0 and mt * (Cout // cand) >= 132:
                n = cand
                break
        if n == 64:
            return self._w[name], 64
        key = f"{name}@{n}"
        if key not in self._w:
            self._w[key] = pack_tc(self._src[name], torch.float16, n).to(self.device)
        return self._w[key], n

    def _ln(self, x32, gw, gb, y32, y16, rows, Cn):
        st = _lib.load().rvcb200_op_layernorm16(C.c_void_p(x32.data_ptr()), C.c_void_p(gw.data_ptr()), C.c_void_p(gb.data_ptr()),
                                                C.c_void_p(y32.data_ptr()), C.c_void_p(y16.data_ptr()), rows, Cn, self.eps,
                                                self._stream)
        if st != 0:
            raise RuntimeError(f"rvcb200_op_layernorm16 failed with status {st}")
        self.last_launches += 1

    # ---- the forward ------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def extract_features(self, source: torch.Tensor = None, version: str = "v2", padding_mask=None, output_layer=None, **kwargs):
        """loaders.py:52-61: [1, n] 16 kHz audio -> [1, frames, 256 (v1) | 768 (v2)] in `source.dtype`."""
        if source is None:
            raise TypeError("extract_features() needs `source`")
        if source.dim() != 2 or source.shape[0] != 1:
            raise ValueError("HubertB200.extract_features handles one utterance per call ([1, n]), like the reference pipeline")
        self._materialize()
        lib, W, dev, H = _lib.load(), self._w, self.device, self.hidden
        # Side effect of the reference kept on purpose: HuggingFace's HubertEncoder draws `torch.rand([])` from the GLOBAL CPU generator
        # once per encoder layer on every forward, training or not (its LayerDrop test).  `VC.vc` draws the synthesizer's noise from
        # the same generator right afterwards (models.py:801), so a drop-in that skipped these draws would produce a different --
        # equally valid, but not the reference's -- noise stream after `torch.manual_seed` (tests/test_pipeline_gpu.py, fixture p4).
        for _ in range(self.rng_draws_per_call):
            torch.rand([])
        n = int(source.shape[1])
        if n < self.conv_kernel[0]:
            raise RuntimeError(f"input of {n} samples is shorter than the feature encoder's first kernel")
        n_layers = (9 if version == "v1" else 12) - 1                        # hidden_states[output_layer - 1]
        if n_layers > self.n_layers:
            raise ValueError("model has fewer encoder layers than the requested output layer")
        self.last_launches = 0
        with torch.cuda.device(dev):
            self._stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            x = source.to(dev, torch.float32).contiguous()
            C0 = self.conv_dim[0]
            K0, S0 = self.conv_kernel[0], self.conv_stride[0]
            L = (n - K0) // S0 + 1
            pad_rows = lambda r: ((r + 1) // 2) * 2 + 2                      # even, and a zero row pair behind the data
            cur = torch.zeros(pad_rows(L), C0, dtype=torch.float16, device=dev)
            stats = torch.empty(2 * C0, dtype=torch.float64, device=dev)
            st = lib.rvcb200_op_hubert_conv0(C.c_void_p(x.data_ptr()), C.c_void_p(W["conv0.w"].data_ptr()),
                                             C.c_void_p(W["conv0.gn_w"].data_ptr()), C.c_void_p(W["conv0.gn_b"].data_ptr()),
                                             C.c_void_p(stats.data_ptr()), C.c_void_p(cur.data_ptr()), 1, n, C0, K0, S0, 1e-5,
                                             cur.numel(), self._stream)
            if st != 0:
                raise RuntimeError(f"rvcb200_op_hubert_conv0 failed with status {st}")
            self.last_launches += 2 if L <= 256 else 3                        # + the fixed-order reduction of the statistics
            feat32 = None
            nconv = len(self.conv_kernel)
            for i in range(1, nconv):
                k = self.conv_kernel[i]
                Lout = (L - k) // 2 + 1
                if Lout < 1:
                    raise RuntimeError("input too short for the feature encoder")
                rows_in = cur.shape[0] // 2                                  # the [L][C0] buffer viewed as [L/2][2 C0]
                last = i == nconv - 1
                n_tile = 256 if (Lout + 127) // 128 >= 148 else 64
                w16 = W[f"conv{i}.w"] if n_tile == 256 else self._conv_w64(i)
                if last:
                    feat32 = torch.empty(Lout, C0, dtype=torch.float32, device=dev)
                    self._gemm(cur.data_ptr(), rows_in, 2 * C0, w16, W["zeros"], C0, Lout, ntaps=2 if k == 3 else 1, n_tile=n_tile,
                               gelu=True, y32=feat32.data_ptr(), ldy32=C0)
                else:
                    nxt = torch.zeros(pad_rows(Lout), C0, dtype=torch.float16, device=dev)
                    self._gemm(cur.data_ptr(), rows_in, 2 * C0, w16, W["zeros"], C0, Lout, ntaps=2 if k == 3 else 1, n_tile=n_tile,
                               gelu=True, y16=nxt.data_ptr(), ldy16=C0)
                    cur = nxt
                L = Lout
            T = L
            # feature projection: LayerNorm(512) -> Linear(512 -> H)
            ln32 = torch.empty(T, C0, dtype=torch.float32, device=dev)
            ln16 = torch.empty(T, C0, dtype=torch.float16, device=dev)
            self._ln(feat32, W["fp.ln_w"], W["fp.ln_b"], ln32, ln16, T, C0)
            h32 = torch.empty(T, H, dtype=torch.float32, device=dev)
            h16 = torch.empty(T, H, dtype=torch.float16, device=dev)
            w16, nt_ = self._tiled("fp.w", T, H)
            self._gemm(ln16.data_ptr(), T, C0, w16, W["fp.b"], H, T, n_tile=nt_, y32=h32.data_ptr(), ldy32=H, y16=h16.data_ptr(), ldy16=H)
            # positional convolution: h + GELU(conv_k128_groups16(h) + b): one launch, an N tile per group (16 launches of 24 CTAs
            # each before: 528 of the 5 100 us of a 60 s utterance, profiles/r2_hubert_launches_60s_v1.csv)
            t32 = torch.empty(T, H, dtype=torch.float32, device=dev)
            cg = H // self.gpos
            self._gemm(h16.data_ptr(), T, cg, W["pos.w"], W["pos.b"], H, T, ntaps=self.kpos, g_off=-(self.kpos // 2), n_tile=cg,
                       ldx16=H, gelu=True, y32=t32.data_ptr(), ldy32=H, res32=h32.data_ptr(), ldr32=H, a_nt_stride=cg)
            self._ln(t32, W["enc.ln_w"], W["enc.ln_b"], h32, h16, T, H)
            # encoder layers (post-norm)
            nh = self.n_heads
            qkv16 = torch.empty(T, 3 * nh * HEAD_PAD, dtype=torch.float16, device=dev)
            att16 = torch.empty(T, nh * HEAD_OUT, dtype=torch.float16, device=dev)
            ff16 = torch.empty(T, self.inter, dtype=torch.float16, device=dev)
            for l in range(n_layers):
                w16, nt_ = self._tiled(f"l{l}.qkv.w", T, 3 * nh * HEAD_PAD)
                self._gemm(h16.data_ptr(), T, H, w16, W[f"l{l}.qkv.b"], 3 * nh * HEAD_PAD, T, n_tile=nt_, y16=qkv16.data_ptr(),
                           ldy16=3 * nh * HEAD_PAD)
                st = lib.rvcb200_op_attention_tc(C.c_void_p(qkv16.data_ptr()), None,      # V is read in place: no V^T scratch
                                                 C.c_void_p(W["ek0"].data_ptr()), C.c_void_p(W["evt0"].data_ptr()), None,
                                                 C.c_void_p(att16.data_ptr()), 1, T, nh, HEAD_OUT, 0, self._stream)
                if st != 0:
                    raise RuntimeError(f"rvcb200_op_attention_tc failed with status {st}")
                self.last_launches += 1
                w16, nt_ = self._tiled(f"l{l}.o.w", T, H)
                self._gemm(att16.data_ptr(), T, nh * HEAD_OUT, w16, W[f"l{l}.o.b"], H, T, n_tile=nt_, y32=t32.data_ptr(), ldy32=H,
                           res32=h32.data_ptr(), ldr32=H)
                self._ln(t32, W[f"l{l}.ln1_w"], W[f"l{l}.ln1_b"], h32, h16, T, H)
                w16, nt_ = self._tiled(f"l{l}.ff1.w", T, self.inter)
                self._gemm(h16.data_ptr(), T, H, w16, W[f"l{l}.ff1.b"], self.inter, T, n_tile=nt_, gelu=True, y16=ff16.data_ptr(),
                           ldy16=self.inter)
                w16, nt_ = self._tiled(f"l{l}.ff2.w", T, H)
                self._gemm(ff16.data_ptr(), T, self.inter, w16, W[f"l{l}.ff2.b"], H, T, n_tile=nt_, y32=t32.data_ptr(), ldy32=H,
                           res32=h32.data_ptr(), ldr32=H)
                self._ln(t32, W[f"l{l}.ln2_w"], W[f"l{l}.ln2_b"], h32, h16, T, H)
            if version == "v1":
                out = torch.empty(T, self.proj_size, dtype=torch.float32, device=dev)
                self._gemm(h16.data_ptr(), T, H, W["final.w"], W["final.b"], self.proj_size, T, y32=out.data_ptr(),
                           ldy32=self.proj_size)
            else:
                out = h32.clone()
            return out.unsqueeze(0).to(source.dtype if source.dtype in (torch.float16, torch.float32) else torch.float32)

    def _conv_w64(self, i):
        """Feature-encoder weights re-tiled for N = 64 (short inputs: few 128-row tiles, so C_out is split over more CTAs)."""
        key = f"conv{i}.w64"
        if key not in self._w:
            w = self._sd[f"feature_extractor.conv_layers.{i}.conv.weight"]
            C0, k = self.conv_dim[0], w.shape[2]
            taps = torch.zeros(2 if k == 3 else 1, 2 * C0, C0)
            taps[0, :C0], taps[0, C0:] = w[:, :, 0].t(), w[:, :, 1].t()
            if k == 3:
                taps[1, :C0] = w[:, :, 2].t()
            self._w[key] = pack_tc(taps, torch.float16, 64).to(self.device)
        return self._w[key]

    def __call__(self, *a, **k):
        raise NotImplementedError("use extract_features(); the training forward is out of scope")
