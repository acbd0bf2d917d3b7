"""GPU: the generic epilogue of the tcgen05 convolution (`rvcb200_op_conv_tc` with `generic = 1`), descriptor by descriptor
as the text encoder / reverse flow (csrc/engine.cu, tensor-core branch) and the HuBERT front end (comfy_rvc_b200/hubert.py)
issue them, against the fp64 restatement of tests/_tc_generic_ref.py.

Which of the kernel's two epilogue forms runs depends on the N tile, not on the modes: the whole-tile form
(`epilogue_lean64`) only when `lean_ok` holds (N = 64 and a list of flag conditions), the pass-by-pass form
(`epilogue_generic16`) otherwise; the residual / running-sum prefetch (`have_pre`) only for N <= 64.  Every case runs at the
N the product uses and at an N that changes the form (or, where no other form is possible, the tiling); both must meet
the fp64 bounds and give the same bits.  `test_lean_form_is_bit_identical_to_pass_by_pass` reruns the N = 64 launches in a child process with
RVCB200_LEAN_EPI=0 (the switch is read once per process) and requires the same bits.

Every output buffer is filled with NaN before the launch and has 128 guard rows after the last batch item; whatever lies
outside the launch's own output columns / rows (sentinels, guard rows, the input columns of a buffer the launch reads and
writes, as the flow's activation buffer) must be bit-identical afterwards.  Input columns the launch must not read are NaN
as well, so a read past `Cin` shows up as a NaN in the result."""
import ctypes as C
import math
import os
import subprocess
import sys

import pytest
import torch

from comfy_rvc_b200 import _lib, weights
from comfy_rvc_b200.config import NAMED_CONFIGS
from tests._tc_generic_ref import generic_ref, row_mask, ulp16

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PADF, GUARD = 32, 128
Y32_TOL = 1e-3          # max abs error of fp32 outputs on O(1) data (the bound of test_tc_gpu.py)
# 16-bit outputs: one fp16 ulp of the fp64 value, plus what the fp32 value can carry before its rounding -- the fp32
# accumulation of up to 3 x 3072 products of O(1) terms and the gate's MUFU ex2 / rcp sigmoid (~1e-6)
Y16_SLACK = 5e-5

CFG = NAMED_CONFIGS["32k_v2"]
H, F_, HALF = CFG.hidden_channels, CFG.filter_channels, CFG.inter_channels // 2
N_WN = CFG.flow_wn_layers
XB = weights.flow_x0_block(CFG)
AW = XB + N_WN * H                       # flow activation buffer [x0 | mask | zeros | acts_0 .. acts_{n-1}]
QKV = 3 * CFG.n_heads * 128              # q|k|v, 128 channels per head (engine.cu)
HID, INTER, HEADS_OUT = 768, 3072, 12 * 96


def _spec(name, Cin, Cout, Ns, *, ntaps=1, g_off=0, x_w=None, x_col=0, y32=None, y16=None, res=None, shapes="enc", **flags):
    """One descriptor.  x_w: width of the activation buffer (row stride); y32 / y16 / res: (buffer, first column, width) --
    buffers with the same name are one allocation; Ns: product N first, then the N that flips the epilogue form."""
    return dict(name=name, Cin=Cin, Cout=Cout, Ns=Ns, ntaps=ntaps, g_off=g_off, x_w=x_w or Cin, x_col=x_col, y32=y32, y16=y16,
                res=res, shapes=shapes, flags=flags)


CASES = [
    # text encoder (engine.cu, TextEncoder on tcgen05)
    _spec("enc.emb", CFG.feat_dim, H, (64, 32), gather=True, alpha=math.sqrt(H), pre_slope=0.1, mask_post=True, mask16=True,
          y32=("y32", 0, H), y16=("y16", 0, H)),
    _spec("enc.qkv", H, QKV, (64, 32), y16=("y16", 0, QKV)),
    _spec("enc.o", H, H, (64, 32), res=("res", 0, H), y32=("y32", 0, H)),
    _spec("enc.ffn1", H, F_, (64, 32), ntaps=CFG.kernel_size, g_off=-(CFG.kernel_size - 1) // 2, relu=True, mask16=True,
          y16=("y16", 0, F_)),
    _spec("enc.ffn2", F_, H, (64, 32), ntaps=CFG.kernel_size, g_off=-(CFG.kernel_size - 1) // 2, mask_pre=True,
          res=("res", 0, H), y32=("y32", 0, H)),
    _spec("enc.proj", H, 2 * CFG.inter_channels, (64, 32), mask_post=True, y32=("y32", 0, 2 * CFG.inter_channels)),
    # reverse flow on folded weights: in_layer j reads [0, xb + jH) of the activation buffer, writes acts_j into it
    *[_spec(f"flow.in{j}", XB + j * H, 2 * H, (64, 32), ntaps=CFG.flow_kernel, g_off=-(CFG.flow_kernel - 1) // 2, x_w=AW,
            cond=True, gate=True, mask16=True, y16=("x", XB + j * H, AW)) for j in range(N_WN)],
    # skip + post: reads the gate outputs, updates the other half of z in place (r - v), fp16 copy into columns [0, half)
    _spec("flow.skip+post", N_WN * H, HALF, (48, 16), x_w=AW, x_col=XB, mask_pre=True, mask_post=True, res_mode=2,
          res=("y32", HALF, CFG.inter_channels), y32=("y32", HALF, CFG.inter_channels), y16=("x", 0, AW)),
    # synthetic: the running sum (accum) with and without the divisor, relu and an output slope (no product launch of the
    # generic kernel sets them; the decoder's epilogue does)
    _spec("syn.accum", H, H, (64, 32), accum=True, y32=("y32", 0, H)),
    _spec("syn.accum_div_relu", H, H, (64, 32), ntaps=3, g_off=-1, relu=True, accum=True, div=3.0, out_slope=0.1,
          mask_post=True, y32=("y32", 0, H), y16=("y16", 0, H)),
    # HuBERT front end (hubert.py): conv stack on the [L/2][2C] view, projections, positional convolution
    _spec("hub.conv_y16", 1024, 512, (64, 256), ntaps=2, gelu=True, y16=("y16", 0, 512), shapes="conv", in_extra=1),
    _spec("hub.conv_y32", 1024, 512, (64, 256), gelu=True, y32=("y32", 0, 512), shapes="conv", in_extra=1),
    _spec("hub.fp", 512, HID, (64, 128, 256), y32=("y32", 0, HID), y16=("y16", 0, HID), shapes="hub"),
    _spec("hub.o", HEADS_OUT, HID, (64, 128, 256), res=("res", 0, HID), y32=("y32", 0, HID), shapes="hub"),
    _spec("hub.ff1", HID, INTER, (64, 256), gelu=True, y16=("y16", 0, INTER), shapes="hub"),
    _spec("hub.ff2", INTER, HID, (64, 128), res=("res", 0, HID), y32=("y32", 0, HID), shapes="hub"),
    _spec("hub.pos", 48, HID, (48,), ntaps=128, g_off=-64, x_w=HID, a_nt_stride=48, gelu=True, res=("res", 0, HID),
          y32=("y32", 0, HID), shapes="hub"),
]
CASE_BY_NAME = {c["name"]: c for c in CASES}

# (B, T, out_len): T not a multiple of 128, lengths T, 128 k +- 1 and 1; the long shapes give every CTA several tiles
SHAPES = {
    "enc": {"short": (3, 700, [700, 383, 1]), "long": (3, 6500, [6500, 4097, 1])},
    "conv": {"short": (1, 1999, None), "long": (1, 19001, None)},       # N = 256 from 18 817 rows on (hubert.py)
    "hub": {"short": (1, 501, None), "long": (1, 2999, None)},          # 2 999 frames = 60 s
}


def lean_ok(c, N):
    """conv_tc.cu `lean_ok` for this descriptor."""
    f = c["flags"]
    res, acc = c["res"] is not None, bool(f.get("accum"))
    gate = bool(f.get("gate"))
    return (N == 64 and not f.get("gather") and f.get("alpha", 1.0) == 1.0 and f.get("pre_slope", 1.0) == 1.0
            and f.get("div", 1.0) == 1.0 and f.get("out_slope", 1.0) == 1.0 and not (res and acc)
            and not (gate and (res or acc or c["y32"] is not None or f.get("relu") or f.get("gelu"))))


def have_pre(c, N):
    """conv_tc.cu: residual / running sum loaded before the accumulator wait."""
    f = c["flags"]
    return not f.get("gate") and N <= 64 and ((c["res"] is not None) != bool(f.get("accum")))


def make_inputs(c, shape):
    """Seeded CPU tensors of one (case, shape): operands exactly representable in fp16, the fp32 side in fp32."""
    B, T, lens = SHAPES[c["shapes"]][shape]
    f = c["flags"]
    g = torch.Generator().manual_seed(sum(map(ord, c["name"])) * 7 + T)
    L_in = T + f.get("in_extra", 0)
    Cin, Cout, nt = c["Cin"], c["Cout"], c["ntaps"]
    Co = Cout // 2 if f.get("gate") else Cout
    read_w = (f["a_nt_stride"] * (Cout // c["Ns"][0] - 1) + Cin) if f.get("a_nt_stride") else Cin
    inp = dict(B=B, T=T, L_in=L_in, Co=Co, lens=lens, read_w=read_w)
    inp["x"] = torch.randn(B, L_in, read_w, generator=g).half()
    inp["w"] = (torch.randn(nt, Cin, Cout, generator=g) / math.sqrt(Cin * nt)).half().float()
    inp["bias"] = torch.randn(Cout, generator=g) * 0.5
    if f.get("cond"):
        inp["cond"] = torch.randn(B, 1024, generator=g) * 0.5              # cond_bstride 1024, the launch's slice at 40
    if f.get("gather"):
        inp["gather"] = torch.randn(256, Cout, generator=g) * 0.5
        inp["gidx"] = torch.randint(0, 256, (B, T), generator=g, dtype=torch.int64)
    if c["res"] is not None:
        inp["res"] = torch.randn(B, T, Co, generator=g)
    if f.get("accum"):
        inp["acc"] = torch.randn(B, T, Co, generator=g)
    return inp


def _buffers(c, inp):
    """Buffer name -> (dtype, width) of every allocation the launch touches."""
    bufs = {"x": (torch.float16, c["x_w"])}
    for key, dt in (("y32", torch.float32), ("y16", torch.float16), ("res", torch.float32)):
        if c[key] is not None:
            name, _, width = c[key]
            bufs.setdefault(name, (dt, width))
    return bufs


def launch(c, inp, N, dev):
    """Runs the descriptor at N tile N; returns (buffers before, buffers after, owned regions) on the CPU."""
    f = c["flags"]
    B, T, L_in, Co = inp["B"], inp["T"], inp["L_in"], inp["Co"]
    rows = B * max(T, L_in) + GUARD
    host = {n: torch.full((rows, w), float("nan"), dtype=dt) for n, (dt, w) in _buffers(c, inp).items()}
    xc = c["x_col"]
    host["x"][:B * L_in, xc:xc + inp["read_w"]] = inp["x"].reshape(B * L_in, -1)
    if c["res"] is not None:
        n, col, _ = c["res"]
        host[n][:B * T, col:col + Co] = inp["res"].reshape(B * T, Co)
    if f.get("accum"):
        n, col, _ = c["y32"]
        host[n][:B * T, col:col + Co] = inp["acc"].reshape(B * T, Co)
    d_bufs = {n: t.to(dev) for n, t in host.items()}
    assert weights.tc_n_for(c["Cout"], N) == N
    w16 = weights.pack_tc(inp["w"], torch.float16, N).to(dev)
    bias = inp["bias"].to(dev)
    keep = [w16, bias]
    d = _lib.TcConvDesc()
    d.x16, d.L_in, d.padf = d_bufs["x"].data_ptr() + 2 * xc, L_in, PADF
    d.w16, d.bias = w16.data_ptr(), bias.data_ptr()
    d.Cin, d.ntaps, d.dil, d.G = c["Cin"], c["ntaps"], 1, 1
    d.g_off[0] = c["g_off"]
    d.N, d.Cout_total = N, c["Cout"]
    d.Lj, d.out_stride, d.Lp_out = T, 1, ((T + 127) // 128) * 128 + 128
    d.generic, d.f32_cl = 1, 1
    d.ldx16 = c["x_w"] if c["x_w"] != c["Cin"] else 0
    d.alpha, d.pre_slope = f.get("alpha", 1.0), f.get("pre_slope", 1.0)
    d.div, d.out_slope = f.get("div", 1.0), f.get("out_slope", 1.0)
    d.gate, d.relu, d.gelu = int(bool(f.get("gate"))), int(bool(f.get("relu"))), int(bool(f.get("gelu")))
    d.mask_pre, d.mask_post, d.mask16 = (int(bool(f.get(k))) for k in ("mask_pre", "mask_post", "mask16"))
    d.accum = int(bool(f.get("accum")))
    d.a_nt_stride = f.get("a_nt_stride", 0)
    if inp["lens"] is not None:
        ol = torch.tensor(inp["lens"], dtype=torch.int32, device=dev)
        keep.append(ol)
        d.out_len = ol.data_ptr()
    if f.get("cond"):
        cd = inp["cond"].to(dev)
        keep.append(cd)
        d.cond, d.cond_bstride = cd.data_ptr() + 4 * 40, cd.shape[1]
    if f.get("gather"):
        gt, gi = inp["gather"].to(dev), inp["gidx"].to(dev)
        keep += [gt, gi]
        d.gather, d.gidx, d.gidx_bstride = gt.data_ptr(), gi.data_ptr(), T
    owned = {}
    if c["y32"] is not None:
        n, col, width = c["y32"]
        d.y32, d.ldy32 = d_bufs[n].data_ptr() + 4 * col, width
        owned.setdefault(n, []).append(col)
    if c["y16"] is not None:
        n, col, width = c["y16"]
        d.y16, d.ldy16 = d_bufs[n].data_ptr() + 2 * col, (width if width != Co else 0)
        owned.setdefault(n, []).append(col)
    if c["res"] is not None:
        n, col, width = c["res"]
        d.res32, d.ldr32, d.res_mode = d_bufs[n].data_ptr() + 4 * col, width, f.get("res_mode", 1)
    st = _lib.load().rvcb200_op_conv_tc(C.byref(d), B, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert st == 0, st
    torch.cuda.synchronize()
    return host, {n: t.cpu() for n, t in d_bufs.items()}, owned


def reference(c, inp, dev):
    """fp64 (v, y16) [B][T][Co] on the device (a checker only)."""
    f = c["flags"]
    dd = lambda t: t.to(dev, torch.float64)
    kw = {k: f[k] for k in ("alpha", "pre_slope", "res_mode", "div", "out_slope", "a_nt_stride") if k in f}
    for k in ("gate", "gelu", "relu", "mask_pre", "mask_post", "mask16"):
        kw[k] = bool(f.get(k))
    if f.get("cond"):
        kw["cond"] = dd(inp["cond"][:, 40:40 + c["Cout"]])
    if f.get("gather"):
        kw["gather"], kw["gidx"] = dd(inp["gather"]), inp["gidx"].to(dev)
    if "res" in inp:
        kw["res"] = dd(inp["res"])
    if "acc" in inp:
        kw["acc"] = dd(inp["acc"])
    if inp["lens"] is not None:
        kw["out_len"] = torch.tensor(inp["lens"])
    return generic_ref(dd(inp["x"]), dd(inp["w"]), dd(inp["bias"]), inp["T"], g_off=c["g_off"], N=c["Ns"][0], **kw)


def _out_view(buf, col, B, T, Co):
    return buf[:B * T, col:col + Co].reshape(B, T, Co)


def check_outputs(c, inp, before, after, owned, ref, N):
    """The fp64 bounds, exact zeros on masked rows, and untouched bits everywhere else.  Returns the max errors."""
    f = c["flags"]
    B, T, Co = inp["B"], inp["T"], inp["Co"]
    v_ref, y16_ref = ref
    dev = v_ref.device
    invalid = ~row_mask(torch.tensor(inp["lens"]) if inp["lens"] is not None else None, B, T, dev)[..., 0]
    errs = {}
    if c["y32"] is not None:
        n, col, _ = c["y32"]
        got = _out_view(after[n], col, B, T, Co).to(dev, torch.float64)
        assert not bool(torch.isnan(got).any()), f"{c['name']} N={N}: NaN in y32 (read past Cin, or an unwritten row)"
        errs["y32"] = (got - v_ref).abs().max().item()
        assert errs["y32"] <= Y32_TOL, (c["name"], N, errs["y32"])
        if f.get("mask_post"):
            assert bool((got[invalid] == 0).all()), f"{c['name']} N={N}: y32 not 0 on a masked row"
    if c["y16"] is not None:
        n, col, _ = c["y16"]
        got = _out_view(after[n], col, B, T, Co).to(dev, torch.float64)
        assert not bool(torch.isnan(got).any()), f"{c['name']} N={N}: NaN in y16"
        bound = ulp16(y16_ref) + Y16_SLACK
        errs["y16 err/bound"] = ((got - y16_ref).abs() / bound).max().item()
        assert errs["y16 err/bound"] <= 1.0, (c["name"], N, "y16 beyond one fp16 ulp", errs["y16 err/bound"])
        if f.get("mask16") or f.get("mask_post"):
            assert bool((got[invalid] == 0).all()), f"{c['name']} N={N}: y16 not 0 on a masked row"
    # everything but the owned output columns of rows [0, B T) keeps its bits (NaN sentinels, guard rows, input columns)
    for n, t in after.items():
        keep = torch.ones_like(t, dtype=torch.bool)
        for col in owned.get(n, []):
            keep[:B * T, col:col + Co] = False
        ib = torch.int16 if t.dtype == torch.float16 else torch.int32
        changed = (t.view(ib) != before[n].view(ib)) & keep
        assert not bool(changed.any()), f"{c['name']} N={N}: buffer {n} changed outside the launch's output " \
                                        f"(first at {changed.nonzero()[0].tolist()})"
    return errs


PARAMS = [(c["name"], s) for c in CASES for s in ("short", "long")]


@pytest.mark.parametrize("name,shape", PARAMS, ids=[f"{n}-{s}" for n, s in PARAMS])
def test_generic_epilogue_matches_fp64(name, shape):
    c = CASE_BY_NAME[name]
    dev = torch.device("cuda", 0)
    inp = make_inputs(c, shape)
    ref = reference(c, inp, dev)
    outs = {}
    for N in c["Ns"]:
        before, after, owned = launch(c, inp, N, dev)
        errs = check_outputs(c, inp, before, after, owned, ref, N)
        outs[N] = after
        print(f"{name} {shape} N={N} ({'lean' if lean_ok(c, N) else 'pass-by-pass'}, prefetch {have_pre(c, N)}): "
              + ", ".join(f"{k} {v:.3e}" for k, v in errs.items()))
    if lean_ok(c, c["Ns"][0]):
        assert not all(lean_ok(c, N) for N in c["Ns"]), "the other N must run the pass-by-pass form"
    # The K loop, and so the accumulation order, does not depend on N, and both forms do the same fp32 arithmetic: every
    # N gives the same bits (measured on a B200 for every case of the table before this was asserted)
    n0 = c["Ns"][0]
    for N in c["Ns"][1:]:
        for b, t in outs[N].items():
            ib = torch.int16 if t.dtype == torch.float16 else torch.int32
            assert torch.equal(t.view(ib), outs[n0][b].view(ib)), f"{name} {shape}: buffer {b} differs between N={n0} and N={N}"


def test_the_cases_cover_both_forms_and_the_prefetch():
    """The table reaches both epilogue forms and both residual paths (fails if a descriptor change moved them)."""
    lean = {c["name"] for c in CASES if lean_ok(c, c["Ns"][0])}
    assert {"enc.qkv", "enc.o", "enc.ffn1", "enc.ffn2", "enc.proj", "flow.in0", "syn.accum"} <= lean
    assert not lean_ok(CASE_BY_NAME["enc.emb"], 64) and not lean_ok(CASE_BY_NAME["flow.skip+post"], 48)
    assert have_pre(CASE_BY_NAME["flow.skip+post"], 48) and have_pre(CASE_BY_NAME["hub.o"], 64)
    assert not have_pre(CASE_BY_NAME["hub.o"], 128) and not have_pre(CASE_BY_NAME["hub.ff2"], 128)


def _dump_n64(path):
    """Child-process side of the lean / pass-by-pass comparison: every N = 64 launch of the table, outputs to `path`."""
    dev = torch.device("cuda", 0)
    res = {}
    for c in CASES:
        if 64 in c["Ns"] and lean_ok(c, 64):
            for s in ("short", "long"):
                res[f"{c['name']}-{s}"] = launch(c, make_inputs(c, s), 64, dev)[1]
    torch.save(res, path)


def test_lean_form_is_bit_identical_to_pass_by_pass(tmp_path):
    """RVCB200_LEAN_EPI=0 (read once per process, conv_tc.cu) forces the pass-by-pass form: the whole-tile form was
    introduced as bit-identical to it, on every N = 64 descriptor of the table."""
    assert os.environ.get("RVCB200_LEAN_EPI", "1") != "0", "this process must run the lean form"
    path = str(tmp_path / "pass_by_pass.pt")
    env = dict(os.environ, RVCB200_LEAN_EPI="0")
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from tests.test_tc_generic_gpu import _dump_n64; _dump_n64({path!r})"
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    child = torch.load(path)
    dev = torch.device("cuda", 0)
    n = 0
    for c in CASES:
        if 64 in c["Ns"] and lean_ok(c, 64):
            for s in ("short", "long"):
                mine = launch(c, make_inputs(c, s), 64, dev)[1]
                for b, t in mine.items():
                    ib = torch.int16 if t.dtype == torch.float16 else torch.int32
                    assert torch.equal(t.view(ib), child[f"{c['name']}-{s}"][b].view(ib)), (c["name"], s, b)
                n += 1
    assert n >= 10


def _valid_desc(keep):
    """A small descriptor the launcher accepts (one tile, N = 64, y32)."""
    dev = torch.device("cuda", 0)
    x = torch.zeros(128, 64, dtype=torch.float16, device=dev)
    w = weights.pack_tc(torch.zeros(1, 64, 64), torch.float16, 64).to(dev)
    b = torch.zeros(64, device=dev)
    y = torch.zeros(128 + GUARD, 64, device=dev)
    keep += [x, w, b, y]
    d = _lib.TcConvDesc()
    d.x16, d.L_in, d.padf, d.w16, d.bias = x.data_ptr(), 128, PADF, w.data_ptr(), b.data_ptr()
    d.Cin, d.ntaps, d.dil, d.G, d.N, d.Cout_total = 64, 1, 1, 1, 64, 64
    d.Lj, d.out_stride, d.Lp_out = 128, 1, 256
    d.generic, d.f32_cl, d.alpha, d.pre_slope, d.div, d.out_slope = 1, 1, 1.0, 1.0, 1.0, 1.0
    d.y32, d.ldy32 = y.data_ptr(), 64
    return d


def test_generic_rejections():
    """Descriptors the launcher must refuse host-side (status 1, nothing launched)."""
    lib, keep = _lib.load(), []
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.rvcb200_op_conv_tc(C.byref(_valid_desc(keep)), 1, st) == 0
    torch.cuda.synchronize()
    d = _valid_desc(keep)
    d.a_nt_stride, d.G = 64, 2                                     # grouped channel slices with phase groups
    d.g_off[1] = 0
    assert lib.rvcb200_op_conv_tc(C.byref(d), 1, st) == 1
    d = _valid_desc(keep)
    d.accum, d.y32 = 1, None                                       # running sum without the buffer that holds it
    assert lib.rvcb200_op_conv_tc(C.byref(d), 1, st) == 1
    d = _valid_desc(keep)
    d.N = 48                                                       # N does not divide Cout_total = 64
    assert lib.rvcb200_op_conv_tc(C.byref(d), 1, st) == 1
    torch.cuda.synchronize()
