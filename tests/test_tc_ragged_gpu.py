"""GPU: ragged batches through the tensor-core text encoder and reverse flow, frame by frame at the mask boundary.

B = 3 items of lengths T, 4 * 128 + 1 and 128 + 1 (one frame past a 128-row tile boundary) in a T = 700 batch.  The taps
`stats`, `z_p` and `z` of the device are compared with `oracle.rvc_oracle.text_encoder` + `flow_reverse` run in float64 on
the fp16-rounded checkpoint, `z_p` formed as `infer` forms it.  Frames >= len must be exactly 0; the worst error over the
last 8 frames before len may not exceed twice the worst error over the rest of the same item -- a mask that leaks across
the boundary (an off-by-one of `out_len`, `mask16`, `mask_pre` / `mask_post`) shows there first, and the ratio needs no
absolute bound.  The whole-item gates of test_tc_gpu.py / test_parity_gpu.py skip exactly these frames."""
import pytest
import torch
import torch.nn.functional as F

from comfy_rvc_b200 import synthetic
from comfy_rvc_b200.config import resolve
from oracle import rvc_oracle
from tests._util import net_infer

pytestmark = pytest.mark.gpu

B, T, LENS, TAIL = 3, 700, [700, 513, 129], 8


def _fold64(sd):
    """fold_weight_norm in float64 on the checkpoint as the device receives it (fp16 on disk)."""
    out = {}
    for k, v in sd.items():
        if k.endswith("weight_v"):
            out[k[:-8] + "weight"] = torch._weight_norm(v.half().double(), sd[k[:-1] + "g"].half().double(), 0)
        elif not k.endswith("weight_g"):
            out[k] = v.half().double()
    return out


@pytest.mark.parametrize("cfg_name,precision", [("32k_v2", "fp16"), ("32k_v2", "bf16"), ("32k_v2:nono", "fp16")])
def test_ragged_tails_of_encoder_and_flow(cfg_name, precision):
    from tests.test_parity_gpu import build_net
    cfg = resolve(cfg_name)
    sd = synthetic.make_state_dict(cfg, seed=3)
    phone, lens, pitch, pitchf, sid = synthetic.make_inputs(cfg, B, T, seed=21, lengths=LENS)
    noise = synthetic.draw_noise(cfg, B, T, seed=22)
    net = build_net(cfg, sd, precision)
    taps = {"stats": None, "z_p": None, "z": None}
    net_infer(net, cfg, (phone, lens, pitch, pitchf, sid), noise, taps)
    torch.cuda.synchronize()
    w = _fold64(sd)
    m_p, logs_p, x_mask = rvc_oracle.text_encoder(w, cfg, phone.double(), pitch if cfg.f0 else None, lens)
    z_p = (m_p + torch.exp(logs_p) * noise[0].double() * 0.66666) * x_mask
    g = F.embedding(sid, w["emb_g.weight"]).unsqueeze(-1)
    z = rvc_oracle.flow_reverse(w, cfg, z_p, x_mask, g)
    refs = {"stats": torch.cat([m_p, logs_p], 1), "z_p": z_p, "z": z}
    for key, ref in refs.items():
        got = taps[key].cpu().double()                                       # [B][T][C], channels-last
        ref = ref.transpose(1, 2)
        err = (got - ref).abs().amax(dim=2)                                  # [B][T] worst channel per frame
        for b, L in enumerate(LENS):
            assert bool((got[b, L:] == 0).all()), f"{key} item {b}: frames >= {L} not zero"
            inner, tail = err[b, :L - TAIL].max().item(), err[b, L - TAIL:L].max().item()
            print(f"{cfg_name} {precision} {key} item {b} (len {L}): interior max|err| {inner:.3e}, last {TAIL} frames {tail:.3e}"
                  f" (|ref| max {ref[b, :L].abs().max().item():.2f})")
            if L < T:
                assert tail <= 2.0 * inner, f"{key} item {b}: error at the mask boundary {tail:.3e} vs interior {inner:.3e}"
