"""GPU: the index blend of `VC.vc` on the device (`IndexIVFFlatB200`, csrc/index_kernels.cu) -- the IVF-Flat nprobe-1 search against
the fp64 oracle with its margin rule, exact ties, determinism, the blend bit for bit against the reference's expression run with
torch on the same device, whole songs against the host path, the sharded song over NCCL, and the C ABI's argument checks."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

import comfy_rvc_b200 as rvc
from comfy_rvc_b200 import IndexIVFFlatB200, _lib, synthetic
from comfy_rvc_b200 import pipeline as pl
from oracle import pipeline_oracle
from tests import _ivf_oracle
from tests._util import load_pipeline_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr())


def _index_case(case, d):
    if case == "flat48":
        return _ivf_oracle.clustered(d, 48, 1, seed=d)
    if case == "flat10k":
        return _ivf_oracle.clustered(d, 10_000, 1, seed=d + 1)
    if case == "ivf50k":
        return _ivf_oracle.clustered(d, 50_000, 1282, seed=d + 2)
    return _ivf_oracle.clustered(d, 20_000, 300, seed=d + 3, skew=True)


def _check_against_oracle(o, x, score, ix):
    """Margin rule: where both fp64 margins exceed tau = 1e-5 (||q||^2 + ||v||^2) the device's neighbour is the oracle's; elsewhere
    the device's list and vector are each within tau of the best.  Returns the fraction of queries in that regime."""
    det = o.detail(x)
    reg = o.in_regime(det)
    assert np.array_equal(ix[reg], det["ix"][reg])
    xd = det["x"]
    for q in np.nonzero(~reg)[0]:
        if ix[q] < 0:
            assert det["ix"][q] < 0 or det["cmargin"][q] <= det["tau_c"][q]
            continue
        l = o.list_of_label[ix[q]]
        dc = ((xd[q] - o.centroids) ** 2).sum(1)
        assert dc[l] - dc.min() <= det["tau_c"][q]
        a, b = o.offs[l], o.offs[l + 1]
        dv = ((xd[q] - o.vectors[a:b]) ** 2).sum(1)
        j = int(np.nonzero(o.labels[a:b] == ix[q])[0][0])
        assert dv[j] - dv.min() <= det["tau_f"][q]
    hit = ix >= 0
    assert np.all(score[~hit] == np.inf)
    pos = np.empty(o.ntotal, dtype=np.int64)
    pos[o.labels] = np.arange(o.ntotal)
    true = ((xd[hit] - o.vectors[pos[ix[hit]]]) ** 2).sum(1)
    assert np.all(np.abs(score[hit] - true) <= det["tau_f"][hit])
    return reg.mean()


@pytest.mark.parametrize("qdtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("case", ["flat48", "flat10k", "ivf50k", "skewed"])
@pytest.mark.parametrize("d", [256, 768])
def test_search_matches_oracle(d, case, qdtype):
    cent, offs, labels, vec = _index_case(case, d)
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device=DEV)
    o = _ivf_oracle.IVFOracle(cent, offs, labels, vec)
    F = 1037                                                              # not a multiple of any tile
    x = _ivf_oracle.queries(vec, F, seed=d)
    if case == "skewed":
        sizes = np.diff(offs)
        assert sizes.max() > 64 and np.any(sizes == 0)                      # a list longer than a vector range, empty lists
        empty = np.nonzero(sizes == 0)[0][:5]
        x[:5] = cent[empty] + 0.01 * np.random.default_rng(1).standard_normal((5, d)).astype(np.float32)
    xt = torch.from_numpy(x).to(DEV).to(qdtype)
    xq = xt.float().cpu().numpy()                                         # what the device searched: fp16 promotes exactly
    score, ix = idx.search_device(xt)
    s1, i1 = score.cpu().numpy(), ix.cpu().numpy()
    score2, ix2 = idx.search_device(xt)
    assert torch.equal(score, score2) and torch.equal(ix, ix2)            # the same bits on every run
    frac = _check_against_oracle(o, xq, s1, i1)
    print(f"d {d} {case} {qdtype}: {frac * 100:.1f} % of queries outside fp32 reach of a tie, {np.mean(i1 < 0) * 100:.1f} % empty")
    assert frac >= 0.9
    if case == "skewed":
        assert np.all(i1[:5] == -1) and np.all(np.isinf(s1[:5]))
    D, I = idx.search(xq)
    assert D.shape == I.shape == (F, 1) and D.dtype == np.float32 and I.dtype == np.int64
    if qdtype == torch.float32:
        assert np.array_equal(I[:, 0], i1) and np.array_equal(D[:, 0], s1)


def _tie_index(d=256):
    """8 lists around 8 centres; centroid 6 duplicates centroid 3 (list 6 holds other vectors); list 2 is long and holds one vector
    twice, at positions 5 and 70 (different vector ranges)."""
    rng = np.random.default_rng(11)
    cent = rng.standard_normal((8, d)).astype(np.float32)
    cent[6] = cent[3]
    sizes = np.array([30, 10, 150, 40, 20, 25, 35, 12])
    owner = np.repeat(np.arange(8), sizes)
    vec = (cent[owner] + 0.35 * rng.standard_normal((sizes.sum(), d))).astype(np.float32)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    vec[offs[2] + 70] = vec[offs[2] + 5]
    labels = rng.permutation(sizes.sum())
    return cent, offs, labels, vec


def test_exact_ties_and_exact_hit():
    cent, offs, labels, vec = _tie_index()
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device=DEV)
    rng = np.random.default_rng(2)
    x = np.stack([
        cent[3] + 0.01 * rng.standard_normal(256),                        # equidistant from centroids 3 and 6: list 3
        vec[offs[2] + 5] + 0.05 * rng.standard_normal(256),               # duplicated vector: position 5, not 70
        vec[offs[4] + 7],                                                 # equal to a stored vector: score 0
    ]).astype(np.float32)
    xt = torch.from_numpy(x).to(DEV)
    score, ix = (t.cpu().numpy() for t in idx.search_device(xt))
    o = _ivf_oracle.IVFOracle(cent, offs, labels, vec)
    assert o.list_of_label[ix[0]] == 3
    assert ix[1] == labels[offs[2] + 5]
    assert ix[2] == labels[offs[4] + 7] and score[2] == 0.0
    out = idx.blend(xt, 0.75, False).cpu().numpy()
    assert np.all(np.isnan(out[2])) and np.all(np.isfinite(out[:2]))      # the reference's 1 / 0: a NaN row


def _bits_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    iv = torch.int16 if a.dtype == torch.float16 else torch.int32
    return bool(torch.equal(na, nb) and torch.equal(a.masked_fill(na, 0).view(iv), b.masked_fill(nb, 0).view(iv)))


@pytest.mark.parametrize("rate", [0.25, 0.75, 1.0])
@pytest.mark.parametrize("fdtype,is_half", [(torch.float32, False), (torch.float16, True), (torch.float16, False)])
def test_blend_bit_exact(fdtype, is_half, rate):
    """Given the device's ids, `blend` equals vc_infer_pipeline.py:61-75 / pipeline.py's host block run with torch on the device."""
    cent, offs, labels, vec = _ivf_oracle.clustered(768, 20_000, 300, seed=4, skew=True)
    vec = vec.astype(np.float16).astype(np.float32)                      # so that a stored vector is an exact hit in fp16 too
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device=DEV)
    o = _ivf_oracle.IVFOracle(cent, offs, labels, vec)
    x = _ivf_oracle.queries(vec, 2999, seed=8, noise=0.6)
    empty = np.nonzero(np.diff(offs) == 0)[0][:3]
    x[:3] = cent[empty]                                                  # empty lists: ix -1, score +inf
    x[3] = vec[17]                                                       # an exact hit: score 0
    x[4] *= 2.5e13                                                       # score ~1e30: w underflows (fp16 feats: inf)
    x[5] *= 2.8e8                                                        # score ~1e20: w subnormal, weight 1.0 (fp16 feats: inf)
    feats = torch.from_numpy(x).to(DEV).to(fdtype).unsqueeze(0)          # [1][F][d], like the front end's output
    score, ix = idx.search_device(feats)
    got = idx.blend_ids(feats, score, ix, rate, is_half)
    big = torch.from_numpy(o.big_npy()).to(DEV)
    w = torch.square(1 / score[:, None])
    w /= w.sum(dim=1, keepdim=True)
    g = big[ix] * w                                                      # np.sum over the k = 1 axis returns the element itself
    if is_half:
        g = g.half()
    want = g.unsqueeze(0) * rate + (1 - rate) * feats
    assert _bits_equal(got, want), (got.dtype, want.dtype)
    assert torch.isnan(got[0, :5]).all(dim=1).tolist() == [True, True, True, True, True]
    if fdtype == torch.float32:                                          # no flush-to-zero: the subnormal w keeps weight 1.0
        assert 9.3e18 < score[5].item() < 2.7e22 and not torch.isnan(got[0, 5]).any()
    assert not torch.isnan(got[0, 6:]).any()
    prev = torch.cuda.get_sync_debug_mode()
    torch.cuda.set_sync_debug_mode("error")                              # enqueue-only: no host synchronisation
    try:
        again = idx.blend(feats, rate, is_half)
    finally:
        torch.cuda.set_sync_debug_mode(prev)
    assert _bits_equal(again, got)
    assert feats.dtype == fdtype and again.data_ptr() != feats.data_ptr()


def _song(case, file_index, index_rate, noise="reference"):
    from tests.test_parity_gpu import build_net
    cfg = case["cfg"]
    net = build_net(cfg, case["sd"], "fp32")
    vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device=DEV), noise=noise)
    vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
    torch.manual_seed(case["rseed"])
    return vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median", file_index,
                       index_rate, 1, 3, cfg.sr, 0, 1.0, case["version"], case["protect"], 160, False, False, None, 50, 1100)


@pytest.mark.parametrize("name", ["p1_40k_v1_4seg", "p2_32k_v2_protect_index"])
def test_song_equals_host_path(name):
    """The device index against the fp64 oracle object over the same arrays, as an `(index, big_npy)` tuple on the host path:
    identical int16 songs (p2: protect < 0.5, so feats0 must stay unblended)."""
    case = load_pipeline_golden(name)
    d = case["cfg"].feat_dim
    cent, offs, labels, vec = _ivf_oracle.clustered(d, 3000, 50, seed=21)
    o = _ivf_oracle.IVFOracle(cent, offs, labels, vec)
    big = o.big_npy()
    host = _song(case, (o, big), 0.75)
    assert o.seen and all(o.in_regime(det).all() for det in o.seen)      # every frame's answer is out of fp32's reach of a tie
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device=DEV)
    dev = _song(case, (idx, big), 0.75)
    assert dev.dtype == np.int16 and np.array_equal(dev, host)
    assert not np.array_equal(dev, _song(case, "", 0.0))                 # the blend changed the song


def test_p2_golden_with_device_flat_index():
    """FakeIndex's vectors as one list (IndexFlatL2), passed alone: the p2 golden's +-1 LSB; and `VC.vc` with the device index
    equals `VC.vc` with the FakeIndex tuple."""
    case = load_pipeline_golden("p2_32k_v2_protect_index")
    fake, big = case["file_index"]
    idx = IndexIVFFlatB200.from_arrays(np.zeros((1, big.shape[1]), np.float32), [0, big.shape[0]], np.arange(big.shape[0]), big,
                                       device=DEV)
    out = _song(case, idx, case["index_rate"])
    gold = case["gold"]["out_i16"]
    d = np.abs(out.astype(np.int32) - gold.astype(np.int32))
    print(f"p2 with the device flat index: int16 max diff {d.max()} LSB, {np.mean(d > 0) * 100:.2f}% samples differ")
    assert out.shape == gold.shape and d.max() <= 1 and np.abs(out).max() == 32440

    from tests.test_parity_gpu import build_net
    cfg = case["cfg"]
    net = build_net(cfg, case["sd"])
    n = 16000 * 2 + 320
    audio0 = synthetic.make_song(3.0, seed=9)[:n]
    coarse, f0 = pipeline_oracle.f0_post(synthetic.pipeline_f0(x=np.zeros(n)), 2)
    pitch = torch.from_numpy(coarse.astype(np.int64)).unsqueeze(0).to(DEV)
    pitchf = torch.from_numpy(f0.astype(np.float32)).unsqueeze(0).to(DEV)
    noise = synthetic.draw_noise(cfg, 1, min(n // 160, 2 * pl.hubert_frames(n)), seed=21)
    orig = net.infer
    net.infer = lambda *a, **k: orig(*a, noise=noise, **k)
    res = []
    for index, b in ((fake, big), (idx, None)):
        vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device=DEV))
        res.append(vc.vc(case["hubert"], net, torch.zeros(1, dtype=torch.int64, device=DEV), audio0, pitch, pitchf, [0, 0, 0], index, b,
                         0.75, "v2", 0.33))
    assert np.array_equal(res[0], res[1])


def _nccl_worker(rank, world, port, name, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        case = load_pipeline_golden(name)
        cfg = case["cfg"]
        net = rvc.SynthesizerTrnMs256NSFsid(*cfg.to_positional(), is_half=False) if cfg.feat_dim == 256 else \
            rvc.SynthesizerTrnMs768NSFsid(*cfg.to_positional(), is_half=False)
        del net.enc_q
        net.load_state_dict({k: v.half() for k, v in case["sd"].items()}, strict=False)
        net.eval().to(f"cuda:{rank}")
        net = net.float().set_precision("fp32")
        idx = IndexIVFFlatB200.from_arrays(*_ivf_oracle.clustered(cfg.feat_dim, 3000, 50, seed=21), device=f"cuda:{rank}")
        vc = pl.VC(cfg.sr, pl.PipelineConfig(*case["tiers"], is_half=False, device=f"cuda:{rank}"), noise="reference")
        vc.f0_method_dict["synthetic"] = synthetic.pipeline_f0
        torch.manual_seed(case["rseed"])
        out = vc.pipeline(case["hubert"], net, 0, case["audio"].copy(), [0, 0, 0], case["f0_up_key"], "synthetic", "median",
                          idx, 0.75, 1, 3, cfg.sr, 0, 1.0, case["version"], case["protect"], 160, False, False, None, 50, 1100,
                          all_ranks=True)
        q.put((rank, out.copy(), vc.last_plan["assignment"]))
    finally:
        dist.destroy_process_group()


def test_sharded_device_index_nccl_is_bit_identical():
    """Two GPUs, one index replica per rank: every rank's song equals the unsharded one bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    name = "p1_40k_v1_4seg"
    case = load_pipeline_golden(name)
    single = _song(case, IndexIVFFlatB200.from_arrays(*_ivf_oracle.clustered(case["cfg"].feat_dim, 3000, 50, seed=21), device=DEV), 0.75)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, name, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = {}
        for _ in procs:
            r, out, assignment = q.get(timeout=900)
            res[r] = (out, assignment)
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
    assert all(len(r) > 0 for r in res[0][1])
    assert np.array_equal(res[0][0], single) and np.array_equal(res[1][0], single)


def test_abi_refuses_bad_arguments():
    lib = _lib.load()
    d, F, nlist = 16, 10, 3
    f = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=DEV)   # noqa: E731
    x, cent, cn = f(F, d), f(nlist, d), f(nlist)
    coarse, offs = f(F, dt=torch.int64), torch.tensor([0, 2, 2, 5], dtype=torch.int32, device=DEV)
    vec, lab, pos = f(5, d), torch.arange(5, device=DEV), torch.arange(5, dtype=torch.int32, device=DEV)
    score, ix, out = f(F), f(F, dt=torch.int64), f(F, d)
    sb = int(lib.rvcb200_op_ivf_scratch_bytes(F, nlist))
    assert sb > 0 and lib.rvcb200_op_ivf_scratch_bytes(-1, nlist) == -1 and lib.rvcb200_op_ivf_scratch_bytes(F, 0) == -1
    scratch = torch.empty(sb, dtype=torch.uint8, device=DEV)

    assign = lambda x_=_p(x), dt=0, ld=d, F_=F, d_=d, c=_p(cent), n=_p(cn), nl=nlist, o=_p(coarse): \
        lib.rvcb200_op_ivf_assign(x_, dt, ld, F_, d_, c, n, nl, o, _st())                              # noqa: E731
    assert assign() == 0
    for kw in (dict(x_=None), dict(dt=2), dict(ld=d - 1), dict(F_=-1), dict(d_=6), dict(d_=0), dict(c=None), dict(n=None), dict(nl=0),
               dict(o=None)):
        assert assign(**kw) == 1, kw

    scan = lambda x_=_p(x), dt=0, ld=d, F_=F, d_=d, c=_p(coarse), nl=nlist, of=_p(offs), v=_p(vec), lb=_p(lab), s=_p(scratch), n=sb, \
        sc=_p(score), i=_p(ix): lib.rvcb200_op_ivf_scan(x_, dt, ld, F_, d_, c, nl, of, v, lb, s, n, sc, i, _st())    # noqa: E731
    assert scan() == 0
    for kw in (dict(x_=None), dict(dt=-1), dict(ld=0), dict(F_=-2), dict(d_=10), dict(c=None), dict(nl=0), dict(of=None), dict(v=None),
               dict(lb=None), dict(s=None), dict(n=sb - 1), dict(sc=None), dict(i=None)):
        assert scan(**kw) == 1, kw

    blend = lambda f_=_p(x), dt=0, ld=d, F_=F, d_=d, sc=_p(score), i=_p(ix), v=_p(vec), p=_p(pos), nt=5, h=0, r=0.5, o=_p(out): \
        lib.rvcb200_op_index_blend(f_, dt, ld, F_, d_, sc, i, v, p, nt, h, r, o, _st())                 # noqa: E731
    assert blend() == 0
    for kw in (dict(f_=None), dict(dt=3), dict(ld=4), dict(F_=-1), dict(d_=18), dict(sc=None), dict(i=None), dict(v=None), dict(p=None),
               dict(nt=0), dict(h=2), dict(r=float("nan")), dict(r=float("inf")), dict(o=None)):
        assert blend(**kw) == 1, kw
    torch.cuda.synchronize()
