"""Device-resident IVF-Flat index for the index blend of `VC.vc` (vc_infer_pipeline.py:59-75) without a host round trip.

    index = IndexIVFFlatB200.from_faiss(faiss.read_index("added_IVF1282_Flat_nprobe_1_x_v2.index"), device="cuda:0")
    vc.pipeline(..., file_index=index, index_rate=0.75, ...)          # or (index, big_npy), or vc.vc(..., index, None, ...)

It performs the search the reference's faiss call does for an `IndexIVFFlat` with METRIC_L2 and nprobe 1: the coarse quantiser
picks one list (lowest centroid index on an exact tie), that list is scanned exhaustively (earliest list position on an exact tie),
and the result is the top-1 in that list.  `IndexFlatL2` is the case of one list holding every vector in id order.  Distances are
fp32 FMA on the CUDA cores (csrc/index_kernels.cu); where two candidates are within fp32 rounding of each other the choice may
differ from faiss's own float rounding, otherwise it is the same neighbour.

`blend` then computes `big_npy[ix] * weight` with the reference's weight `w / w`, w = float32(1 / score)^2 (exactly 1.0, or NaN
for a score of 0 -- a query equal to a stored vector -- and for scores whose w over- or underflows), rounds to fp16 with
`is_half`, and blends with `index_rate` using the roundings of the reference's torch expression, into a new buffer.
"""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import numpy as np
import torch

from . import _lib

_DT = {torch.float32: 0, torch.float16: 1}


def _p(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(t.data_ptr())


class IndexIVFFlatB200:
    """IVF-Flat (nprobe 1, L2) index held on one device: fp32 centroids and their squared norms, CSR list offsets, and the
    vectors and labels in list order.  Labels are a permutation of 0..ntotal-1 (RVC adds its vectors in order and indexes
    `big_npy = reconstruct_n(0, ntotal)` by label).  Stands in for the faiss object: `d`, `ntotal`, `nprobe`, `reconstruct_n`,
    `search(x, k=1)`."""

    nprobe = 1

    def __init__(self, centroids, list_offsets, labels, vectors, device="cuda:0"):
        cent = np.ascontiguousarray(_host(centroids), dtype=np.float32)
        offs = np.asarray(_host(list_offsets))
        lab = np.asarray(_host(labels))
        vec = np.ascontiguousarray(_host(vectors), dtype=np.float32)
        if cent.ndim != 2 or cent.shape[0] < 1:
            raise ValueError("centroids must be [nlist >= 1][d]")
        nlist, d = cent.shape
        if d < 4 or d % 4 != 0:
            raise ValueError(f"d = {d}: the device index needs d % 4 == 0")
        if vec.ndim != 2 or vec.shape[1] != d:
            raise ValueError(f"vectors must be [ntotal][{d}]")
        ntotal = vec.shape[0]
        if ntotal < 1 or ntotal >= 2 ** 31:
            raise ValueError("the index needs 1 <= ntotal < 2^31 vectors")
        if offs.shape != (nlist + 1,) or not np.issubdtype(offs.dtype, np.integer):
            raise ValueError(f"list_offsets must be {nlist + 1} integers (CSR)")
        if offs[0] != 0 or offs[-1] != ntotal or np.any(np.diff(offs) < 0):
            raise ValueError("list_offsets must rise from 0 to ntotal")
        if lab.shape != (ntotal,) or not np.issubdtype(lab.dtype, np.integer):
            raise ValueError(f"labels must be {ntotal} integers")
        if lab.min() < 0 or lab.max() >= ntotal or np.bincount(lab, minlength=ntotal).max() != 1:
            raise ValueError("labels must be a permutation of 0..ntotal-1")
        dev = torch.device(device)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        pos = np.empty(ntotal, dtype=np.int32)
        pos[lab] = np.arange(ntotal, dtype=np.int32)
        self.d, self.ntotal, self.nlist, self.device = int(d), int(ntotal), int(nlist), dev
        self.centroids = torch.from_numpy(cent).to(dev)
        self.cnorm = torch.from_numpy(np.einsum("ij,ij->i", cent, cent, dtype=np.float32)).to(dev)
        self.list_offsets = torch.from_numpy(offs.astype(np.int32)).to(dev)
        self.labels = torch.from_numpy(lab.astype(np.int64)).to(dev)
        self.vectors = torch.from_numpy(vec).to(dev)
        self.pos_of_label = torch.from_numpy(pos).to(dev)

    @classmethod
    def from_arrays(cls, centroids, list_offsets, labels, vectors, device="cuda:0") -> "IndexIVFFlatB200":
        """centroids [nlist][d]; list_offsets [nlist + 1] (CSR: list l holds rows list_offsets[l]..list_offsets[l + 1] - 1 of
        `vectors` / `labels`, in the list's stored order); labels [ntotal], a permutation of 0..ntotal-1; vectors [ntotal][d]."""
        return cls(centroids, list_offsets, labels, vectors, device)

    @classmethod
    def from_faiss(cls, index, device="cuda:0") -> "IndexIVFFlatB200":
        """Copy a faiss `IndexIVFFlat` (METRIC_L2, nprobe 1) or `IndexFlatL2` to the device.  Uses only these faiss calls:
        `faiss.extract_index_ivf` (raises for a non-IVF index), `faiss.METRIC_L2`, `faiss.rev_swig_ptr`; the IVF object's
        `nlist`, `nprobe`, `d`, `metric_type`, `code_size`, `quantizer.reconstruct_n`, `invlists.list_size` / `get_ids` /
        `get_codes`; for a flat index its `d`, `ntotal`, `metric_type`, `code_size` and `reconstruct_n`.  Refuses (ValueError)
        nprobe != 1, a metric other than L2, codes that are not raw fp32 (code_size != 4 * d) and labels that are not a
        permutation of 0..ntotal-1.  A transform wrapper (IndexPreTransform) is refused by its changed `d`; an IndexIDMap or
        IndexRefine wrapper is not detected and must not be passed (`extract_index_ivf` unwraps it, and the inner index's ids
        would be taken as labels); RVC writes plain IndexIVFFlat files.  This method has been checked against a stand-in object
        exposing exactly the calls above, not against the faiss library itself."""
        import faiss
        try:
            ivf = faiss.extract_index_ivf(index)
        except Exception:  # noqa: BLE001 -- not an IVF index: IndexFlatL2 is one list of every vector in id order
            ivf = None
        if ivf is None:
            d = int(index.d)
            if int(index.metric_type) != int(faiss.METRIC_L2):
                raise ValueError("only METRIC_L2 indices run on the device")
            if int(getattr(index, "code_size", -1)) != 4 * d:
                raise ValueError("only raw fp32 codes (IndexFlatL2 or IndexIVFFlat) run on the device")
            n = int(index.ntotal)
            return cls(np.zeros((1, d), np.float32), np.array([0, n]), np.arange(n), index.reconstruct_n(0, n), device)
        d, nlist = int(ivf.d), int(ivf.nlist)
        if d != int(index.d):
            raise ValueError("the IVF index is wrapped in a transform; only a plain IndexIVFFlat runs on the device")
        if int(ivf.nprobe) != 1:
            raise ValueError(f"nprobe = {ivf.nprobe}: the device index searches one list (nprobe 1) only")
        if int(ivf.metric_type) != int(faiss.METRIC_L2):
            raise ValueError("only METRIC_L2 indices run on the device")
        if int(ivf.code_size) != 4 * d:
            raise ValueError(f"code_size {ivf.code_size} != 4 * d: only raw fp32 codes (IVF-Flat) run on the device")
        cent = np.asarray(ivf.quantizer.reconstruct_n(0, nlist), dtype=np.float32).reshape(nlist, d)
        inv = ivf.invlists
        sizes = np.array([int(inv.list_size(l)) for l in range(nlist)], dtype=np.int64)
        offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        labels = np.empty(int(offs[-1]), dtype=np.int64)
        vectors = np.empty((int(offs[-1]), d), dtype=np.float32)
        for l in range(nlist):
            n = int(sizes[l])
            if n:
                labels[offs[l]: offs[l + 1]] = faiss.rev_swig_ptr(inv.get_ids(l), n)
                codes = np.asarray(faiss.rev_swig_ptr(inv.get_codes(l), n * 4 * d), dtype=np.uint8)
                vectors[offs[l]: offs[l + 1]] = codes.view(np.float32).reshape(n, d)
        return cls(cent, offs, labels, vectors, device)

    # ---- faiss-compatible surface --------------------------------------------------------------------------------
    def reconstruct_n(self, i0: int, n: int) -> np.ndarray:
        """Vectors with labels i0..i0+n-1, fp32 [n][d] on the host (`big_npy` of pitch_extraction.py:64)."""
        if i0 < 0 or n < 0 or i0 + n > self.ntotal:
            raise ValueError("reconstruct_n: range outside 0..ntotal")
        return self.vectors[self.pos_of_label[i0: i0 + n].long()].cpu().numpy()

    def search(self, x, k: int = 1) -> Tuple[np.ndarray, np.ndarray]:
        """faiss's `search` for k = 1: (D float32 [n][1], I int64 [n][1]) on the host; I = -1, D = +inf where the chosen list is empty."""
        if k != 1:
            raise ValueError("the device index returns the top-1 only (k = 1)")
        q = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)).to(self._cuda())
        with torch.cuda.device(self.device):
            score, ix = self.search_device(q)
        return score.cpu().numpy()[:, None], ix.cpu().numpy()[:, None]

    # ---- the device path --------------------------------------------------------------------------------------------
    def _cuda(self) -> torch.device:
        if self.device.type != "cuda":
            raise RuntimeError("IndexIVFFlatB200 searches on a CUDA device only; there is no CPU fallback")
        return self.device

    def _queries(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() == 3 and x.shape[0] == 1:
            x = x[0]
        if x.dim() != 2 or x.shape[1] != self.d:
            raise ValueError(f"queries must be [F][{self.d}] (or [1][F][{self.d}])")
        if x.dtype not in _DT:
            raise ValueError(f"queries must be float32 or float16, not {x.dtype}")
        if x.device != self._cuda():
            raise ValueError(f"queries on {x.device}, index on {self.device}")
        if x.stride(1) != 1:
            x = x.contiguous()
        return x

    def _ld(self, x: torch.Tensor) -> int:
        return x.stride(0) if x.shape[0] > 1 else self.d                      # a single row may report any stride

    def search_device(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-1 of every row of x ([F][d] or [1][F][d], fp32 / fp16, on the index's device): (score fp32 [F], ix int64 [F]),
        enqueued on the current stream with no host synchronisation."""
        x = self._queries(x)
        F_ = int(x.shape[0])
        lib = _lib.load()
        dev = self.device
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        coarse = torch.empty(F_, dtype=torch.int64, device=dev)
        scratch = torch.empty(max(int(lib.rvcb200_op_ivf_scratch_bytes(F_, self.nlist)), 1), dtype=torch.uint8, device=dev)
        score = torch.empty(F_, dtype=torch.float32, device=dev)
        ix = torch.empty(F_, dtype=torch.int64, device=dev)
        dt = _DT[x.dtype]
        _lib.check(lib.rvcb200_op_ivf_assign(_p(x), dt, self._ld(x), F_, self.d, _p(self.centroids), _p(self.cnorm), self.nlist,
                                             _p(coarse), stream), None, "ivf_assign")
        _lib.check(lib.rvcb200_op_ivf_scan(_p(x), dt, self._ld(x), F_, self.d, _p(coarse), self.nlist, _p(self.list_offsets),
                                           _p(self.vectors), _p(self.labels), _p(scratch), scratch.numel(), _p(score), _p(ix), stream),
                   None, "ivf_scan")
        return score, ix

    def blend_ids(self, feats: torch.Tensor, score: torch.Tensor, ix: torch.Tensor, index_rate: float, is_half: bool) -> torch.Tensor:
        """The gather, weight and blend of vc_infer_pipeline.py:61-75 for given search results (`rvcb200_op_index_blend`)."""
        shape = feats.shape
        x = self._queries(feats)
        F_ = int(x.shape[0])
        if score.shape != (F_,) or ix.shape != (F_,) or score.dtype != torch.float32 or ix.dtype != torch.int64:
            raise ValueError("score / ix must be float32 / int64 [F]")
        out_dtype = torch.float16 if (is_half and x.dtype == torch.float16) else torch.float32
        out = torch.empty(F_, self.d, dtype=out_dtype, device=self.device)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.load().rvcb200_op_index_blend(_p(x), _DT[x.dtype], self._ld(x), F_, self.d, _p(score.contiguous()),
                                                      _p(ix.contiguous()), _p(self.vectors), _p(self.pos_of_label), self.ntotal,
                                                      1 if is_half else 0, float(index_rate), _p(out), stream), None, "index_blend")
        return out.view(shape)

    def blend(self, feats: torch.Tensor, index_rate: float, is_half: bool) -> torch.Tensor:
        """`feats` ([1][F][d] or [F][d], fp32 / fp16, on the index's device) blended with its nearest stored vectors exactly as
        vc_infer_pipeline.py:59-75 computes it, into a new buffer (`feats` is left as it is).  The result is fp16 when `is_half`
        and `feats` is fp16, fp32 otherwise (torch's promotion).  Enqueue-only: scratch comes from the caching allocator on
        the current stream and nothing waits for the device."""
        with torch.cuda.device(self._cuda()):
            score, ix = self.search_device(feats)
            return self.blend_ids(feats, score, ix, index_rate, is_half)


def _host(a):
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
