"""CPU: the device index's host side -- the fp64 IVF oracle, `IndexIVFFlatB200.from_arrays` / `from_faiss` (layout and refusals;
a CPU-resident index is only a container, it never searches) and the reference's blend weight rule."""
import sys
import types

import numpy as np
import pytest
import torch

from comfy_rvc_b200 import IndexIVFFlatB200, synthetic
from tests import _ivf_oracle


def test_oracle_with_one_list_agrees_with_fake_index():
    for d in (256, 768):
        fake = synthetic.FakeIndex(d, seed=5)
        big = fake.big_npy
        o = _ivf_oracle.IVFOracle(np.zeros((1, d)), [0, big.shape[0]], np.arange(big.shape[0]), big)
        x = torch.randn(300, d, generator=torch.Generator().manual_seed(d)).numpy()
        D0, I0 = fake.search(x, k=1)
        D1, I1 = o.search(x, k=1)
        assert I1.dtype == np.int64 and D1.dtype == np.float32 and I1.shape == D1.shape == (300, 1)
        assert np.array_equal(I0, I1)
        np.testing.assert_allclose(D1, D0, rtol=1e-6)
        assert np.array_equal(o.big_npy(), big)


def test_oracle_tie_rules_and_empty_list():
    d = 8
    cent = np.zeros((3, d))
    cent[1, 0] = 4.0
    cent[2] = cent[1]                                     # duplicated centroid: the lower index wins
    vec = np.zeros((4, d))
    vec[0, 0], vec[1, 0], vec[2, 0], vec[3, 0] = 4.5, 3.0, 3.0, 5.0
    o = _ivf_oracle.IVFOracle(cent, [0, 0, 4, 4], [3, 1, 0, 2], vec)   # list 0 empty, list 1 holds everything, list 2 empty
    x = np.zeros((3, d))
    x[0, 0] = 3.3                                         # nearest stored value 3.0 at positions 1 and 2: position 1 (label 1)
    x[1, 0] = 0.1                                         # list 0: empty
    x[2, 0] = 4.5                                         # equal to the vector at position 0: distance 0
    D, I = o.search(x)
    assert I[:, 0].tolist() == [1, -1, 3]
    assert D[1, 0] == np.inf and D[2, 0] == 0.0
    det = o.seen[-1]
    assert det["list"].tolist() == [1, 0, 1]


def test_weight_rule_matches_the_numpy_expression():
    """vc_infer_pipeline.py:63-64 (`np.square(1 / score)`, `weight /= weight.sum(axis=1, keepdims=True)`) for k = 1."""
    score = np.array([[0.0], [1e-30], [1e-20], [3.5], [0.125], [1e19], [1e30], [np.float32(3.4028235e38)], [np.inf]], dtype=np.float32)
    with np.errstate(divide="ignore", over="ignore", under="ignore", invalid="ignore"):
        w = np.square(1 / score)
        w /= w.sum(axis=1, keepdims=True)
    got = _ivf_oracle.weight_rule(score[:, 0])
    assert w.dtype == got.dtype == np.float32
    assert np.array_equal(np.isnan(w[:, 0]), np.isnan(got))
    assert np.array_equal(w[:, 0][~np.isnan(got)], got[~np.isnan(got)])
    assert np.isnan(got).tolist() == [True, True, True, False, False, False, True, True, True]   # 1e19: w is subnormal, not 0
    assert np.all(got[~np.isnan(got)] == 1.0)


def _arrays(d=16, nlist=5, N=40, seed=0):
    return _ivf_oracle.clustered(d, N, nlist, seed=seed)


def test_from_arrays_layout():
    cent, offs, labels, vec = _arrays()
    idx = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device="cpu")
    assert (idx.d, idx.ntotal, idx.nlist, idx.nprobe) == (16, 40, 5, 1)
    assert idx.list_offsets.dtype == torch.int32 and idx.list_offsets.tolist() == offs.tolist()
    assert idx.labels.dtype == torch.int64 and idx.labels.tolist() == labels.tolist()
    assert torch.equal(idx.vectors, torch.from_numpy(vec)) and torch.equal(idx.centroids, torch.from_numpy(cent))
    np.testing.assert_allclose(idx.cnorm.numpy(), (cent.astype(np.float64) ** 2).sum(1), rtol=1e-6)
    pos = idx.pos_of_label.numpy()
    assert np.array_equal(labels[pos], np.arange(40))
    big = idx.reconstruct_n(0, 40)                        # by label, like faiss's reconstruct_n
    o = _ivf_oracle.IVFOracle(cent, offs, labels, vec)
    assert np.array_equal(big, o.big_npy())
    assert np.array_equal(idx.reconstruct_n(7, 3), big[7:10])
    with pytest.raises(ValueError):
        idx.search(np.zeros((2, 16), np.float32), k=2)
    with pytest.raises(RuntimeError):                     # no CPU fallback
        idx.search(np.zeros((2, 16), np.float32))
    # tensors are accepted too
    idx2 = IndexIVFFlatB200.from_arrays(*(torch.from_numpy(a) for a in (cent, offs, labels, vec)), device="cpu")
    assert torch.equal(idx2.pos_of_label, idx.pos_of_label)


@pytest.mark.parametrize("case", ["dup_label", "label_range", "neg_label", "offs_start", "offs_end", "offs_down", "offs_len",
                                  "d_mod4", "vec_d", "no_lists", "float_labels", "empty"])
def test_from_arrays_refusals(case):
    cent, offs, labels, vec = _arrays()
    offs = offs.copy()
    labels = labels.copy()
    if case == "dup_label":
        labels[3] = labels[4]
    elif case == "label_range":
        labels[labels.argmax()] = 40
    elif case == "neg_label":
        labels[labels.argmin()] = -1
    elif case == "offs_start":
        offs[0] = 1
    elif case == "offs_end":
        offs[-1] = 39
    elif case == "offs_down":
        offs[2], offs[3] = offs[3], offs[2] - 1
    elif case == "offs_len":
        offs = offs[:-1]
    elif case == "d_mod4":
        cent, vec = cent[:, :14], vec[:, :14]
    elif case == "vec_d":
        vec = vec[:, :12]
    elif case == "no_lists":
        cent, offs = cent[:0], np.array([0])
    elif case == "float_labels":
        labels = labels.astype(np.float32)
    elif case == "empty":
        cent, offs, labels, vec = cent, np.zeros(6, np.int64), labels[:0], vec[:0]
    with pytest.raises(ValueError):
        IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device="cpu")


# ---- from_faiss against a stand-in that exposes exactly the faiss calls from_faiss documents ---------------------------------
class _Ptr:
    def __init__(self, arr):
        self.arr = arr


def _fake_faiss():
    m = types.ModuleType("faiss")
    m.METRIC_L2, m.METRIC_INNER_PRODUCT = 1, 0

    def extract_index_ivf(index):
        if not isinstance(index, _FakeIVF):
            raise RuntimeError("could not extract IVF index")
        return index

    def rev_swig_ptr(ptr, n):
        assert ptr.arr.size == n, "rev_swig_ptr called with a length other than the list's"
        return ptr.arr
    m.extract_index_ivf, m.rev_swig_ptr = extract_index_ivf, rev_swig_ptr
    return m


class _FakeQuantizer:
    def __init__(self, cent):
        self._cent = cent

    def reconstruct_n(self, i0, n):
        return self._cent[i0: i0 + n].copy()


class _FakeInvlists:
    def __init__(self, offs, labels, vec):
        self._offs, self._labels, self._vec = offs, labels, vec

    def list_size(self, l):
        return int(self._offs[l + 1] - self._offs[l])

    def get_ids(self, l):
        return _Ptr(self._labels[self._offs[l]: self._offs[l + 1]].astype(np.int64))

    def get_codes(self, l):
        return _Ptr(np.ascontiguousarray(self._vec[self._offs[l]: self._offs[l + 1]]).view(np.uint8).reshape(-1))


class _FakeIVF:
    def __init__(self, cent, offs, labels, vec, nprobe=1, metric_type=1, code_size=None):
        self.d, self.nlist, self.nprobe, self.metric_type = cent.shape[1], cent.shape[0], nprobe, metric_type
        self.code_size = 4 * self.d if code_size is None else code_size
        self.quantizer = _FakeQuantizer(cent)
        self.invlists = _FakeInvlists(offs, labels, vec)


class _FakeFlat:
    def __init__(self, vec, metric_type=1, code_size=None):
        self.d, self.ntotal, self.metric_type = vec.shape[1], vec.shape[0], metric_type
        self.code_size = 4 * self.d if code_size is None else code_size
        self._vec = vec

    def reconstruct_n(self, i0, n):
        return self._vec[i0: i0 + n].copy()


@pytest.fixture
def fake_faiss(monkeypatch):
    monkeypatch.setitem(sys.modules, "faiss", _fake_faiss())


def test_from_faiss_ivf_flat(fake_faiss):
    cent, offs, labels, vec = _ivf_oracle.clustered(16, 60, 6, seed=3, skew=True)
    assert np.any(np.diff(offs) == 0)                     # an empty list on the way
    idx = IndexIVFFlatB200.from_faiss(_FakeIVF(cent, offs, labels, vec), device="cpu")
    ref = IndexIVFFlatB200.from_arrays(cent, offs, labels, vec, device="cpu")
    for name in ("centroids", "cnorm", "list_offsets", "labels", "vectors", "pos_of_label"):
        assert torch.equal(getattr(idx, name), getattr(ref, name)), name


def test_from_faiss_flat_is_one_list(fake_faiss):
    fake = synthetic.FakeIndex(256, seed=5)
    idx = IndexIVFFlatB200.from_faiss(_FakeFlat(fake.big_npy), device="cpu")
    assert idx.nlist == 1 and idx.list_offsets.tolist() == [0, 48] and idx.labels.tolist() == list(range(48))
    assert np.array_equal(idx.reconstruct_n(0, 48), fake.big_npy)


@pytest.mark.parametrize("what", ["nprobe", "metric", "code_size", "labels", "flat_metric", "flat_code_size"])
def test_from_faiss_refusals(fake_faiss, what):
    cent, offs, labels, vec = _arrays()
    if what == "nprobe":
        index = _FakeIVF(cent, offs, labels, vec, nprobe=4)
    elif what == "metric":
        index = _FakeIVF(cent, offs, labels, vec, metric_type=0)
    elif what == "code_size":
        index = _FakeIVF(cent, offs, labels, vec, code_size=16)          # e.g. 8-bit scalar quantiser codes
    elif what == "labels":
        bad = labels.copy()
        bad[0] = bad[1]
        index = _FakeIVF(cent, offs, bad, vec)
    elif what == "flat_metric":
        index = _FakeFlat(vec, metric_type=0)
    else:
        index = _FakeFlat(vec, code_size=8)
    with pytest.raises(ValueError):
        IndexIVFFlatB200.from_faiss(index, device="cpu")
