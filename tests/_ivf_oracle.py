"""fp64 restatement of the search faiss runs for an IndexIVFFlat with METRIC_L2 and nprobe 1 (IndexFlatL2: one list of every
vector in id order), the reference's blend weight, and seeded clustered test indices.

Tie rules: the coarse step takes the lowest centroid index among equal distances; the fine step scans the list in stored order and
keeps the earliest position among equal distances (faiss's heap replaces on a strict <).  An empty list gives (+inf, -1)."""
from __future__ import annotations

import numpy as np


def weight_rule(score: np.ndarray) -> np.ndarray:
    """vc_infer_pipeline.py:63-64 for k = 1 as single fp32 roundings: w = float32(1 / score)^2, weight = w / w."""
    s = np.asarray(score, dtype=np.float32)
    with np.errstate(divide="ignore", over="ignore", under="ignore", invalid="ignore"):
        r = np.float32(1.0) / s
        w = r * r
        return w / w


class IVFOracle:
    """`.search(x, k=1)` like the faiss object, computed in fp64; `detail(x)` adds the lists, the margins and the norms the GPU tests
    compare against."""

    def __init__(self, centroids, list_offsets, labels, vectors):
        self.centroids = np.asarray(centroids, dtype=np.float64)
        self.offs = np.asarray(list_offsets, dtype=np.int64)
        self.labels = np.asarray(labels, dtype=np.int64)
        self.vectors = np.asarray(vectors, dtype=np.float64)
        self.d = self.centroids.shape[1]
        self.ntotal = self.vectors.shape[0]
        self.nlist = self.centroids.shape[0]
        self.list_of_label = np.empty(self.ntotal, dtype=np.int64)
        for l in range(self.nlist):
            self.list_of_label[self.labels[self.offs[l]: self.offs[l + 1]]] = l
        self.seen = []                                  # detail() of every search() call

    def big_npy(self) -> np.ndarray:
        out = np.empty((self.ntotal, self.d), dtype=np.float32)
        out[self.labels] = self.vectors.astype(np.float32)
        return out

    @staticmethod
    def _sqdist(x: np.ndarray, y: np.ndarray) -> np.ndarray:
        return np.maximum((x * x).sum(1)[:, None] - 2.0 * x @ y.T + (y * y).sum(1)[None, :], 0.0)

    def detail(self, x) -> dict:
        x = np.asarray(x, dtype=np.float64)
        F = x.shape[0]
        dc = self._sqdist(x, self.centroids)
        lst = np.argmin(dc, axis=1)                                          # first minimum: lowest centroid index
        part = np.sort(dc, axis=1)
        cmargin = part[:, 1] - part[:, 0] if self.nlist > 1 else np.full(F, np.inf)
        dist = np.full(F, np.inf)
        ix = np.full(F, -1, dtype=np.int64)
        fmargin = np.full(F, np.inf)
        vnorm = np.zeros(F)
        for l in np.unique(lst):
            q = np.nonzero(lst == l)[0]
            a, b = self.offs[l], self.offs[l + 1]
            if a == b:
                continue
            dv = self._sqdist(x[q], self.vectors[a:b])
            j = np.argmin(dv, axis=1)                                        # first minimum: earliest list position
            dist[q] = dv[np.arange(len(q)), j]
            ix[q] = self.labels[a + j]
            vnorm[q] = (self.vectors[a + j] ** 2).sum(1)
            if b - a > 1:
                s = np.sort(dv, axis=1)
                fmargin[q] = s[:, 1] - s[:, 0]
        qn = (x * x).sum(1)
        cn = (self.centroids[lst] ** 2).sum(1)
        return dict(list=lst, ix=ix, dist=dist, cmargin=cmargin, fmargin=fmargin, tau_c=1e-5 * (qn + cn), tau_f=1e-5 * (qn + vnorm),
                    x=x)

    def in_regime(self, det: dict) -> np.ndarray:
        """Queries whose answer fp32 arithmetic cannot flip: both margins above tau = 1e-5 (||q||^2 + ||v||^2)."""
        return (det["cmargin"] > det["tau_c"]) & (det["fmargin"] > det["tau_f"])

    def search(self, x, k: int = 1):
        assert k == 1
        det = self.detail(x)
        self.seen.append(det)
        return det["dist"].astype(np.float32)[:, None], det["ix"][:, None]


def clustered(d: int, N: int, nlist: int, seed: int = 0, skew: bool = False, spread: float = 0.35):
    """A seeded index shaped like RVC's: nlist cluster centres (the centroids), N vectors around them, lists in cluster order and
    labels a random permutation.  skew: power-law list sizes with some empty lists.  Returns (centroids, offsets, labels, vectors)."""
    rng = np.random.default_rng(seed)
    cent = rng.standard_normal((nlist, d)).astype(np.float32)
    if nlist == 1:
        cent[:] = 0.0
        sizes = np.array([N])
    elif skew:
        w = 1.0 / np.arange(1, nlist + 1) ** 1.1
        w[rng.choice(nlist, max(1, nlist // 10), replace=False)] = 0.0      # empty lists
        sizes = rng.multinomial(N, w / w.sum())
    else:
        sizes = rng.multinomial(N, np.full(nlist, 1.0 / nlist))
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    owner = np.repeat(np.arange(nlist), sizes)
    vec = (cent[owner] + spread * rng.standard_normal((N, d))).astype(np.float32)
    if nlist == 1:
        vec = rng.standard_normal((N, d)).astype(np.float32)
    labels = rng.permutation(N).astype(np.int64)
    return cent, offs, labels, vec


def queries(vec: np.ndarray, F: int, seed: int = 1, noise: float = 0.3) -> np.ndarray:
    """F queries near random stored vectors (like frames of the voice the index was built from)."""
    rng = np.random.default_rng(seed)
    src = rng.integers(0, vec.shape[0], F)
    return (vec[src] + noise * rng.standard_normal((F, vec.shape[1]))).astype(np.float32)
