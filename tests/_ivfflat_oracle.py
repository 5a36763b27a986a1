"""NumPy restatement of Faiss's IndexIVFFlat, for the IVFFlat tests (test infrastructure only).

Follows upstream faiss/IndexIVF.cpp + faiss/IndexIVFFlat.cpp (~v1.7.4, recalled like the rest of oracle/faiss_shim.py,
whose Clustering and flat indexes it builds on; PARITY UNPINNED):
  - IndexIVF::IndexIVF: is_trained = (quantizer.ntotal == nlist); spherical clustering for inner product;
  - Level1Quantizer::train_q1: Clustering with niter 10 (seed 1234, <= 256 points per centroid), skipped when the
    quantizer already holds nlist centroids;
  - IndexIVF::add_with_ids(n, x, nullptr): ids ntotal + i, list = quantizer top-1 (lowest id on ties), appended in
    insertion order, so ids ascend inside every list;
  - IndexIVF::search: quantizer.search(x, min(nprobe, nlist)), then IVFFlatScanner over each probed list with the
    direct FP32 formulas fvec_inner_product / fvec_L2sqr (no norm expansion).  The top-k is taken in this
    repository's canonical (distance, id) order over the scanned set (lexsort), not Faiss's heap order.
"""
from __future__ import annotations

import numpy as np

from oracle import faiss_shim as fs

FLT_MAX = float(np.finfo(np.float32).max)


class IndexIVFFlat:
    def __init__(self, quantizer: fs.IndexFlat, d: int, nlist: int, metric: int = fs.METRIC_L2):
        if quantizer.d != d:
            raise RuntimeError("quantizer dimension differs from the index dimension")
        self.quantizer, self.d, self.nlist, self.metric_type = quantizer, int(d), int(nlist), int(metric)
        self.cp = fs.ClusteringParameters()
        self.cp.niter = 10
        self.cp.spherical = self.metric_type == fs.METRIC_INNER_PRODUCT
        self.nprobe = 1
        self.is_trained = quantizer.ntotal == self.nlist
        self.reset()

    def reset(self) -> None:
        self.ids = [np.zeros(0, np.int64) for _ in range(self.nlist)]
        self.vecs = [np.zeros((0, self.d), np.float32) for _ in range(self.nlist)]
        self.ntotal = 0

    def train(self, x) -> None:
        x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
        if self.quantizer.ntotal != self.nlist:
            clus = fs.Clustering(self.d, self.nlist, self.cp)
            self.quantizer.reset()
            clus.train(x, self.quantizer)
        self.is_trained = True

    def assign(self, x) -> np.ndarray:
        return self.quantizer.search(np.ascontiguousarray(x, dtype=np.float32), 1)[1].ravel()

    def add(self, x) -> None:
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
        self.add_preassigned(x, self.assign(x))

    def add_preassigned(self, x, assign) -> None:
        x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
        ids = np.arange(self.ntotal, self.ntotal + x.shape[0], dtype=np.int64)
        for l in np.unique(assign):
            sel = assign == l
            self.ids[l] = np.concatenate([self.ids[l], ids[sel]])
            self.vecs[l] = np.concatenate([self.vecs[l], x[sel]])
        self.ntotal += x.shape[0]

    def assignment(self) -> np.ndarray:
        """List number of every vector, in insertion order."""
        out = np.empty(self.ntotal, np.int64)
        for l in range(self.nlist):
            out[self.ids[l]] = l
        return out

    def probes(self, x) -> np.ndarray:
        x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
        return self.quantizer.search(x, min(self.nprobe, self.nlist))[1]

    def search(self, x, k: int, probes=None):
        x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
        nq = x.shape[0]
        ip = self.metric_type == fs.METRIC_INNER_PRODUCT
        D = np.full((nq, k), -FLT_MAX if ip else FLT_MAX, dtype=np.float32)
        I = np.full((nq, k), -1, dtype=np.int64)
        if nq == 0 or self.ntotal == 0 or not self.is_trained:
            return D, I
        coarse = self.probes(x) if probes is None else probes
        for qi in range(nq):
            lists = [l for l in coarse[qi] if l >= 0 and self.ids[l].size]
            if not lists:
                continue
            y = np.concatenate([self.vecs[l] for l in lists])
            ids = np.concatenate([self.ids[l] for l in lists])
            if ip:
                s = np.einsum("jd,d->j", y, x[qi], dtype=np.float32)
                order = np.lexsort((ids, -s))[:k]
            else:
                diff = y - x[qi]
                s = np.einsum("jd,jd->j", diff, diff, dtype=np.float32)
                order = np.lexsort((ids, s))[:k]
            D[qi, :order.size], I[qi, :order.size] = s[order], ids[order]
        return D, I
