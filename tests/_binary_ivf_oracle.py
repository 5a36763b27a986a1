"""NumPy restatement of faiss.IndexBinaryIVF (faiss/IndexBinaryIVF.cpp, ~1.7.4), from memory, for the binary IVF tests.

Built on tests/_binary_oracle.py (Hamming distances) and oracle.faiss_shim (Clustering):
  - IndexBinaryIVF::IndexBinaryIVF: is_trained = (quantizer.ntotal == nlist), cp.niter = 10;
  - train: codes decoded to +-1 floats (bit j of byte i -> coordinate 8 i + j, LSB first, 1 -> +1, 0 -> -1), L2
    Clustering (seed 1234, <= 256 points per centroid), centroids thresholded back (> 0 -> 1);
  - add: ids ntotal + i, list = quantizer Hamming top-1 (lowest list id on ties), appended in insertion order;
  - search: quantizer top-min(nprobe, nlist) probes, exact Hamming over the probed lists, top-k in this repository's
    canonical (distance, id) order (not Faiss's heap order), padded with id -1 / 2^31 - 1;
  - range_search: distance < radius over the probed lists, by probe rank, then by position in the list.
"""
from __future__ import annotations

import numpy as np

from oracle import faiss_shim as fs
from tests._binary_oracle import INT32_MAX, hamming, knn_from_distances


def binary_to_real(codes: np.ndarray) -> np.ndarray:
    return np.unpackbits(np.asarray(codes, np.uint8), axis=1, bitorder="little").astype(np.float32) * 2 - 1


def real_to_binary(x: np.ndarray) -> np.ndarray:
    return np.packbits(np.asarray(x) > 0, axis=1, bitorder="little")


class IndexBinaryIVF:
    def __init__(self, quantizer_codes: np.ndarray | None, d: int, nlist: int):
        self.d, self.code_size, self.nlist = int(d), int(d) // 8, int(nlist)
        self.quantizer = np.zeros((0, self.code_size), np.uint8) if quantizer_codes is None else quantizer_codes
        self.nprobe = 1
        self.is_trained = self.quantizer.shape[0] == self.nlist
        self.reset()

    def reset(self) -> None:
        self.ids = [np.zeros(0, np.int64) for _ in range(self.nlist)]
        self.codes = [np.zeros((0, self.code_size), np.uint8) for _ in range(self.nlist)]
        self.ntotal = 0

    def train(self, x) -> None:
        x = np.asarray(x, np.uint8)
        if self.quantizer.shape[0] != self.nlist:
            cp = fs.ClusteringParameters()
            cp.niter = 10
            clus = fs.Clustering(self.d, self.nlist, cp)
            flat = fs.IndexFlatL2(self.d)
            clus.train(binary_to_real(x), flat)
            self.quantizer = real_to_binary(flat.reconstruct_n())
        self.is_trained = True

    def assign(self, x) -> np.ndarray:
        return knn_from_distances(hamming(np.asarray(x, np.uint8), self.quantizer), 1)[1].ravel()

    def add(self, x) -> None:
        assert self.is_trained
        x = np.asarray(x, np.uint8)
        self.add_preassigned(x, self.assign(x))

    def add_preassigned(self, x, assign) -> None:
        x = np.asarray(x, np.uint8)
        ids = np.arange(self.ntotal, self.ntotal + x.shape[0], dtype=np.int64)
        for l in np.unique(assign):
            sel = assign == l
            self.ids[l] = np.concatenate([self.ids[l], ids[sel]])
            self.codes[l] = np.concatenate([self.codes[l], x[sel]])
        self.ntotal += x.shape[0]

    def assignment(self) -> np.ndarray:
        out = np.empty(self.ntotal, np.int64)
        for l in range(self.nlist):
            out[self.ids[l]] = l
        return out

    def probes(self, x) -> np.ndarray:
        return knn_from_distances(hamming(np.asarray(x, np.uint8), self.quantizer), min(self.nprobe, self.nlist))[1]

    def _scanned(self, probes_row):
        lists = [l for l in probes_row if l >= 0 and self.ids[l].size]
        if not lists:
            return np.zeros((0, self.code_size), np.uint8), np.zeros(0, np.int64)
        return np.concatenate([self.codes[l] for l in lists]), np.concatenate([self.ids[l] for l in lists])

    def search(self, x, k: int, probes=None):
        x = np.asarray(x, np.uint8)
        nq = x.shape[0]
        D = np.full((nq, k), INT32_MAX, np.int32)
        I = np.full((nq, k), -1, np.int64)
        if nq == 0 or self.ntotal == 0 or not self.is_trained:
            return D, I
        coarse = self.probes(x) if probes is None else probes
        for qi in range(nq):
            y, ids = self._scanned(coarse[qi])
            if not ids.size:
                continue
            dist = hamming(x[qi:qi + 1], y)[0]
            order = np.lexsort((ids, dist))[:k]
            D[qi, :order.size], I[qi, :order.size] = dist[order], ids[order]
        return D, I

    def range_search(self, x, radius: int, probes=None):
        x = np.asarray(x, np.uint8)
        nq = x.shape[0]
        lims = np.zeros(nq + 1, np.uint64)
        Ds, Is = [], []
        if nq and self.ntotal and self.is_trained:
            coarse = self.probes(x) if probes is None else probes
            for qi in range(nq):
                y, ids = self._scanned(coarse[qi])           # probe rank, then list position
                dist = hamming(x[qi:qi + 1], y)[0] if ids.size else np.zeros(0, np.int32)
                hit = dist < radius
                Ds.append(dist[hit].astype(np.int32))
                Is.append(ids[hit])
                lims[qi + 1] = lims[qi] + hit.sum()
        D = np.concatenate(Ds) if Ds else np.zeros(0, np.int32)
        I = np.concatenate(Is) if Is else np.zeros(0, np.int64)
        return lims, D, I
