"""NumPy restatement of faiss.IndexBinaryFlat (faiss/IndexBinaryFlat.cpp, faiss/utils/hamming.cpp, ~1.7.4), from memory.

Distances are popcounts of XORed uint64 words (np.bitwise_count), exact integers.  search returns the k smallest
(distance, id) pairs in that order -- among equal distances the lowest ids -- padded with id -1 / 2^31 - 1 (the neutral
value of Faiss's CMax<int32> heap, recalled); range_search keeps distance < radius, in ascending id."""
import numpy as np

INT32_MAX = 2**31 - 1


def _words(codes: np.ndarray) -> np.ndarray:
    """uint8 rows [n, code_size] -> uint64 words [n, ceil(code_size / 8)] (zero bytes appended)."""
    n, cs = codes.shape
    pad = np.zeros((n, (cs + 7) // 8 * 8), np.uint8)
    pad[:, :cs] = codes
    return pad.view(np.uint64)


def hamming(q: np.ndarray, x: np.ndarray, block_bytes: int = 1 << 28) -> np.ndarray:
    """[nq, nb] int32 Hamming distances between the rows of q and x (uint8 codes)."""
    qw, xw = _words(q), _words(x)
    out = np.empty((qw.shape[0], xw.shape[0]), np.int32)
    step = max(1, block_bytes // max(1, 8 * xw.shape[0] * xw.shape[1]))
    for i in range(0, qw.shape[0], step):
        out[i:i + step] = np.bitwise_count(qw[i:i + step, None, :] ^ xw[None, :, :]).sum(-1, dtype=np.int32)
    return out


def knn_from_distances(dist: np.ndarray, k: int):
    """(D int32 [nq, k], I int64 [nq, k]): the k smallest (distance, id) keys of every row, padded past ntotal."""
    nq, nb = dist.shape
    D = np.full((nq, k), INT32_MAX, np.int32)
    I = np.full((nq, k), -1, np.int64)
    kk = min(k, nb)
    if nq == 0 or kk == 0:
        return D, I
    key = dist.astype(np.int64) * nb + np.arange(nb, dtype=np.int64)[None, :]      # unique: (distance, id) order
    part = np.argpartition(key, kk - 1, axis=1)[:, :kk] if kk < nb else np.broadcast_to(np.arange(nb), (nq, nb))
    order = np.take_along_axis(part, np.argsort(np.take_along_axis(key, part, 1), axis=1), 1)
    I[:, :kk] = order
    D[:, :kk] = np.take_along_axis(dist, order, 1)
    return D, I


def range_from_distances(dist: np.ndarray, radius: int):
    """(lims uint64 [nq + 1], D int32, I int64): every id with distance < radius, ascending id per query."""
    hit = dist < radius
    lims = np.zeros(dist.shape[0] + 1, np.uint64)
    np.cumsum(hit.sum(1), out=lims[1:])
    rows, cols = np.nonzero(hit)           # row-major: ascending id inside a row
    return lims, dist[rows, cols].astype(np.int32), cols.astype(np.int64)


class IndexBinaryFlat:
    def __init__(self, d: int):
        if d % 8 != 0:
            raise RuntimeError("Error: 'd % 8 == 0' failed")
        self.d, self.code_size = d, d // 8
        self.codes = np.zeros((0, self.code_size), np.uint8)

    @property
    def ntotal(self) -> int:
        return self.codes.shape[0]

    def add(self, x) -> None:
        x = np.asarray(x)
        assert x.dtype == np.uint8 and x.shape[1] == self.code_size
        self.codes = np.concatenate([self.codes, x])

    def search(self, x, k: int):
        return knn_from_distances(hamming(np.asarray(x), self.codes), k)

    def range_search(self, x, radius: int):
        return range_from_distances(hamming(np.asarray(x), self.codes), radius)
