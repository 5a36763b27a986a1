"""B200-resident drop-in for the slice of the ``faiss`` module the reference calls.

Same names and call contracts as faiss (IndexFlatIP / IndexFlatL2 / Kmeans / normalize_L2 /
read_index / write_index), so the reference's own ``kmeans_faiss.py``, ``utils.py``,
``bag_of_visual_words.py`` and ``engine.py`` run unmodified on top of it
(``sys.modules["faiss"] = image_search_engine_b200.faiss_compat`` -- see INTEGRATION.md).

Reference call sites (under /root/reference/backend):
  kmeans_faiss.py:29-44,49   utils.py:300-327   engine.py:53-55,116,131
  bag_of_visual_words.py:187,194,213   siamese/test_index.py:53-54

Inputs may be NumPy arrays (host: copied to the GPU, results returned as NumPy with
Faiss's shapes/dtypes) or CUDA tensors (zero-copy, results returned as CUDA tensors).
All arithmetic runs in libise kernels; there is no CPU path.
"""
from __future__ import annotations

import struct
import threading
import time

import numpy as np
import torch

from . import ops
from ._lib import METRIC_IP, METRIC_L2, IseError

METRIC_INNER_PRODUCT = METRIC_IP
# METRIC_L2 imported above keeps faiss's value (1)

# faiss/utils/distances.cpp: below this many queries Faiss skips the BLAS expansion
distance_compute_blas_threshold = 20

_FLT_MAX = float(np.finfo(np.float32).max)


def _as_host_f32(x) -> np.ndarray:
    a = np.asarray(x)  # shares memory with np.matrix (SURVEY quirk Q4)
    if a.ndim != 2:
        raise AssertionError("expected a 2-D array")
    return a


def _to_device(x, dtype=torch.float32) -> tuple[torch.Tensor, bool]:
    """Returns (cuda tensor [n, d], input_was_torch_cuda)."""
    dev = ops.require_cuda()
    if isinstance(x, torch.Tensor):
        if x.dim() != 2:
            raise AssertionError("expected a 2-D tensor")
        if x.is_cuda:
            t = x if x.dtype in (torch.float32, torch.uint8) else x.to(torch.float32)
            return (t if t.stride(1) == 1 else t.contiguous()), True
        t = x
    else:
        a = _as_host_f32(x)
        if a.dtype == np.uint8:
            pass  # ORB / BRISK bytes travel as bytes; the float32 cast happens on the device
        elif a.dtype != np.float32:
            a = a.astype(np.float32)
        t = torch.from_numpy(np.ascontiguousarray(a))
    if t.dtype not in (torch.float32, torch.uint8):
        t = t.to(torch.float32)
    return t.to(dev, non_blocking=True), False


def normalize_L2(x) -> None:
    """faiss.normalize_L2: in place on the caller's buffer (utils.py:303 relies on that)."""
    if isinstance(x, torch.Tensor) and x.is_cuda:
        ops.normalize_l2_(x)
        return
    a = np.asarray(x)
    if a.dtype != np.float32 or a.ndim != 2 or not a.flags.c_contiguous:
        raise TypeError("normalize_L2 needs a C-contiguous float32 2-D array")
    dev = ops.require_cuda()
    t = torch.from_numpy(a).to(dev)
    ops.normalize_l2_(t)
    a[...] = t.cpu().numpy()


class IndexFlat:
    """Flat (exhaustive) index whose vectors live in HBM."""

    def __init__(self, d: int, metric: int = METRIC_L2):
        self.d = int(d)
        self.metric_type = int(metric)
        self.metric_arg = 0.0
        self.is_trained = True
        self.verbose = False
        self._chunks: list[torch.Tensor] = []
        self._ntotal = 0
        self._xb: torch.Tensor | None = None
        self._op: ops.Operand | None = None
        self._lock = threading.Lock()
        # "verified": coarse tensor-core pass + exact FP32 re-score with a proven candidate list;
        # "split": FP32-grade split products for every tile (see ops.search_topk)
        self.precision = "verified"

    # ---- storage ----
    @property
    def ntotal(self) -> int:
        return self._ntotal

    def add(self, x) -> None:
        t, _ = _to_device(x)
        if t.shape[1] != self.d:
            raise AssertionError(f"add: expected (n, {self.d}) array")
        if t.dtype != torch.float32:
            t = t.to(torch.float32)
        with self._lock:
            self._chunks.append(t.clone() if isinstance(x, torch.Tensor) and x.is_cuda else t)
            self._ntotal += t.shape[0]
            self._xb = None
            self._op = None

    def train(self, x) -> None:
        pass

    def reset(self) -> None:
        with self._lock:
            self._chunks, self._ntotal, self._xb, self._op = [], 0, None, None

    def _database(self) -> torch.Tensor:
        with self._lock:
            if self._xb is None:
                if not self._chunks:
                    dev = ops.require_cuda()
                    self._xb = torch.zeros((0, self.d), dtype=torch.float32, device=dev)
                elif len(self._chunks) == 1:
                    self._xb = self._chunks[0]
                else:
                    self._xb = torch.cat(self._chunks, dim=0)
                    self._chunks = [self._xb]
            return self._xb

    def _operand(self) -> ops.Operand:
        xb = self._database()
        with self._lock:
            if self._op is None:
                self._op = ops.attach_sample(ops.prepare_operand(xb))
            return self._op

    # ---- search ----
    def search(self, x, k: int):
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        q, was_cuda = _to_device(x)
        if q.shape[1] != self.d:
            raise AssertionError(f"search: expected (n, {self.d}) array")
        D, I = self._search_device(q, k)
        if was_cuda:
            return D, I
        return D.cpu().numpy(), I.cpu().numpy()

    def _search_device(self, q: torch.Tensor, k: int, need_distances: bool = True):
        """need_distances=False skips the exact FP32 re-score (callers that only use the ids, e.g.
        quantisation); the returned scores are then the tensor-core accumulator values."""
        nq = q.shape[0]
        largest = self.metric_type == METRIC_INNER_PRODUCT
        pad = -_FLT_MAX if largest else _FLT_MAX
        if self._ntotal == 0 or nq == 0:
            D = torch.full((nq, k), pad, dtype=torch.float32, device=q.device)
            I = torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
            return D, I
        kk = min(k, ops.MAX_TOPK)
        if k > ops.MAX_TOPK and self._ntotal > ops.MAX_TOPK:
            # beyond the fused-selection limit: exact pair scores + repeated masked selection passes (any k, like Faiss)
            qf = q if q.dtype == torch.float32 else q.to(torch.float32)
            return ops.search_exact_any_k(qf.contiguous(), self._database(), self.metric_type, k)
        if nq < distance_compute_blas_threshold:
            qf = q if q.dtype == torch.float32 else q.to(torch.float32)
            D, I = ops.flat_search_exact(qf.contiguous(), self._database(), self.metric_type, kk)
        else:
            b = self._operand()
            # nearest-column queries over raw float32 descriptors (quantisation: FaissKMeans.transform): the row
            # preparation runs inside the contraction kernel
            fused = ops.assign_fused(q, b, self.metric_type) if (kk == 1 and q.dtype == torch.float32) else None
            if fused is not None:
                D, I, a = fused
                if need_distances:
                    ops.rescore_topk_(q, self._database(), a, b, self.metric_type, D, I)
            else:
                a = ops.prepare_operand(q, rows=True)
                D, I = ops.search_topk(q, a, self._database(), b, self.metric_type, kk, precision=self.precision,
                                       need_distances=need_distances)
        if kk < k:
            Dp = torch.full((nq, k), pad, dtype=torch.float32, device=q.device)
            Ip = torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
            Dp[:, :kk], Ip[:, :kk] = D, I
            D, I = Dp, Ip
        return D, I

    def range_search(self, x, radius: float):
        """faiss IndexFlat::range_search: every stored vector scoring better than ``radius`` (IP: > radius, L2: squared
        distance < radius; strict, in FP32).  Returns (lims [nq + 1], D, I): the results of query i are
        D[lims[i]:lims[i+1]] / I[...] in ascending id.  NumPy input gives NumPy output (lims uint64, like Faiss's
        size_t array); CUDA tensors give CUDA tensors (lims int64)."""
        q, was_cuda = _to_device(x)
        if q.shape[1] != self.d:
            raise AssertionError(f"range_search: expected (n, {self.d}) array")
        lims, D, I = self._range_search_device(q, radius)
        if was_cuda:
            return lims, D, I
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    def _range_search_device(self, q: torch.Tensor, radius: float):
        nq = q.shape[0]
        if self._ntotal == 0 or nq == 0:
            return ops._range_empty(nq, q.device)
        if nq < distance_compute_blas_threshold:
            qf = q if q.dtype == torch.float32 else q.to(torch.float32)
            return ops.range_search_exact(qf.contiguous(), self._database(), self.metric_type, radius)
        b = self._operand()
        a = ops.prepare_operand(q, rows=True)
        return ops.range_search(q, a, self._database(), b, self.metric_type, radius)

    def assign(self, x, k: int = 1):
        return self.search(x, k)[1]

    def reconstruct(self, i: int) -> np.ndarray:
        return self._database()[int(i)].cpu().numpy()

    def reconstruct_n(self, i0: int = 0, ni: int = -1) -> np.ndarray:
        if ni < 0:
            ni = self._ntotal - i0
        return self._database()[i0:i0 + ni].cpu().numpy()

    def __repr__(self):
        name = "IndexFlatIP" if self.metric_type == METRIC_INNER_PRODUCT else "IndexFlatL2"
        return f"<image_search_engine_b200.{name} d={self.d} ntotal={self.ntotal} (HBM resident)>"

    # joblib/pickle: persist like faiss.serialize_index would (host copy of the vectors)
    def __getstate__(self):
        return {"d": self.d, "metric_type": self.metric_type, "xb": self.reconstruct_n()}

    def __setstate__(self, st):
        self.__init__(st["d"], st["metric_type"])
        if st["xb"].shape[0]:
            self.add(st["xb"])


class IndexFlatIP(IndexFlat):
    def __init__(self, d: int, metric: int = METRIC_INNER_PRODUCT):
        super().__init__(d, METRIC_INNER_PRODUCT)


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int, metric: int = METRIC_L2):
        super().__init__(d, METRIC_L2)


class IndexIVFPQ:
    """faiss.IndexIVFPQ as the reference builds it (utils.py:311-325): ``IndexIVFPQ(IndexFlatL2(d), d, 8, 16, 8)``,
    ``nprobe = 5``, ``train(data)`` then ``add(data)``; L2, by_residual.

    Training is the hot path's own machinery: level-1 clustering (nlist centroids, niter = 10) and one k-means
    per sub-quantizer (256 centroids on d/M-dimensional residual slices, niter = 25, seed 1234, at most 65 536
    training rows) run on the tensor-core assign + update kernels; vectors are encoded with the fused top-1
    assign; search probes the ``nprobe`` nearest lists and scans their codes with a shared-memory look-up table
    (``ise_ivfpq_scan``) followed by the canonical top-k selection.  Approximate by construction (8-bit codes):
    returned distances are sum_m |(q - c_list)_m - pq_m[code_m]|^2 like Faiss's.
    """

    def __init__(self, quantizer, d, nlist, M, nbits_per_idx, metric=METRIC_L2):
        if metric != METRIC_L2:
            raise NotImplementedError("the reference builds IndexIVFPQ with the default L2 metric only")
        if int(d) % int(M) != 0:
            raise RuntimeError("The dimension of the vector (d) should be a multiple of the number of "
                               "subquantizers (M)")
        if int(nbits_per_idx) != 8:
            raise NotImplementedError("8-bit codes only (utils.py:321)")
        self.quantizer, self.d, self.nlist = quantizer, int(d), int(nlist)
        self.M, self.nbits, self.ksub, self.dsub = int(M), 8, 256, int(d) // int(M)
        self.nprobe, self.by_residual, self.is_trained, self.metric_type = 1, True, False, METRIC_L2
        self.niter_coarse, self.pq_cp = 10, ClusteringParameters()
        self.pq_centroids = None            # [M, ksub, dsub] float32 (device)
        self._sub_index = None              # one flat L2 index per sub-quantizer (encoding)
        self._codes = self._ids = self._assign = None    # insertion order
        self._sorted = None                 # (codes, ids, list_offsets) grouped by list
        self._lock = threading.RLock()

    @property
    def ntotal(self) -> int:
        return 0 if self._ids is None else int(self._ids.shape[0])

    # -- training --
    def set_trained_state(self, coarse_centroids, pq_centroids) -> None:
        """Installs externally trained quantizers (lock-step tests against the oracle)."""
        cc, _ = _to_device(np.ascontiguousarray(coarse_centroids, dtype=np.float32))
        self.quantizer.reset()
        self.quantizer.add(cc)
        pq, _ = _to_device(np.ascontiguousarray(pq_centroids, dtype=np.float32).reshape(self.M * self.ksub, self.dsub))
        self._install_pq(pq.reshape(self.M, self.ksub, self.dsub))

    def _install_pq(self, pq: torch.Tensor) -> None:
        self.pq_centroids = pq.contiguous()
        self._sub_index = []
        for m in range(self.M):
            ix = IndexFlatL2(self.dsub)
            ix.add(self.pq_centroids[m])
            self._sub_index.append(ix)
        self.is_trained = True

    def train(self, x) -> None:
        xd, _ = _to_device(x)
        xd = xd.to(torch.float32)
        if xd.shape[1] != self.d:
            raise AssertionError(f"train: expected (n, {self.d}) array")
        if not (self.quantizer.ntotal == self.nlist):                      # IndexIVF::train_q1
            km = Kmeans(self.d, self.nlist, niter=self.niter_coarse, seed=1234)
            km.train(xd)
            self.quantizer.reset()
            self.quantizer.add(km.index._database())
        nmax = self.pq_cp.max_points_per_centroid * self.ksub              # train_residual: fvecs_maybe_subsample
        if xd.shape[0] > nmax:
            perm = ops.rand_perm_prefix(xd.shape[0], self.pq_cp.seed, nmax)
            xd = xd.index_select(0, torch.from_numpy(perm).to(xd.device))
        _, assign = self.quantizer._search_device(xd, 1, need_distances=False)
        res = ops.ivfpq_residual(xd, self.quantizer._database(), assign)
        pq = torch.empty((self.M, self.ksub, self.dsub), dtype=torch.float32, device=xd.device)
        for m in range(self.M):                                            # ProductQuantizer::train, Train_default
            km = Kmeans(self.dsub, self.ksub, niter=self.pq_cp.niter, seed=self.pq_cp.seed)
            km.train(res[:, m * self.dsub:(m + 1) * self.dsub].contiguous())
            pq[m] = km.index._database()
        self._install_pq(pq)

    # -- add / search --
    def _encode(self, xd: torch.Tensor):
        _, assign = self.quantizer._search_device(xd, 1, need_distances=False)
        assign = assign.reshape(-1)
        res = ops.ivfpq_residual(xd, self.quantizer._database(), assign)
        codes = torch.empty((xd.shape[0], self.M), dtype=torch.uint8, device=xd.device)
        for m in range(self.M):
            _, c = self._sub_index[m]._search_device(res[:, m * self.dsub:(m + 1) * self.dsub].contiguous(), 1,
                                                     need_distances=False)
            codes[:, m] = c.reshape(-1).to(torch.uint8)
        return assign, codes

    def add(self, x) -> None:
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        xd, _ = _to_device(x)
        xd = xd.to(torch.float32)
        if xd.shape[1] != self.d:
            raise AssertionError(f"add: expected (n, {self.d}) array")
        assign, codes = self._encode(xd)
        ids = torch.arange(self.ntotal, self.ntotal + xd.shape[0], dtype=torch.int64, device=xd.device)
        with self._lock:
            self._codes = codes if self._codes is None else torch.cat([self._codes, codes])
            self._assign = assign if self._assign is None else torch.cat([self._assign, assign])
            self._ids = ids if self._ids is None else torch.cat([self._ids, ids])
            self._sorted = None

    def _lists(self):
        with self._lock:
            if self._sorted is None:
                order = torch.argsort(self._assign, stable=True)           # lists keep insertion order
                counts = torch.bincount(self._assign, minlength=self.nlist)
                off = torch.zeros((self.nlist + 1,), dtype=torch.int64, device=counts.device)
                off[1:] = torch.cumsum(counts, 0)
                self._sorted = (self._codes.index_select(0, order).contiguous(), self._ids.index_select(0, order), off)
            return self._sorted

    def search(self, x, k: int):
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        q, was_cuda = _to_device(x)
        q = q.to(torch.float32)
        if q.shape[1] != self.d:
            raise AssertionError(f"search: expected (n, {self.d}) array")
        nq = q.shape[0]
        D = torch.full((nq, k), _FLT_MAX, dtype=torch.float32, device=q.device)
        I = torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
        if nq and self.ntotal:
            codes, ids, off = self._lists()
            _, probes = self.quantizer._search_device(q, min(self.nprobe, self.nlist), need_distances=False)
            for q0 in range(0, nq, 4096):                                  # bounds the [nq, ntotal] distance matrix
                qs = q[q0:q0 + 4096].contiguous()
                dist = ops.ivfpq_scan(qs, self.quantizer._database(), probes[q0:q0 + 4096], self.pq_centroids, codes, off)
                Dv, pos = ops.scores_topk_any_k_(dist, METRIC_L2, k)
                ok = pos >= 0
                I[q0:q0 + 4096] = torch.where(ok, ids[pos.clamp(min=0)], torch.full_like(pos, -1))
                D[q0:q0 + 4096] = Dv
        if was_cuda:
            return D, I
        return D.cpu().numpy(), I.cpu().numpy()

    def reset(self) -> None:
        with self._lock:
            self._codes = self._ids = self._assign = self._sorted = None

    # joblib / pickle: quantizers and codes as host arrays
    def __getstate__(self):
        host = lambda t: None if t is None else t.cpu().numpy()
        return dict(d=self.d, nlist=self.nlist, M=self.M, nprobe=self.nprobe, coarse=self.quantizer.reconstruct_n(),
                    pq=host(self.pq_centroids), codes=host(self._codes), assign=host(self._assign))

    def __setstate__(self, st):
        self.__init__(IndexFlatL2(st["d"]), st["d"], st["nlist"], st["M"], 8)
        self.nprobe = st["nprobe"]
        if st["pq"] is not None:
            self.set_trained_state(st["coarse"], st["pq"])
        if st["codes"] is not None:
            dev = ops.require_cuda()
            self._codes = torch.from_numpy(st["codes"]).to(dev)
            self._assign = torch.from_numpy(st["assign"]).to(dev)
            self._ids = torch.arange(self._codes.shape[0], dtype=torch.int64, device=dev)

    def __repr__(self):
        return (f"<image_search_engine_b200.IndexIVFPQ d={self.d} nlist={self.nlist} M={self.M} nprobe={self.nprobe} "
                f"ntotal={self.ntotal} (HBM resident)>")


# ------------------------------------------------------------------------------------------
# flat index file format (faiss/impl/index_write.cpp), so existing models/*.faiss files open
# ------------------------------------------------------------------------------------------
def write_index(index: IndexFlat, fname) -> None:
    if isinstance(index, IndexIVFPQ):
        raise NotImplementedError("only flat indexes are written in Faiss's file format; an IndexIVFPQ can be pickled")
    xb = index.reconstruct_n() if index.ntotal else np.zeros((0, index.d), np.float32)
    fourcc = b"IxFI" if index.metric_type == METRIC_INNER_PRODUCT else b"IxF2"
    with open(str(fname), "wb") as f:
        f.write(fourcc)
        f.write(struct.pack("<i", index.d))
        f.write(struct.pack("<q", index.ntotal))
        f.write(struct.pack("<q", 1 << 20))
        f.write(struct.pack("<q", 1 << 20))
        f.write(struct.pack("<B", 1))
        f.write(struct.pack("<i", index.metric_type))
        if index.metric_type > 1:
            f.write(struct.pack("<f", index.metric_arg))
        f.write(struct.pack("<Q", index.ntotal * index.d))
        f.write(np.ascontiguousarray(xb, dtype="<f4").tobytes())


def read_index(fname) -> IndexFlat:
    with open(str(fname), "rb") as f:
        fourcc = f.read(4)
        if fourcc not in (b"IxFI", b"IxF2", b"IxFl"):
            raise RuntimeError(f"unsupported index type {fourcc!r}: only flat indexes are on the hot path")
        (d,) = struct.unpack("<i", f.read(4))
        (ntotal,) = struct.unpack("<q", f.read(8))
        f.read(16)
        f.read(1)
        (metric,) = struct.unpack("<i", f.read(4))
        if metric > 1:
            f.read(4)
        (count,) = struct.unpack("<Q", f.read(8))
        if count != ntotal * d:
            raise RuntimeError("corrupt flat index payload")
        xb = np.frombuffer(f.read(count * 4), dtype="<f4").reshape(ntotal, d)
    idx = IndexFlatIP(d) if metric == METRIC_INNER_PRODUCT else IndexFlatL2(d)
    if ntotal:
        idx.add(xb)
    return idx


# ------------------------------------------------------------------------------------------
# k-means (faiss/Clustering.cpp + python/extra_wrappers.py Kmeans)
# ------------------------------------------------------------------------------------------
class ClusteringParameters:
    def __init__(self):
        self.niter = 25
        self.nredo = 1
        self.verbose = False
        self.spherical = False
        self.int_centroids = False
        self.update_index = False
        self.frozen_centroids = False
        self.min_points_per_centroid = 39
        self.max_points_per_centroid = 256
        self.seed = 1234
        self.decode_block_size = 32768


class Kmeans:
    """faiss.Kmeans with the Lloyd iterations on the B200.

    Per iteration: centroid planes (prepare) -> fused assign (tcgen05 contraction + argmax) ->
    scatter-add update -> mean / split-empty / renorm.  The multi-GPU variant (rows sharded over
    ranks, one NCCL all-reduce of the sum|count buffer per iteration) is parallel.ShardedKmeans.
    """

    def __init__(self, d, k, **kwargs):
        self.d = int(d)
        self.k = int(k)
        self.cp = ClusteringParameters()
        for key, v in kwargs.items():
            if key == "gpu":
                continue  # everything already runs on the GPU
            getattr(self.cp, key)
            setattr(self.cp, key, v)
        self.centroids = None
        self.obj = None
        self.iteration_stats = None
        self.index = None
        self.trace = None  # optional list: per-iteration device snapshots for lock-step tests
        self.precision = "verified"  # see ops.search_topk

    # -- helpers --
    def _post_process(self, cent: torch.Tensor):
        if self.cp.spherical:
            ops.normalize_l2_(cent)
        if self.cp.int_centroids:
            raise NotImplementedError("int_centroids is never set by the reference")

    def train(self, x, weights=None, init_centroids=None):
        if weights is not None:
            raise NotImplementedError("weights are never passed by the reference")
        cp, d, k = self.cp, self.d, self.k
        xd, _ = _to_device(x)
        n = xd.shape[0]
        assert xd.shape[1] == d
        if n < k:
            raise RuntimeError("Number of training points (%d) should be at least as large as number of "
                               "clusters (%d)" % (n, k))
        if n > k * cp.max_points_per_centroid:
            # Clustering::train validates ALL of its input before sub-sampling; without sub-sampling the check rides
            # on the operand conversion pass below
            if xd.dtype == torch.float32 and ops.has_nonfinite(xd):
                raise RuntimeError("input contains NaN's or Inf's")
            nsub = k * cp.max_points_per_centroid
            perm = ops.rand_perm_prefix(n, cp.seed, nsub)
            xd = xd.index_select(0, torch.from_numpy(perm).to(xd.device))
            n = nsub
        self.index = IndexFlatIP(d) if cp.spherical else IndexFlatL2(d)
        if n == k:
            cent = xd.to(torch.float32).clone()
            self.centroids = cent.cpu().numpy()
            self.iteration_stats = [dict(obj=0.0, time=0.0, time_search=0.0, imbalance_factor=1.0, nsplit=0)]
            self.obj = np.array([0.0])
            self.index.add(cent)
            return 0.0
        from .parallel import DeviceOps, lloyd_train      # the Lloyd loop is shared with the multi-GPU ShardedKmeans
        if k >= 1024:
            ops.split_plan_warm(min(k * 2048, 1 << 28))
        # row operand: one pass, per-row scales; the same pass rejects NaN / Inf like Clustering::train does
        a_op = ops.compact_operand(ops.prepare_operand(xd, rows=True), reject_nonfinite=True)
        cent, stats = lloyd_train(cp, d, k, xd, n, a_op, DeviceOps(),
                                  init_rows=lambda seed, n_input: self._initial_rows(xd, n, seed, n_input, k),
                                  init_centroids=init_centroids, trace=self.trace, precision=self.precision)
        self.index.add(cent)
        self.centroids = cent.cpu().numpy().reshape(k, d)
        self.iteration_stats = stats
        self.obj = np.array([s["obj"] for s in stats])
        return self.obj[-1] if self.obj.size else 0.0

    def _initial_rows(self, xd, n, seed, n_input, k):
        """centroids[i] = x[perm[i]] for i in [n_input, k) with perm = rand_perm(nx, seed)."""
        perm = ops.rand_perm_prefix(n, seed, k)[n_input:k]
        return xd.index_select(0, torch.from_numpy(perm).to(xd.device)).to(torch.float32)

    def assign(self, x):
        assert self.centroids is not None, "should train before assigning"
        D, I = self.index.search(x, 1)
        return D.ravel(), I.ravel()
