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

import operator
import struct
import threading
import time

import numpy as np
import torch

from . import ops
from ._lib import METRIC_IP, METRIC_L2, IseError

METRIC_INNER_PRODUCT = METRIC_IP
# METRIC_L2 imported above keeps faiss's value (1)

# faiss/utils/distances.cpp: below this many queries Faiss skips the BLAS expansion (the flat searches decide on
# ops.BLAS_THRESHOLD; this is faiss's name for the same value, read by engine.py)
distance_compute_blas_threshold = ops.BLAS_THRESHOLD


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
        return ops.flat_search(q, self._database(), self.metric_type, k, operand=self._operand, precision=self.precision,
                               need_distances=need_distances)

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
        return ops.flat_range_search(q, self._database(), self.metric_type, radius, operand=self._operand)

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
    assign; search probes the ``nprobe`` nearest lists and scans only their codes: the (query, probe) pairs are
    grouped by list, each pair gets one look-up table, and the partial top-k lists are merged (``ise_ivfpq_search``),
    so time and memory follow the probed lists.  For k > 128 (or M * ksub > 8192) the search scans into a
    [min(nq, 4096), ntotal] distance matrix (``ise_ivfpq_scan``) followed by the top-k selection instead.  Both return
    the same distances, sum_m |(q - c_list)_m - pq_m[code_m]|^2 like Faiss's; approximate by construction (8-bit
    codes).  Results are in the canonical (distance, id) order: among equal distances the lowest ids win.
    ``range_search`` filters the same lists by a radius (``ise_ivfpq_range_count`` / ``_fill``) in Faiss's probe order.
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
        """(codes, ids, list offsets, host list sizes): the codes grouped by list, rebuilt after add / reset."""
        with self._lock:
            if self._sorted is None:
                order = torch.argsort(self._assign, stable=True)           # lists keep insertion order (= ascending id)
                counts = torch.bincount(self._assign, minlength=self.nlist)
                off = torch.zeros((self.nlist + 1,), dtype=torch.int64, device=counts.device)
                off[1:] = torch.cumsum(counts, 0)
                self._sorted = (self._codes.index_select(0, order).contiguous(), self._ids.index_select(0, order), off,
                                counts.cpu().numpy())
            return self._sorted

    def _probes(self, q: torch.Tensor) -> torch.Tensor:
        return self.quantizer._search_device(q, min(self.nprobe, self.nlist), need_distances=False)[1]

    def _grouped(self, k: int) -> bool:
        """search scans the probed lists grouped by list; otherwise into a dense [min(nq, 4096), ntotal] matrix"""
        return k <= ops.MAX_TOPK and self.M * self.ksub <= ops.IVFPQ_MAX_TABLE

    def search(self, x, k: int):
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        q, was_cuda = _to_device(x)
        q = q.to(torch.float32)
        if q.shape[1] != self.d:
            raise AssertionError(f"search: expected (n, {self.d}) array")
        nq = q.shape[0]
        if not (nq and self.ntotal):
            D, I = ops.topk_padding(nq, k, METRIC_L2, q.device)
        elif self._grouped(k):
            codes, ids, off, sizes = self._lists()
            D, I = ops.ivfpq_search(q.contiguous(), self.quantizer._database(), self.pq_centroids, codes, ids, off,
                                    int(sizes.max()), self._probes(q), k)
        else:
            D, I = ops.topk_padding(nq, k, METRIC_L2, q.device)
            codes, ids, off, _ = self._lists()
            probes = self._probes(q)
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

    def range_search(self, x, radius: float):
        """IndexIVF::range_search: probe min(nprobe, nlist) lists as ``search`` does and return every stored code of
        them whose distance (the one ``search`` returns) is below ``radius``: strict, radius cast to float32.  Returns
        (lims [nq + 1], D, I); the results of query i are D[lims[i]:lims[i+1]] / I[...] in Faiss's scan order: by probe
        rank (nearest list first), then by position in the list (ids ascend inside a list).  NumPy input gives NumPy
        output (lims uint64); CUDA tensors give CUDA tensors (lims int64).  An untrained or empty index returns no
        results."""
        radius = float(radius)
        q, was_cuda = _to_device(x)
        if q.shape[1] != self.d:
            raise AssertionError(f"range_search: expected (n, {self.d}) array")
        q = q.to(torch.float32).contiguous()
        nq = q.shape[0]
        if nq and self.ntotal and self.is_trained:
            codes, ids, off, sizes = self._lists()
            lims, D, I = ops.ivfpq_range_search(q, self.quantizer._database(), self.pq_centroids, codes, ids, off,
                                                int(sizes.max()), self._probes(q), radius)
        else:
            lims, D, I = ops.range_empty(nq, q.device)
        if was_cuda:
            return lims, D, I
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    def get_list_size(self, list_no: int) -> int:
        sizes = self._lists()[3] if self.ntotal else np.zeros(self.nlist, np.int64)
        return int(sizes[int(list_no)])

    def get_list_ids(self, list_no: int) -> np.ndarray:
        """Ids stored in one list, in list order (InvertedLists::get_ids)."""
        if not self.ntotal:
            return np.zeros(0, np.int64)
        _, ids, off, _ = self._lists()
        l = int(list_no)
        return ids[int(off[l]):int(off[l + 1])].cpu().numpy()

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


class _InvertedLists:
    """The list-sorted storage of the IVF indexes (IndexIVFFlat: FP32 vectors, IndexBinaryIVF: padded code rows): one
    device copy of the rows grouped by list with their ids and list offsets; rows added since the last search are merged
    into it lazily at the next search.  Subclasses set ``nlist`` and ``_lock`` and call ``_clear`` in __init__."""

    def _clear(self) -> None:
        self._rows = self._ids = self._off = None   # list-sorted rows, their ids, list offsets [nlist + 1] (device)
        self._sizes = np.zeros(self.nlist, np.int64)   # host copy of the list sizes
        self._pending = []                              # (rows, list numbers, ids) added since the last search
        self._ntotal = 0

    @property
    def ntotal(self) -> int:
        return self._ntotal

    def _list_numbers(self, list_nos, n: int, device) -> torch.Tensor:
        lists = torch.as_tensor(np.asarray(list_nos) if not isinstance(list_nos, torch.Tensor) else list_nos)
        lists = lists.to(device=device, dtype=torch.int64).reshape(-1)
        if lists.shape[0] != n:
            raise AssertionError("add_preassigned: one list number per vector")
        if lists.shape[0] and not (0 <= int(lists.min()) and int(lists.max()) < self.nlist):
            raise AssertionError(f"add_preassigned: list numbers must lie in [0, {self.nlist})")
        return lists

    def _append(self, rows: torch.Tensor, lists: torch.Tensor) -> None:
        """Appends device rows (ids ntotal + i) to the given lists, in order."""
        sizes = torch.bincount(lists, minlength=self.nlist).cpu().numpy()
        with self._lock:
            ids = torch.arange(self._ntotal, self._ntotal + rows.shape[0], dtype=torch.int64, device=rows.device)
            self._pending.append((rows.contiguous(), lists, ids))
            self._sizes += sizes
            self._ntotal += rows.shape[0]

    def _lists(self):
        """Merges the pending rows into the list-sorted storage (stable by list: ids keep ascending in every list)."""
        with self._lock:
            if self._pending:
                first = self._pending[0][0]
                dev = first.device
                old = self._rows is not None
                parts_l = [torch.repeat_interleave(torch.arange(self.nlist, device=dev), torch.diff(self._off))] if old else []
                parts_l += [p[1] for p in self._pending]
                order = torch.argsort(torch.cat(parts_l), stable=True)
                dest = torch.empty_like(order)
                dest[order] = torch.arange(order.shape[0], device=dev)
                rows_all = torch.empty((self._ntotal,) + tuple(first.shape[1:]), dtype=first.dtype, device=dev)
                ids = torch.empty((self._ntotal,), dtype=torch.int64, device=dev)
                r0 = 0
                for rows, row_ids in ([(self._rows, self._ids)] if old else []) + [(p[0], p[2]) for p in self._pending]:
                    pos = dest[r0:r0 + rows.shape[0]]
                    rows_all.index_copy_(0, pos, rows)
                    ids.index_copy_(0, pos, row_ids)
                    r0 += rows.shape[0]
                off = np.zeros(self.nlist + 1, np.int64)
                np.cumsum(self._sizes, out=off[1:])
                self._rows, self._ids, self._off = rows_all, ids, torch.from_numpy(off).to(dev)
                self._pending = []
            return self._rows, self._ids, self._off

    def _insertion_order(self):
        """(rows, list numbers) in insertion order (ids 0 .. ntotal - 1), on the device: what pickling stores."""
        rows, ids, off = self._lists()
        xb = torch.empty_like(rows)
        xb[ids] = rows
        assign = torch.empty_like(ids)
        assign[ids] = torch.repeat_interleave(torch.arange(self.nlist, device=ids.device), torch.diff(off))
        return xb, assign

    def reset(self) -> None:
        with self._lock:
            self._clear()

    def get_list_size(self, list_no: int) -> int:
        return int(self._sizes[int(list_no)])

    def get_list_ids(self, list_no: int) -> np.ndarray:
        """Ids stored in one list, in list order (InvertedLists::get_ids)."""
        _, ids, off = self._lists() if self._ntotal else (None, None, None)
        if ids is None:
            return np.zeros(0, np.int64)
        l = int(list_no)
        return ids[int(off[l]):int(off[l + 1])].cpu().numpy()


class IndexIVFFlat(_InvertedLists):
    """faiss.IndexIVFFlat (faiss/IndexIVFFlat.cpp, ~1.7.4): an inverted file whose lists hold the raw FP32 vectors, so
    a search scans only the ``nprobe`` probed lists yet returns exact FP32 distances.  ``range_search`` filters the
    same lists by a radius (``ise_ivfflat_range_count`` / ``_fill``) and returns its results in Faiss's probe order.

    Training is the level-1 clustering of ``IndexIVFPQ`` (niter 10, seed 1234, spherical for inner product); vectors
    go to their quantizer top-1 list; a search probes ``min(nprobe, nlist)`` lists through the quantizer and scans
    them with ``ise_ivfflat_search`` (pairs grouped by list, exact FP32 scan, canonical merge).  Storage is one
    list-sorted FP32 copy of the vectors with their ids and list offsets; rows added since the last search are merged
    into it lazily at the next search.

    Ties: among exactly equal distances the lowest ids win (the flat index's canonical (distance, id) order, SURVEY
    Q5).  Faiss's heap keeps the first-scanned candidate when a tie falls exactly on the k-th place, which can be a
    higher id from an earlier-probed list; this index deliberately returns the canonical order instead.
    """

    def __init__(self, quantizer, d, nlist, metric=METRIC_L2):
        """IndexIVF::IndexIVF: the index is trained when the quantizer already holds nlist centroids."""
        if int(metric) not in (METRIC_L2, METRIC_INNER_PRODUCT):
            raise NotImplementedError("IndexIVFFlat supports METRIC_L2 and METRIC_INNER_PRODUCT")
        if quantizer.d != int(d):
            raise RuntimeError(f"quantizer dimension {quantizer.d} differs from the index dimension {int(d)}")
        self.quantizer, self.d, self.nlist, self.metric_type = quantizer, int(d), int(nlist), int(metric)
        self.nprobe = 1
        self.is_trained = quantizer.ntotal == self.nlist
        self._lock = threading.RLock()
        self._clear()

    def train(self, x) -> None:
        """Level1Quantizer::train_q1: k-means (niter 10, seed 1234, <= 256 points per centroid, spherical for inner
        product) unless the quantizer already holds nlist centroids; the centroids replace the quantizer's content."""
        xd, _ = _to_device(x)
        if xd.shape[1] != self.d:
            raise AssertionError(f"train: expected (n, {self.d}) array")
        if self.quantizer.ntotal != self.nlist:
            km = Kmeans(self.d, self.nlist, niter=10, seed=1234, spherical=self.metric_type == METRIC_INNER_PRODUCT)
            km.train(xd)
            self.quantizer.reset()
            self.quantizer.add(km.index._database())
        self.is_trained = True

    def add(self, x) -> None:
        """IndexIVF::add_with_ids(n, x, nullptr): ids ntotal + i, list = the quantizer's top-1 (lowest id on ties)."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        xd, _ = _to_device(x)
        if xd.shape[1] != self.d:
            raise AssertionError(f"add: expected (n, {self.d}) array")
        xd = xd.to(torch.float32)
        _, assign = self.quantizer._search_device(xd, 1, need_distances=False)
        self.add_preassigned(xd, assign.reshape(-1))

    def add_preassigned(self, x, list_nos) -> None:
        """IndexIVF::add_core with precomputed_idx: appends x (ids ntotal + i) to the given lists, in order."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        xd, was_cuda = _to_device(x)
        if xd.shape[1] != self.d:
            raise AssertionError(f"add: expected (n, {self.d}) array")
        xd = xd.to(torch.float32)
        if was_cuda and xd.data_ptr() == x.data_ptr():
            xd = xd.clone()
        self._append(xd, self._list_numbers(list_nos, xd.shape[0], xd.device))

    def search(self, x, k: int):
        """IndexIVF::search: probe min(nprobe, nlist) lists, exact FP32 scan (IVFFlatScanner: fvec_inner_product /
        fvec_L2sqr), top-k in the canonical (distance, id) order; padding id -1 / -+FLT_MAX."""
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        if k > ops.MAX_TOPK:
            raise NotImplementedError(f"IndexIVFFlat.search supports k <= {ops.MAX_TOPK}")
        q, was_cuda = _to_device(x)
        if q.shape[1] != self.d:
            raise AssertionError(f"search: expected (n, {self.d}) array")
        q = q.to(torch.float32).contiguous()
        nq = q.shape[0]
        if nq and self._ntotal and self.is_trained:
            xs, ids, off = self._lists()
            _, probes = self.quantizer._search_device(q, min(self.nprobe, self.nlist), need_distances=False)
            D, I = ops.ivfflat_search(q, xs, ids, off, int(self._sizes.max()), probes, self.metric_type, k)
        else:
            D, I = ops.topk_padding(nq, k, self.metric_type, q.device)
        if was_cuda:
            return D, I
        return D.cpu().numpy(), I.cpu().numpy()

    def range_search(self, x, radius: float):
        """IndexIVF::range_search: probe min(nprobe, nlist) lists as ``search`` does and return every vector of them
        whose exact FP32 score (IVFFlatScanner's direct formulas) beats ``radius``: IP dis > radius, L2 squared
        distance < radius, both strict, radius cast to float32.  Returns (lims [nq + 1], D, I); the results of query i
        are D[lims[i]:lims[i+1]] / I[...] in Faiss's scan order: by probe rank (nearest list first), then by position
        in the list (ids ascend inside a list).  This differs from IndexFlat.range_search, whose results come in
        ascending id.  NumPy input gives NumPy output (lims uint64); CUDA tensors give CUDA tensors (lims int64).  An
        untrained or empty index returns no results."""
        q, was_cuda = _to_device(x)
        if q.shape[1] != self.d:
            raise AssertionError(f"range_search: expected (n, {self.d}) array")
        q = q.to(torch.float32).contiguous()
        nq = q.shape[0]
        if nq and self._ntotal and self.is_trained:
            xs, ids, off = self._lists()
            _, probes = self.quantizer._search_device(q, min(self.nprobe, self.nlist), need_distances=False)
            lims, D, I = ops.ivfflat_range_search(q, xs, ids, off, int(self._sizes.max()), probes, self.metric_type,
                                                  radius)
        else:
            lims, D, I = ops.range_empty(nq, q.device)
        if was_cuda:
            return lims, D, I
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    # joblib / pickle: trained state, vectors and list numbers in insertion order (host arrays)
    def __getstate__(self):
        st = dict(d=self.d, nlist=self.nlist, metric_type=self.metric_type, nprobe=self.nprobe,
                  quantizer_metric=self.quantizer.metric_type, is_trained=self.is_trained,
                  coarse=self.quantizer.reconstruct_n(), xb=None, assign=None)
        if self._ntotal:
            xb, assign = self._insertion_order()
            st["xb"], st["assign"] = xb.cpu().numpy(), assign.cpu().numpy()
        return st

    def __setstate__(self, st):
        quantizer = IndexFlat(st["d"], st["quantizer_metric"])
        if st["coarse"].shape[0]:
            quantizer.add(st["coarse"])
        self.__init__(quantizer, st["d"], st["nlist"], st["metric_type"])
        self.nprobe, self.is_trained = st["nprobe"], st["is_trained"]
        if st["xb"] is not None:
            self.add_preassigned(st["xb"], st["assign"])

    def __repr__(self):
        return (f"<image_search_engine_b200.IndexIVFFlat d={self.d} nlist={self.nlist} nprobe={self.nprobe} "
                f"ntotal={self.ntotal} (HBM resident)>")


def _binary_rows(x, code_size: int, what: str):
    """uint8 code rows [n, code_size] as given (NumPy array or tensor), checked without device work: another dtype raises
    TypeError like faiss's _check_dtype_uint8, another shape AssertionError."""
    a = x if isinstance(x, torch.Tensor) else np.asarray(x)
    if a.dtype != (torch.uint8 if isinstance(a, torch.Tensor) else np.uint8):
        raise TypeError(f"{what}: binary codes must be uint8, got {a.dtype}")
    if a.ndim != 2 or a.shape[1] != code_size:
        raise AssertionError(f"{what}: expected (n, {code_size}) uint8 array")
    return a


class IndexBinaryFlat:
    """faiss.IndexBinaryFlat (faiss/IndexBinaryFlat.cpp, faiss/utils/hamming.cpp, ~1.7.4): exhaustive search over
    packed binary codes -- ORB (d = 256 bits), BRISK / FREAK (512), dHash (64) -- by Hamming distance.

    ``d`` is in bits (a multiple of 8, at most 2048: the scan keeps a query's words in registers); ``code_size = d // 8``.
    Codes are uint8 rows [n, code_size], NumPy or CUDA tensors, with ids ntotal + i; they live in HBM with each row
    padded with zero bytes to a multiple of 16.  ``search`` returns (D int32, I int64) sorted by (distance, id): among
    equal distances the lowest ids win, also when the tie falls on the k-th place.  ``range_search`` keeps every code with
    distance < radius, in ascending id, with the same distances.  Both run ``ise_binary_knn`` /
    ``ise_binary_range_count`` + ``_fill`` (XOR + popcount on CUDA cores, no [nq, ntotal] matrix).  Restated from
    memory like the rest of the Faiss semantics here (tests/_binary_oracle.py); no parity run against Faiss itself.
    """

    def __init__(self, d: int):
        d = int(d)
        if d <= 0 or d % 8 != 0:
            raise RuntimeError("Error: 'd % 8 == 0' failed")     # FAISS_THROW_IF_NOT in IndexBinary::IndexBinary
        if d // 8 > ops.BINARY_MAX_CODE_SIZE:
            raise NotImplementedError(f"IndexBinaryFlat supports d <= {8 * ops.BINARY_MAX_CODE_SIZE} bits")
        self.d, self.code_size = d, d // 8
        self.is_trained = True
        self.verbose = False
        self._lock = threading.Lock()
        self._chunks: list[torch.Tensor] = []    # padded device rows [n, pitch], in id order
        self._ntotal = 0
        self._codes: torch.Tensor | None = None  # their concatenation, built at the next search

    @property
    def ntotal(self) -> int:
        return self._ntotal

    def _device_rows(self, a) -> tuple[torch.Tensor, bool]:
        """Checked rows -> (zero-padded contiguous copy [n, pitch] on the device, input_was_cuda)."""
        dev = ops.require_cuda()
        was_cuda = isinstance(a, torch.Tensor) and a.is_cuda
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        rows = torch.zeros((t.shape[0], ops.binary_pitch(self.code_size)), dtype=torch.uint8, device=dev)
        rows[:, :self.code_size] = t.to(dev, non_blocking=True)
        return rows, was_cuda

    def add(self, x) -> None:
        rows, _ = self._device_rows(_binary_rows(x, self.code_size, "add"))
        with self._lock:
            self._chunks.append(rows)
            self._ntotal += rows.shape[0]
            self._codes = None

    def train(self, x) -> None:
        pass

    def reset(self) -> None:
        with self._lock:
            self._chunks, self._ntotal, self._codes = [], 0, None

    def _database(self) -> torch.Tensor:
        with self._lock:
            if self._codes is None:
                if not self._chunks:
                    dev = ops.require_cuda()
                    self._codes = torch.zeros((0, ops.binary_pitch(self.code_size)), dtype=torch.uint8, device=dev)
                else:
                    self._codes = self._chunks[0] if len(self._chunks) == 1 else torch.cat(self._chunks)
                    self._chunks = [self._codes]
            return self._codes

    def search(self, x, k: int):
        """hammings_knn_hc: the k nearest codes of every query, (D int32 [nq, k], I int64 [nq, k]) in the canonical
        (distance, id) order; when k > ntotal the tail is id -1 with D = 2^31 - 1 (the neutral value of Faiss's
        CMax<int32> heap, recalled rather than checked against Faiss).  1 <= k <= 128."""
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        if k > ops.MAX_TOPK:
            raise NotImplementedError(f"IndexBinaryFlat.search supports k <= {ops.MAX_TOPK}")
        q, was_cuda = self._device_rows(_binary_rows(x, self.code_size, "search"))
        db = self._database()
        if q.shape[0] and db.shape[0]:
            D, I = ops.binary_knn(q, db, self.code_size, k)
        else:
            D = torch.full((q.shape[0], k), 2**31 - 1, dtype=torch.int32, device=q.device)
            I = torch.full((q.shape[0], k), -1, dtype=torch.int64, device=q.device)
        if was_cuda:
            return D, I
        return D.cpu().numpy(), I.cpu().numpy()

    def range_search(self, x, radius: int):
        """hamming_range_search: every stored code with Hamming distance < radius (strict).  Returns (lims [nq + 1], D
        int32, I int64); the results of query i are D[lims[i]:lims[i+1]] / I[...] in ascending id.  NumPy input gives
        NumPy output (lims uint64, like Faiss's size_t array); CUDA tensors give CUDA tensors (lims int64)."""
        radius = operator.index(radius)
        q, was_cuda = self._device_rows(_binary_rows(x, self.code_size, "range_search"))
        lims, D, I = ops.binary_range_search(q, self._database(), self.code_size, radius)
        if was_cuda:
            return lims, D, I
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    def reconstruct(self, i: int) -> np.ndarray:
        return self._database()[int(i), :self.code_size].cpu().numpy()

    def reconstruct_n(self, i0: int = 0, ni: int = -1) -> np.ndarray:
        if ni < 0:
            ni = self._ntotal - i0
        return self._database()[i0:i0 + ni, :self.code_size].cpu().numpy()

    def __repr__(self):
        return f"<image_search_engine_b200.IndexBinaryFlat d={self.d} ntotal={self.ntotal} (HBM resident)>"

    # joblib / pickle: the codes as a host array
    def __getstate__(self):
        return {"d": self.d, "codes": self.reconstruct_n() if self._ntotal else np.zeros((0, self.code_size), np.uint8)}

    def __setstate__(self, st):
        self.__init__(st["d"])
        if st["codes"].shape[0]:
            self.add(st["codes"])


class IndexBinaryIVF(_InvertedLists):
    """faiss.IndexBinaryIVF (faiss/IndexBinaryIVF.cpp, ~1.7.4, recalled rather than checked against Faiss, like the rest
    of the Faiss semantics here; tests/_binary_ivf_oracle.py): an inverted file of binary codes whose probed lists are
    scanned by exact Hamming distance, for collections where IndexBinaryFlat's exhaustive scan is too slow.

    ``quantizer`` is an IndexBinaryFlat of the same ``d`` (bits, a multiple of 8, at most 2048) holding the nlist list
    codes.  ``train`` decodes a sample of the codes to +-1 floats, runs the L2 k-means of IndexIVFFlat (niter 10, seed
    1234, <= 256 points per centroid) and thresholds the centroids back to bits.  A code goes to the quantizer's Hamming
    top-1 (lowest list id on ties).  ``search`` probes ``min(nprobe, nlist)`` lists through the quantizer and returns
    (D int32, I int64) in the canonical (distance, id) order over their codes (``ise_binary_ivf_search``); as in
    IndexIVFFlat, this deliberately differs from Faiss's heap, which can keep a higher id from an earlier-probed list
    when a tie falls on the k-th place.  ``range_search`` keeps every code of the same lists with distance < radius, in
    Faiss's scan order: by probe rank, then by position in the list.  Codes live in HBM grouped by list, rows
    zero-padded to a multiple of 16 bytes."""

    def __init__(self, quantizer: IndexBinaryFlat, d: int, nlist: int):
        d = int(d)
        if d <= 0 or d % 8 != 0:
            raise RuntimeError("Error: 'd % 8 == 0' failed")
        if d // 8 > ops.BINARY_MAX_CODE_SIZE:
            raise NotImplementedError(f"IndexBinaryIVF supports d <= {8 * ops.BINARY_MAX_CODE_SIZE} bits")
        if quantizer.d != d:
            raise RuntimeError(f"quantizer dimension {quantizer.d} differs from the index dimension {d}")
        self.quantizer, self.d, self.code_size, self.nlist = quantizer, d, d // 8, int(nlist)
        self.nprobe = 1
        self.is_trained = quantizer.ntotal == self.nlist
        self.verbose = False
        self._lock = threading.RLock()
        self._clear()

    def train(self, x) -> None:
        """IndexBinaryIVF::train: unless the quantizer already holds nlist codes, k-means (L2, niter 10, seed 1234) on the
        codes decoded to +-1 floats, centroids thresholded back to bits (> 0 -> 1).  Only the <= 256 * nlist sampled
        codes are decoded, the sample Kmeans would draw (rand_perm prefix), which gives the result of decoding all."""
        a = _binary_rows(x, self.code_size, "train")
        if self.quantizer.ntotal != self.nlist:
            codes, _ = self.quantizer._device_rows(a)
            n, nmax = codes.shape[0], self.nlist * ClusteringParameters().max_points_per_centroid
            if n < self.nlist:
                raise RuntimeError("Number of training points (%d) should be at least as large as number of "
                                   "clusters (%d)" % (n, self.nlist))
            if n > nmax:
                perm = ops.rand_perm_prefix(n, 1234, nmax)
                codes = codes.index_select(0, torch.from_numpy(perm).to(codes.device))
            km = Kmeans(self.d, self.nlist, niter=10, seed=1234)
            km.train(ops.binary_to_real(codes, self.code_size))
            self.quantizer.reset()
            self.quantizer.add(ops.real_to_binary(km.index._database().contiguous(), self.code_size))
        self.is_trained = True

    def _assign(self, rows: torch.Tensor) -> torch.Tensor:
        """Quantizer Hamming top-1 of padded device rows (lowest list id on ties)."""
        return ops.binary_knn(rows, self.quantizer._database(), self.code_size, 1)[1].reshape(-1)

    def add(self, x) -> None:
        """IndexBinaryIVF::add_with_ids(n, x, nullptr): ids ntotal + i, list = the quantizer's top-1."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        rows, _ = self.quantizer._device_rows(_binary_rows(x, self.code_size, "add"))
        self._append(rows, self._assign(rows))

    def add_preassigned(self, x, list_nos) -> None:
        """IndexBinaryIVF::add_core with precomputed_idx: appends x (ids ntotal + i) to the given lists, in order."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        rows, _ = self.quantizer._device_rows(_binary_rows(x, self.code_size, "add"))
        self._append(rows, self._list_numbers(list_nos, rows.shape[0], rows.device))

    def _probes(self, q: torch.Tensor) -> torch.Tensor:
        nprobe = min(self.nprobe, self.nlist)
        return ops.binary_knn(q, self.quantizer._database(), self.code_size, nprobe)[1]

    def _check_nprobe(self) -> None:
        if min(self.nprobe, self.nlist) > ops.MAX_TOPK:
            raise NotImplementedError(f"IndexBinaryIVF probes at most {ops.MAX_TOPK} lists")

    def search(self, x, k: int):
        """IndexBinaryIVF::search: the k nearest codes of the min(nprobe, nlist) probed lists, (D int32 [nq, k], I int64
        [nq, k]) in the canonical (distance, id) order; fewer than k results leave id -1 / 2^31 - 1.  1 <= k <= 128."""
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")
        if k > ops.MAX_TOPK:
            raise NotImplementedError(f"IndexBinaryIVF.search supports k <= {ops.MAX_TOPK}")
        a = _binary_rows(x, self.code_size, "search")
        self._check_nprobe()
        q, was_cuda = self.quantizer._device_rows(a)
        nq = q.shape[0]
        if nq and self._ntotal and self.is_trained:
            codes, ids, off = self._lists()
            D, I = ops.binary_ivf_search(q, codes, ids, off, int(self._sizes.max()), self._probes(q), self.code_size, k)
        else:
            D = torch.full((nq, k), 2**31 - 1, dtype=torch.int32, device=q.device)
            I = torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
        if was_cuda:
            return D, I
        return D.cpu().numpy(), I.cpu().numpy()

    def range_search(self, x, radius: int):
        """IndexBinaryIVF::range_search: every code of the probed lists with Hamming distance < radius (strict), with the
        distances ``search`` returns.  Returns (lims [nq + 1], D int32, I int64); the results of query i are
        D[lims[i]:lims[i+1]] / I[...] by probe rank, then by position in the list (ids ascend inside a list).  NumPy
        input gives NumPy output (lims uint64); CUDA tensors give CUDA tensors (lims int64)."""
        radius = operator.index(radius)
        a = _binary_rows(x, self.code_size, "range_search")
        self._check_nprobe()
        q, was_cuda = self.quantizer._device_rows(a)
        nq = q.shape[0]
        if nq and self._ntotal and self.is_trained:
            codes, ids, off = self._lists()
            lims, D, I = ops.binary_ivf_range_search(q, codes, ids, off, int(self._sizes.max()), self._probes(q),
                                                     self.code_size, radius)
        else:
            lims, D, I = ops.range_empty(nq, q.device)
            D = D.to(torch.int32)
        if was_cuda:
            return lims, D, I
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    # joblib / pickle: quantizer codes, nprobe, codes and list numbers in insertion order (host arrays)
    def __getstate__(self):
        st = dict(d=self.d, nlist=self.nlist, nprobe=self.nprobe, is_trained=self.is_trained,
                  coarse=self.quantizer.__getstate__()["codes"], codes=None, assign=None)
        if self._ntotal:
            rows, assign = self._insertion_order()
            st["codes"], st["assign"] = rows[:, :self.code_size].cpu().numpy(), assign.cpu().numpy()
        return st

    def __setstate__(self, st):
        quantizer = IndexBinaryFlat(st["d"])
        if st["coarse"].shape[0]:
            quantizer.add(st["coarse"])
        self.__init__(quantizer, st["d"], st["nlist"])
        self.nprobe, self.is_trained = st["nprobe"], st["is_trained"]
        if st["codes"] is not None:
            self.add_preassigned(st["codes"], st["assign"])

    def __repr__(self):
        return (f"<image_search_engine_b200.IndexBinaryIVF d={self.d} nlist={self.nlist} nprobe={self.nprobe} "
                f"ntotal={self.ntotal} (HBM resident)>")


# ------------------------------------------------------------------------------------------
# flat index file format (faiss/impl/index_write.cpp), so existing models/*.faiss files open
# ------------------------------------------------------------------------------------------
def write_index(index: IndexFlat, fname) -> None:
    if isinstance(index, (IndexBinaryFlat, IndexBinaryIVF)):
        name = type(index).__name__
        raise NotImplementedError("Faiss writes binary indexes with write_index_binary (IBxF / IBwF), which is not "
                                  f"provided; an {name} can be pickled")
    if isinstance(index, (IndexIVFPQ, IndexIVFFlat)):
        name = type(index).__name__
        raise NotImplementedError(f"only flat indexes are written in Faiss's file format; an {name} can be pickled")
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
