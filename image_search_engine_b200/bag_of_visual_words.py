"""Drop-in for backend/bag_of_visual_words.py: BOVW (:40-120), run_clustering (:123-134),
train_bovw_model (:137-204) and load_cluster_model (:207-216).

What changes underneath: instead of one small Faiss search + one np.histogram call per image in a
Python loop (:98-106), all images' descriptors are packed into one matrix + an offsets vector,
quantised by ONE fused tcgen05 assign launch and binned by ONE histogram launch.  The per-image
results are identical to the loop's.

Kept quirks (SURVEY section 8a): np.histogram(idx, bins=k) bins over [min(idx), max(idx)] rather than
[0, k) (Q1) -- reproduced bit-exactly by ``hist_mode="numpy_compat"`` (default); ``"bincount"``
gives the intended word-id histogram.  ``transform`` ignores X when ``self.descriptions`` is set.
"""
from __future__ import annotations

import os
import threading
import time
from pathlib import Path

import joblib
import numpy as np
import torch
from sklearn.base import BaseEstimator
from sklearn.pipeline import Pipeline

from . import faiss_compat as faiss
from . import ops
from ._lib import HIST_BINCOUNT, HIST_NUMPY_COMPAT
from .kmeans_faiss import FaissKMeans
from .utils import OkapiTransformer, create_search_index

_HIST_MODES = {"numpy_compat": HIST_NUMPY_COMPAT, "bincount": HIST_BINCOUNT}
# Rate of the clear that runs beside the assign in histograms_device.  Any HBM stream beside the assign slows it: on a
# B200 (1000 W) at C2, 328 MB written unpaced cost the assign ~40-49 us and paced to 1-2 TB/s ~17-22 us (measured,
# profiles/microbench_hist_zeroed.py has the step-level A/B).  At 2 TB/s the clear lasts ~170 us, under a fifth of the
# C2 assign (100 descriptors of d = 128 per image).
_CLEAR_GB_PER_S = 2000.0


def describe_dataset(describer, X, prediction=False):
    """Input contract of the hot path (descriptors.py:104-139): a list with one (n_i, d) uint8/float32
    array per image.  Feature extraction (OpenCV / CNN) is upstream of the retrieval core: the host
    application's ``descriptors.describe_dataset`` is used when importable; a describer may also be any
    callable ``paths -> list[np.ndarray]``; a list of arrays passes through unchanged."""
    if isinstance(X, PackedDescriptions):
        return X
    if isinstance(X, (list, tuple)) and len(X) and isinstance(X[0], (np.ndarray, torch.Tensor)):
        return list(X)
    if callable(describer):
        return describer(X)
    try:
        from descriptors import describe_dataset as host_describe  # the reference's own module
    except Exception as exc:  # pragma: no cover - depends on the host application
        raise RuntimeError("no descriptor extractor available: pass descriptor arrays, a callable, "
                           "or put the application's descriptors.py on sys.path") from exc
    return host_describe(describer, X, prediction=prediction) if prediction else host_describe(describer, X)


class PackedDescriptions:
    """All images' descriptors as ONE [N, d] matrix (uint8 or float32) plus an int64 offsets vector
    (image i owns rows [offsets[i], offsets[i+1])).  This is the ragged-ingestion format of the GPU
    path: build it once (``pack_descriptions(list, pin=True)`` puts it in pinned host memory) and hand
    it to ``BOVW.transform`` / ``run_clustering`` instead of the Python list."""

    def __init__(self, matrix, offsets):
        self.matrix = matrix
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)

    def __len__(self):
        return self.offsets.shape[0] - 1

    def pin(self):
        if isinstance(self.matrix, np.ndarray):
            self.matrix = torch.from_numpy(self.matrix)
        if not self.matrix.is_cuda and not self.matrix.is_pinned():
            self.matrix = self.matrix.pin_memory()
        return self


def pack_descriptions(descriptions, pin=False):
    """list[(n_i, d)] -> (matrix [N, d], offsets int64 [n_img + 1]); dtype uint8 or float32."""
    if isinstance(descriptions, PackedDescriptions):
        return descriptions.matrix, descriptions.offsets
    if pin:
        m, o = pack_descriptions(descriptions)
        return PackedDescriptions(m, o).pin()
    if len(descriptions) == 0:
        raise ValueError("no images to quantise")
    counts = np.fromiter((len(x) for x in descriptions), dtype=np.int64, count=len(descriptions))
    offsets = np.zeros(len(descriptions) + 1, dtype=np.int64)
    np.cumsum(counts, out=offsets[1:])
    if isinstance(descriptions[0], torch.Tensor):
        return torch.cat(list(descriptions), dim=0), offsets
    same_u8 = all(x.dtype == np.uint8 for x in descriptions)
    mat = np.concatenate(descriptions, axis=0)
    if not same_u8 and mat.dtype != np.float32:
        mat = mat.astype(np.float32)
    return mat, offsets


class _ListPacker:
    """list[(n_i, d) float32 | uint8 ndarray] -> rows of a PERSISTENT pinned buffer (``bufs`` caches it across calls),
    copied by ``ise_pack_rows`` on host threads instead of one single-threaded np.concatenate
    (bag_of_visual_words.py:128) followed by a pin_memory copy.  float32 descriptors whose values are all integers in
    [0, 255] (OpenCV SIFT, ORB as float) can be narrowed to uint8 on the way: a quarter of the PCIe bytes, and the
    device widens uint8 for free.  Images are packed range by range (``pack(i0, i1, wire)``), so a caller can overlap
    the packing of the next chunk with the transfer and the kernels of the previous one.  ``ok`` is False when the
    list is not a plain list of C-contiguous same-dtype 2-D arrays (the caller then takes the generic path)."""

    def __init__(self, descriptions, bufs: dict, nthreads: int | None = None):
        import ctypes as C
        import os
        from . import _lib
        self.ok = False
        n_img = len(descriptions)
        if n_img == 0:
            return
        ptrs = np.empty(n_img, dtype=np.uint64)
        counts = np.empty(n_img, dtype=np.int64)
        try:
            from . import _fastlist                 # C walker (csrc/fastlist.c): ~20 ns per image
        except ImportError:                          # not built: same checks in the interpreter (~1.6 us per image)
            _fastlist = None
        if _fastlist is not None:
            got = _fastlist.walk(descriptions, ptrs.ctypes.data, counts.ctypes.data)
            if got is None:
                return
            dt, d = (np.dtype(np.float32), got[1]) if got[0] == 0 else (np.dtype(np.uint8), got[1])
        else:
            first = descriptions[0]
            if not isinstance(first, np.ndarray) or first.ndim != 2 or first.dtype not in (np.float32, np.uint8):
                return
            dt, d = first.dtype, int(first.shape[1])
            for i, a in enumerate(descriptions):
                if not isinstance(a, np.ndarray) or a.dtype != dt or a.ndim != 2 or a.shape[1] != d or not a.flags.c_contiguous:
                    return
                ptrs[i] = a.ctypes.data
                counts[i] = a.shape[0]
        offsets = np.zeros(n_img + 1, dtype=np.int64)
        np.cumsum(counts, out=offsets[1:])
        if int(offsets[-1]) == 0:
            return
        self._finish(descriptions, ptrs, offsets, int(d), dt == np.uint8, bufs, nthreads)

    def _finish(self, keep, ptrs, offsets, d, src_u8, bufs, nthreads):
        import ctypes as C
        from . import _lib
        self._keep = keep                            # the arrays must outlive the raw pointers
        self.ptrs, self.offsets, self.n_img, self.n_rows, self.d = ptrs, offsets, len(offsets) - 1, int(offsets[-1]), d
        self.src_u8 = src_u8
        self.bufs, self._lib, self._C = bufs, _lib, C
        self.nthreads = nthreads or self.default_threads()
        self.ok = True

    @staticmethod
    def default_threads() -> int:
        """The host cores this process may use, shared with the other ranks of the node (torchrun: LOCAL_WORLD_SIZE)."""
        import os
        try:
            cores = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            cores = os.cpu_count() or 1
        ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1))
        env = os.environ.get("ISE_PACK_THREADS")
        if env:
            return max(1, int(env))
        # two cores stay free for the calling thread (it feeds the copy engine and launches the kernels) and the driver
        return max(2, min(16, cores // ranks - 2))

    @classmethod
    def from_matrix(cls, mat: torch.Tensor, bufs: dict, block_rows: int = 4096, nthreads: int | None = None):
        """The same packer over an already packed float32 host matrix, cut into blocks of rows (its "images"): used to
        NARROW integer-valued descriptors to uint8 on the way to the device when the host has the cores for it."""
        self = cls.__new__(cls)
        self.ok = False
        n, d = int(mat.shape[0]), int(mat.shape[1])
        if n == 0 or mat.dtype != torch.float32 or mat.is_cuda or not mat.is_contiguous():
            return self
        starts = np.arange(0, n, block_rows, dtype=np.int64)
        offsets = np.append(starts, np.int64(n))
        ptrs = (np.uint64(mat.data_ptr()) + starts.astype(np.uint64) * np.uint64(d * 4)).astype(np.uint64)
        self._finish(mat, ptrs, offsets, d, False, bufs, nthreads)
        return self

    def wire_dtypes(self, try_u8: bool = True):
        """Wire formats to try, in order."""
        if self.src_u8:
            return [torch.uint8]
        return [torch.uint8, torch.float32] if try_u8 else [torch.float32]

    def view(self, wire: torch.dtype) -> torch.Tensor:
        kind = "u8" if wire == torch.uint8 else "f32"
        b = self.bufs.get(kind)
        if b is None or b.numel() < self.n_rows * self.d:
            b = torch.empty((max(self.n_rows * self.d, 1),), dtype=wire, pin_memory=True)
            self.bufs[kind] = b
        return b[: self.n_rows * self.d].view(self.n_rows, self.d)

    def pack(self, i0: int, i1: int, wire: torch.dtype) -> bool:
        """Copies images [i0, i1) to their rows of view(wire); False = a float32 value does not fit uint8."""
        C, _lib = self._C, self._lib
        ok = C.c_int(0)
        _lib.check(_lib.load().ise_pack_rows(
            C.c_void_p(self.ptrs.ctypes.data), C.c_void_p(self.offsets.ctypes.data), int(i0), int(i1), self.d,
            _lib.DTYPE_U8 if self.src_u8 else _lib.DTYPE_F32, _lib.DTYPE_U8 if wire == torch.uint8 else _lib.DTYPE_F32,
            C.c_void_p(self.view(wire).data_ptr()), self.nthreads, C.byref(ok)))
        return bool(ok.value)

    def begin(self, image_cuts: np.ndarray, wire: torch.dtype) -> None:
        """Starts packing the image ranges [image_cuts[c], image_cuts[c + 1]) in the background, in order."""
        C, _lib = self._C, self._lib
        self.end()
        self._cuts = np.ascontiguousarray(image_cuts, dtype=np.int64)
        job = C.c_void_p()
        _lib.check(_lib.load().ise_pack_begin(
            C.c_void_p(self.ptrs.ctypes.data), C.c_void_p(self.offsets.ctypes.data), C.c_void_p(self._cuts.ctypes.data),
            len(self._cuts) - 1, self.d, _lib.DTYPE_U8 if self.src_u8 else _lib.DTYPE_F32,
            _lib.DTYPE_U8 if wire == torch.uint8 else _lib.DTYPE_F32, C.c_void_p(self.view(wire).data_ptr()),
            self.nthreads, C.byref(job)))
        self._job = job

    def wait(self, chunk: int) -> bool:
        """Blocks until chunk ``chunk`` is in the pinned buffer; False = a float32 value does not fit uint8."""
        C, _lib = self._C, self._lib
        ok = C.c_int(0)
        _lib.check(_lib.load().ise_pack_wait(self._job, int(chunk), C.byref(ok)))
        return bool(ok.value)

    def poll(self, chunk: int):
        """(done, ok) without blocking: done = the workers have finished the chunk; ok = no value refused so far."""
        C, _lib = self._C, self._lib
        done, ok = C.c_int(0), C.c_int(0)
        _lib.check(_lib.load().ise_pack_poll(self._job, int(chunk), C.byref(done), C.byref(ok)))
        return bool(done.value), bool(ok.value)

    def claim(self, chunk: int) -> bool:
        """Takes a chunk the workers have not started away from them (the caller sends it in its source format)."""
        C, _lib = self._C, self._lib
        got = C.c_int(0)
        _lib.check(_lib.load().ise_pack_claim(self._job, int(chunk), C.byref(got)))
        return bool(got.value)

    def end(self) -> None:
        job = self.__dict__.pop("_job", None)
        if job is not None:
            self._lib.load().ise_pack_end(job)


def _pack_list_into(descriptions, bufs: dict, try_u8: bool = True, nthreads: int | None = None):
    """The whole list in one go: PackedDescriptions in the persistent pinned buffer, or None (see _ListPacker)."""
    pk = _ListPacker(descriptions, bufs, nthreads)
    if not pk.ok:
        return None
    for wire in pk.wire_dtypes(try_u8):
        if pk.pack(0, pk.n_img, wire):
            return PackedDescriptions(pk.view(wire), pk.offsets)
    return None


def _narrow_on_the_wire(mat, n_chunks: int) -> bool:
    """Whether a packed float32 host matrix is worth narrowing to uint8 for the host -> device copy: the narrowing pass
    reads the matrix once on host threads, so it only pays when this process has cores (and memory bandwidth) to spare
    -- measured: 1 - 2 ranks per node yes; 8 ranks sharing the host no (profiles/r02_findings.md section 3).
    ISE_NARROW_PINNED=0 / 1 overrides."""
    import os
    if not isinstance(mat, torch.Tensor) or mat.is_cuda or mat.dtype != torch.float32 or not mat.is_pinned():
        return False
    if not mat.is_contiguous() or mat.shape[0] < 8192 * n_chunks:
        return False
    env = os.environ.get("ISE_NARROW_PINNED")
    if env is not None:
        return env == "1"
    return _ListPacker.default_threads() >= 6


class BOVW(BaseEstimator):
    """Bag of Visual Words: describe -> cluster (codebook) -> quantise -> per-image histogram."""

    def __init__(self, describer, n_clusters=10, hist_mode="numpy_compat"):
        self.describer = describer
        self.n_clusters = n_clusters
        self.hist_mode = hist_mode

    def __getstate__(self):
        # copy first: on Python >= 3.11 BaseEstimator.__getstate__ hands back the LIVE __dict__, and popping from it
        # would drop the caches of the estimator being pickled
        state = dict(super().__getstate__())
        for key in ("_pipe_cache", "_csr_cache", "_csr_bufs", "_pipe_lock", "_pack_bufs", "_last_transfer",
                    "_clear_streams"):   # CUDA streams / events / staging buffers / locks are not persisted
            state.pop(key, None)
        return state

    def _lock(self):
        """Guards the cached staging buffers, pinned result buffers, side streams and events of the pipelined host
        paths (histograms_host / transform_csr): the reference serves queries from a threaded Flask server
        (engine.py:137) and fans transform out over joblib threads (bag_of_visual_words.py:108-113), so two threads
        may call the same BOVW at once; the pipelines are then serialised per object instead of overwriting each
        other's buffers."""
        lk = self.__dict__.get("_pipe_lock")
        if lk is None:
            lk = self.__dict__.setdefault("_pipe_lock", threading.RLock())
        return lk

    def fit(self, X, y=None):
        self.descriptions = describe_dataset(self.describer, X)
        self.clusterer = run_clustering(self.descriptions, self.n_clusters)
        return self

    def transform(self, X, y=None, output="numpy", out=None):
        """float64 (n_images, n_clusters) histogram matrix; ``output="device"`` keeps it in HBM,
        ``out=`` is an optional pinned CPU tensor that receives the result."""
        descriptions = getattr(self, "descriptions", None)
        if descriptions is None:
            descriptions = describe_dataset(self.describer, X, prediction=True)
        if output != "device" and out is not None:
            return self.histograms_host(descriptions, out)
        H = self.histograms_device(descriptions)
        if output == "device":
            return H
        return _to_host(H, out)

    def histograms_host(self, descriptions, out: torch.Tensor, *, okapi: OkapiTransformer | None = None,
                        n_chunks: int = 8) -> np.ndarray:
        with self._lock():
            return self._histograms_host(descriptions, out, okapi=okapi, n_chunks=n_chunks)

    def _histograms_host(self, descriptions, out: torch.Tensor, *, okapi: OkapiTransformer | None = None,
                         n_chunks: int = 8) -> np.ndarray:
        """Host descriptors in, host histogram matrix out, with the three legs overlapped: the images are
        cut into ``n_chunks`` groups and chunk i+1's H2D copy, chunk i's kernels and chunk i-1's D2H copy
        run concurrently on three streams (PCIe is full duplex).  ``out`` must be a pinned CPU tensor
        [n_images, n_clusters] (float64 or float32); ``pack_descriptions(..., pin=True)`` pins the input."""
        if self.hist_mode not in _HIST_MODES:
            raise ValueError(f"hist_mode must be one of {sorted(_HIST_MODES)}")
        dev = ops.require_cuda()
        mat, offsets = pack_descriptions(descriptions)
        if isinstance(mat, np.ndarray):
            mat = torch.from_numpy(mat)
        n_img = len(offsets) - 1
        if tuple(out.shape) != (n_img, int(self.n_clusters)) or not out.is_pinned():
            raise ValueError("out must be a pinned CPU tensor of shape (n_images, n_clusters)")
        if mat.is_cuda or n_img < 2 * n_chunks:
            H = self.histograms_device(descriptions, okapi=okapi, out_dtype=out.dtype)
            return _to_host(H, out)
        kw = dict(mode=_HIST_MODES[self.hist_mode], out_dtype=out.dtype)
        if okapi is not None:
            total = float(offsets[-1] - offsets[0])
            kw.update(okapi=True, k1=okapi.k1, k2=okapi.k2, b=okapi.b, avgdl=total / n_img)   # batch-wide avgdl
        # chunk boundaries in images, balanced by descriptor count
        targets = offsets[0] + (offsets[-1] - offsets[0]) * np.arange(1, n_chunks) / n_chunks
        cuts = np.unique(np.concatenate([[0], np.searchsorted(offsets, targets), [n_img]])).astype(np.int64)
        max_rows = int(max(offsets[i1] - offsets[i0] for i0, i1 in zip(cuts[:-1], cuts[1:])))
        max_imgs = int(np.diff(cuts).max())
        # Device staging buffers, streams and events are created once and reused: allocating per call
        # through the caching allocator across three streams forces cudaMalloc/cudaFree churn that
        # costs more than the copies themselves (profiles/r01_findings.md).
        NB = 3
        key = (max_rows, int(mat.shape[1]), mat.dtype, max_imgs, int(self.n_clusters), out.dtype, str(dev))
        pc = self.__dict__.get("_pipe_cache")
        if pc is None or pc["key"] != key:
            pc = dict(key=key, s_in=torch.cuda.Stream(), s_out=torch.cuda.Stream(),
                      xd=[torch.empty((max_rows, mat.shape[1]), dtype=mat.dtype, device=dev) for _ in range(NB)],
                      H=[torch.empty((max_imgs, int(self.n_clusters)), dtype=out.dtype, device=dev) for _ in range(NB)],
                      ev_in=[torch.cuda.Event() for _ in range(NB)], ev_c=[torch.cuda.Event() for _ in range(NB)],
                      ev_out=[torch.cuda.Event() for _ in range(NB)])
            self.__dict__["_pipe_cache"] = pc
        main, s_in, s_out = torch.cuda.current_stream(), pc["s_in"], pc["s_out"]
        off_dev = torch.from_numpy(offsets).to(dev)
        s_in.wait_stream(main)
        s_out.wait_stream(main)
        for ci, (i0, i1) in enumerate(zip(cuts[:-1], cuts[1:])):
            b = ci % NB
            r0, r1 = int(offsets[i0]), int(offsets[i1])
            ni, nr = int(i1 - i0), r1 - r0
            xd, H = pc["xd"][b][:nr], pc["H"][b][:ni]
            with torch.cuda.stream(s_in):
                if ci >= NB:
                    s_in.wait_event(pc["ev_c"][b])        # kernels of chunk ci-NB are done with this buffer
                xd.copy_(mat[r0:r1], non_blocking=True)
                pc["ev_in"][b].record(s_in)
            main.wait_event(pc["ev_in"][b])
            if ci >= NB:
                main.wait_event(pc["ev_out"][b])          # D2H of chunk ci-NB has drained this H buffer
            words = self.clusterer.transform_device(xd)
            ops.bovw_histogram(words, off_dev[i0:i1 + 1] - r0, int(self.n_clusters), out=H, **kw)
            pc["ev_c"][b].record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(pc["ev_c"][b])
                out[int(i0):int(i1)].copy_(H, non_blocking=True)
                pc["ev_out"][b].record(s_out)
        s_out.synchronize()
        return out.numpy()

    # ---- CSR path: what `Pipeline([bovw, tfidf]).transform(...)` returns in the reference is a scipy CSR
    # matrix (utils.py:153-202); building it on the device never materialises the dense matrix ----
    def _csr_kwargs(self, okapi):
        if self.hist_mode not in _HIST_MODES:
            raise ValueError(f"hist_mode must be one of {sorted(_HIST_MODES)}")
        kw = dict(mode=_HIST_MODES[self.hist_mode])
        if okapi is not None:
            kw.update(okapi=True, k1=okapi.k1, k2=okapi.k2, b=okapi.b)
        return kw

    def csr_device(self, descriptions, *, okapi: OkapiTransformer | None = None, out_dtype=torch.float64):
        """(indptr int32, indices int32, data) CUDA tensors of the histogram (+ Okapi tf) matrix; the used length
        of indices / data is indptr[-1]."""
        dev = ops.require_cuda()
        mat, offsets = pack_descriptions(descriptions)
        xd = mat.to(dev, non_blocking=True) if isinstance(mat, torch.Tensor) else \
            torch.from_numpy(mat).to(dev, non_blocking=True)
        off = torch.from_numpy(offsets).to(dev, non_blocking=True)
        words = self.clusterer.transform_device(xd)
        return ops.bovw_histogram_csr(words, off, int(self.n_clusters), out_dtype=out_dtype, **self._csr_kwargs(okapi))

    def transform_csr(self, X=None, *, okapi: OkapiTransformer | None = None, n_chunks: int = 8, copy: bool = True):
        with self._lock():
            return self._transform_csr(X, okapi=okapi, n_chunks=n_chunks, copy=copy)

    def _transform_csr(self, X=None, *, okapi: OkapiTransformer | None = None, n_chunks: int = 8, copy: bool = True):
        """Host descriptors in, scipy CSR float64 (n_images, n_clusters) out == OkapiTransformer().transform(
        BOVW.transform(X)) of the reference (``okapi=None``: the plain histogram as CSR).  The host -> device copy
        of the descriptors is cut into ``n_chunks`` pieces overlapped with the quantisation of the previous
        piece; the ids stay in HBM, the CSR arrays are built there for the whole batch and come back in one
        small copy (~12 B per non-zero instead of 8 B per matrix cell).  ``copy=False`` returns a matrix that
        aliases this object's pinned result buffers (valid until the next call)."""
        import scipy.sparse as sp
        # like transform(): cached descriptions win over X (bag_of_visual_words.py:89-92), except that an explicit
        # PackedDescriptions batch is always taken as given
        descriptions = X if isinstance(X, PackedDescriptions) else getattr(self, "descriptions", None)
        if descriptions is None:
            descriptions = describe_dataset(self.describer, X, prediction=True)
        dev = ops.require_cuda()
        k = int(self.n_clusters)
        packer = None
        if isinstance(descriptions, (list, tuple)) and len(descriptions) >= 2 * n_chunks and k <= ops.CSR_MAX_BINS:
            # the reference's own input contract (a Python list with one array per image): packed chunk by chunk,
            # on host threads, straight into a persistent pinned buffer (uint8 on the wire when the values allow it);
            # chunk i + 1 is packed while chunk i is on its way to the device and being quantised
            packer = _ListPacker(descriptions, self.__dict__.setdefault("_pack_bufs", {}))
            if not packer.ok:
                packer = None
        if k > ops.CSR_MAX_BINS:
            # codebooks beyond the shared-memory counter budget: dense kernel, CSR conversion on the host
            H = self.histograms_device(descriptions, okapi=okapi)
            return sp.csr_matrix(H.cpu().numpy())
        # attempts, in order: (packer or None, wire dtype or None = "send `mat` as it is")
        if packer is not None:
            offsets = packer.offsets
            mat = packer.view(packer.wire_dtypes()[0])
            attempts = [(packer, w) for w in packer.wire_dtypes()]
        else:
            mat, offsets = pack_descriptions(descriptions)
            if isinstance(mat, np.ndarray):
                mat = torch.from_numpy(mat)
            attempts = [(None, None)]
            if _narrow_on_the_wire(mat, n_chunks):
                # pinned float32 matrix on a host with cores to spare: integer-valued descriptors (OpenCV SIFT, ORB as
                # float) cross PCIe as uint8 -- a quarter of the bytes, narrowed block by block on host threads while
                # the previous chunk is copied and quantised; any other value makes the first block refuse at once
                npk = _ListPacker.from_matrix(mat, self.__dict__.setdefault("_pack_bufs", {}))
                if npk.ok:
                    attempts = [(npk, torch.uint8), (None, None)]
        n_img, n_rows = len(offsets) - 1, int(mat.shape[0])
        kw = self._csr_kwargs(okapi)
        off_dev = torch.from_numpy(offsets).to(dev, non_blocking=True)
        sent_bytes, wire_name = int(mat.numel() * mat.element_size()), str(mat.dtype).replace("torch.", "")
        if packer is None and (mat.is_cuda or n_img < 2 * n_chunks or not mat.is_pinned()):
            words = self.clusterer.transform_device(mat.to(dev, non_blocking=True))
        else:
            # chunked H2D (copy stream) overlapped with the assign of the previous chunk (current stream); staging
            # buffers per wire dtype, NB deep
            NB = 3
            caches = self.__dict__.get("_csr_cache")
            if caches is None or caches.get("dev") != str(dev):
                caches = {"dev": str(dev), "s_in": torch.cuda.Stream()}
                self.__dict__["_csr_cache"] = caches
            main, s_in = torch.cuda.current_stream(), caches["s_in"]
            s_in.wait_stream(main)
            ncol = int(mat.shape[1])
            src_mat = mat
            words = torch.empty((n_rows,), dtype=torch.int64, device=dev)

            def pool(max_rows, dtype, depth=NB):
                key = (max_rows, ncol, dtype, depth)
                pc = caches.get(key)
                if pc is None:
                    for old in [q for q in caches if isinstance(q, tuple) and q[:2] != key[:2]]:
                        del caches[old]          # staging buffers of another batch shape
                    pc = dict(xd=[torch.empty((max_rows, ncol), dtype=dtype, device=dev) for _ in range(depth)],
                              ev_in=[torch.cuda.Event() for _ in range(depth)], ev_c=[torch.cuda.Event() for _ in range(depth)],
                              depth=depth)
                    caches[key] = pc
                pc["used"] = 0
                return pc

            def send(pc, rows, r0, r1):
                """rows (pinned host) -> staging buffer -> words[r0:r1]; returns the event of the copy"""
                i = pc["used"]
                pc["used"] = i + 1
                b = i % pc["depth"]
                xd = pc["xd"][b][: int(r1 - r0)]
                with torch.cuda.stream(s_in):
                    if i >= pc["depth"]:
                        s_in.wait_event(pc["ev_c"][b])
                    xd.copy_(rows, non_blocking=True)
                    pc["ev_in"][b].record(s_in)
                main.wait_event(pc["ev_in"][b])
                words[int(r0):int(r1)] = self.clusterer.transform_device(xd)
                pc["ev_c"][b].record(main)
                return pc["ev_in"][b]

            def unit_chunks(pk):
                """whole packer units (images / row blocks) per chunk, balanced by rows"""
                uc = np.unique(np.searchsorted(pk.offsets, np.linspace(0, n_rows, n_chunks + 1))).astype(np.int64)
                uc[0], uc[-1] = 0, pk.n_img
                return uc, pk.offsets[uc]

            for pk, wire in attempts:
                fits = True
                if pk is None:
                    # the matrix as it is, in order
                    cuts = np.unique(np.linspace(0, n_rows, n_chunks + 1).astype(np.int64))
                    pc = pool(int(np.diff(cuts).max()), src_mat.dtype)
                    for r0, r1 in zip(cuts[:-1], cuts[1:]):
                        send(pc, src_mat[int(r0):int(r1)], r0, r1)
                    sent_bytes, wire_name = int(src_mat.numel() * src_mat.element_size()), str(src_mat.dtype).replace("torch.", "")
                elif pk is packer:
                    # list input: chunk c is sent once the background job has packed it; a value that is not an integer
                    # in [0, 255] makes the uint8 attempt start over with float32 on the wire
                    uc, cuts = unit_chunks(pk)
                    buf = pk.view(wire)
                    pc = pool(int(np.diff(cuts).max()), buf.dtype)
                    pk.begin(uc, wire)
                    try:
                        for ci, (r0, r1) in enumerate(zip(cuts[:-1], cuts[1:])):
                            if r1 <= r0:
                                continue
                            if not pk.wait(ci):
                                fits = False
                                break
                            send(pc, buf[int(r0):int(r1)], r0, r1)
                    finally:
                        pk.end()
                    sent_bytes, wire_name = int(buf.numel() * buf.element_size()), str(buf.dtype).replace("torch.", "")
                else:
                    # pinned float32 matrix, two-ended: the workers narrow chunks to uint8 from the FRONT; whenever the copy
                    # engine has room and no narrowed chunk is ready, a chunk is claimed from the BACK and sent as float32
                    # -- the two meet where the host's and PCIe's bandwidth balance.  A value that does not fit uint8 stops
                    # the narrowing; the chunks already sent stay valid, the rest goes as float32.
                    uc, cuts = unit_chunks(pk)
                    buf = pk.view(torch.uint8)
                    max_rows = int(np.diff(cuts).max())
                    pu, pf = pool(max_rows, torch.uint8), pool(max_rows, torch.float32, depth=4)
                    front, back, narrowing, inflight, sent_bytes, n_u8 = 0, len(cuts) - 2, True, [], 0, 0
                    trace = [] if os.environ.get("ISE_TRACE_WIRE") else None
                    t_begin = time.perf_counter()
                    pk.begin(uc, torch.uint8)
                    try:
                        while front <= back:
                            if not narrowing:
                                r0, r1 = int(cuts[front]), int(cuts[front + 1])
                                send(pf, src_mat[r0:r1], r0, r1)
                                sent_bytes += (r1 - r0) * ncol * 4
                                front += 1
                                continue
                            done, ok = pk.poll(front)
                            if not ok:
                                narrowing = False
                                continue
                            if done:
                                r0, r1 = int(cuts[front]), int(cuts[front + 1])
                                send(pu, buf[r0:r1], r0, r1)
                                if trace is not None:
                                    trace.append(("u8", front, round((time.perf_counter() - t_begin) * 1e3, 2)))
                                sent_bytes += (r1 - r0) * ncol
                                n_u8 += 1
                                front += 1
                                continue
                            inflight = [e for e in inflight if not e.query()]
                            if len(inflight) < 3 and back > front and pk.claim(back):
                                r0, r1 = int(cuts[back]), int(cuts[back + 1])
                                inflight.append(send(pf, src_mat[r0:r1], r0, r1))
                                if trace is not None:
                                    trace.append(("f32", back, round((time.perf_counter() - t_begin) * 1e3, 2)))
                                sent_bytes += (r1 - r0) * ncol * 4
                                back -= 1
                                continue
                            time.sleep(2e-5)
                    finally:
                        pk.end()
                    n_all = len(cuts) - 1
                    if trace is not None:
                        print("wire trace (kind, chunk, ms):", trace, flush=True)
                    wire_name = "uint8" if n_u8 == n_all else ("float32" if n_u8 == 0 else f"uint8 ({n_u8} of {n_all} chunks) + float32")
                if fits:
                    break
                # the pinned rows of the abandoned attempt may still be in flight: let the copies drain before the buffers
                # are reused / re-packed
                s_in.synchronize()
        # what crossed PCIe on the way in (bench.py reports it)
        self.__dict__["_last_transfer"] = dict(h2d_bytes=int(sent_bytes + offsets.nbytes), wire=wire_name, rows=n_rows)
        # persistent device + pinned result buffers (indptr | indices | data), grown on demand
        rb = self.__dict__.get("_csr_bufs")
        if rb is None or rb["cap"] < max(n_rows, 1) or rb["n_img"] < n_img or rb["dev"] != str(dev):
            cap = max(n_rows, 1)
            rb = dict(cap=cap, n_img=n_img, dev=str(dev),
                      d=(torch.empty((n_img + 1,), dtype=torch.int32, device=dev),
                         torch.empty((cap,), dtype=torch.int32, device=dev),
                         torch.empty((cap,), dtype=torch.float64, device=dev)),
                      h=(torch.empty((n_img + 1,), dtype=torch.int32, pin_memory=True),
                         torch.empty((cap,), dtype=torch.int32, pin_memory=True),
                         torch.empty((cap,), dtype=torch.float64, pin_memory=True)))
            self.__dict__["_csr_bufs"] = rb
        d_ptr, d_idx, d_dat = rb["d"]
        h_ptr, h_idx, h_dat = rb["h"]
        ops.bovw_histogram_csr(words, off_dev, k, out=(d_ptr[: n_img + 1], d_idx, d_dat), **kw)
        h_ptr[: n_img + 1].copy_(d_ptr[: n_img + 1], non_blocking=True)
        # the non-zero count is only known on the device: ship the upper bound (one entry per descriptor)
        h_idx[:n_rows].copy_(d_idx[:n_rows], non_blocking=True)
        h_dat[:n_rows].copy_(d_dat[:n_rows], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        indptr = h_ptr[: n_img + 1].numpy()
        nnz = int(indptr[-1])
        indices, data = h_idx[:nnz].numpy(), h_dat[:nnz].numpy()
        if copy:
            indptr, indices, data = indptr.copy(), indices.copy(), data.copy()
        return sp.csr_matrix((data, indices, indptr), shape=(n_img, k), copy=False)

    def histograms_device(self, descriptions, *, okapi: OkapiTransformer | None = None,
                          out_dtype=torch.float64) -> torch.Tensor:
        """One assign launch + one histogram launch for all images; optional fused Okapi weighting.  The result matrix
        is cleared on a side stream while the assign runs, and the histogram then writes only the non-zero bins."""
        if self.hist_mode not in _HIST_MODES:
            raise ValueError(f"hist_mode must be one of {sorted(_HIST_MODES)}")
        dev = ops.require_cuda()
        mat, offsets = pack_descriptions(descriptions)
        xd = mat.to(dev, non_blocking=True) if isinstance(mat, torch.Tensor) else \
            torch.from_numpy(mat).to(dev, non_blocking=True)
        off = torch.empty((len(offsets),), dtype=torch.int64, device=dev)
        out = torch.empty((len(offsets) - 1, int(self.n_clusters)), dtype=out_dtype, device=dev)
        main = torch.cuda.current_stream()
        allocated = main.record_event()
        side = self.__dict__.setdefault("_clear_streams", {}).get(dev.index)
        if side is None:
            side = self.__dict__["_clear_streams"].setdefault(dev.index, torch.cuda.Stream(device=dev))
        # the assign is enqueued first; the clear's blocks fit beside its CTAs on every SM (csrc/bovw.cu, clear_kernel).
        # Only the histogram reads the offsets, so their upload goes to the side stream too, off the assign's path.
        words = self.clusterer.transform_device(xd)
        side.wait_event(allocated)
        with torch.cuda.stream(side):
            off.copy_(torch.from_numpy(offsets), non_blocking=True)
            ops.clear_(out, _CLEAR_GB_PER_S)
        # the current stream waits for the side stream before `off` / `out` are used, returned or freed: the caching
        # allocator only orders them on the current stream
        main.wait_stream(side)
        kw = {}
        if okapi is not None:
            kw = dict(okapi=True, k1=okapi.k1, k2=okapi.k2, b=okapi.b)
        return ops.bovw_histogram(words, off, int(self.n_clusters), mode=_HIST_MODES[self.hist_mode],
                                  out_dtype=out_dtype, out=out, zeroed=True, **kw)

    def fit_transform(self, X, y=None):
        self.fit(X)
        return self.transform(X)


def _to_host(t: torch.Tensor, out: torch.Tensor | None = None) -> np.ndarray:
    """Device -> NumPy.  ``out`` (a pinned CPU tensor of the same shape) makes the copy a single DMA."""
    if out is not None:
        out.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out.numpy()
    return t.cpu().numpy()


def run_clustering(descriptions, n_clusters):
    """Codebook training over all descriptors with the reference's defaults n_init=3, max_iter=25."""
    print("Starting clustering...")
    mat, _ = pack_descriptions(descriptions)
    clusterer = FaissKMeans(n_clusters)
    clusterer.fit(mat)
    print("Clustering finished.")
    return clusterer


def load_cluster_model(n_clusters, index=None):
    if isinstance(index, (str, Path)):
        index = faiss.read_index(str(index))
    return FaissKMeans(n_clusters=n_clusters, index=index)


def train_bovw_model(images_paths, describer, config=None):
    """Offline index build (bag_of_visual_words.py:137-204), same two-argument call as the reference
    (indexer.py:37).  ``config`` supplies NUM_CLUSTERS, the three artefact paths and, with
    BOVW_HYPERPARAMETERS_SEARCH, the cluster-count grid (:149-181); when omitted it is the host application's own
    ``config.Config()``, which is what the reference's module-level ``config = Config()`` (:37) resolves to."""
    if config is None:
        try:
            from config import Config      # the application's backend/config.py, like bag_of_visual_words.py:32,37
        except Exception as exc:
            raise RuntimeError("train_bovw_model(images_paths, describer): no `config` module with a `Config` class "
                               "on sys.path (the reference's backend/config.py); pass config= explicitly") from exc
        config = Config()
    print(f"Received {len(images_paths)} images to process")
    pipeline = Pipeline([("bovw", BOVW(describer, n_clusters=config.NUM_CLUSTERS)), ("tfidf", OkapiTransformer())])
    if getattr(config, "BOVW_HYPERPARAMETERS_SEARCH", False):
        # cluster-count grid search (:149-181): every candidate is a full fit on the GPU; the scorer labels all
        # cached descriptors with one assign launch.  n_jobs stays 1: the candidates share one device.
        from sklearn.model_selection import GridSearchCV
        from . import utils as _utils
        _utils.CLUSTER_EVAL_SAMPLE_SIZE = getattr(config, "CLUSTER_EVAL_SAMPLE_SIZE", _utils.CLUSTER_EVAL_SAMPLE_SIZE)
        _utils.CLUSTER_EVAL_N_SAMPLES = getattr(config, "CLUSTER_EVAL_N_SAMPLES", _utils.CLUSTER_EVAL_N_SAMPLES)
        clusters_to_test = np.unique(np.linspace(config.MIN_NUM_CLUSTERS, config.MAX_NUM_CLUSTERS,
                                                 config.NUM_CLUSTERS_TO_TEST).round().astype(int))
        search = GridSearchCV(estimator=pipeline, param_grid={"bovw__n_clusters": clusters_to_test}, n_jobs=1,
                              verbose=1, scoring=_utils.calc_sampled_cluster_score)
        search.fit(images_paths)
        print("Search finished.")
        print(f"Best score: {search.best_score_:.3f}")
        print(f"Best parameters: {search.best_params_}")
        pipeline = search.best_estimator_
        bovw, tfidf = pipeline.named_steps["bovw"], pipeline.named_steps["tfidf"]
    else:
        bovw, tfidf = pipeline.named_steps["bovw"], pipeline.named_steps["tfidf"]
        bovw.fit(images_paths)
    # GPU-resident build: histogram + Okapi fused, float32 rows, normalise + add without leaving HBM
    H = bovw.histograms_device(bovw.descriptions, okapi=tfidf, out_dtype=torch.float32)
    tfidf.fit(H)
    tfidf.finish_device_(H)    # opt-in corrected mode (OkapiTransformer(compat=False)): idf + row norm; no-op by default
    print("Saving KMeans index", bovw.clusterer.index)
    faiss.write_index(bovw.clusterer.index, str(config.BOVW_KMEANS_INDEX_PATH))
    index = create_search_index(H)
    print("Saving final index", index)
    faiss.write_index(index, str(config.BOVW_INDEX_PATH))
    print("Saving pipeline", pipeline)
    bovw.clusterer = None      # the index is persisted separately, like the reference (:198-202)
    bovw.descriptions = None
    joblib.dump(pipeline, str(config.BOVW_PIPELINE_PATH), compress=0)
    return pipeline, index
