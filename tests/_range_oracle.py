"""NumPy restatement of Faiss's flat range search, for the range-search tests (test infrastructure only).

Follows upstream faiss/IndexFlat.cpp IndexFlat::range_search -> faiss/utils/distances.cpp range_search_inner_product /
range_search_L2sqr (~v1.7.4, recalled like the rest of oracle/faiss_shim.py, whose knn regimes and constants it reuses;
PARITY UNPINNED).  There is no reference call site: range search is an extension mirroring Faiss's API.
"""
from __future__ import annotations

import numpy as np

from oracle import faiss_shim as fs


def range_search(x: np.ndarray, y: np.ndarray, radius: float, metric: int, y_norms: np.ndarray | None = None):
    """range_search_inner_product / range_search_L2sqr.

    Same two regimes as faiss_shim.knn: n < 20 direct per-pair formulas, n >= 20 the BLAS expansion with L2 =
    |x|^2+|y|^2-2<x,y> clamped at 0.  IP keeps dis > radius, L2 keeps dis < radius (squared), both strict and in
    float32 (radius is cast).  Results of a query follow the database scan order, i.e. ascending id.
    Returns (lims uint64 [n+1] -- Faiss copies its size_t array; recalled, not checked --, D float32, I int64).
    """
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32)
    nx = x.shape[0]
    ny = y.shape[0]
    r = np.float32(radius)
    largest = metric == fs.METRIC_INNER_PRODUCT
    lims = np.zeros(nx + 1, dtype=np.uint64)
    if nx == 0 or ny == 0:
        return lims, np.zeros(0, np.float32), np.zeros(0, np.int64)
    blas = nx >= fs.distance_compute_blas_threshold
    if not largest and blas:
        x_norms = fs.fvec_norms_L2sqr(x)
        if y_norms is None:
            y_norms = fs.fvec_norms_L2sqr(y)
    bs_x, bs_y = fs.distance_compute_blas_query_bs, fs.distance_compute_blas_database_bs
    D_rows = [[] for _ in range(nx)]
    I_rows = [[] for _ in range(nx)]
    for i0 in range(0, nx, bs_x):
        i1 = min(nx, i0 + bs_x)
        xb = x[i0:i1]
        for j0 in range(0, ny, bs_y):
            j1 = min(ny, j0 + bs_y)
            yb = y[j0:j1]
            if blas:
                ip = xb @ yb.T
                if largest:
                    s = ip
                else:
                    s = x_norms[i0:i1, None] + y_norms[None, j0:j1] - np.float32(2.0) * ip
                    np.maximum(s, np.float32(0.0), out=s)
            elif largest:
                s = np.einsum("id,jd->ij", xb, yb, dtype=np.float32)
            else:
                diff = xb[:, None, :] - yb[None, :, :]
                s = np.einsum("ijd,ijd->ij", diff, diff, dtype=np.float32)
            s = s.astype(np.float32, copy=False)
            keep = (s > r) if largest else (s < r)
            for i in np.nonzero(keep.any(axis=1))[0]:
                cols = np.nonzero(keep[i])[0]
                D_rows[i0 + i].append(s[i, cols])
                I_rows[i0 + i].append(cols.astype(np.int64) + j0)
    counts = np.array([sum(a.size for a in row) for row in I_rows], dtype=np.uint64)
    np.cumsum(counts, out=lims[1:])
    D = np.concatenate([a for row in D_rows for a in row]) if lims[-1] else np.zeros(0, np.float32)
    I = np.concatenate([a for row in I_rows for a in row]) if lims[-1] else np.zeros(0, np.int64)
    return lims, D.astype(np.float32, copy=False), I.astype(np.int64, copy=False)


def index_range_search(index: fs.IndexFlat, x, radius: float):
    """IndexFlat::range_search on an oracle flat index (Python wrapper: returns lims, D, I)."""
    x = np.asarray(x)
    if x.ndim != 2 or x.shape[1] != index.d:
        raise AssertionError("range_search: expected (n, %d) array" % index.d)
    y = index.reconstruct_n()
    y_norms = fs.fvec_norms_L2sqr(y) if index.metric_type == fs.METRIC_L2 else None
    return range_search(np.ascontiguousarray(x, dtype=np.float32), y, radius, index.metric_type, y_norms)
