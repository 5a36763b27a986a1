"""NumPy restatement of Faiss's IndexIVF::range_search for IndexIVFFlat, for the IVFFlat range tests (test
infrastructure only).

Follows upstream faiss/IndexIVF.cpp range_search -> range_search_preassigned (parallel_mode 0) and
faiss/IndexIVFFlat.cpp IVFFlatScanner::scan_codes_range (~v1.7.4, recalled like tests/_ivfflat_oracle.py, whose index
it reads; PARITY UNPINNED):
  - the quantizer probes min(nprobe, nlist) lists, as for search;
  - per query, the probes are visited in rank order (probe -1 and empty lists skipped), and each list's vectors in list
    order (ascending id);
  - every vector is scored with the direct FP32 formulas fvec_inner_product / fvec_L2sqr and kept when IP dis > radius
    or L2 dis < radius (strict; radius cast to float32), in visiting order.
"""
from __future__ import annotations

import numpy as np

from oracle import faiss_shim as fs
from tests._ivfflat_oracle import IndexIVFFlat


def range_search(index: IndexIVFFlat, x, radius: float, probes=None):
    """Returns (lims uint64 [nq + 1], D float32, I int64); query i's results are D / I[lims[i]:lims[i+1]]."""
    x = np.ascontiguousarray(np.asarray(x), dtype=np.float32)
    nq = x.shape[0]
    lims = np.zeros(nq + 1, np.uint64)
    if nq == 0 or index.ntotal == 0 or not index.is_trained:
        return lims, np.zeros(0, np.float32), np.zeros(0, np.int64)
    coarse = index.probes(x) if probes is None else probes
    r = np.float32(radius)
    ip = index.metric_type == fs.METRIC_INNER_PRODUCT
    D, I, counts = [], [], np.zeros(nq, np.uint64)
    for qi in range(nq):
        for l in coarse[qi]:
            if l < 0 or index.ids[l].size == 0:
                continue
            y = index.vecs[l]
            if ip:
                s = np.einsum("jd,d->j", y, x[qi], dtype=np.float32)
                keep = s > r
            else:
                diff = y - x[qi]
                s = np.einsum("jd,jd->j", diff, diff, dtype=np.float32)
                keep = s < r
            D.append(s[keep])
            I.append(index.ids[l][keep])
            counts[qi] += int(keep.sum())
    np.cumsum(counts, out=lims[1:])
    D = np.concatenate(D).astype(np.float32, copy=False) if lims[-1] else np.zeros(0, np.float32)
    I = np.concatenate(I).astype(np.int64, copy=False) if lims[-1] else np.zeros(0, np.int64)
    return lims, D, I


def scan_keys(probes: np.ndarray, assignment: np.ndarray, list_ids, lims, I):
    """(probe rank, list position) of every result: Faiss's visiting order, strictly increasing within a query.
    assignment[id] = list of the id, list_ids[l] = ids of list l in list order."""
    lims = np.asarray(lims).astype(np.int64)
    I = np.asarray(I)
    rank = np.empty(I.size, np.int64)
    pos = np.empty(I.size, np.int64)
    where = {}
    for i in range(lims.size - 1):
        seg = I[lims[i]:lims[i + 1]]
        if seg.size == 0:
            continue
        rank_of = {int(l): r for r, l in reversed(list(enumerate(probes[i])))}
        lst = assignment[seg]
        rank[lims[i]:lims[i + 1]] = [rank_of[int(l)] for l in lst]
        for j, (l, v) in enumerate(zip(lst, seg)):
            m = where.get(int(l))
            if m is None:
                m = where[int(l)] = {int(v2): p for p, v2 in enumerate(list_ids[int(l)])}
            pos[lims[i] + j] = m[int(v)]
    return rank, pos


def assert_scan_order(probes, assignment, list_ids, lims, I):
    """Within every query the results come in strictly increasing (probe rank, list position)."""
    rank, pos = scan_keys(probes, assignment, list_ids, lims, I)
    lims = np.asarray(lims).astype(np.int64)
    for i in range(lims.size - 1):
        r, p = rank[lims[i]:lims[i + 1]], pos[lims[i]:lims[i + 1]]
        ok = (np.diff(r) > 0) | ((np.diff(r) == 0) & (np.diff(p) > 0))
        assert ok.all(), f"query {i}: results out of (probe rank, list position) order"
