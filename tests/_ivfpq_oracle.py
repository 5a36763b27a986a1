"""NumPy restatement of Faiss's IndexIVFPQ search and range search over given quantizers and lists, for the IVFPQ tests
(test infrastructure only).

Follows upstream faiss/IndexIVF.cpp search / range_search -> *_preassigned and faiss/IndexIVFPQ.cpp IVFPQScanner
(by_residual, L2, no precomputed tables; scan_codes / scan_codes_range) (~v1.7.4, recalled, PARITY UNPINNED):
  - a probed list l gives the residual r = q - coarse[l] and the look-up table tab[m][c] = |r_m - pq[m][c]|^2 over the
    m-th d/M-dimensional slice;
  - a code's distance is dis = 0; dis += tab[m][code[m]] for m = 0 .. M-1, in float32 and in that order;
  - range search visits the probes in rank order (probe -1 and empty lists skipped), each list in list order
    (ascending id), and keeps dis < radius (strict; radius cast to float32) in visiting order;
  - search returns the k smallest distances in the canonical (distance, id) order, padded with id -1 / FLT_MAX.
    (Faiss's heap can keep a higher id from an earlier-probed list when a tie falls on the k-th place; this project
    returns the canonical order instead, like its other indexes.)
Lists are given as ``codes_by_list[l]`` (uint8 [n_l, M]) and ``ids_by_list[l]`` (int64 [n_l], ascending).
"""
from __future__ import annotations

import numpy as np

FLT_MAX = float(np.finfo(np.float32).max)


def table(q, coarse_row, pq):
    """tab[m, c] (float32 [M, ksub]) for query q against the list whose centroid is coarse_row; pq [M, ksub, dsub]."""
    M, ksub, dsub = pq.shape
    r = (np.asarray(q, np.float32) - np.asarray(coarse_row, np.float32)).reshape(M, 1, dsub)
    t = r - pq
    return np.einsum("mcj,mcj->mc", t, t, dtype=np.float32)


def list_distances(tab, codes):
    """dis[i] of every code row (float32), summed over m in order."""
    dis = np.zeros(codes.shape[0], np.float32)
    for m in range(codes.shape[1]):
        dis += tab[m, codes[:, m]]
    return dis


def range_search(q, coarse, pq, codes_by_list, ids_by_list, probes, radius):
    """Returns (lims uint64 [nq + 1], D float32, I int64); query i's results are D / I[lims[i]:lims[i+1]]."""
    q = np.ascontiguousarray(q, np.float32)
    nq = q.shape[0]
    r = np.float32(radius)
    lims = np.zeros(nq + 1, np.uint64)
    D, I = [], []
    for i in range(nq):
        n = 0
        for l in probes[i]:
            if l < 0 or ids_by_list[l].size == 0:
                continue
            dis = list_distances(table(q[i], coarse[l], pq), codes_by_list[l])
            keep = dis < r
            D.append(dis[keep])
            I.append(ids_by_list[l][keep])
            n += int(keep.sum())
        lims[i + 1] = lims[i] + n
    D = np.concatenate(D).astype(np.float32) if lims[-1] else np.zeros(0, np.float32)
    I = np.concatenate(I).astype(np.int64) if lims[-1] else np.zeros(0, np.int64)
    return lims, D, I


def search(q, coarse, pq, codes_by_list, ids_by_list, probes, k):
    """(D float32 [nq, k], I int64 [nq, k]) in the canonical (distance, id) order over the probed lists."""
    q = np.ascontiguousarray(q, np.float32)
    nq = q.shape[0]
    D = np.full((nq, k), FLT_MAX, np.float32)
    I = np.full((nq, k), -1, np.int64)
    for i in range(nq):
        dis, ids = [], []
        for l in probes[i]:
            if l < 0 or ids_by_list[l].size == 0:
                continue
            dis.append(list_distances(table(q[i], coarse[l], pq), codes_by_list[l]))
            ids.append(ids_by_list[l])
        if not dis:
            continue
        dis, ids = np.concatenate(dis), np.concatenate(ids)
        o = np.lexsort((ids, dis))[:k]
        D[i, :o.size], I[i, :o.size] = dis[o], ids[o]
    return D, I


def distances64(q, coarse, pq, codes, assign):
    """FP64 distance of every query to every code (codes [n, M] in id order, assign[id] = its list)."""
    q = np.asarray(q, np.float64)
    M, ksub, dsub = pq.shape
    recon = np.asarray(pq, np.float64)[np.arange(M)[None, :], codes.astype(np.int64)].reshape(codes.shape[0], -1)
    x = np.asarray(coarse, np.float64)[assign] + recon     # the vector the code stands for
    return ((q[:, None, :] - x[None, :, :]) ** 2).sum(2)
