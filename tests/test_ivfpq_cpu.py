"""CPU: the NumPy restatement of IndexIVFPQ search / range search (tests/_ivfpq_oracle.py) against an FP64 brute force
over the probed lists, its scan order, and every list probed against a plain filter over every code."""
import numpy as np
import pytest

from tests import _ivfpq_oracle as ref
from tests._ivfflat_range_oracle import assert_scan_order


def _index(rng, n=1500, d=32, M=8, nlist=12, ksub=256):
    coarse = (3.0 * rng.standard_normal((nlist, d))).astype(np.float32)
    pq = rng.standard_normal((M, ksub, d // M)).astype(np.float32)
    codes = rng.integers(0, ksub, (n, M)).astype(np.uint8)
    assign = rng.integers(0, nlist, n)
    assign[:3] = 0
    assign[assign == nlist - 1] = 0                       # list nlist - 1 stays empty
    ids_by_list = [np.nonzero(assign == l)[0].astype(np.int64) for l in range(nlist)]
    codes_by_list = [codes[i] for i in ids_by_list]
    return coarse, pq, codes, assign, codes_by_list, ids_by_list


def _probes(rng, q, coarse, nprobe):
    d2 = ((q[:, None, :].astype(np.float64) - coarse[None]) ** 2).sum(2)
    pr = np.argsort(d2, 1, kind="stable")[:, :nprobe]
    pr[0, -1] = -1                                        # a missing probe
    return pr


def _probed(assign, probes):
    return (assign[None, :, None] == probes[:, None, :]).any(2)


@pytest.mark.parametrize("nprobe", [1, 3, 12])
def test_range_restatement_against_fp64(nprobe):
    rng = np.random.default_rng(nprobe)
    coarse, pq, codes, assign, cbl, ibl = _index(rng)
    q = (coarse[rng.integers(0, coarse.shape[0], 20)] + rng.standard_normal((20, coarse.shape[1]))).astype(np.float32)
    pr = _probes(rng, q, coarse, nprobe)
    s = ref.distances64(q, coarse, pq, codes, assign)
    probed = _probed(assign, pr)
    radius = float(np.median(s[probed]))
    lims, D, I = ref.range_search(q, coarse, pq, cbl, ibl, pr, radius)
    assert lims.dtype == np.uint64 and lims[-1] > 0
    lims = lims.astype(np.int64)
    for i in range(q.shape[0]):
        ids = I[lims[i]:lims[i + 1]]
        tau = 1e-4 * np.max(s[i][probed[i]], initial=1.0)
        sure = np.nonzero(probed[i] & (s[i] < radius - tau))[0]
        assert np.isin(sure, ids).all()
        assert probed[i][ids].all() and (s[i][ids] < radius + tau).all()
        np.testing.assert_allclose(D[lims[i]:lims[i + 1]], s[i][ids], rtol=1e-5, atol=tau)


@pytest.mark.parametrize("k", [1, 10, 200])
def test_search_restatement_against_fp64(k):
    rng = np.random.default_rng(k)
    coarse, pq, codes, assign, cbl, ibl = _index(rng)
    q = (coarse[rng.integers(0, coarse.shape[0], 15)] + rng.standard_normal((15, coarse.shape[1]))).astype(np.float32)
    pr = _probes(rng, q, coarse, 3)
    s = ref.distances64(q, coarse, pq, codes, assign)
    probed = _probed(assign, pr)
    D, I = ref.search(q, coarse, pq, cbl, ibl, pr, k)
    for i in range(q.shape[0]):
        cand = np.nonzero(probed[i])[0]
        n = min(k, cand.size)
        assert (I[i, n:] == -1).all() and (D[i, n:] == ref.FLT_MAX).all()
        assert probed[i][I[i, :n]].all() and len(set(I[i, :n])) == n
        np.testing.assert_allclose(D[i, :n], s[i][I[i, :n]], rtol=1e-5, atol=1e-3)
        assert (np.diff(D[i, :n]) >= 0).all()
        kth = np.sort(s[i][cand])[n - 1]
        assert (s[i][I[i, :n]] <= kth + 1e-3 * max(1.0, kth)).all()


def test_range_results_come_in_scan_order():
    rng = np.random.default_rng(5)
    coarse, pq, codes, assign, cbl, ibl = _index(rng)
    q = (coarse[rng.integers(0, coarse.shape[0], 25)] + rng.standard_normal((25, coarse.shape[1]))).astype(np.float32)
    pr = _probes(rng, q, coarse, 5)
    s = ref.distances64(q, coarse, pq, codes, assign)
    lims, D, I = ref.range_search(q, coarse, pq, cbl, ibl, pr, float(np.quantile(s, 0.3)))
    assert lims[-1] > 0
    assert_scan_order(pr, assign, ibl, lims, I)


def test_every_list_probed_equals_a_plain_filter():
    rng = np.random.default_rng(6)
    coarse, pq, codes, assign, cbl, ibl = _index(rng)
    nlist = coarse.shape[0]
    q = (coarse[rng.integers(0, nlist, 10)] + rng.standard_normal((10, coarse.shape[1]))).astype(np.float32)
    pr = np.tile(np.arange(nlist), (q.shape[0], 1))
    radius = float(np.quantile(ref.distances64(q, coarse, pq, codes, assign), 0.2))
    lims, D, I = ref.range_search(q, coarse, pq, cbl, ibl, pr, radius)
    lims = lims.astype(np.int64)
    for i in range(q.shape[0]):
        dis = np.array([ref.list_distances(ref.table(q[i], coarse[assign[j]], pq), codes[j:j + 1])[0]
                        for j in range(codes.shape[0])], np.float32)
        keep = np.nonzero(dis < np.float32(radius))[0]
        o = np.argsort(I[lims[i]:lims[i + 1]], kind="stable")
        np.testing.assert_array_equal(I[lims[i]:lims[i + 1]][o], keep)
        np.testing.assert_array_equal(D[lims[i]:lims[i + 1]][o], dis[keep])
    Dk, Ik = ref.search(q, coarse, pq, cbl, ibl, pr, 7)
    for i in range(q.shape[0]):
        dis = np.concatenate([ref.list_distances(ref.table(q[i], coarse[l], pq), cbl[l]) for l in range(nlist)])
        ids = np.concatenate(ibl)
        o = np.lexsort((ids, dis))[:7]
        np.testing.assert_array_equal(Ik[i], ids[o])
        np.testing.assert_array_equal(Dk[i], dis[o])
