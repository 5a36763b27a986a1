"""IndexIVFPQ search and range search grouped by list (ise_ivfpq_search, ise_ivfpq_range_count / _fill): bit equality
with the dense path (ise_ivfpq_scan into an [nq, ntotal] matrix), Faiss's range order, edge cases, the query batching
that bounds the look-up tables, the workspace bound, an index whose dense matrix could not be allocated, and the
index API (list introspection, pickling, recall)."""
import pickle

import numpy as np
import pytest
import torch

from tests import _ivfpq_oracle as ref
from tests._ivfflat_range_oracle import assert_scan_order

pytestmark = pytest.mark.gpu

FLT_MAX = np.finfo(np.float32).max


def _install(coarse, pq, codes, assign, nprobe):
    """A GPU IndexIVFPQ holding the given quantizers and codes (ids = row numbers), without training."""
    from image_search_engine_b200 import faiss_compat as fc
    nlist, d = coarse.shape
    M = pq.shape[0]
    ix = fc.IndexIVFPQ(fc.IndexFlatL2(d), d, nlist, M, 8)
    ix.set_trained_state(np.asarray(coarse), np.asarray(pq))
    ix._codes = torch.as_tensor(codes).cuda().contiguous()
    ix._assign = torch.as_tensor(assign).cuda().to(torch.int64)
    ix._ids = torch.arange(ix._codes.shape[0], dtype=torch.int64, device="cuda")
    ix._sorted = None
    ix.nprobe = nprobe
    return ix


def _random_index(rng, n, d, M, nlist, nprobe, skew=None):
    coarse = (4.0 * rng.standard_normal((nlist, d))).astype(np.float32)
    pq = rng.standard_normal((M, 256, d // M)).astype(np.float32)
    codes = rng.integers(0, 256, (n, M)).astype(np.uint8)
    assign = rng.integers(0, nlist, n).astype(np.int64)
    if skew is not None:
        assign[:skew] = 0
    return _install(coarse, pq, codes, assign, nprobe), coarse


def _queries(rng, coarse, nq):
    return (coarse[rng.integers(0, coarse.shape[0], nq)] +
            rng.standard_normal((nq, coarse.shape[1]))).astype(np.float32)


def _probes(ix, qd):
    return ix._probes(qd)


def _dense(ix, qd, probes):
    """The dense path's [nq, ntotal] distance matrix (list-sorted positions, +inf outside the probed lists)."""
    from image_search_engine_b200 import ops
    codes, ids, off, _ = ix._lists()
    return ops.ivfpq_scan(qd, ix.quantizer._database(), probes, ix.pq_centroids, codes, off)


def _expected_topk(ix, dist, k):
    """(D, I) from the dense matrix: D from the dense path's selection, I the (distance, id) lexsort on the host."""
    from image_search_engine_b200 import ops
    _, ids, _, _ = ix._lists()
    nq, nt = dist.shape
    Dv, _ = ops.scores_topk_any_k_(dist.clone(), ops.METRIC_L2, k)
    kth = torch.kthvalue(dist, min(k, nt), dim=1).values
    rows, cols = torch.nonzero((dist <= kth[:, None]) & torch.isfinite(dist), as_tuple=True)
    vals = dist[rows, cols].cpu().numpy()
    rows, idv = rows.cpu().numpy(), ids[cols].cpu().numpy()
    o = np.lexsort((idv, vals, rows))
    rows, idv = rows[o], idv[o]
    first = np.searchsorted(rows, np.arange(nq))
    rank = np.arange(rows.size) - first[rows]
    I = np.full((nq, k), -1, np.int64)
    keep = rank < k
    I[rows[keep], rank[keep]] = idv[keep]
    return Dv.cpu().numpy(), I


def _assert_search_equals_dense(ix, q, k):
    qd = torch.from_numpy(q).cuda()
    D, I = ix.search(qd, k)
    De, Ie = _expected_topk(ix, _dense(ix, qd, _probes(ix, qd)), k)
    np.testing.assert_array_equal(D.cpu().numpy().view(np.uint32), De.view(np.uint32))
    np.testing.assert_array_equal(I.cpu().numpy(), Ie)
    return D, I


def _expected_range(ix, dist, probes, radius):
    """Every dense entry with dis < radius, in (probe rank, list position) order."""
    _, ids, off, _ = ix._lists()
    dist, ids, off, probes = dist.cpu().numpy(), ids.cpu().numpy(), off.cpu().numpy(), probes.cpu().numpy()
    r = np.float32(radius)
    lims, D, I = [0], [], []
    for i in range(dist.shape[0]):
        n = 0
        for l in probes[i]:
            if l < 0:
                continue
            seg = dist[i, off[l]:off[l + 1]]
            keep = np.nonzero(seg < r)[0]
            D.append(seg[keep])
            I.append(ids[off[l] + keep])
            n += keep.size
        lims.append(lims[-1] + n)
    cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
    return np.array(lims, np.uint64), cat(D, np.float32), cat(I, np.int64)


def _assert_range_equals_dense(ix, q, radius):
    qd = torch.from_numpy(q).cuda()
    probes = _probes(ix, qd)
    lims, D, I = ix.range_search(q, radius)
    le, De, Ie = _expected_range(ix, _dense(ix, qd, probes), probes, radius)
    np.testing.assert_array_equal(lims, le)
    np.testing.assert_array_equal(I, Ie)
    np.testing.assert_array_equal(D.view(np.uint32), De.view(np.uint32))
    return lims, D, I


_DM = [(d, M) for d in (64, 96, 128, 512) for M in (8, 16, 32) if d % M == 0]


@pytest.mark.parametrize("nlist", [8, 64, 1024])
@pytest.mark.parametrize("d,M", _DM)
def test_search_bit_equal_to_dense_path(d, M, nlist):
    rng = np.random.default_rng(d * 7 + M + nlist)
    ix, coarse = _random_index(rng, 10_000, d, M, nlist, 1)
    q = _queries(rng, coarse, 5000)
    for nprobe in (1, 5, nlist):
        ix.nprobe = nprobe
        for nq in (1, 7, 5000):
            for k in (1, 10, 128):
                _assert_search_equals_dense(ix, q[:nq], k)


@pytest.mark.parametrize("nlist", [8, 64])
@pytest.mark.parametrize("d,M", [(64, 8), (96, 32), (128, 16), (512, 16)])
def test_range_bit_equal_to_dense_path_and_to_search(d, M, nlist):
    rng = np.random.default_rng(d + M + nlist)
    ix, coarse = _random_index(rng, 6000, d, M, nlist, 1)
    q = _queries(rng, coarse, 150)
    for nprobe in (1, 5, nlist):
        ix.nprobe = nprobe
        D, I = ix.search(q, 128)
        for col in (9, 99):                                    # about 10 and 100 results per query
            radius = float(np.median(D[:, col]))
            lims, Dr, Ir = _assert_range_equals_dense(ix, q, radius)
            assert lims[-1] > 0
            assign = ix._assign.cpu().numpy()
            list_ids = [ix.get_list_ids(l) for l in range(nlist)]
            assert_scan_order(_probes(ix, torch.from_numpy(q).cuda()).cpu().numpy(), assign, list_ids, lims, Ir)
            for i in range(q.shape[0]):                        # the distance search returns for the same pair
                seg = slice(int(lims[i]), int(lims[i + 1]))
                common, a, b = np.intersect1d(Ir[seg], I[i], return_indices=True)
                np.testing.assert_array_equal(Dr[seg][a].view(np.uint32), D[i][b].view(np.uint32))


def test_edge_cases():
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(1)
    d, M, nlist = 64, 8, 16
    ix, coarse = _random_index(rng, 3000, d, M, nlist, 4)
    q = _queries(rng, coarse, 30)
    # nq = 0
    D, I = ix.search(q[:0], 5)
    assert D.shape == (0, 5) and I.shape == (0, 5)
    lims, D, I = ix.range_search(q[:0], 10.0)
    assert lims.dtype == np.uint64 and lims.tolist() == [0] and D.size == 0 and I.size == 0
    # radius <= 0: nothing
    for r in (0.0, -1.0):
        lims, D, I = ix.range_search(q, r)
        assert (lims == 0).all() and D.size == 0
    # nprobe > nlist probes every list
    ix.nprobe = nlist + 7
    _assert_search_equals_dense(ix, q, 10)
    _assert_range_equals_dense(ix, q, float(np.median(ix.search(q, 20)[0][:, -1])))
    # probed empty lists
    assign = rng.integers(0, 4, 3000)
    ix2 = _install(coarse, ix.pq_centroids.cpu().numpy(), ix._codes.cpu().numpy(), assign, nlist)
    assert all(ix2.get_list_size(l) == 0 for l in range(4, nlist))
    _assert_search_equals_dense(ix2, q, 10)
    _assert_range_equals_dense(ix2, q, float(np.median(ix2.search(q, 20)[0][:, -1])))
    # k larger than what the probed lists hold
    ix3 = _install(coarse, ix.pq_centroids.cpu().numpy(), ix._codes.cpu().numpy()[:40], assign[:40], 1)
    D, I = _assert_search_equals_dense(ix3, q, 128)
    assert (I[:, 40:] == -1).all() and (D[:, 40:] == float(FLT_MAX)).all()
    # empty (trained) and untrained indexes
    empty = _install(coarse, ix.pq_centroids.cpu().numpy(), np.zeros((0, M), np.uint8), np.zeros(0, np.int64), 4)
    untrained = fc.IndexIVFPQ(fc.IndexFlatL2(d), d, nlist, M, 8)
    for e in (empty, untrained):
        D, I = e.search(q, 5)
        assert (I == -1).all() and (D == FLT_MAX).all()
        lims, D, I = e.range_search(q, 1e9)
        assert lims.shape == (31,) and (lims == 0).all() and D.size == 0 and I.size == 0
        assert e.get_list_size(3) == 0 and e.get_list_ids(3).size == 0
    # argument errors before any device work
    with pytest.raises(AssertionError):
        ix.range_search(q[:, :10], 1.0)
    with pytest.raises((TypeError, ValueError)):
        ix.range_search(q, "far")


def test_duplicated_codes_tie_on_lowest_ids():
    rng = np.random.default_rng(2)
    d, M, nlist, n = 32, 8, 8, 4000
    coarse = (4.0 * rng.standard_normal((nlist, d))).astype(np.float32)
    pq = rng.standard_normal((M, 256, d // M)).astype(np.float32)
    codes = rng.integers(0, 256, (n, M)).astype(np.uint8)
    assign = rng.integers(0, nlist, n)
    dup = np.nonzero(assign == 3)[0]
    codes[dup] = codes[dup[0]]                               # one code, many ids: exact ties
    ix = _install(coarse, pq, codes, assign, 2)
    q = (coarse[3] + 0.1 * rng.standard_normal((20, d))).astype(np.float32)
    D, I = _assert_search_equals_dense(ix, q, 50)
    I = I.cpu().numpy()
    assert (I[:, :50] == dup[:50]).all()                     # ascending ids among the tied codes
    _assert_range_equals_dense(ix, q, float(D[0, 0]) * 1.0001 + 1e-3)


def test_skewed_list_split_into_chunks():
    rng = np.random.default_rng(3)
    ix, coarse = _random_index(rng, 120_000, 64, 16, 64, 3, skew=100_000)   # list 0 holds ~100k codes
    q = _queries(rng, coarse, 40)
    q[:10] = coarse[0] + rng.standard_normal((10, 64)).astype(np.float32)
    for nq in (1, 40):
        for k in (10, 128):
            _assert_search_equals_dense(ix, q[:nq], k)
    D, _ = ix.search(q, 100)
    _assert_range_equals_dense(ix, q, float(np.median(D[:, -1])))


def test_lut_batching(monkeypatch):
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(4)
    ix, coarse = _random_index(rng, 8000, 64, 16, 32, 6)
    q = _queries(rng, coarse, 50)
    D0, I0 = ix.search(q, 20)
    l0, Dr0, Ir0 = ix.range_search(q, float(np.median(D0[:, -1])))
    monkeypatch.setattr(ops, "IVFPQ_LUT_BUDGET", 3 * 6 * 16 * 256 * 4 + 17)   # 3 queries per call
    assert ops.ivfpq_batch(6, 16, 256) == 3
    D1, I1 = _assert_search_equals_dense(ix, q, 20)
    np.testing.assert_array_equal(D1.cpu().numpy(), D0)
    np.testing.assert_array_equal(I1.cpu().numpy(), I0)
    l1, Dr1, Ir1 = _assert_range_equals_dense(ix, q, float(np.median(D0[:, -1])))
    np.testing.assert_array_equal(l1, l0)
    np.testing.assert_array_equal(Ir1, Ir0)
    np.testing.assert_array_equal(Dr1, Dr0)
    assert ops.last_search_stats["mode"] == "ivfpq-range" and ops.last_search_stats["results"] == int(l0[-1])


def test_workspace_bound_and_every_range_slot_written():
    from image_search_engine_b200 import _lib, ops
    rng = np.random.default_rng(5)
    nq, d, M, nlist, nprobe, k = 2000, 64, 16, 256, 8, 10
    ix, coarse = _random_index(rng, 200_000, d, M, nlist, nprobe)
    qd = torch.from_numpy(_queries(rng, coarse, nq)).cuda()
    codes, ids, off, sizes = ix._lists()
    max_len = int(sizes.max())
    probes = _probes(ix, qd)
    tables = 4 * nq * nprobe * M * 256
    ws = ops.ivfpq_search_workspace_bytes(nq, nprobe, nlist, max_len, M, 256, k)
    S = min(-(-max_len // 1024), max(1, 256 // nprobe), max(1, (1 << 24) // (nq * nprobe * k)))
    assert tables <= ws <= tables + 12 * nq * nprobe * S * k * 257 // 256 + 16 * nq * nprobe + 24 * (nlist + 1) + (64 << 20)
    wr = ops.ivfpq_range_workspace_bytes(nq, nprobe, nlist, max_len, M, 256)
    S = min(-(-max_len // 1024), max(1, 256 // nprobe), max(1, (1 << 22) // (nq * nprobe)))
    assert tables <= wr <= tables + 16 * (nq * nprobe * S + 1) + 16 * nq * nprobe + 24 * (nlist + 1) + (64 << 20)
    # the C ABI with sentinel-filled outputs and slack past the total: every slot below lims[nq] is written, none past
    radius = float(np.median(ix.search(qd[:100], 30)[0][:, -1].cpu().numpy()))
    lib, ctx = _lib.load(), _lib.ctx(torch.cuda.current_device())
    wsb = torch.empty((wr,), dtype=torch.uint8, device="cuda")
    lims = torch.empty((nq + 1,), dtype=torch.int64, device="cuda")
    cent, pq = ix.quantizer._database(), ix.pq_centroids
    _lib.check(lib.ise_ivfpq_range_count(ctx, ops._ptr(qd), nq, d, ops._ptr(cent), nlist, ops._ptr(pq), M, 256,
                                         ops._ptr(codes), ops._ptr(ids), ops._ptr(off), max_len, ops._ptr(probes),
                                         nprobe, radius, ops._ptr(lims), ops._ptr(wsb), wr, ops._stream()))
    total = int(lims[-1])
    assert total > nq
    D = torch.full((total + 64,), float("nan"), dtype=torch.float32, device="cuda")
    I = torch.full((total + 64,), -7, dtype=torch.int64, device="cuda")
    _lib.check(lib.ise_ivfpq_range_fill(ctx, nq, d, nlist, M, 256, ops._ptr(codes), ops._ptr(ids), ops._ptr(off),
                                        max_len, nprobe, radius, ops._ptr(D), ops._ptr(I), ops._ptr(wsb), wr,
                                        ops._stream()))
    assert not torch.isnan(D[:total]).any() and (I[:total] >= 0).all()
    assert torch.isnan(D[total:]).all() and (I[total:] == -7).all()
    l2, D2, I2 = ix.range_search(qd, radius)
    assert torch.equal(l2, lims) and torch.equal(D2, D[:total]) and torch.equal(I2, I[:total])
    # a workspace one byte short is refused
    with pytest.raises(_lib.IseError):
        _lib.check(lib.ise_ivfpq_range_count(ctx, ops._ptr(qd), nq, d, ops._ptr(cent), nlist, ops._ptr(pq), M, 256,
                                             ops._ptr(codes), ops._ptr(ids), ops._ptr(off), max_len, ops._ptr(probes),
                                             nprobe, radius, ops._ptr(lims), ops._ptr(wsb), wr - 1, ops._stream()))


def test_index_beyond_the_dense_matrix():
    """About 20 M codes: the dense path's [4096, ntotal] matrix would need 330 GB; the grouped path searches 10 000
    queries and range-searches them, and a sampled subset equals the dense path bit for bit."""
    from image_search_engine_b200 import faiss_compat as fc
    n, d, M, nlist = 20_000_000, 32, 8, 1024
    g = torch.Generator(device="cuda").manual_seed(6)
    rng = np.random.default_rng(6)
    coarse = (4.0 * rng.standard_normal((nlist, d))).astype(np.float32)
    pq = rng.standard_normal((M, 256, d // M)).astype(np.float32)
    ix = fc.IndexIVFPQ(fc.IndexFlatL2(d), d, nlist, M, 8)
    ix.set_trained_state(coarse, pq)
    ix._codes = torch.randint(0, 256, (n, M), generator=g, device="cuda", dtype=torch.uint8)
    ix._assign = torch.randint(0, nlist, (n,), generator=g, device="cuda", dtype=torch.int64)
    ix._ids = torch.arange(n, dtype=torch.int64, device="cuda")
    ix._sorted = None
    ix.nprobe = 8
    assert 4096 * ix.ntotal * 4 > torch.cuda.get_device_properties(0).total_memory
    q = _queries(rng, coarse, 10_000)
    qd = torch.from_numpy(q).cuda()
    D, I = ix.search(qd, 10)
    assert (I >= 0).all()
    sample = rng.choice(10_000, 32, replace=False)
    De, Ie = _expected_topk(ix, _dense(ix, qd[sample], _probes(ix, qd[sample])), 10)
    np.testing.assert_array_equal(D[sample].cpu().numpy().view(np.uint32), De.view(np.uint32))
    np.testing.assert_array_equal(I[sample].cpu().numpy(), Ie)
    radius = float(D[:, 9].median())
    lims, Dr, Ir = ix.range_search(qd, radius)
    assert 10_000 <= int(lims[-1]) <= 100 * 10_000
    ls = lims.cpu().numpy()
    le, De, Ie = _expected_range(ix, _dense(ix, qd[sample], _probes(ix, qd[sample])), _probes(ix, qd[sample]), radius)
    got_I = np.concatenate([Ir[ls[i]:ls[i + 1]].cpu().numpy() for i in sample])
    got_D = np.concatenate([Dr[ls[i]:ls[i + 1]].cpu().numpy() for i in sample])
    np.testing.assert_array_equal(np.diff(ls)[sample], np.diff(le.astype(np.int64)))
    np.testing.assert_array_equal(got_I, Ie)
    np.testing.assert_array_equal(got_D.view(np.uint32), De.view(np.uint32))


def test_list_introspection_and_pickle():
    rng = np.random.default_rng(7)
    ix, coarse = _random_index(rng, 5000, 64, 16, 32, 4)
    assign = ix._assign.cpu().numpy()
    for l in range(32):
        assert ix.get_list_size(l) == int((assign == l).sum())
        np.testing.assert_array_equal(ix.get_list_ids(l), np.nonzero(assign == l)[0])
    q = _queries(rng, coarse, 40)
    D, I = ix.search(q, 10)
    lims, Dr, Ir = ix.range_search(q, float(np.median(D[:, -1])))
    again = pickle.loads(pickle.dumps(ix))
    assert repr(again) == repr(ix)
    D2, I2 = again.search(q, 10)
    l2, Dr2, Ir2 = again.range_search(q, float(np.median(D[:, -1])))
    np.testing.assert_array_equal(D2, D)
    np.testing.assert_array_equal(I2, I)
    np.testing.assert_array_equal(l2, lims)
    np.testing.assert_array_equal(Ir2, Ir)
    np.testing.assert_array_equal(Dr2, Dr)


def test_recall_no_worse_than_the_oracle_index():
    from image_search_engine_b200 import faiss_compat as fc
    from oracle import faiss_shim as fs
    rng = np.random.default_rng(8)
    n, d, k, nlist = 4000, 64, 10, 16
    cent = 3.0 * rng.standard_normal((30, d))
    x = (cent[rng.integers(0, 30, n)] + rng.standard_normal((n, d))).astype(np.float32)
    q = x[:300] + 0.05 * rng.standard_normal((300, d)).astype(np.float32)
    flat = fc.IndexFlatL2(d)
    flat.add(x)
    _, If = flat.search(q, k)
    ix = fc.IndexIVFPQ(fc.IndexFlatL2(d), d, nlist, 16, 8)
    ix.train(x)
    ix.add(x)
    oracle = fs.IndexIVFPQ(fs.IndexFlatL2(d), d, nlist, 16, 8)
    oracle.train(x)
    oracle.add(x)
    for nprobe in (1, 4):
        ix.nprobe = oracle.nprobe = nprobe
        _, I = ix.search(q, k)
        _, Io = oracle.search(q, k)
        recall = np.mean([len(set(a) & set(b)) / k for a, b in zip(I, If)])
        recall_o = np.mean([len(set(a) & set(b)) / k for a, b in zip(Io, If)])
        assert recall >= recall_o - 0.05, (nprobe, recall, recall_o)
