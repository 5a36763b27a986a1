"""IndexBinaryFlat on the GPU, bit for bit against the NumPy restatement (tests/_binary_oracle.py): search and range search
over code widths that are and are not multiples of 16 bytes, every threads-per-query and column-split regime, heavy
ties, edge cases, CUDA tensors, pickling, the workspace bound and a 1 M x 256-bit check."""
import pickle

import numpy as np
import pytest
import torch

from tests._binary_oracle import (INT32_MAX, IndexBinaryFlat as OracleBinaryFlat, hamming, knn_from_distances,
                                  range_from_distances)

pytestmark = pytest.mark.gpu


def _gpu(d, *parts):
    from image_search_engine_b200 import faiss_compat as fc
    ix = fc.IndexBinaryFlat(d)
    for p in parts:
        ix.add(p)
    return ix


def _assert_range_equal(got, want):
    lims, D, I = got
    assert lims.dtype == np.uint64 and D.dtype == np.int32 and I.dtype == np.int64
    for g, w in zip((lims, D, I), want):
        assert np.array_equal(g, w)


def _assert_range_matches_search(lims, RD, RI, D, I):
    """For every id both calls return, the range distance equals the search distance."""
    for i in range(D.shape[0]):
        ids, dis = RI[lims[i]:lims[i + 1]], RD[lims[i]:lims[i + 1]]
        common, a, b = np.intersect1d(ids, I[i], return_indices=True)
        assert np.array_equal(dis[a], D[i, b])


@pytest.mark.parametrize("nq", [1, 7, 500, 5000])
@pytest.mark.parametrize("d", [8, 24, 64, 256, 512, 520, 2048])
def test_search_bit_exact(d, nq):
    rng = np.random.default_rng(d * 10 + nq)
    nb = 3000 if d >= 512 else 6000
    x = rng.integers(0, 256, (nb, d // 8), dtype=np.uint8)
    q = rng.integers(0, 256, (nq, d // 8), dtype=np.uint8)
    q[: nq // 2] = x[rng.integers(0, nb, nq // 2)]                      # distance 0 hits
    ix = _gpu(d, x[:1000], x[1000:])
    dist = hamming(q, x)
    for k in (1, 2, 10, 128):
        D, I = ix.search(q, k)
        assert D.dtype == np.int32 and I.dtype == np.int64 and D.shape == (nq, k)
        Dr, Ir = knn_from_distances(dist, k)
        assert np.array_equal(I, Ir), k
        assert np.array_equal(D, Dr), k


def test_search_single_chunk_grid():
    """A batch large enough that every column chunk is the whole database (one partial list per query)."""
    rng = np.random.default_rng(5)
    x = rng.integers(0, 256, (3000, 8), dtype=np.uint8)
    q = rng.integers(0, 256, (80_000, 8), dtype=np.uint8)
    D, I = _gpu(64, x).search(q, 10)
    Dr, Ir = knn_from_distances(hamming(q, x), 10)
    assert np.array_equal(I, Ir) and np.array_equal(D, Dr)


@pytest.mark.parametrize("kind", ["duplicates", "alphabet4"])
@pytest.mark.parametrize("nq", [1, 7, 40, 300])
def test_heavy_ties_lowest_ids_win(kind, nq):
    rng = np.random.default_rng(nq + (kind == "duplicates"))
    d, nb = 256, 40_000
    if kind == "duplicates":
        base = rng.integers(0, 256, (25, d // 8), dtype=np.uint8)
        x = base[rng.integers(0, 25, nb)]                               # ~1600 copies of every code, spread over ids
        q = base[rng.integers(0, 25, nq)]
    else:
        x = rng.integers(0, 16, (nb, d // 8), dtype=np.uint8)           # 4 live bits per byte: few distinct distances
        q = rng.integers(0, 16, (nq, d // 8), dtype=np.uint8)
    ix = _gpu(d, x)
    dist = hamming(q, x)
    cut_ties = False
    for k in (1, 2, 10, 128):
        D, I = ix.search(q, k)
        Dr, Ir = knn_from_distances(dist, k)
        assert np.array_equal(I, Ir) and np.array_equal(D, Dr), (kind, k)
        kth = Dr[:, -1][:, None]
        cut_ties |= bool(((dist == kth).sum(1) > (Dr == kth).sum(1)).any())
    assert cut_ties        # some k-th distance is shared by more codes than fit: the tie falls on the k-th place


def test_edge_cases():
    rng = np.random.default_rng(2)
    d = 64
    x = rng.integers(0, 256, (37, 8), dtype=np.uint8)
    q = rng.integers(0, 256, (9, 8), dtype=np.uint8)
    ix = _gpu(d, x)
    dist = hamming(q, x)
    for k in (36, 37, 38, 128):                                          # k < ntotal, ==, >
        D, I = ix.search(q, k)
        Dr, Ir = knn_from_distances(dist, k)
        assert np.array_equal(I, Ir) and np.array_equal(D, Dr)
    assert (ix.search(q, 128)[1][:, 37:] == -1).all() and (ix.search(q, 128)[0][:, 37:] == INT32_MAX).all()
    D, I = ix.search(np.zeros((0, 8), np.uint8), 5)                     # nq = 0
    assert D.shape == (0, 5) and I.shape == (0, 5) and D.dtype == np.int32
    lims, RD, RI = ix.range_search(np.zeros((0, 8), np.uint8), 3)
    assert lims.shape == (1,) and lims[0] == 0 and RD.size == 0 and RD.dtype == np.int32
    empty = _gpu(d)                                                      # empty index
    D, I = empty.search(q, 4)
    assert (I == -1).all() and (D == INT32_MAX).all() and D.dtype == np.int32
    lims, RD, RI = empty.range_search(q, 65)
    assert (lims == 0).all() and lims.dtype == np.uint64 and RD.size == 0 and RI.size == 0
    zeros = _gpu(d, np.zeros((700, 8), np.uint8))                       # all-zero codes: every distance ties
    D, I = zeros.search(np.zeros((3, 8), np.uint8), 10)
    assert (D == 0).all() and (I == np.arange(10)).all()
    lims, RD, RI = zeros.range_search(np.zeros((3, 8), np.uint8), 1)
    assert np.array_equal(lims, [0, 700, 1400, 2100]) and (RD == 0).all() and np.array_equal(RI[:700], np.arange(700))


@pytest.mark.parametrize("nq", [1, 7, 500])
@pytest.mark.parametrize("d", [64, 256, 520])
def test_range_search_bit_exact(d, nq):
    rng = np.random.default_rng(d + nq)
    nb = 20_000
    centers = rng.integers(0, 256, (40, d // 8), dtype=np.uint8)
    flips = np.packbits(rng.random((nb, d)) < 0.08, axis=1)              # clusters: distances spread from 0 up
    x = centers[rng.integers(0, 40, nb)] ^ flips
    q = x[rng.integers(0, nb, nq)] ^ np.packbits(rng.random((nq, d)) < 0.02, axis=1)
    ix = _gpu(d, x)
    dist = hamming(q, x)
    D, I = ix.search(q, 128)
    for radius in (0, 1, d // 4, d + 1):
        got = ix.range_search(q, radius)
        want = range_from_distances(dist, radius)
        _assert_range_equal(got, want)
        if radius == 0:
            assert got[0][-1] == 0
        if radius == d + 1:
            assert got[0][-1] == nq * nb
        _assert_range_matches_search(*got, D, I)


def test_cuda_tensors_in_and_out_pickle_reset_reconstruct():
    rng = np.random.default_rng(9)
    d = 512
    x = rng.integers(0, 256, (5000, 64), dtype=np.uint8)
    q = x[:50] ^ np.packbits(rng.random((50, d)) < 0.05, axis=1)
    ix = _gpu(d, torch.from_numpy(x[:2000]).cuda(), x[2000:])
    D, I = ix.search(q, 10)
    Dt, It = ix.search(torch.from_numpy(q).cuda(), 10)
    assert Dt.is_cuda and It.is_cuda and Dt.dtype == torch.int32 and It.dtype == torch.int64
    assert np.array_equal(Dt.cpu().numpy(), D) and np.array_equal(It.cpu().numpy(), I)
    lims, RD, RI = ix.range_search(q, 60)
    tl, tD, tI = ix.range_search(torch.from_numpy(q).cuda(), 60)
    assert tl.is_cuda and tl.dtype == torch.int64 and tD.dtype == torch.int32
    assert np.array_equal(tl.cpu().numpy(), lims) and np.array_equal(tD.cpu().numpy(), RD)
    assert np.array_equal(tI.cpu().numpy(), RI)
    assert np.array_equal(ix.reconstruct(4321), x[4321]) and ix.reconstruct(4321).dtype == np.uint8
    assert np.array_equal(ix.reconstruct_n(1990, 20), x[1990:2010]) and np.array_equal(ix.reconstruct_n(), x)
    assert "IndexBinaryFlat" in repr(ix) and "ntotal=5000" in repr(ix)
    ix2 = pickle.loads(pickle.dumps(ix))
    assert ix2.ntotal == 5000 and ix2.d == d
    D2, I2 = ix2.search(q, 10)
    assert np.array_equal(D2, D) and np.array_equal(I2, I)
    ix.reset()
    assert ix.ntotal == 0
    ix.add(x[2500:])
    D3, I3 = ix.search(q, 10)
    oracle = OracleBinaryFlat(d)
    oracle.add(x[2500:])
    Dr, Ir = oracle.search(q, 10)
    assert np.array_equal(D3, Dr) and np.array_equal(I3, Ir)


def test_workspace_within_stated_bound():
    from image_search_engine_b200 import ops
    for nq, nb, cs, k in [(1, 10_000_000, 8, 10), (500, 1_000_000, 32, 2), (10_000, 1_000_000, 64, 128),
                          (200_000, 50_000, 32, 128), (7, 300, 256, 1)]:
        ws = ops.binary_knn_workspace_bytes(nq, nb, cs, k)
        assert 0 < ws <= 12 * max(1 << 24, nq * k) + 4 * nq * k + 768, (nq, nb, k, ws)
        rws = ops.binary_range_workspace_bytes(nq, nb, cs)
        assert 0 < rws <= 16 * (max(1 << 22, nq) + 1) + 512 + (64 << 20), (nq, nb, rws)
    # a search allocates its workspace and outputs, never an [nq, ntotal] matrix
    rng = np.random.default_rng(3)
    x = torch.from_numpy(rng.integers(0, 256, (400_000, 32), dtype=np.uint8)).cuda()
    q = x[:4000].clone()
    ix = _gpu(256, x)
    ix.search(q, 10)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    ix.search(q, 10)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base <= ops.binary_knn_workspace_bytes(4000, 400_000, 32, 10) + (4 << 20)


def test_full_size_1m_256_bit():
    rng = np.random.default_rng(2024)
    nb, d = 1_000_000, 256
    x = rng.integers(0, 256, (nb, d // 8), dtype=np.uint8)
    x[rng.integers(0, nb, 20_000)] = x[rng.integers(0, nb, 20_000)]     # some exact duplicates
    ix = _gpu(d, x)
    nq = 10_000
    q = x[rng.integers(0, nb, nq)] ^ np.packbits(rng.random((nq, d)) < 0.1, axis=1)
    D, I = ix.search(q, 10)
    lims, RD, RI = ix.range_search(q, 40)
    rows = rng.choice(nq, 500, replace=False)
    dist = hamming(q[rows], x)
    Dr, Ir = knn_from_distances(dist, 10)
    assert np.array_equal(I[rows], Ir) and np.array_equal(D[rows], Dr)
    rl, rD, rI = range_from_distances(dist, 40)
    for j, i in enumerate(rows):
        assert np.array_equal(RI[lims[i]:lims[i + 1]], rI[rl[j]:rl[j + 1]])
        assert np.array_equal(RD[lims[i]:lims[i + 1]], rD[rl[j]:rl[j + 1]])
    _assert_range_matches_search(lims, RD, RI, D, I)
