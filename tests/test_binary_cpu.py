"""IndexBinaryFlat without a GPU: the NumPy restatement against an np.unpackbits brute force (ties included), and the
GPU class's argument checks before any device work / loud failure."""
import numpy as np
import pytest
import torch

from tests._binary_oracle import INT32_MAX, IndexBinaryFlat, hamming


def _brute(q, x):
    """Hamming distances bit by bit."""
    return (np.unpackbits(q, axis=1)[:, None, :] != np.unpackbits(x, axis=1)[None, :, :]).sum(-1)


@pytest.mark.parametrize("d", [8, 24, 64, 72, 256, 520])
def test_oracle_distances_match_unpackbits(d):
    rng = np.random.default_rng(d)
    x = rng.integers(0, 256, (300, d // 8), dtype=np.uint8)
    q = rng.integers(0, 256, (17, d // 8), dtype=np.uint8)
    assert np.array_equal(hamming(q, x), _brute(q, x))


@pytest.mark.parametrize("k", [1, 2, 10, 128, 400])
def test_oracle_search_and_range_are_brute_force_with_ties(k):
    rng = np.random.default_rng(k)
    d = 32
    base = rng.integers(0, 16, (12, d // 8), dtype=np.uint8)          # few distinct codes: many equal distances
    x = base[rng.integers(0, 12, 350)]
    q = np.concatenate([base[:3], rng.integers(0, 16, (5, d // 8), dtype=np.uint8)])
    ix = IndexBinaryFlat(d)
    ix.add(x[:100])
    ix.add(x[100:])
    D, I = ix.search(q, k)
    dist = _brute(q, x)
    ref = np.lexsort((np.broadcast_to(np.arange(x.shape[0]), dist.shape), dist), axis=1)[:, :k]
    kk = min(k, x.shape[0])
    assert np.array_equal(I[:, :kk], ref)
    assert np.array_equal(D[:, :kk], np.take_along_axis(dist, ref, 1))
    assert (I[:, kk:] == -1).all() and (D[:, kk:] == INT32_MAX).all()
    for radius in (0, 1, 5, d + 1):
        lims, RD, RI = ix.range_search(q, radius)
        for i in range(q.shape[0]):
            ids = np.nonzero(dist[i] < radius)[0]
            assert np.array_equal(RI[lims[i]:lims[i + 1]], ids)
            assert np.array_equal(RD[lims[i]:lims[i + 1]], dist[i, ids])


def test_gpu_class_checks_arguments_before_device_work():
    from image_search_engine_b200 import faiss_compat
    for d in (0, 7, 12, 260):
        with pytest.raises(RuntimeError):
            faiss_compat.IndexBinaryFlat(d)
    with pytest.raises(NotImplementedError):
        faiss_compat.IndexBinaryFlat(2056)
    ix = faiss_compat.IndexBinaryFlat(256)
    assert ix.code_size == 32 and ix.ntotal == 0 and ix.is_trained and ix.d == 256
    with pytest.raises(TypeError):
        ix.add(np.zeros((4, 32), np.float32))
    with pytest.raises(TypeError):
        ix.add(torch.zeros((4, 32), dtype=torch.int8))
    with pytest.raises(TypeError):
        ix.search(np.zeros((1, 32), np.int64), 5)
    with pytest.raises(AssertionError):
        ix.add(np.zeros((4, 31), np.uint8))
    with pytest.raises(AssertionError):
        ix.search(np.zeros((1, 33), np.uint8), 5)
    with pytest.raises(AssertionError):
        ix.range_search(np.zeros(32, np.uint8), 5)
    with pytest.raises(AssertionError):
        ix.search(np.zeros((1, 32), np.uint8), 0)
    with pytest.raises(NotImplementedError):
        ix.search(np.zeros((1, 32), np.uint8), 129)
    with pytest.raises(NotImplementedError):
        faiss_compat.write_index(ix, "unused.faiss")
    assert ix.ntotal == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_binary_fails_loudly_without_gpu():
    from image_search_engine_b200 import IseError, faiss_compat
    x = np.zeros((64, 8), np.uint8)
    ix = faiss_compat.IndexBinaryFlat(64)
    with pytest.raises(IseError):
        ix.add(x)
    with pytest.raises(IseError):
        ix.search(x, 5)
    with pytest.raises(IseError):
        ix.range_search(x, 3)
