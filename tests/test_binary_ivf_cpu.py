"""IndexBinaryIVF without a GPU: the NumPy restatement against an np.unpackbits brute force over the probed lists (ties
included), known answers for the training conversion, the GPU class's argument checks before any device work, and the
loud failure."""
import numpy as np
import pytest
import torch

from tests._binary_ivf_oracle import IndexBinaryIVF, binary_to_real, real_to_binary
from tests._binary_oracle import INT32_MAX


def _brute(q, x):
    return (np.unpackbits(q, axis=1)[:, None, :] != np.unpackbits(x, axis=1)[None, :, :]).sum(-1)


@pytest.mark.parametrize("nprobe", [1, 3, 6])
def test_oracle_search_and_range_are_brute_force_over_probed_lists(nprobe):
    rng = np.random.default_rng(nprobe)
    d, nlist = 32, 6
    base = rng.integers(0, 16, (10, d // 8), dtype=np.uint8)           # few distinct codes: many ties
    x = base[rng.integers(0, 10, 400)]
    q = np.concatenate([base[:3], rng.integers(0, 16, (5, d // 8), dtype=np.uint8)])
    ix = IndexBinaryIVF(rng.integers(0, 256, (nlist, d // 8), dtype=np.uint8), d, nlist)
    ix.nprobe = nprobe
    ix.add(x[:150])
    ix.add(x[150:])
    # top-1 assignment with the lowest list id on ties
    dq = _brute(x, ix.quantizer)
    assert np.array_equal(ix.assignment(), np.lexsort((np.broadcast_to(np.arange(nlist), dq.shape), dq), axis=1)[:, 0])
    probes = ix.probes(q)
    dp = _brute(q, ix.quantizer)
    assert np.array_equal(probes, np.lexsort((np.broadcast_to(np.arange(nlist), dp.shape), dp), axis=1)[:, :nprobe])
    assign, dist = ix.assignment(), _brute(q, x)
    for k in (1, 10, 128, 500):
        D, I = ix.search(q, k)
        for i in range(q.shape[0]):
            cand = np.nonzero(np.isin(assign, probes[i]))[0]
            ref = cand[np.lexsort((cand, dist[i, cand]))][:k]
            assert np.array_equal(I[i, :ref.size], ref) and np.array_equal(D[i, :ref.size], dist[i, ref])
            assert (I[i, ref.size:] == -1).all() and (D[i, ref.size:] == INT32_MAX).all()
    for radius in (0, 1, 5, d + 1):
        lims, RD, RI = ix.range_search(q, radius)
        for i in range(q.shape[0]):
            ref = np.concatenate([np.nonzero((assign == l) & (dist[i] < radius))[0] for l in probes[i]])
            assert np.array_equal(RI[lims[i]:lims[i + 1]], ref)
            assert np.array_equal(RD[lims[i]:lims[i + 1]], dist[i, ref])


def test_conversion_known_answers():
    codes = np.array([[0b00000001, 0b10000000], [0xFF, 0x00]], np.uint8)
    x = binary_to_real(codes)
    assert x.dtype == np.float32 and x.shape == (2, 16)
    assert x[0].tolist() == [1] + [-1] * 14 + [1]                     # LSB first, 0 -> -1
    assert x[1].tolist() == [1] * 8 + [-1] * 8
    assert np.array_equal(real_to_binary(x), codes)
    c = np.array([[0.0, 0.5, -0.5, 0.0, 1e-30, -0.0, 2.0, 0.0]], np.float32)
    assert real_to_binary(c).tolist() == [[0b01010010]]                 # exact zeros (and -0) give bit 0


def test_gpu_class_checks_arguments_before_device_work():
    from image_search_engine_b200 import faiss_compat as fc
    for d in (0, 7, 12):
        with pytest.raises(RuntimeError):
            fc.IndexBinaryIVF(fc.IndexBinaryFlat(8), d, 4)
    with pytest.raises(NotImplementedError):
        fc.IndexBinaryIVF(fc.IndexBinaryFlat(2048), 2056, 4)
    with pytest.raises(RuntimeError):
        fc.IndexBinaryIVF(fc.IndexBinaryFlat(128), 256, 4)              # quantizer d mismatch
    ix = fc.IndexBinaryIVF(fc.IndexBinaryFlat(256), 256, 16)
    assert ix.code_size == 32 and ix.nprobe == 1 and not ix.is_trained and ix.ntotal == 0
    with pytest.raises(TypeError):
        ix.train(np.zeros((64, 32), np.float32))
    with pytest.raises(TypeError):
        ix.search(torch.zeros((1, 32), dtype=torch.int8), 5)
    with pytest.raises(TypeError):
        ix.range_search(np.zeros((1, 32), np.int64), 5)
    with pytest.raises(AssertionError):
        ix.train(np.zeros((64, 31), np.uint8))
    with pytest.raises(AssertionError):
        ix.search(np.zeros((1, 33), np.uint8), 5)
    with pytest.raises(AssertionError):
        ix.search(np.zeros((1, 32), np.uint8), 0)
    with pytest.raises(NotImplementedError):
        ix.search(np.zeros((1, 32), np.uint8), 129)
    with pytest.raises(RuntimeError, match="is_trained"):
        ix.add(np.zeros((4, 32), np.uint8))
    big = fc.IndexBinaryIVF(fc.IndexBinaryFlat(64), 64, 200)
    big.nprobe = 129
    with pytest.raises(NotImplementedError):
        big.search(np.zeros((1, 8), np.uint8), 5)
    with pytest.raises(NotImplementedError):
        big.range_search(np.zeros((1, 8), np.uint8), 5)
    with pytest.raises(NotImplementedError):
        fc.write_index(ix, "unused.faiss")
    assert ix.ntotal == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_binary_ivf_fails_loudly_without_gpu():
    from image_search_engine_b200 import IseError, faiss_compat as fc
    x = np.zeros((64, 8), np.uint8)
    ix = fc.IndexBinaryIVF(fc.IndexBinaryFlat(64), 64, 4)
    with pytest.raises(IseError):
        ix.train(x)
    with pytest.raises(IseError):
        ix.search(x, 5)
    with pytest.raises(IseError):
        ix.range_search(x, 3)
