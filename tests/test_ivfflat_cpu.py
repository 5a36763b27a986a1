"""IndexIVFFlat without a GPU: the NumPy restatement against FP64 brute force, the inverted-list invariants, and the
GPU class's argument checks / loud failure."""
import numpy as np
import pytest
import torch

from oracle import faiss_shim as fs
from tests._ivfflat_oracle import IndexIVFFlat
from tests._util import assert_topk_parity, scores64, unit_rows


def _clustered(rng, n, d, centers=24):
    c = 3.0 * rng.standard_normal((centers, d)).astype(np.float32)
    return (c[rng.integers(0, centers, n)] + rng.standard_normal((n, d))).astype(np.float32)


@pytest.mark.parametrize("metric_ip", [False, True])
def test_oracle_all_lists_probed_is_brute_force(metric_ip):
    rng = np.random.default_rng(11 + metric_ip)
    n, d, nlist, nq, k = 1500, 24, 16, 40, 10
    x = unit_rows(rng, n, d) if metric_ip else _clustered(rng, n, d)
    q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    quant = fs.IndexFlatIP(d) if metric_ip else fs.IndexFlatL2(d)
    ix = IndexIVFFlat(quant, d, nlist, fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    assert not ix.is_trained
    ix.train(x)
    assert ix.is_trained and quant.ntotal == nlist
    ix.add(x[:700])
    ix.add(x[700:])
    ix.nprobe = nlist
    D, I = ix.search(q, k)
    s = scores64(q, x, metric_ip)
    ref = np.argsort(-s if metric_ip else s, axis=1, kind="stable")[:, :k]
    assert_topk_parity(I, ref, q, x, metric_ip)
    np.testing.assert_allclose(D, np.take_along_axis(s, I, 1), rtol=1e-4, atol=1e-4)
    assert (np.diff(D, axis=1) <= 0).all() if metric_ip else (np.diff(D, axis=1) >= 0).all()


def test_oracle_list_invariants_after_several_adds():
    rng = np.random.default_rng(3)
    d, nlist = 16, 8
    x = _clustered(rng, 900, d)
    ix = IndexIVFFlat(fs.IndexFlatL2(d), d, nlist)
    ix.train(x)
    for a, b in ((0, 100), (100, 101), (101, 600), (600, 900)):
        ix.add(x[a:b])
    all_ids = np.concatenate(ix.ids)
    assert np.array_equal(np.sort(all_ids), np.arange(900))            # every id exactly once
    for l in range(nlist):
        assert (np.diff(ix.ids[l]) > 0).all()                           # ids ascend inside a list
        assert np.array_equal(ix.vecs[l], x[ix.ids[l]])
    assert np.array_equal(ix.assignment(), ix.assign(x))
    ix.reset()
    assert ix.ntotal == 0 and ix.is_trained
    D, I = ix.search(x[:2], 3)
    assert (I == -1).all() and (D == np.finfo(np.float32).max).all()


def test_gpu_class_checks_quantizer_dimension_before_device_work():
    from image_search_engine_b200 import faiss_compat
    with pytest.raises(RuntimeError):
        faiss_compat.IndexIVFFlat(faiss_compat.IndexFlatL2(8), 16, 4)
    with pytest.raises(NotImplementedError):
        faiss_compat.IndexIVFFlat(faiss_compat.IndexFlatL2(8), 8, 4, metric=7)
    ix = faiss_compat.IndexIVFFlat(faiss_compat.IndexFlatIP(8), 8, 4, faiss_compat.METRIC_INNER_PRODUCT)
    assert not ix.is_trained and ix.nprobe == 1 and ix.ntotal == 0 and ix.nlist == 4
    with pytest.raises(RuntimeError, match="is_trained"):
        ix.add(np.zeros((4, 8), np.float32))
    with pytest.raises(NotImplementedError):
        ix.search(np.zeros((1, 8), np.float32), 129)
    with pytest.raises(NotImplementedError):
        faiss_compat.write_index(ix, "unused.faiss")


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_ivfflat_fails_loudly_without_gpu():
    from image_search_engine_b200 import IseError, faiss_compat
    x = np.zeros((64, 8), np.float32)
    ix = faiss_compat.IndexIVFFlat(faiss_compat.IndexFlatL2(8), 8, 4)
    with pytest.raises(IseError):
        ix.train(x)
    with pytest.raises(IseError):
        ix.search(x, 5)
