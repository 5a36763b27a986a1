"""IndexIVFFlat range search without a GPU: the NumPy restatement (tests/_ivfflat_range_oracle.py) against FP64 brute
force over the probed lists, its (probe rank, list position) order, and equality with the flat range search when every
list is probed."""
import numpy as np
import pytest
import torch

from oracle import faiss_shim as fs
from tests._ivfflat_oracle import IndexIVFFlat
from tests._ivfflat_range_oracle import assert_scan_order, range_search
from tests._range_oracle import range_search as flat_range_search
from tests._util import EPS32, near_tie_tol, scores64, unit_rows


def _clustered(rng, n, d, centers=24):
    c = 3.0 * rng.standard_normal((centers, d)).astype(np.float32)
    return (c[rng.integers(0, centers, n)] + rng.standard_normal((n, d))).astype(np.float32)


def _tau(x, y, metric_ip, factor=16.0):
    t = near_tie_tol(x, y, factor)
    if not metric_ip:
        t = 2 * t + factor * EPS32 * ((x.astype(np.float64) ** 2).sum(1) + (y.astype(np.float64) ** 2).sum(1).max())
    return t


def _index(rng, metric_ip, n=1500, d=24, nlist=16):
    x = unit_rows(rng, n, d) if metric_ip else _clustered(rng, n, d)
    ix = IndexIVFFlat(fs.IndexFlatIP(d) if metric_ip else fs.IndexFlatL2(d), d, nlist,
                      fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    ix.train(x)
    ix.add(x[:700])
    ix.add(x[700:])
    return ix, x


def _radius(s, metric_ip, per_query):
    return float(np.quantile(s, 1 - per_query / s.shape[1]) if metric_ip else np.quantile(s, per_query / s.shape[1]))


@pytest.mark.parametrize("nprobe", [1, 4])
@pytest.mark.parametrize("metric_ip", [False, True])
def test_restatement_against_fp64_over_probed_lists(metric_ip, nprobe):
    rng = np.random.default_rng(40 + 2 * nprobe + metric_ip)
    ix, x = _index(rng, metric_ip)
    ix.nprobe = nprobe
    q = x[rng.integers(0, x.shape[0], 30)] + 0.05 * rng.standard_normal((30, x.shape[1])).astype(np.float32)
    s = scores64(q, x, metric_ip)
    radius = _radius(s, metric_ip, 40)
    probes = ix.probes(q)
    lims, D, I = range_search(ix, q, radius)
    assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
    assert lims[0] == 0 and (np.diff(lims.astype(np.int64)) >= 0).all() and D.shape == I.shape == (int(lims[-1]),)
    assert lims[-1] > 0
    assign = ix.assignment()
    tau = _tau(q, x, metric_ip)
    for i in range(q.shape[0]):
        seg = slice(int(lims[i]), int(lims[i + 1]))
        probed = np.isin(assign, probes[i])
        margin = (s[i] - radius) if metric_ip else (radius - s[i])
        sure = np.nonzero(probed & (margin > tau[i]))[0]
        assert np.isin(sure, I[seg]).all()
        assert probed[I[seg]].all() and (margin[I[seg]] >= -tau[i]).all()
        np.testing.assert_allclose(D[seg], s[i, I[seg]], rtol=1e-4, atol=tau[i])
    assert_scan_order(probes, assign, ix.ids, lims, I)


@pytest.mark.parametrize("metric_ip", [False, True])
def test_all_lists_probed_is_the_flat_range_search(metric_ip):
    rng = np.random.default_rng(7 + metric_ip)
    ix, x = _index(rng, metric_ip)
    ix.nprobe = ix.nlist
    q = x[rng.integers(0, x.shape[0], 25)] + 0.05 * rng.standard_normal((25, x.shape[1])).astype(np.float32)
    radius = _radius(scores64(q, x, metric_ip), metric_ip, 60)
    lims, D, I = range_search(ix, q, radius)
    lf, Df, If = flat_range_search(q, x, radius, ix.metric_type)
    s = scores64(q, x, metric_ip)
    tau = _tau(q, x, metric_ip)
    for i in range(q.shape[0]):
        a = set(I[int(lims[i]):int(lims[i + 1])].tolist())
        b = set(If[int(lf[i]):int(lf[i + 1])].tolist())
        for j in a ^ b:                                   # the two formulas may disagree only next to the radius
            assert abs(s[i, j] - radius) <= tau[i]
    assert_scan_order(ix.probes(q), ix.assignment(), ix.ids, lims, I)


def test_empty_and_untrained_restatement():
    d = 8
    ix = IndexIVFFlat(fs.IndexFlatL2(d), d, 4)
    lims, D, I = range_search(ix, np.zeros((3, d), np.float32), 1.0)
    assert (lims == 0).all() and lims.shape == (4,) and D.size == I.size == 0
    lims, D, I = range_search(ix, np.zeros((0, d), np.float32), 1.0)
    assert lims.shape == (1,) and lims[0] == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_gpu_range_search_fails_loudly_without_gpu():
    from image_search_engine_b200 import IseError, faiss_compat
    ix = faiss_compat.IndexIVFFlat(faiss_compat.IndexFlatL2(8), 8, 4)
    with pytest.raises(IseError):
        ix.range_search(np.zeros((2, 8), np.float32), 1.0)
