"""IndexFlat.range_search on the B200: parity with the oracle (FP64 scores, near-radius ids exempt), the coarse bound on
adversarial operands, overflow re-runs, edge cases and agreement with search."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from tests._util import EPS32, near_tie_tol, orb_like, scores64, sift_like, unit_rows

pytestmark = pytest.mark.gpu


def _index(metric_ip, d):
    from image_search_engine_b200 import faiss_compat
    return faiss_compat.IndexFlatIP(d) if metric_ip else faiss_compat.IndexFlatL2(d)


def _tau(x, y, metric_ip, factor=16.0):
    t = near_tie_tol(x, y, factor)
    if not metric_ip:
        t = 2 * t + factor * EPS32 * ((x.astype(np.float64) ** 2).sum(1) + (y.astype(np.float64) ** 2).sum(1).max())
    return t


def _assert_range_parity(lims, D, I, x, y, radius, metric_ip, rows=None):
    """Per query: ids strictly ascending, every id clearing the radius by more than tau present, none missing it by
    more than tau; distances equal to the FP64 scores to rtol 1e-4."""
    lims = np.asarray(lims).astype(np.int64)
    D, I = np.asarray(D), np.asarray(I)
    nq = x.shape[0]
    assert lims.shape == (nq + 1,) and lims[0] == 0 and np.all(np.diff(lims) >= 0)
    assert D.shape == I.shape == (lims[-1],) and D.dtype == np.float32 and I.dtype == np.int64
    rows = range(nq) if rows is None else rows
    s = scores64(x[list(rows)], y, metric_ip)
    tau = _tau(x[list(rows)], y, metric_ip)
    for j, i in enumerate(rows):
        ids = I[lims[i]:lims[i + 1]]
        assert np.all(np.diff(ids) > 0), f"row {i}: ids not ascending"
        margin = (s[j] - radius) if metric_ip else (radius - s[j])
        sure = np.nonzero(margin > tau[j])[0]
        assert np.isin(sure, ids).all(), f"row {i}: {np.setdiff1d(sure, ids)[:5]} missing"
        assert (margin[ids] >= -tau[j]).all(), f"row {i}: returned ids miss the radius by more than tau"
        np.testing.assert_allclose(D[lims[i]:lims[i + 1]], s[j, ids], rtol=1e-4, atol=tau[j])


def _radius_for(x, y, metric_ip, per_query):
    s = scores64(x, y, metric_ip)
    q = per_query / y.shape[0]
    return float(np.quantile(s, 1 - q) if metric_ip else np.quantile(s, q))


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("d", [64, 100, 2048])
def test_range_parity_both_regimes(metric_ip, d):
    rng = np.random.default_rng(d + (0 if metric_ip else 1))
    y = unit_rows(rng, 4000, d)
    x = y[rng.integers(0, 4000, 300)] + 0.3 * unit_rows(rng, 300, d)
    index = _index(metric_ip, d)
    index.add(y)
    for nq in (5, 300):
        for per_query in (10, 300):
            radius = _radius_for(x[:nq], y, metric_ip, per_query)
            lims, D, I = index.range_search(x[:nq], radius)
            assert lims.dtype == np.uint64
            _assert_range_parity(lims, D, I, x[:nq], y, radius, metric_ip)
            assert per_query / 3 < lims[-1] / nq < 3 * per_query


def test_range_multicast_cluster_shape():
    """d = 2048 with 65 536 database rows: the B hi plane is 256 MB (the collect runs with multicast clusters)."""
    from image_search_engine_b200 import faiss_compat, ops
    dev = ops.require_cuda()
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    n, d, nq = 65536, 2048, 300
    y = torch.randn((n, d), generator=gen, device=dev)
    y /= y.norm(dim=1, keepdim=True)
    x = y[:nq] + 0.5 * torch.randn((nq, d), generator=gen, device=dev) / d ** 0.5
    index = faiss_compat.IndexFlatIP(d)
    index.add(y)
    lims, D, I = index.range_search(x, 0.06)
    assert ops.search_stats()["mode"] == "range"
    yh, xh = y.cpu().numpy(), x.cpu().numpy()
    _assert_range_parity(lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy(), xh, yh, 0.06, True, rows=range(48))
    assert 20 < int(lims[-1]) / nq < 2000


@pytest.mark.parametrize("metric_ip", [True, False])
def test_range_overflow_rerun_matches_large_cap(metric_ip):
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(5)
    y = unit_rows(rng, 5000, 128)
    x = unit_rows(rng, 200, 128)
    radius = _radius_for(x, y, metric_ip, 60)
    index = _index(metric_ip, 128)
    index.add(y)
    q = torch.from_numpy(x).cuda()
    a = ops.prepare_operand(q, rows=True)
    big = ops.range_search(q, a, index._database(), index._operand(), index.metric_type, radius, _cap=8192)
    assert ops.search_stats()["overflow_rows"] == 0
    small = ops.range_search(q, a, index._database(), index._operand(), index.metric_type, radius, _cap=16)
    st = ops.search_stats()
    assert st["overflow_rows"] > 0 and st["results"] == int(big[0][-1])
    for u, v in zip(big, small):
        assert torch.equal(u, v)
    _assert_range_parity(*(t.cpu().numpy() for t in small), x, y, radius, metric_ip)


@pytest.mark.parametrize("metric_ip", [True, False])
def test_range_adversarial_bound(metric_ip):
    from tests.test_gpu_fullsize import _adversarial
    rng = np.random.default_rng(2049)
    a, b = _adversarial(rng, 256, 6000, 2048)
    index = _index(metric_ip, 2048)
    index.add(b)
    s = scores64(a[:1], b, metric_ip)[0]
    radius = float(np.median(s))                    # among the near-duplicates of one base row
    lims, D, I = index.range_search(a, radius)
    _assert_range_parity(lims, D, I, a, b, radius, metric_ip)
    assert lims[-1] > 0


def test_range_edges():
    from image_search_engine_b200 import faiss_compat
    rng = np.random.default_rng(9)
    d = 128
    # empty index, nq = 0
    index = faiss_compat.IndexFlatIP(d)
    lims, D, I = index.range_search(unit_rows(rng, 30, d), 0.1)
    assert lims.tolist() == [0] * 31 and D.size == 0 and I.size == 0
    y = sift_like(rng, 3000, d)                     # integer rows: every FP32 score is exact
    index.add(y)
    lims, D, I = index.range_search(y[:0], 0.1)
    assert lims.tolist() == [0] and D.size == 0
    for nq in (5, 300):
        own = rng.integers(0, 3000, nq)
        x = y[own]
        # nothing / everything
        lims, D, I = index.range_search(x, 1e30)
        assert lims.tolist() == [0] * (nq + 1)
        lims, D, I = index.range_search(x, -1e30)
        assert (np.diff(lims.astype(np.int64)) == 3000).all()
        assert np.array_equal(I.reshape(nq, 3000), np.broadcast_to(np.arange(3000), (nq, 3000)))
        # radius = an exact FP32 score that occurs (the self-match of query 0): excluded, strictly
        s = scores64(x, y, True)
        radius = float(s[0, own[0]])
        assert np.float32(radius) == radius
        lims, D, I = index.range_search(x, radius)
        lims = lims.astype(np.int64)
        for i in range(nq):
            assert np.array_equal(I[lims[i]:lims[i + 1]], np.nonzero(s[i] > radius)[0])
        assert own[0] not in I[lims[0]:lims[1]]
    # L2 with the radius at an exact squared distance
    l2 = faiss_compat.IndexFlatL2(d)
    l2.add(y)
    x = y[rng.integers(0, 3000, 300)] + 1
    s = scores64(x, y, False)
    radius = float(np.sort(s[0])[20])
    lims, D, I = l2.range_search(x, radius)
    lims = lims.astype(np.int64)
    for i in range(300):
        assert np.array_equal(I[lims[i]:lims[i + 1]], np.nonzero(s[i] < radius)[0])
        np.testing.assert_array_equal(D[lims[i]:lims[i + 1]], s[i, s[i] < radius].astype(np.float32))


def test_range_uint8_queries_and_cuda_io_and_add_reset():
    from image_search_engine_b200 import faiss_compat
    from oracle import faiss_shim as fs
    from tests._range_oracle import range_search
    rng = np.random.default_rng(13)
    yb = orb_like(rng, 2500, 32)
    index = faiss_compat.IndexFlatIP(32)
    index.add(yb[:1000].astype(np.float32))
    index.add(yb[1000:].astype(np.float32))                 # several add() calls
    xb = yb[rng.integers(0, 2500, 300)]
    s = scores64(xb, yb, True)
    radius = float(np.quantile(s, 1 - 50 / 2500))
    for nq in (5, 300):
        lims, D, I = index.range_search(xb[:nq], radius)     # uint8 queries (integer scores: exact)
        want = range_search(xb[:nq].astype(np.float32), yb.astype(np.float32), radius, fs.METRIC_INNER_PRODUCT)
        assert np.array_equal(lims, want[0]) and np.array_equal(I, want[2]) and np.array_equal(D, want[1])
        # CUDA in -> CUDA out
        lc, Dc, Ic = index.range_search(torch.from_numpy(xb[:nq]).cuda(), radius)
        assert lc.is_cuda and Dc.is_cuda and Ic.is_cuda and lc.dtype == torch.int64
        assert np.array_equal(lc.cpu().numpy(), want[0].astype(np.int64)) and np.array_equal(Ic.cpu().numpy(), want[2])
    index.reset()
    lims, D, I = index.range_search(xb[:30], radius)
    assert lims.tolist() == [0] * 31
    index.add(yb[:100].astype(np.float32))
    lims, D, I = index.range_search(xb[:30], radius)
    want = range_search(xb[:30].astype(np.float32), yb[:100].astype(np.float32), radius, fs.METRIC_INNER_PRODUCT)
    assert np.array_equal(lims, want[0]) and np.array_equal(I, want[2])


@pytest.mark.parametrize("metric_ip", [True, False])
def test_range_contains_search_hits_beyond_radius(metric_ip):
    rng = np.random.default_rng(17)
    y = unit_rows(rng, 20000, 256)
    x = y[rng.integers(0, 20000, 400)] + 0.2 * unit_rows(rng, 400, 256)
    index = _index(metric_ip, 256)
    index.add(y)
    radius = _radius_for(x[:50], y, metric_ip, 30)
    Ds, Is = index.search(x, 50)
    lims, D, I = index.range_search(x, radius)
    lims = lims.astype(np.int64)
    for i in range(400):
        beat = Is[i][(Ds[i] > radius) if metric_ip else (Ds[i] < radius)]
        assert np.isin(beat, I[lims[i]:lims[i + 1]]).all(), f"row {i}"


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_range_search_on_two_gpus():
    script = Path(__file__).parent / "multi_gpu_range_check.py"
    env = dict(os.environ, NCCL_DEBUG="WARN")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", str(script)],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and "MULTI_GPU_RANGE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
