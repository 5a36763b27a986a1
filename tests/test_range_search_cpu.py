"""CPU: the range-search restatement (tests/_range_oracle.py) against an FP64 brute force, and
ShardedIndexFlat.range_search at world size 2 over gloo with that restatement standing in for the device kernels
(the local_ops seam of parallel.py)."""
import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import faiss_shim as fs
from tests._range_oracle import index_range_search, range_search
from tests.test_parallel_gloo import OracleOps, _free_port


def _brute(x, y, radius, metric):
    """FP64 scores; per query the ids beating radius (strictly) and the scores."""
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    if metric == fs.METRIC_INNER_PRODUCT:
        s = x64 @ y64.T
        return s, s > radius
    s = ((x64[:, None, :] - y64[None, :, :]) ** 2).sum(-1)
    return s, s < radius


def _check_layout(lims, D, I, nq, ny):
    assert lims.dtype == np.uint64 and lims.shape == (nq + 1,) and lims[0] == 0
    assert np.all(np.diff(lims.astype(np.int64)) >= 0)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == I.shape == (int(lims[-1]),)
    for i in range(nq):
        ids = I[int(lims[i]):int(lims[i + 1])]
        assert np.all(np.diff(ids) > 0) and (ids.size == 0 or (ids[0] >= 0 and ids[-1] < ny))


@pytest.mark.parametrize("metric", [fs.METRIC_INNER_PRODUCT, fs.METRIC_L2])
@pytest.mark.parametrize("nq", [5, 40])          # direct formulas / BLAS expansion
def test_oracle_range_search_integer_rows_exact_and_strict(metric, nq):
    # integer rows: every FP32 score is exact, so the FP64 brute force must agree bit for bit and the radius can be set
    # to a score that occurs -- that column must be excluded (strict comparison)
    rng = np.random.default_rng(3 + nq)
    y = rng.integers(0, 8, (1500, 24)).astype(np.float32)
    x = y[rng.integers(0, 1500, nq)].copy()
    s64, _ = _brute(x, y, 0, metric)
    radius = float(np.sort(s64[0])[::-1][30] if metric == fs.METRIC_INNER_PRODUCT else np.sort(s64[0])[30])
    lims, D, I = range_search(x, y, radius, metric)
    _check_layout(lims, D, I, nq, y.shape[0])
    s64, keep = _brute(x, y, radius, metric)
    on_radius = 0
    for i in range(nq):
        ids = I[int(lims[i]):int(lims[i + 1])]
        assert np.array_equal(ids, np.nonzero(keep[i])[0])
        np.testing.assert_array_equal(D[int(lims[i]):int(lims[i + 1])], s64[i, ids].astype(np.float32))
        on_radius += int((s64[i] == radius).sum())
        assert not np.any(s64[i, ids] == radius)
    assert on_radius > 0, "no score equals the radius: strictness was not exercised"


@pytest.mark.parametrize("metric", [fs.METRIC_INNER_PRODUCT, fs.METRIC_L2])
@pytest.mark.parametrize("nq", [3, 25])
def test_oracle_range_search_float_rows_match_fp64(metric, nq):
    rng = np.random.default_rng(11)
    y = rng.standard_normal((2100, 40)).astype(np.float32)
    x = rng.standard_normal((nq, 40)).astype(np.float32)
    radius = 12.0 if metric == fs.METRIC_INNER_PRODUCT else 55.0
    lims, D, I = range_search(x, y, radius, metric)
    _check_layout(lims, D, I, nq, y.shape[0])
    s64, keep = _brute(x, y, radius, metric)
    tau = 1e-4 * np.abs(s64).max()
    for i in range(nq):
        ids = I[int(lims[i]):int(lims[i + 1])]
        sure = set(np.nonzero(keep[i] & (np.abs(s64[i] - radius) > tau))[0])
        maybe = set(np.nonzero(np.abs(s64[i] - radius) <= tau)[0])
        assert sure <= set(ids) <= sure | maybe
        np.testing.assert_allclose(D[int(lims[i]):int(lims[i + 1])], s64[i, ids], rtol=1e-4, atol=1e-3)
    assert lims[-1] > 10 * nq


def test_oracle_index_range_search_and_edges():
    rng = np.random.default_rng(5)
    y = rng.standard_normal((300, 16)).astype(np.float32)
    for metric, cls in ((fs.METRIC_INNER_PRODUCT, fs.IndexFlatIP), (fs.METRIC_L2, fs.IndexFlatL2)):
        index = cls(16)
        lims, D, I = index_range_search(index, y[:4], 1.0)                         # empty index
        assert lims.tolist() == [0] * 5 and D.size == 0 and I.size == 0
        index.add(y[:100])
        index.add(y[100:])
        q = np.asmatrix(y[:30])
        got = index_range_search(index, q, 3.0)
        want = range_search(y[:30], y, 3.0, metric)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)
        lims, D, I = index_range_search(index, y[:0], 3.0)                         # nq = 0
        assert lims.tolist() == [0] and D.size == 0


def _data():
    rng = np.random.default_rng(21)
    db = rng.standard_normal((1501, 24)).astype(np.float32)
    db[744:758] = db[751] + 0.05 * rng.standard_normal((14, 24)).astype(np.float32)   # a cluster across the shard cut
    db[1200] = db[3]                                                              # exact cross-shard duplicate
    q = db[rng.integers(0, 1501, 40)] + 0.01 * rng.standard_normal((40, 24)).astype(np.float32)
    q[0] = db[3]
    q[1] = db[751]
    return db, q


RADII = {fs.METRIC_INNER_PRODUCT: 9.0, fs.METRIC_L2: 12.0}


class RangeOracleOps(OracleOps):
    def range_search(self, q, q_op, db, b_op, metric, radius, id_base):
        lims, D, I = range_search(q_op.numpy(), b_op.numpy(), radius, metric)
        return torch.from_numpy(lims.astype(np.int64)), torch.from_numpy(D), torch.from_numpy(I + id_base)


def _worker(rank, world, port, out):
    import os
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from image_search_engine_b200.parallel import ShardedIndexFlat, shard_bounds
        db, q = _data()
        bd = shard_bounds(db.shape[0], world)
        res = {}
        for metric in (fs.METRIC_INNER_PRODUCT, fs.METRIC_L2):
            idx = ShardedIndexFlat(24, metric, local_ops=RangeOracleOps())
            idx.add_local(db[bd[rank]:bd[rank + 1]])
            for nq in (5, 40):
                lims, D, I = idx.range_search(q[:nq], RADII[metric])
                res[(metric, nq)] = (lims.numpy().copy(), D.numpy().copy(), I.numpy().copy())
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_sharded_range_search_world_size_2_matches_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    db, q = _data()
    cut = 751
    for metric in (fs.METRIC_INNER_PRODUCT, fs.METRIC_L2):
        for nq in (5, 40):
            want = range_search(q[:nq], db, RADII[metric], metric)
            for r in (out[0], out[1]):
                lims, D, I = r[(metric, nq)]
                assert np.array_equal(lims, want[0].astype(np.int64))
                assert np.array_equal(I, want[2])
                np.testing.assert_allclose(D, want[1], rtol=1e-6, atol=1e-6)
            lims, _, I = out[0][(metric, nq)]
            ids1 = I[lims[1]:lims[2]]
            assert ids1.min() < cut <= ids1.max(), "matches of query 1 do not straddle the shard cut"
            ids0 = I[lims[0]:lims[1]]
            assert 3 in ids0 and 1200 in ids0
