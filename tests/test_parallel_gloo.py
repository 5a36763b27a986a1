"""CPU, world_size 2 over gloo: the sharding / collective control flow of parallel.py, with the oracle
standing in for the device kernels (local_ops seam).  The product default (DeviceOps) is exercised on
the GPU box by tests/test_gpu_api.py and bench.py --gpus N."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import faiss_shim as fs


class OracleOps:
    """Same interface as parallel.DeviceOps, NumPy/oracle arithmetic on CPU tensors."""

    def device(self):
        return torch.device("cpu")

    def to_local(self, x):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        return t if t.dtype in (torch.float32, torch.uint8) else t.to(torch.float32)

    def prepare(self, x, reuse=False, rows=False, reject_nonfinite=False):
        return x

    def new_buffers(self, k, d, dev):
        accum = torch.empty((k * d + k,), dtype=torch.float32)
        return accum, accum[:k * d].view(k, d), accum[k * d:], torch.zeros((1,), dtype=torch.float64)

    def assign(self, x, a_op, cent, metric, precision="verified"):
        D, I = fs.knn(a_op.numpy().astype(np.float32), cent.numpy(), 1, metric)
        return torch.from_numpy(D), torch.from_numpy(I)

    def accumulate(self, x, assign, dis, sums, counts, obj, cent=None, metric=None, a_op=None):
        a = assign.numpy().ravel()
        np.add.at(counts.numpy(), a, np.float32(1))
        np.add.at(sums.numpy(), a, x.numpy().astype(np.float32))
        obj += float(dis.numpy().astype(np.float64).sum())

    def finalize(self, sums, counts, cent, n_global, spherical, obj):
        c, h = cent.numpy(), counts.numpy().copy()
        c[:] = 0
        nz = h != 0
        c[nz] = sums.numpy()[nz] * (np.float32(1) / h[nz])[:, None]
        ns = fs.split_clusters(c.shape[1], c.shape[0], n_global, h, c)
        if spherical:
            fs.normalize_L2(c)
        return ns, float(obj.item())

    def normalize(self, cent):
        fs.normalize_L2(cent.numpy())

    def search(self, q, db, b_op, metric, k, id_base):
        D, I = fs.knn(q.numpy(), b_op.numpy(), k, metric)
        I = np.where(I >= 0, I + id_base, -1)
        return torch.from_numpy(D), torch.from_numpy(I)

    def merge(self, Dg, Ig, metric):
        g, m, k = Dg.shape
        D = Dg.numpy().transpose(1, 0, 2).reshape(m, g * k)
        I = Ig.numpy().transpose(1, 0, 2).reshape(m, g * k)
        key = -D if metric == fs.METRIC_INNER_PRODUCT else D
        ikey = np.where(I < 0, np.iinfo(np.int64).max, I)
        order = np.lexsort((ikey, key), axis=1)[:, :k]
        return torch.from_numpy(np.take_along_axis(D, order, 1)), torch.from_numpy(np.take_along_axis(I, order, 1))


def _data():
    rng = np.random.default_rng(12)
    centers = rng.standard_normal((12, 16)).astype(np.float32) * 4
    x = centers[rng.integers(0, 12, 3001)] + rng.standard_normal((3001, 16)).astype(np.float32)
    x[:1500] = x[0]  # heavy duplicates: several initial centroids coincide -> empty clusters -> split path
    db = rng.standard_normal((1501, 24)).astype(np.float32)
    db[700] = db[3]  # cross-shard exact tie: lower id must win
    q = db[rng.integers(0, 1501, 40)] + 0.01 * rng.standard_normal((40, 24)).astype(np.float32)
    q[0] = db[3]
    return x, db, q


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from image_search_engine_b200.parallel import ShardedIndexFlat, ShardedKmeans, shard_bounds
        x, db, q = _data()
        res = {}
        b = shard_bounds(x.shape[0], world)
        for name, kw in [("spherical", dict(k=16, spherical=True, niter=5, seed=42, nredo=2)),
                         ("l2_subsample", dict(k=8, spherical=False, niter=4, seed=7))]:
            k = kw.pop("k")
            km = ShardedKmeans(16, k, local_ops=OracleOps(), **kw)
            km.train(x[b[rank]:b[rank + 1]])
            res[name] = (km.centroids.copy(), km.obj.copy(), [s["nsplit"] for s in km.iteration_stats])
        bd = shard_bounds(db.shape[0], world)
        for metric in (fs.METRIC_INNER_PRODUCT, fs.METRIC_L2):
            idx = ShardedIndexFlat(24, metric, local_ops=OracleOps())
            idx.add_local(db[bd[rank]:bd[rank + 1]])
            assert idx.ntotal == db.shape[0] and idx.id_base == bd[rank]
            D, I = idx.search(q, 10)
            res[f"search{metric}"] = (D.numpy().copy(), I.numpy().copy())
        out[rank] = res
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.timeout(300)
def test_world_size_2_matches_single_process():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    x, db, q = _data()
    r0, r1 = out[0], out[1]
    # k-means: both ranks end with identical centroids, equal (to FP32 sum-order noise) to one process
    for name, kw in [("spherical", dict(k=16, spherical=True, niter=5, seed=42, nredo=2)),
                     ("l2_subsample", dict(k=8, spherical=False, niter=4, seed=7))]:
        k = kw.pop("k")
        assert np.array_equal(r0[name][0], r1[name][0]) and np.array_equal(r0[name][1], r1[name][1])
        ref = fs.Kmeans(16, k, **kw)
        ref.train(x)
        np.testing.assert_allclose(r0[name][0], ref.centroids, rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(r0[name][1], ref.obj, rtol=1e-4)  # Faiss sums obj in FP32, sequentially
        assert r0[name][2] == [s["nsplit"] for s in ref.iteration_stats]
    assert sum(r0["spherical"][2]) > 0, "split path was not exercised"
    # sharded search == unsharded search, including the cross-shard tie
    for metric in (fs.METRIC_INNER_PRODUCT, fs.METRIC_L2):
        D, I = fs.knn(q, db, 10, metric)
        for r in (r0, r1):
            assert np.array_equal(r[f"search{metric}"][1], I)
            np.testing.assert_allclose(r[f"search{metric}"][0], D, rtol=1e-6, atol=1e-6)
    assert r0[f"search{fs.METRIC_INNER_PRODUCT}"][1][0, 0] == 3
