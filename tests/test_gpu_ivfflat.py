"""IndexIVFFlat on the GPU: lock-step with the NumPy restatement (tests/_ivfflat_oracle.py), exactness against the flat
index when every list is probed, edge cases, training, workspace bound and a benchmark-size FP64 check."""
import pickle

import numpy as np
import pytest
import torch

from oracle import faiss_shim as fs
from tests._ivfflat_oracle import IndexIVFFlat as OracleIVFFlat
from tests._util import assert_topk_parity, scores64, unit_rows

pytestmark = pytest.mark.gpu

FLT_MAX = float(np.finfo(np.float32).max)


def _clustered(rng, n, d, centers=24, spread=3.0):
    c = spread * rng.standard_normal((centers, d)).astype(np.float32)
    return (c[rng.integers(0, centers, n)] + rng.standard_normal((n, d))).astype(np.float32)


def _data(rng, n, d, metric_ip):
    x = _clustered(rng, n, d)
    if metric_ip:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def _gpu_index(centroids, metric_ip, nlist=None):
    from image_search_engine_b200 import faiss_compat as fc
    d = centroids.shape[1]
    quant = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    quant.add(centroids)
    return fc.IndexIVFFlat(quant, d, nlist or centroids.shape[0], fc.METRIC_INNER_PRODUCT if metric_ip else fc.METRIC_L2)


def _gpu_assignment(ix):
    out = np.full(ix.ntotal, -1, np.int64)
    for l in range(ix.nlist):
        out[ix.get_list_ids(l)] = l
    return out


def _probes(ix, q):
    qd = torch.from_numpy(np.ascontiguousarray(q, dtype=np.float32)).cuda()
    return ix.quantizer._search_device(qd, min(ix.nprobe, ix.nlist), need_distances=False)[1].cpu().numpy()


def _assert_sorted(D, metric_ip):
    assert (np.diff(D, axis=1) <= 0).all() if metric_ip else (np.diff(D, axis=1) >= 0).all()


@pytest.mark.parametrize("d", [64, 100, 2048])
@pytest.mark.parametrize("metric_ip", [False, True])
def test_ivfflat_lockstep_with_oracle(metric_ip, d):
    rng = np.random.default_rng(d + 7 * metric_ip)
    n, nlist, nq, k = 3000, 16, 80, 10
    x = _data(rng, n, d, metric_ip)
    q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    ref = OracleIVFFlat(fs.IndexFlatIP(d) if metric_ip else fs.IndexFlatL2(d), d, nlist,
                        fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    ref.train(x)
    ref.add(x[:1200])
    ref.add(x[1200:])
    cent = ref.quantizer.reconstruct_n()
    ix = _gpu_index(cent, metric_ip)
    assert ix.is_trained
    ix.train(x)                                                       # quantizer holds nlist centroids: no clustering
    np.testing.assert_array_equal(ix.quantizer.reconstruct_n(), cent)
    ix.add(x[:1200])
    ix.add(x[1200:])
    assert ix.ntotal == n
    assign, ref_assign = _gpu_assignment(ix), ref.assignment()
    assert (assign >= 0).all()
    bad = np.nonzero(assign != ref_assign)[0]
    assert bad.size <= 0.005 * n                                      # coarse near ties only
    if bad.size:
        s = scores64(x[bad], cent, metric_ip)
        gap = np.abs(s[np.arange(bad.size), assign[bad]] - s[np.arange(bad.size), ref_assign[bad]])
        assert (gap <= 1e-3 * np.abs(s).max()).all()
    for l in range(nlist):
        assert (np.diff(ix.get_list_ids(l)) > 0).all()
    ix.reset()
    ix.add_preassigned(x, ref_assign)                                 # the oracle's lists
    for nprobe in (1, 4):
        ix.nprobe = ref.nprobe = nprobe
        D, I = ix.search(q, k)
        assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (nq, k)
        Dr, Ir = ref.search(q, k, probes=_probes(ix, q))
        assert_topk_parity(I, Ir, q, x, metric_ip)
        same = I == Ir
        np.testing.assert_allclose(D[same], Dr[same], rtol=1e-4, atol=1e-5 * np.abs(Dr).max())
        _assert_sorted(D, metric_ip)


@pytest.mark.parametrize("nlist", [64, 1024])
@pytest.mark.parametrize("metric_ip", [False, True])
def test_ivfflat_all_lists_probed_equals_flat(metric_ip, nlist):
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(nlist + metric_ip)
    n, d, nq, k = 20000, 48, 300, 20
    x = _data(rng, n, d, metric_ip)
    q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    ix = _gpu_index(x[rng.choice(n, nlist, replace=False)], metric_ip)
    ix.add(x)
    ix.nprobe = nlist                                                 # nprobe * chunks > 256 lists: two-level merge
    D, I = ix.search(q, k)
    flat = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    flat.add(x)
    Df, If = flat.search(q, k)
    assert_topk_parity(I, If, q, x, metric_ip)
    s = scores64(q, x, metric_ip)
    np.testing.assert_allclose(D, np.take_along_axis(s, I, 1), rtol=1e-4, atol=1e-5 * np.abs(s).max())
    _assert_sorted(D, metric_ip)


def test_ivfflat_edge_cases():
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(5)
    d, nlist, n = 37, 8, 300                                          # d % 4 != 0: scalar loads
    x = np.rint(_clustered(rng, n, d) * 10).clip(0, 255).astype(np.float32)
    ix = _gpu_index(x[:nlist].copy(), False)
    # untrained and empty indexes return padding
    un = fc.IndexIVFFlat(fc.IndexFlatL2(d), d, nlist)
    D, I = un.search(x[:3], 5)
    assert not un.is_trained and (I == -1).all() and (D == FLT_MAX).all()
    D, I = ix.search(x[:3], 5)
    assert (I == -1).all() and (D == FLT_MAX).all()
    # lists 0, 2, 5 only: the others are empty
    lists = np.array([0, 2, 5])[rng.integers(0, 3, n)]
    ix.add_preassigned(x, lists)
    assert [ix.get_list_size(l) for l in range(nlist)] == list(np.bincount(lists, minlength=nlist))
    ref = OracleIVFFlat(fs.IndexFlatL2(d), d, nlist)
    ref.quantizer.add(x[:nlist])
    ref.is_trained = True
    ref.add_preassigned(x, lists)
    ix.nprobe = 100                                                   # clamped to nlist
    D, I = ix.search(x[:50], 10)
    Dr, Ir = ref.search(x[:50], 10, probes=np.tile(np.arange(nlist), (50, 1)))
    assert_topk_parity(I, Ir, x[:50], x, False)
    # k above the scanned count: exact padding
    ix.nprobe = 1
    q1 = x[:1]
    pr = _probes(ix, q1)[0, 0]
    D, I = ix.search(q1, 128)
    held = ix.get_list_size(pr)
    assert ((I[0] >= 0).sum() == held) and (I[0, held:] == -1).all() and (D[0, held:] == FLT_MAX).all()
    assert set(I[0, :held]) == set(ix.get_list_ids(pr))
    D1, I1 = ix.search(q1, 1)
    assert I1[0, 0] == I[0, 0] and D1[0, 0] == D[0, 0]
    with pytest.raises(NotImplementedError):
        ix.search(q1, 129)
    D, I = ix.search(x[:0], 4)
    assert D.shape == (0, 4) and I.shape == (0, 4)
    # uint8 queries equal their float32 values
    ix.nprobe = 3
    Du, Iu = ix.search(x[:40].astype(np.uint8), 7)
    Df, If = ix.search(x[:40], 7)
    assert np.array_equal(Iu, If) and np.array_equal(Du, Df)
    # CUDA tensors in -> CUDA tensors out, same values
    Dt, It = ix.search(torch.from_numpy(x[:40]).cuda(), 7)
    assert Dt.is_cuda and It.is_cuda and Dt.dtype == torch.float32 and It.dtype == torch.int64
    assert np.array_equal(It.cpu().numpy(), If) and np.array_equal(Dt.cpu().numpy(), Df)
    # pickle round trip
    ix2 = pickle.loads(pickle.dumps(ix))
    assert ix2.ntotal == n and ix2.nprobe == 3 and ix2.is_trained
    D2, I2 = ix2.search(x[:40], 7)
    assert np.array_equal(I2, If) and np.array_equal(D2, Df)
    # reset + a new add (uint8 rows)
    ix.reset()
    assert ix.ntotal == 0 and ix.is_trained
    ix.add(x[:100].astype(np.uint8))
    assert ix.ntotal == 100 and sum(ix.get_list_size(l) for l in range(nlist)) == 100
    ix.nprobe = nlist
    D, I = ix.search(x[:5], 1)
    assert (I[:, 0] == np.arange(5)).all() and (D[:, 0] == 0).all()


@pytest.mark.parametrize("metric_ip", [False, True])
def test_ivfflat_exact_duplicates_lowest_id_wins(metric_ip):
    rng = np.random.default_rng(21)
    d, nlist, n = 32, 4, 400
    x = unit_rows(rng, n, d)
    v = x[7].copy()
    for i in (90, 200, 301):                                          # duplicates of row 7
        x[i] = v
    lists = rng.integers(0, nlist, n)
    lists[[7, 200]] = 1                                               # two copies in one list ...
    lists[[90, 301]] = [2, 3]                                         # ... and one in each of two others
    ix = _gpu_index(unit_rows(rng, nlist, d), metric_ip)
    ix.add_preassigned(x, lists)
    ix.nprobe = nlist
    D, I = ix.search(np.stack([v, v]), 6)
    assert (I[:, :4] == [7, 90, 200, 301]).all()
    assert (D[:, :4] == D[:, :1]).all()
    ix.nprobe = 1                                                     # with only one list probed: its copies, in id order
    D, I = ix.search(v[None], 3)
    l = _probes(ix, v[None])[0, 0]
    dup = sorted(i for i in (7, 90, 200, 301) if lists[i] == l)
    assert list(I[0, :len(dup)]) == dup


def test_ivfflat_skewed_list_is_split_into_chunks():
    rng = np.random.default_rng(8)
    d, nlist, n, k = 64, 16, 40000, 10
    x = _data(rng, n, d, False)
    lists = np.where(rng.random(n) < 0.9, 3, rng.integers(0, nlist, n))          # list 3 holds ~90 %
    cent = x[rng.choice(n, nlist, replace=False)]
    cent[3] = x[lists == 3][5]
    ix = _gpu_index(cent, False)
    ix.add_preassigned(x, lists)
    ref = OracleIVFFlat(fs.IndexFlatL2(d), d, nlist)
    ref.quantizer.add(ix.quantizer.reconstruct_n())
    ref.is_trained = True
    ref.add_preassigned(x, lists)
    for nq, nprobe in ((1, 1), (1, 4), (200, 2)):
        q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
        q[0] = x[lists == 3][5]
        ix.nprobe = nprobe
        D, I = ix.search(q, k)
        Dr, Ir = ref.search(q, k, probes=_probes(ix, q))
        assert_topk_parity(I, Ir, q, x, False)
        np.testing.assert_allclose(D, Dr, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("metric_ip", [False, True])
def test_ivfflat_training_end_to_end(metric_ip):
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(31 + metric_ip)
    n, d, nlist, nq, k = 8000, 32, 40, 200, 10
    x = _data(rng, n, d, metric_ip)
    q = x[rng.integers(0, n, nq)] + 0.1 * rng.standard_normal((nq, d)).astype(np.float32)
    quant = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    metric = fc.METRIC_INNER_PRODUCT if metric_ip else fc.METRIC_L2
    ix = fc.IndexIVFFlat(quant, d, nlist, metric)
    ix.train(x)
    km = fc.Kmeans(d, nlist, niter=10, seed=1234, spherical=metric_ip)
    km.train(x)
    # same code path; the centroid sums of the Lloyd update may round differently from run to run (a few ulps)
    np.testing.assert_allclose(ix.quantizer.reconstruct_n(), km.centroids, rtol=2e-6, atol=1e-6)
    ix.add(x)
    ix.nprobe = 4
    _, I = ix.search(q, k)
    ref = OracleIVFFlat(fs.IndexFlatIP(d) if metric_ip else fs.IndexFlatL2(d), d, nlist,
                        fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    ref.train(x)
    ref.add(x)
    ref.nprobe = 4
    _, Ir = ref.search(q, k)
    flat = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    flat.add(x)
    _, If = flat.search(q, k)
    recall = np.mean([len(set(a) & set(b)) / k for a, b in zip(I, If)])
    recall_ref = np.mean([len(set(a) & set(b)) / k for a, b in zip(Ir, If)])
    assert recall >= recall_ref - 0.05, (recall, recall_ref)


def test_ivfflat_search_builds_no_dense_matrix():
    from image_search_engine_b200 import ops
    nq, ntotal, d, nlist, nprobe, k = 4096, 1_000_000, 32, 1024, 16, 10
    g = torch.Generator(device="cuda").manual_seed(4)
    xd = torch.randn((ntotal, d), generator=g, device="cuda")
    ix = _gpu_index(xd[:nlist].cpu().numpy(), False)
    ix.add(xd)
    ix.nprobe = nprobe
    q = xd[:nq] + 0.1
    ix.search(q[:20], k)                                              # builds the list-sorted storage
    xs, ids, off = ix._lists()
    _, probes = ix.quantizer._search_device(q, nprobe, need_distances=False)
    max_len = int(ix._sizes.max())
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    D, I = ops.ivfflat_search(q, xs, ids, off, max_len, probes, ix.metric_type, k)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    ws = ops.ivfflat_search_workspace_bytes(nq, nprobe, nlist, max_len, k)
    assert rise <= ws + 2 * nq * k * 12 + (4 << 20), (rise, ws)
    assert ws <= 12 * max(1 << 24, nq * nprobe * k) * 257 // 256 + 16 * nq * nprobe + 24 * (nlist + 1) + (64 << 20)
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    D2, I2 = ix.search(q, k)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < nq * ntotal * 4 // 20
    assert torch.equal(I2, I) and torch.equal(D2, D)


def test_ivfflat_benchmark_size_fp64_check():
    rng = np.random.default_rng(12)
    ntotal, d, nlist, nprobe, nq, k = 1_000_000, 512, 4096, 32, 10_000, 10
    g = torch.Generator(device="cuda").manual_seed(12)
    centers = torch.randn((4096, d), generator=g, device="cuda")
    xd = centers[torch.randint(0, 4096, (ntotal,), generator=g, device="cuda")] + \
        0.5 * torch.randn((ntotal, d), generator=g, device="cuda")
    xd /= xd.norm(dim=1, keepdim=True)
    ix = _gpu_index(xd[torch.randint(0, ntotal, (nlist,), generator=g, device="cuda")].cpu().numpy(), True)
    ix.add(xd)
    ix.nprobe = nprobe
    q = xd[torch.randint(0, ntotal, (nq,), generator=g, device="cuda")] + \
        0.05 * torch.randn((nq, d), generator=g, device="cuda")
    D, I = ix.search(q, k)
    rows = rng.choice(nq, 100, replace=False)
    qs = q[rows].cpu().numpy()
    probes = ix.quantizer._search_device(q[rows].contiguous(), nprobe, need_distances=False)[1].cpu().numpy()
    D, I = D[rows].cpu().numpy(), I[rows].cpu().numpy()
    lists = {}
    ref_I = np.empty_like(I)
    for r in range(rows.size):
        cand = np.concatenate([lists.setdefault(l, ix.get_list_ids(l)) for l in probes[r]])
        y = xd[torch.from_numpy(cand).cuda()].cpu().numpy().astype(np.float64)
        s = y @ qs[r].astype(np.float64)
        order = np.lexsort((cand, -s))[:k]
        ref_I[r] = cand[order]
        s_of = dict(zip(cand.tolist(), s.tolist()))
        got = np.array([s_of[i] for i in I[r]])                       # every returned id lies in a probed list
        np.testing.assert_allclose(D[r], got, rtol=1e-4, atol=1e-6)
        # ids as assert_topk_parity: a mismatch is an FP32 near tie (tau = 16 eps |q| max|y|, unit rows)
        tau = 16 * np.finfo(np.float32).eps * np.linalg.norm(qs[r].astype(np.float64))
        diff = I[r] != ref_I[r]
        assert (np.abs(got[diff] - s[order][diff]) <= tau).all()
    assert (I != ref_I).any(axis=1).mean() <= 0.01
