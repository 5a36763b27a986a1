"""IndexIVFFlat.range_search on the GPU: bit equality with the NumPy restatement (tests/_ivfflat_range_oracle.py) on
integer data, FP64 parity on float data, agreement with search, edge cases, a skewed list split into chunks, the
workspace bound and a benchmark-size FP64 check."""
import pickle

import numpy as np
import pytest
import torch

from oracle import faiss_shim as fs
from tests._ivfflat_oracle import IndexIVFFlat as OracleIVFFlat
from tests._ivfflat_range_oracle import assert_scan_order, range_search as oracle_range_search
from tests._util import EPS32, near_tie_tol, scores64, sift_like, unit_rows

pytestmark = pytest.mark.gpu


def _clustered(rng, n, d, centers=24, spread=3.0):
    c = spread * rng.standard_normal((centers, d)).astype(np.float32)
    return (c[rng.integers(0, centers, n)] + rng.standard_normal((n, d))).astype(np.float32)


def _tau(x, y, metric_ip, factor=16.0):
    t = near_tie_tol(x, y, factor)
    if not metric_ip:
        t = 2 * t + factor * EPS32 * ((x.astype(np.float64) ** 2).sum(1) + (y.astype(np.float64) ** 2).sum(1).max())
    return t


def _pair(cent, x, lists, metric_ip):
    """The GPU index and the restatement holding the same centroids and lists."""
    from image_search_engine_b200 import faiss_compat as fc
    d, nlist = x.shape[1], cent.shape[0]
    quant = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    quant.add(cent)
    ix = fc.IndexIVFFlat(quant, d, nlist, fc.METRIC_INNER_PRODUCT if metric_ip else fc.METRIC_L2)
    ix.add_preassigned(x, lists)
    ref = OracleIVFFlat(fs.IndexFlatIP(d) if metric_ip else fs.IndexFlatL2(d), d, nlist,
                        fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    ref.quantizer.add(cent)
    ref.is_trained = True
    ref.add_preassigned(x, lists)
    return ix, ref


def _probes(ix, q):
    qd = torch.from_numpy(np.ascontiguousarray(q, dtype=np.float32)).cuda()
    return ix.quantizer._search_device(qd, min(ix.nprobe, ix.nlist), need_distances=False)[1].cpu().numpy()


def _assert_order(ix, ref, q, lims, I):
    assert_scan_order(_probes(ix, q), ref.assignment(), ref.ids, lims, I)


def _probed(lists, probes):
    """probed[i, j]: vector j lies in one of query i's probed lists."""
    return (lists[None, :, None] == probes[:, None, :]).any(2)


def _radius_probed(s, probed, metric_ip, per_query):
    """A radius that keeps about per_query of each query's probed vectors (median over the queries)."""
    kth = []
    for i in range(s.shape[0]):
        v = np.sort(s[i, probed[i]])
        if metric_ip:
            v = v[::-1]
        if v.size:
            kth.append(v[min(per_query, v.size) - 1])
    return float(np.median(kth))


def _assert_parity(lims, D, I, q, x, probed, radius, metric_ip):
    """Membership against FP64 over the probed lists (ids within tau of the radius exempt), D to rtol 1e-4."""
    lims = np.asarray(lims).astype(np.int64)
    s = scores64(q, x, metric_ip)
    tau = _tau(q, x, metric_ip)
    for i in range(q.shape[0]):
        ids = I[lims[i]:lims[i + 1]]
        margin = (s[i] - radius) if metric_ip else (radius - s[i])
        sure = np.nonzero(probed[i] & (margin > tau[i]))[0]
        assert np.isin(sure, ids).all(), f"query {i}: {np.setdiff1d(sure, ids)[:5]} missing"
        assert probed[i][ids].all(), f"query {i}: a result outside the probed lists"
        assert (margin[ids] >= -tau[i]).all(), f"query {i}: results miss the radius by more than tau"
        np.testing.assert_allclose(D[lims[i]:lims[i + 1]], s[i, ids], rtol=1e-4, atol=tau[i])


@pytest.mark.parametrize("d", [128, 2048])
@pytest.mark.parametrize("metric_ip", [False, True])
def test_integer_data_equals_restatement_bit_for_bit(metric_ip, d):
    """Integer rows whose FP32 partial sums are all exact: lims, D and I equal the restatement, order included."""
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(d + metric_ip)
    n, nlist, nq = 4000, 16, 60
    x = sift_like(rng, n, d) if d == 128 else rng.integers(0, 8, (n, d)).astype(np.float32)
    q = sift_like(rng, nq, d) if d == 128 else rng.integers(0, 8, (nq, d)).astype(np.float32)
    cent = x[rng.choice(n, nlist, replace=False)]
    lists = np.argmax(scores64(x, cent, True), 1) if metric_ip else np.argmin(scores64(x, cent, False), 1)
    ix, ref = _pair(cent, x, lists, metric_ip)
    s = scores64(q, x, metric_ip)
    flat = fc.IndexFlatIP(d) if metric_ip else fc.IndexFlatL2(d)
    flat.add(x)
    for nprobe in (1, 4, nlist):
        ix.nprobe = nprobe
        pr = _probes(ix, q)
        radius = _radius_probed(s, _probed(lists, pr), metric_ip, 100)
        lims, D, I = ix.range_search(q, radius)
        assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
        lr, Dr, Ir = oracle_range_search(ref, q, radius, probes=pr)
        assert lims[-1] > 0
        np.testing.assert_array_equal(lims, lr)
        np.testing.assert_array_equal(I, Ir)
        np.testing.assert_array_equal(D, Dr)
        _assert_order(ix, ref, q, lims, I)
        if nprobe == nlist:
            lf, Df, If = flat.range_search(q, radius)
            np.testing.assert_array_equal(lims, lf)
            for i in range(nq):
                seg = slice(int(lims[i]), int(lims[i + 1]))
                o = np.argsort(I[seg], kind="stable")
                np.testing.assert_array_equal(I[seg][o], If[seg])
                np.testing.assert_array_equal(D[seg][o], Df[seg])


@pytest.mark.parametrize("per_query", [10, 300])
@pytest.mark.parametrize("d", [64, 100, 2048])
@pytest.mark.parametrize("metric_ip", [False, True])
def test_float_data_parity_with_fp64(metric_ip, d, per_query):
    rng = np.random.default_rng(3 * d + metric_ip + per_query)
    n, nlist, nq, nprobe = 3000, 16, 40, 4
    x = _clustered(rng, n, d)
    if metric_ip:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
    q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    cent = x[rng.choice(n, nlist, replace=False)]
    lists = np.argmax(scores64(x, cent, True), 1) if metric_ip else np.argmin(scores64(x, cent, False), 1)
    ix, ref = _pair(cent, x, lists, metric_ip)
    ix.nprobe = nprobe
    pr = _probes(ix, q)
    probed = _probed(lists, pr)
    radius = _radius_probed(scores64(q, x, metric_ip), probed, metric_ip, per_query)
    lims, D, I = ix.range_search(q, radius)
    assert lims[-1] >= nq * per_query // 4
    _assert_parity(lims, D, I, q, x, probed, radius, metric_ip)
    _assert_order(ix, ref, q, lims, I)


@pytest.mark.parametrize("metric_ip", [False, True])
def test_agrees_with_search_bit_for_bit(metric_ip):
    rng = np.random.default_rng(17 + metric_ip)
    n, d, nlist, nq, k = 6000, 48, 32, 100, 40
    x = _clustered(rng, n, d)
    if metric_ip:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
    q = x[rng.integers(0, n, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    cent = x[rng.choice(n, nlist, replace=False)]
    lists = np.argmax(scores64(x, cent, True), 1) if metric_ip else np.argmin(scores64(x, cent, False), 1)
    ix, _ = _pair(cent, x, lists, metric_ip)
    ix.nprobe = 4
    pr = _probes(ix, q)
    probed = _probed(lists, pr)
    radius = np.float32(_radius_probed(scores64(q, x, metric_ip), probed, metric_ip, 25))
    Ds, Is = ix.search(q, k)
    lims, D, I = ix.range_search(q, radius)
    lims = lims.astype(np.int64)
    full = 0
    for i in range(nq):
        got = dict(zip(I[lims[i]:lims[i + 1]].tolist(), D[lims[i]:lims[i + 1]].tolist()))
        beat = (Is[i] >= 0) & ((Ds[i] > radius) if metric_ip else (Ds[i] < radius))
        for j, v in zip(Is[i][beat], Ds[i][beat]):
            assert j in got and np.float32(got[j]) == v, f"query {i}: id {j}"
        if k >= lims[i + 1] - lims[i]:
            full += 1
            assert set(got) == set(Is[i][beat].tolist())
    assert full >= nq // 2


def test_edge_cases():
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(5)
    d, nlist, n = 37, 8, 300                                          # d % 4 != 0: scalar loads
    x = np.rint(_clustered(rng, n, d) * 10).clip(0, 255).astype(np.float32)
    cent = x[:nlist].copy()
    # untrained, empty, nq = 0
    un = fc.IndexIVFFlat(fc.IndexFlatL2(d), d, nlist)
    for index in (un, _pair(cent, x[:0], np.zeros(0, np.int64), False)[0]):
        lims, D, I = index.range_search(x[:3], 1e30)
        assert lims.dtype == np.uint64 and lims.shape == (4,) and (lims == 0).all()
        assert D.shape == I.shape == (0,) and D.dtype == np.float32 and I.dtype == np.int64
    lists = np.array([0, 2, 5])[rng.integers(0, 3, n)]               # the other lists stay empty
    ix, ref = _pair(cent, x, lists, False)
    lims, D, I = ix.range_search(x[:0], 1e30)
    assert lims.shape == (1,) and lims[0] == 0 and D.size == 0
    with pytest.raises(AssertionError):
        ix.range_search(np.zeros((2, d + 1), np.float32), 1.0)
    # radius +-1e30: every vector of the probed lists in probe order, or nothing
    for nprobe in (2, nlist):
        ix.nprobe = nprobe
        q = x[:20]
        pr = _probes(ix, q)
        lims, D, I = ix.range_search(q, 1e30)
        for i in range(q.shape[0]):
            want = np.concatenate([ix.get_list_ids(l) for l in pr[i]])
            np.testing.assert_array_equal(I[int(lims[i]):int(lims[i + 1])], want)
        lims, D, I = ix.range_search(q, -1e30)
        assert (lims == 0).all() and I.size == 0
    # a radius equal to an exactly occurring score excludes that vector (strict test); integer data: exact scores
    ix.nprobe = nlist
    s = scores64(x[:1], x, False)[0]
    j = int(np.argsort(s)[10])
    lims, D, I = ix.range_search(x[:1], float(s[j]))
    assert j not in set(I.tolist()) and (D < s[j]).all()
    lims, D, I = ix.range_search(x[:1], float(s[j]) + 0.5)
    assert j in set(I.tolist())
    # uint8 queries equal their float32 values; CUDA in -> CUDA out
    ix.nprobe = 3
    radius = float(np.quantile(scores64(x[:40], x, False), 0.2))
    lf, Df, If = ix.range_search(x[:40], radius)
    lu, Du, Iu = ix.range_search(x[:40].astype(np.uint8), radius)
    assert np.array_equal(lu, lf) and np.array_equal(Iu, If) and np.array_equal(Du, Df)
    lt, Dt, It = ix.range_search(torch.from_numpy(x[:40]).cuda(), radius)
    assert lt.is_cuda and Dt.is_cuda and It.is_cuda
    assert lt.dtype == torch.int64 and Dt.dtype == torch.float32 and It.dtype == torch.int64
    assert np.array_equal(lt.cpu().numpy(), lf.astype(np.int64)) and np.array_equal(It.cpu().numpy(), If)
    assert np.array_equal(Dt.cpu().numpy(), Df)
    lr, Dr, Ir = oracle_range_search(ref, x[:40], radius, probes=_probes(ix, x[:40]))
    assert np.array_equal(lf, lr) and np.array_equal(If, Ir) and np.array_equal(Df, Dr)
    # pickle round trip
    ix2 = pickle.loads(pickle.dumps(ix))
    l2, D2, I2 = ix2.range_search(x[:40], radius)
    assert np.array_equal(l2, lf) and np.array_equal(I2, If) and np.array_equal(D2, Df)
    # rows added after a search are merged in first
    extra = np.rint(_clustered(rng, 50, d) * 10).clip(0, 255).astype(np.float32)
    xl = np.array([1, 2, 7])[rng.integers(0, 3, 50)]
    ix.add_preassigned(extra, xl)
    ref.add_preassigned(extra, xl)
    la, Da, Ia = ix.range_search(x[:40], radius)
    lr, Dr, Ir = oracle_range_search(ref, x[:40], radius, probes=_probes(ix, x[:40]))
    assert np.array_equal(la, lr) and np.array_equal(Ia, Ir) and np.array_equal(Da, Dr)
    assert ix.ntotal == n + 50
    # reset
    ix.reset()
    lims, D, I = ix.range_search(x[:5], 1e30)
    assert (lims == 0).all() and I.size == 0


@pytest.mark.parametrize("metric_ip", [False, True])
def test_exact_duplicates_across_lists_in_probe_order(metric_ip):
    rng = np.random.default_rng(21)
    d, nlist, n = 32, 4, 400
    x = unit_rows(rng, n, d)
    v = x[7].copy()
    for i in (90, 200, 301):
        x[i] = v
    lists = rng.integers(0, nlist, n)
    lists[[7, 200]] = 1
    lists[[90, 301]] = [2, 3]
    cent = unit_rows(rng, nlist, d)
    ix, ref = _pair(cent, x, lists, metric_ip)
    ix.nprobe = nlist
    q = np.stack([v, v])
    s_dup = scores64(v[None], v[None], metric_ip)[0, 0]
    radius = s_dup - 1e-3 if metric_ip else 1e-3                      # only the copies (unit rows, random others)
    lims, D, I = ix.range_search(q, radius)
    pr = _probes(ix, q)
    rank = {int(l): r for r, l in enumerate(pr[0])}
    want = sorted((7, 90, 200, 301), key=lambda i: (rank[int(lists[i])], i))
    for r in range(2):
        assert list(I[int(lims[r]):int(lims[r + 1])]) == want
        assert (D[int(lims[r]):int(lims[r + 1])] == D[int(lims[r])]).all()
    lr, Dr, Ir = oracle_range_search(ref, q, radius, probes=pr)
    assert np.array_equal(lims, lr) and np.array_equal(I, Ir)


def test_skewed_list_keeps_order_across_chunks():
    """One list holds ~90 % of 40 k rows and is split into chunks; integer rows make the comparison exact."""
    rng = np.random.default_rng(8)
    d, nlist, n = 64, 16, 40000
    x = sift_like(rng, n, d)
    lists = np.where(rng.random(n) < 0.9, 3, rng.integers(0, nlist, n))
    cent = x[rng.choice(n, nlist, replace=False)]
    cent[3] = x[lists == 3][5]
    ix, ref = _pair(cent, x, lists, False)
    for nq, nprobe in ((1, 1), (1, 4), (200, 2)):
        q = sift_like(rng, nq, d)
        q[0] = x[lists == 3][5]
        ix.nprobe = nprobe
        pr = _probes(ix, q)
        radius = float(np.quantile(scores64(q, x, False), 0.3))     # thousands of hits in the long list
        lims, D, I = ix.range_search(q, radius)
        lr, Dr, Ir = oracle_range_search(ref, q, radius, probes=pr)
        assert int(lims[1]) > 5000
        assert np.array_equal(lims, lr) and np.array_equal(I, Ir) and np.array_equal(D, Dr)
        _assert_order(ix, ref, q, lims, I)


def test_workspace_bound_and_every_slot_written():
    from image_search_engine_b200 import _lib, ops
    nq, ntotal, d, nlist, nprobe = 4096, 1_000_000, 32, 1024, 16
    g = torch.Generator(device="cuda").manual_seed(4)
    xd = torch.randn((ntotal, d), generator=g, device="cuda")
    ix, _ = _pair(xd[:nlist].cpu().numpy(), np.zeros((0, d), np.float32), np.zeros(0, np.int64), False)
    ix.add(xd)
    ix.nprobe = nprobe
    q = xd[:nq] + 0.1
    radius = 40.0                                                     # tens to hundreds of hits per query
    ix.range_search(q[:20], radius)                                   # builds the list-sorted storage
    xs, ids, off = ix._lists()
    _, probes = ix.quantizer._search_device(q, nprobe, need_distances=False)
    max_len = int(ix._sizes.max())
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    lims, D, I = ops.ivfflat_range_search(q, xs, ids, off, max_len, probes, ix.metric_type, radius)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    ws = ops.ivfflat_range_workspace_bytes(nq, nprobe, nlist, max_len)
    total = int(lims[-1])
    assert total > nq and ops.last_search_stats["mode"] == "ivf-range" and ops.last_search_stats["results"] == total
    assert rise <= ws + 8 * (nq + 1) + 12 * total + (4 << 20), (rise, ws)
    S = min(-(-max_len // 64), max(1, 256 // nprobe), max(1, (1 << 22) // (nq * nprobe)))
    assert ws <= 16 * (nq * nprobe * S + 1) + 16 * nq * nprobe + 24 * (nlist + 1) + (64 << 20)
    # the C ABI with sentinel-filled outputs and slack past the total: every slot below lims[nq] is written, none past
    lib, ctx = _lib.load(), _lib.ctx(torch.cuda.current_device())
    wsb = torch.empty((ws,), dtype=torch.uint8, device="cuda")
    lims2 = torch.empty((nq + 1,), dtype=torch.int64, device="cuda")
    args = (ctx, ops._ptr(q), nq, d, ops._ptr(xs), ops._ptr(ids), ops._ptr(off), nlist, max_len)
    _lib.check(lib.ise_ivfflat_range_count(*args, ops._ptr(probes), nprobe, ix.metric_type, radius, ops._ptr(lims2),
                                           ops._ptr(wsb), ws, ops._stream()))
    assert torch.equal(lims2, lims)
    D2 = torch.full((total + 1000,), float("nan"), device="cuda")
    I2 = torch.full((total + 1000,), -7, dtype=torch.int64, device="cuda")
    _lib.check(lib.ise_ivfflat_range_fill(*args, nprobe, ix.metric_type, radius, ops._ptr(D2), ops._ptr(I2),
                                          ops._ptr(wsb), ws, ops._stream()))
    assert not torch.isnan(D2[:total]).any() and (I2[:total] >= 0).all()
    assert torch.isnan(D2[total:]).all() and (I2[total:] == -7).all()
    assert torch.equal(D2[:total], D) and torch.equal(I2[:total], I)


def test_benchmark_size_fp64_check():
    rng = np.random.default_rng(12)
    ntotal, d, nlist, nprobe, nq = 1_000_000, 512, 4096, 32, 10_000
    g = torch.Generator(device="cuda").manual_seed(12)
    centers = torch.randn((4096, d), generator=g, device="cuda")
    xd = centers[torch.randint(0, 4096, (ntotal,), generator=g, device="cuda")] + \
        0.5 * torch.randn((ntotal, d), generator=g, device="cuda")
    xd /= xd.norm(dim=1, keepdim=True)
    cent = xd[torch.randint(0, ntotal, (nlist,), generator=g, device="cuda")].cpu().numpy()
    ix, _ = _pair(cent, np.zeros((0, d), np.float32), np.zeros(0, np.int64), True)
    ix.add(xd)
    ix.nprobe = nprobe
    q = xd[torch.randint(0, ntotal, (nq,), generator=g, device="cuda")] + \
        0.05 * torch.randn((nq, d), generator=g, device="cuda")
    Ds, _ = ix.search(q[:200], 50)
    radius = float(torch.median(Ds[:, -1]).item())                   # about 50 results per query
    lims, D, I = ix.range_search(q, radius)
    lims, D, I = lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
    assert lims[-1] > 10 * nq
    rows = rng.choice(nq, 100, replace=False)
    qs = q[rows].cpu().numpy()
    probes = ix.quantizer._search_device(q[rows].contiguous(), nprobe, need_distances=False)[1].cpu().numpy()
    lists = {}
    for r, i in enumerate(rows):
        cand = np.concatenate([lists.setdefault(l, ix.get_list_ids(l)) for l in probes[r]])
        y = xd[torch.from_numpy(cand).cuda()].cpu().numpy().astype(np.float64)
        s = y @ qs[r].astype(np.float64)
        tau = 16 * EPS32 * np.linalg.norm(qs[r].astype(np.float64))
        got = I[lims[i]:lims[i + 1]]
        sure = cand[s - radius > tau]
        assert np.isin(sure, got).all()
        pos = {int(c): j for j, c in enumerate(cand)}                # probe order, then list order
        order = np.array([pos[int(v)] for v in got])
        assert (np.diff(order) > 0).all()
        s_got = s[order]
        assert (s_got - radius >= -tau).all()
        np.testing.assert_allclose(D[lims[i]:lims[i + 1]], s_got, rtol=1e-4, atol=1e-6)
