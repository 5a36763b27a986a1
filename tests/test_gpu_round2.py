"""GPU tests of the round-2 boundary work: O(nnz) Okapi on CSR input, the opt-in corrected tf-idf mode, k beyond
the fused-selection limit, thread safety of the cached host pipelines, and the sharded index's equality with the flat
index and its empty shard handling.  All through the public Python surface, i.e. through the C ABI."""
import threading
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from tests._util import assert_topk_parity, sift_like, unit_rows

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).parent / "golden"


def _okapi_ref(H, k1=1.0, k2=1.0, b=0.75):
    """utils.py:180-200 restated on a dense float64 matrix (zeros stay zero)."""
    H = np.asarray(H, dtype=np.float64)
    dl = H.sum(axis=1, keepdims=True)
    t = H * k1
    with np.errstate(invalid="ignore", divide="ignore"):
        out = t / (t + k2 * (1 - b + b * (dl / dl.mean())))
    return np.where(H != 0, out, 0.0)


def test_okapi_sparse_in_sparse_out():
    from image_search_engine_b200 import OkapiTransformer
    rng = np.random.default_rng(7)
    H = np.zeros((300, 1000))
    for i in range(300):
        w = rng.integers(0, 1000, rng.integers(1, 120))
        np.add.at(H[i], w, 1.0)
    H[17] = 0                                            # an empty document
    want = _okapi_ref(H)
    X = sp.csr_matrix(H)
    T = OkapiTransformer().transform(X)                  # copy=True: the input is left alone
    assert sp.issparse(T) and T.format == "csr" and T.dtype == np.float64
    assert np.array_equal(X.toarray(), H)
    assert np.array_equal(T.indices, X.indices) and np.array_equal(T.indptr, X.indptr)
    np.testing.assert_allclose(T.toarray(), want, rtol=1e-15, atol=0)
    T2 = OkapiTransformer().transform(X, copy=False)     # in place on the caller's matrix, like the reference
    assert T2 is X
    np.testing.assert_allclose(X.toarray(), want, rtol=1e-15, atol=0)
    # other parameters, CSC input, a single row (dl / avgdl == 1)
    T3 = OkapiTransformer(k1=1.5, k2=0.5, b=0.3).transform(sp.csc_matrix(H))
    np.testing.assert_allclose(T3.toarray(), _okapi_ref(H, 1.5, 0.5, 0.3), rtol=1e-15, atol=0)
    T4 = OkapiTransformer().transform(sp.csr_matrix(H[:1]))
    np.testing.assert_allclose(T4.toarray(), H[:1] / (H[:1] + 1.0), rtol=1e-15, atol=0)
    empty = OkapiTransformer().transform(sp.csr_matrix((5, 8)))
    assert empty.shape == (5, 8) and empty.nnz == 0


def test_okapi_opt_in_idf_and_norm_known_answer():
    """compat=False: tf weights x fitted idf, then row normalisation -- checked against the closed form on a tiny
    hand-made matrix and against the dense device path (GPU-resident index build)."""
    from image_search_engine_b200 import OkapiTransformer, ops
    H = np.array([[2, 0, 1, 0],
                  [0, 3, 1, 0],
                  [1, 1, 0, 0],
                  [0, 0, 4, 0],
                  [1, 0, 0, 5]], dtype=np.float64)
    n = H.shape[0]
    df = (H != 0).sum(0)
    idf = np.log((n - df + 0.5) / (df + 0.5))
    tf = _okapi_ref(H)
    for norm in ("l2", "l1", None):
        ok = OkapiTransformer(compat=False, norm=norm).fit(H)
        np.testing.assert_allclose(ok.idf_, idf, rtol=1e-15)
        want = tf * idf[None, :]
        if norm == "l2":
            want = want / np.sqrt((want ** 2).sum(1, keepdims=True))
        elif norm == "l1":
            want = want / np.abs(want).sum(1, keepdims=True)
        got = ok.transform(H)
        assert sp.issparse(got)
        np.testing.assert_allclose(got.toarray(), want, rtol=1e-14, atol=1e-300)
        dev = ops.require_cuda()
        Hd = torch.from_numpy(H).to(dev)
        got_d = ok.transform(Hd)
        assert got_d.is_cuda and torch.equal(Hd, torch.from_numpy(H).to(dev))     # copy=True
        np.testing.assert_allclose(got_d.cpu().numpy(), want, rtol=1e-14, atol=1e-300)
        got_f = ok.transform(Hd.to(torch.float32)).cpu().numpy()
        np.testing.assert_allclose(got_f, want, rtol=2e-6, atol=1e-30)
    # use_idf=False keeps only the normalisation; the default (compat) ignores both, like the reference
    ok = OkapiTransformer(compat=False, use_idf=False).fit(H)
    np.testing.assert_allclose(ok.transform(H).toarray(), tf / np.sqrt((tf ** 2).sum(1, keepdims=True)), rtol=1e-14)
    np.testing.assert_allclose(OkapiTransformer().fit(H).transform(H).toarray(), tf, rtol=1e-15)


@pytest.mark.parametrize("metric_ip", [True, False])
def test_search_with_k_beyond_the_fused_limit(metric_ip):
    """Faiss's IndexFlat.search takes any k; k > 128 goes through exact pair scores + masked selection passes."""
    from image_search_engine_b200 import faiss_compat
    from oracle import faiss_shim as fs
    rng = np.random.default_rng(11)
    db = unit_rows(rng, 3000, 48)
    db[100] = db[5]                                      # exact tie: lower id first
    q = db[rng.integers(0, 3000, 30)] + 0.05 * rng.standard_normal((30, 48)).astype(np.float32)
    q[0] = db[5]
    idx = faiss_compat.IndexFlatIP(48) if metric_ip else faiss_compat.IndexFlatL2(48)
    idx.add(db)
    for k in (129, 300):
        D, I = idx.search(q, k)
        assert D.shape == (30, k) and I.dtype == np.int64
        Dr, Ir = fs.knn(q, db, k, fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
        assert_topk_parity(I, Ir, q, db, metric_ip, max_mismatch_frac=0.5)
        np.testing.assert_allclose(D, Dr, rtol=1e-4, atol=1e-5)
        assert list(I[0, :2]) == [5, 100]
        assert all(len(set(row)) == k for row in I)      # no id returned twice across the passes
    D, I = idx.search(q[:3], 3500)                       # k > ntotal > 128: padded like Faiss
    assert (I[:, 3000:] == -1).all() and (I[:, :3000] >= 0).all()
    assert sorted(I[0, :3000]) == list(range(3000))
    pad = -np.finfo(np.float32).max if metric_ip else np.finfo(np.float32).max
    assert (D[:, 3000:] == pad).all()


def test_concurrent_pipelined_transforms_share_one_bovw():
    """Two threads calling transform_csr / histograms_host on ONE BOVW (threaded Flask server, joblib threads):
    the cached staging buffers are guarded, so every call returns its own correct matrix."""
    from image_search_engine_b200 import BOVW, FaissKMeans, OkapiTransformer, faiss_compat
    from image_search_engine_b200.bag_of_visual_words import pack_descriptions
    rng = np.random.default_rng(5)
    k, d = 256, 64
    cent = unit_rows(rng, k, d)
    gi = faiss_compat.IndexFlatIP(d)
    gi.add(cent)
    bovw = BOVW(None, n_clusters=k)
    bovw.clusterer = FaissKMeans(k, index=gi)
    batches = []
    for s in range(2):
        descs = [sift_like(rng, int(rng.integers(30, 90)), d) for _ in range(200)]
        batches.append(pack_descriptions(descs, pin=True))
    ok = OkapiTransformer()
    want = [bovw.transform_csr(b, okapi=ok, n_chunks=4).toarray() for b in batches]
    got, errs = {}, []

    def work(t):
        try:
            for it in range(6):
                m = bovw.transform_csr(batches[t], okapi=ok, n_chunks=4, copy=True).toarray()
                out = torch.empty((200, k), dtype=torch.float64, pin_memory=True)
                h = bovw.histograms_host(batches[t], out, okapi=ok, n_chunks=4).copy()
                got[(t, it)] = (m, h)
        except Exception as e:  # pragma: no cover
            errs.append(e)

    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs
    for (t, it), (m, h) in got.items():
        assert np.array_equal(m, want[t]) and np.array_equal(h, want[t]), (t, it)


def test_sharded_index_small_batches_and_empty_shard():
    """world = 1 (no process group): the sharded index runs the unsharded index's dispatch (ops.flat_search /
    ops.flat_range_search) -- the exact kernel below 20 queries, the fused top-1 or the tensor-core path above -- so
    both return the same bits; a shard without rows answers with padded lists instead of raising; k beyond the fused
    limit is refused before any work."""
    from image_search_engine_b200 import faiss_compat
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2, IseError
    from image_search_engine_b200.parallel import ShardedIndexFlat
    rng = np.random.default_rng(3)
    db = rng.standard_normal((5000, 40)).astype(np.float32)
    qf = db[:40] + 1e-4 * rng.standard_normal((40, 40)).astype(np.float32)
    qu = rng.integers(0, 256, (40, 40), dtype=np.uint8)
    for metric in (METRIC_IP, METRIC_L2):
        six = ShardedIndexFlat(40, metric)
        six.add_local(db)
        flat = faiss_compat.IndexFlatIP(40) if metric == METRIC_IP else faiss_compat.IndexFlatL2(40)
        flat.add(db)
        for q in (qf, qu):
            for nq in (7, 40):
                for k in (1, 5, 10, 100):
                    D, I = six.search(q[:nq], k)
                    Dr, Ir = flat.search(q[:nq], k)
                    assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr), \
                        (metric, q.dtype, nq, k)                                                # same kernels, same bits
                radius = float(np.median(Dr[:, 50]))
                got = six.range_search(q[:nq], radius)
                want = flat.range_search(q[:nq], radius)
                assert want[0][-1] > 0, (metric, q.dtype, nq)
                for a, b in zip(got, want):
                    a = a.cpu().numpy()
                    assert np.array_equal(a, b.astype(a.dtype)), (metric, q.dtype, nq)
        with pytest.raises(IseError, match=r"topk must be in \[1, 128\]"):
            six.search(qf, 200)
    empty = ShardedIndexFlat(40, METRIC_L2)
    empty.add_local(np.zeros((0, 40), np.float32))
    D, I = empty.search(qf[:7], 5)
    assert (I.cpu().numpy() == -1).all() and (D.cpu().numpy() == np.finfo(np.float32).max).all()


@pytest.mark.parametrize("metric_ip", [True, False])
def test_flat_search_id_base_shifts_only_the_ids(metric_ip):
    """ops.flat_search with id_base = 1000 (a shard's global ids) returns the id_base = 0 ids plus 1000 and the same
    distances, on the direct-formula, tensor-core and fused top-1 paths."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(8)
    metric = METRIC_IP if metric_ip else METRIC_L2
    dev = ops.require_cuda()
    db = torch.from_numpy(rng.standard_normal((1000, 64)).astype(np.float32)).to(dev)
    q = torch.from_numpy(rng.standard_normal((120_000, 64)).astype(np.float32)).to(dev)
    op = ops.attach_sample(ops.prepare_operand(db))
    for nq, k in ((7, 10), (40, 1), (40, 10), (120_000, 1)):
        D0, I0 = ops.flat_search(q[:nq], db, metric, k, operand=lambda: op)
        mode = ops.search_stats()["mode"]
        D1, I1 = ops.flat_search(q[:nq], db, metric, k, operand=lambda: op, id_base=1000)
        assert ops.search_stats()["mode"] == mode
        assert torch.equal(I1, I0 + 1000) and torch.equal(D1, D0), (nq, k)
    assert mode.startswith("fused"), mode


# ---------------------------------------------------------------------------------------------------------------
# single-pass row preparation (per-row power-of-two scales) and the atomics-free k-means update
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [128, 32, 100, 256, 512, 640, 30])
def test_prepare_rows_single_pass(d):
    """Row operands: every row is scaled by its own power of two; hi + lo reconstruct the row to ~22 bits, norms are the
    exact FP32 sums, pad columns are zero, NaN / Inf are reported.  d = 640 (> 512) and d = 30 (not a multiple of 4)
    fall back to the two-pass kernels and must satisfy the same contract."""
    from image_search_engine_b200 import ops
    dev = ops.require_cuda()
    rng = np.random.default_rng(d)
    x = (rng.standard_normal((3001, d)) * np.exp2(rng.integers(-12, 12, (3001, 1)))).astype(np.float32)
    x[5] = 0                                              # an all-zero row keeps scale 1
    op = ops.prepare_operand(torch.from_numpy(x).to(dev), rows=True)
    assert op.row_inv is not None and op.lo is not None
    inv = op.row_inv.cpu().numpy()
    assert (inv == np.exp2(np.round(np.log2(inv)))).all()                  # powers of two
    scaled_max = np.abs(x).max(1) / inv
    single_pass = d % 4 == 0 and d <= 512
    if single_pass:
        nz = np.abs(x).max(1) > 0
        assert ((scaled_max[nz] >= 8192) & (scaled_max[nz] < 16384)).all() and inv[5] == 1.0
        assert float(op.meta[0]) == 1.0 and float(op.meta[1]) == 1.0
    rec = (op.hi.float() + op.lo.float()).cpu().numpy()[:, :d] * inv[:, None]
    # ~22 bits relative to the magnitude the scale was chosen for: the row's own maximum (single pass) or the tensor's
    ref_mag = np.abs(x).max(1, keepdims=True) if single_pass else np.abs(x).max()
    assert (np.abs(rec - x) <= ref_mag * 2.0 ** -21 + 1e-30).all()
    assert (op.hi.cpu().numpy()[:, d:] == 0).all()
    np.testing.assert_allclose(op.norms.cpu().numpy(), (x.astype(np.float64) ** 2).sum(1), rtol=2e-6)
    assert float(op.meta[2]) != 0.0 and float(op.meta[7]) == 0.0
    np.testing.assert_allclose(float(op.meta[4]), (x.astype(np.float64) ** 2).sum(1).max(), rtol=2e-6)
    for bad in (np.nan, np.inf, -np.inf):
        y = x.copy()
        y[1234, d // 2] = bad
        assert float(ops.prepare_operand(torch.from_numpy(y).to(dev), rows=True).meta[7]) != 0.0
        assert ops.has_nonfinite(torch.from_numpy(y).to(dev)) and not ops.has_nonfinite(torch.from_numpy(x).to(dev))


def test_prepare_rows_exact_rows_skip_their_lo_store():
    """Integer-valued rows are exact in one plane: no lo store at all when every row is (LO_NONZERO stays 0); when
    only SOME rows are, the skipped rows' lo parts are zeroed by the fix-up so the plane can be read as a whole."""
    from image_search_engine_b200 import ops
    dev = ops.require_cuda()
    rng = np.random.default_rng(77)
    s = sift_like(rng, 20000, 128)
    for _ in range(2):
        poison = torch.full((20000, 128), float("nan"), dtype=torch.float16, device=dev)
        del poison
        op = ops.prepare_operand(torch.from_numpy(s).to(dev), rows=True)
    assert float(op.meta[2]) == 0.0
    inv = op.row_inv.cpu().numpy()
    assert np.array_equal(op.hi.float().cpu().numpy() * inv[:, None], s)
    assert ops.compact_operand(op).lo is None
    mixed = s.copy()
    mixed[::7] += rng.standard_normal((len(mixed[::7]), 128)).astype(np.float32) * 0.37
    for _ in range(2):
        poison = torch.full((20000, 128), float("nan"), dtype=torch.float16, device=dev)
        del poison
        om = ops.prepare_operand(torch.from_numpy(mixed).to(dev), rows=True)
    assert 0.0 < float(om.meta[2]) < 2.0 ** -22          # inexact rows exist; the value is their largest relative residual^2
    lo = om.lo.float().cpu().numpy()
    assert not np.isnan(lo).any()
    exact_rows = np.ones(20000, bool)
    exact_rows[::7] = False
    assert (lo[exact_rows] == 0).all() and (np.abs(lo[~exact_rows]).max(1) > 0).all()
    rec = (om.hi.float().cpu().numpy() + lo) * om.row_inv.cpu().numpy()[:, None]
    assert (np.abs(rec - mixed) <= np.abs(mixed).max(1, keepdims=True) * 2.0 ** -21).all()


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("m,n,d,k,kind", [(3000, 4096, 128, 1, "sift"), (2000, 700, 64, 1, "scaled"), (500, 30000, 96, 10, "scaled"),
                                           (300, 70000, 128, 40, "unit"), (150, 5000, 512, 100, "scaled")])
def test_row_scaled_operands_through_the_search_paths(metric_ip, m, n, d, k, kind):
    """gemm_select / gemm_collect / rescore_select with per-row scales on the A side: rows of wildly different magnitude
    (2^-10 .. 2^10) must come out with the oracle's ids and real-unit distances."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    from oracle import faiss_shim as fs
    dev = ops.require_cuda()
    rng = np.random.default_rng(m + n + d + k)
    db = unit_rows(rng, n, d)
    if kind == "sift":
        q = sift_like(rng, m, d)
    else:
        q = db[rng.integers(0, n, m)] + 0.05 * rng.standard_normal((m, d)).astype(np.float32)
        if kind == "scaled":
            q = (q * np.exp2(rng.integers(-10, 10, (m, 1)))).astype(np.float32)
    qd, dbd = torch.from_numpy(q).to(dev), torch.from_numpy(db).to(dev)
    a = ops.prepare_operand(qd, rows=True)
    b = ops.attach_sample(ops.prepare_operand(dbd))
    metric = METRIC_IP if metric_ip else METRIC_L2
    Dr, Ir = fs.knn(q, db, k, fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    for precision in ("verified", "split"):
        D, I = ops.search_topk(qd, a, dbd, b, metric, k, precision=precision)
        assert_topk_parity(I.cpu().numpy(), Ir, q, db, metric_ip, max_mismatch_frac=0.05 if kind != "scaled" else 0.6)
        scale_tol = 1e-4 * np.abs(Dr).max(1, keepdims=True) + 1e-6
        assert (np.abs(D.cpu().numpy() - Dr) <= 1e-4 * np.abs(Dr) + scale_tol).all(), precision
    # raw kernel output (no exact re-score): the accumulator is rescaled by the row's own factor
    val, idx = ops.gemm_select(a, b, metric, min(k, 32))
    kk = min(k, 32)
    tol = 2e-3 * (np.abs(Dr[:, :kk]) + (np.linalg.norm(q, axis=1, keepdims=True) ** 2 if not metric_ip else 0)) + 1e-6
    assert (np.abs(val.cpu().numpy() - Dr[:, :kk]) <= tol).all()


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("n,d,k,kind", [(50000, 128, 4096, "sift"), (30000, 32, 512, "orb"), (20000, 64, 300, "float"),
                                          (9000, 256, 1000, "float"), (6000, 100, 64, "float"), (40000, 128, 20000, "sift"),
                                          (3000, 8, 16, "float"), (5000, 2048, 40, "float"), (700, 30, 9, "float")])
def test_sorted_gather_accumulate_equals_oracle(metric_ip, n, d, k, kind):
    """Counting sort + chunked gather-reduce vs a float64 scatter-add: counts exact, sums / objective within FP32
    reassociation.  k = 20000 takes the global-atomic histogram (no shared-memory bins); d = 30 (rows not 4-column
    aligned) falls back to the atomic kernel; two calls into the same buffers add up (shards / ranks)."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    dev = ops.require_cuda()
    rng = np.random.default_rng(n + d + k)
    x = orb_like_(rng, n, d) if kind == "orb" else sift_like(rng, n, d) if kind == "sift" else \
        rng.standard_normal((n, d)).astype(np.float32)
    assign = rng.integers(0, max(1, k - 3), n).astype(np.int64)      # last 3 clusters stay empty
    assign[: n // 10] = assign[0]                                     # one big cluster: long runs, many chunks
    cent = unit_rows(rng, k, d)
    xf = x.astype(np.float32)
    sums_ref = np.zeros((k, d), np.float64)
    np.add.at(sums_ref, assign, xf.astype(np.float64))
    counts_ref = np.bincount(assign, minlength=k).astype(np.float32)
    c64 = cent.astype(np.float64)[assign]
    obj_ref = float((xf * c64).sum()) if metric_ip else float(((xf - c64) ** 2).sum())
    xd, ad, cd = torch.from_numpy(x).to(dev), torch.from_numpy(assign).to(dev), torch.from_numpy(cent).to(dev)
    accum = torch.zeros(k * d + k, device=dev)
    sums, counts = accum[:k * d].view(k, d), accum[k * d:]
    obj = torch.zeros(1, dtype=torch.float64, device=dev)
    metric = METRIC_IP if metric_ip else METRIC_L2
    ws = ops.kmeans_accumulate_sorted(xd, ad, sums, counts, obj, centroids=cd, metric=metric)
    assert np.array_equal(counts.cpu().numpy(), counts_ref)
    np.testing.assert_allclose(sums.cpu().numpy(), sums_ref, rtol=2e-5, atol=2e-5 * np.abs(sums_ref).max())
    assert abs(float(obj.item()) - obj_ref) <= 1e-5 * abs(obj_ref) + 1e-3
    if x.dtype == np.float32:                                          # same sums from the FP16 hi plane when it is exact
        a_op = ops.compact_operand(ops.prepare_operand(xd, rows=True))
        accum.zero_()
        obj.zero_()
        ws = ops.kmeans_accumulate_sorted(xd, ad, sums, counts, obj, centroids=cd, metric=metric, workspace=ws, exact_op=a_op)
        assert (a_op.lo is None) == (kind == "sift")
        assert np.array_equal(counts.cpu().numpy(), counts_ref)
        np.testing.assert_allclose(sums.cpu().numpy(), sums_ref, rtol=2e-5, atol=2e-5 * np.abs(sums_ref).max())
        assert abs(float(obj.item()) - obj_ref) <= 1e-5 * abs(obj_ref) + 1e-3
    half = n // 2                                                      # second call: buffers accumulate, workspace reused
    accum.zero_()
    obj.zero_()
    ws = ops.kmeans_accumulate_sorted(xd[:half], ad[:half], sums, counts, obj, centroids=cd, metric=metric, workspace=ws)
    ops.kmeans_accumulate_sorted(xd[half:], ad[half:], sums, counts, obj, centroids=cd, metric=metric, workspace=ws)
    assert np.array_equal(counts.cpu().numpy(), counts_ref)
    np.testing.assert_allclose(sums.cpu().numpy(), sums_ref, rtol=2e-5, atol=2e-5 * np.abs(sums_ref).max())
    assert abs(float(obj.item()) - obj_ref) <= 1e-5 * abs(obj_ref) + 1e-3


def orb_like_(rng, n, d):
    return rng.integers(0, 256, size=(n, d), dtype=np.uint8)


def test_kmeans_train_rejects_nonfinite_and_warms_the_split_stream():
    from image_search_engine_b200 import FaissKMeans
    rng = np.random.default_rng(9)
    x = sift_like(rng, 6000, 32)
    FaissKMeans(16, n_init=1, max_iter=2).fit(x)
    y = x.copy()
    y[4321, 7] = np.nan
    with pytest.raises(RuntimeError, match="NaN"):
        FaissKMeans(16, n_init=1, max_iter=2).fit(y)
    big = np.tile(x, (2, 1))                                       # 12000 rows > 256 * 16: the sub-sampled path validates ALL rows
    big[11999, 0] = np.inf
    with pytest.raises(RuntimeError, match="NaN"):
        FaissKMeans(16, n_init=1, max_iter=2).fit(big)


def test_transform_csr_from_a_python_list_of_arrays():
    """The reference's input contract is a list with one (n_i, d) array per image: it is packed by the C list walker +
    ise_pack_rows into a persistent pinned buffer -- uint8 on the wire when every value is an integer in [0, 255] --
    and must give exactly the matrix of the pre-packed path, for ragged lists with empty images too."""
    from image_search_engine_b200 import BOVW, FaissKMeans, OkapiTransformer, faiss_compat
    from image_search_engine_b200.bag_of_visual_words import _pack_list_into, pack_descriptions
    rng = np.random.default_rng(15)
    k, d = 512, 128
    gi = faiss_compat.IndexFlatIP(d)
    gi.add(unit_rows(rng, k, d))
    bovw = BOVW(None, n_clusters=k)
    bovw.clusterer = FaissKMeans(k, index=gi)
    ok = OkapiTransformer()
    sizes = rng.integers(0, 160, 300)
    sizes[7] = 0
    ints = [sift_like(rng, int(s), d) for s in sizes]                       # integer-valued float32 -> uint8 on the wire
    general = [a + np.float32(0.25) for a in ints]                          # not integers -> float32 on the wire
    bytes_ = [a.astype(np.uint8) for a in ints]                             # ORB-style uint8 input
    for descs, wire in ((ints, torch.uint8), (general, torch.float32), (bytes_, torch.uint8)):
        bufs = {}
        packed = _pack_list_into(descs, bufs)
        assert packed is not None and packed.matrix.dtype == wire and packed.matrix.is_pinned()
        mat, off = pack_descriptions(descs)
        assert np.array_equal(packed.offsets, off)
        assert np.array_equal(packed.matrix.numpy().astype(np.float32), np.asarray(mat, dtype=np.float32))
        packed2 = _pack_list_into(descs, bufs)                              # the pinned buffer is reused
        assert packed2.matrix.data_ptr() == packed.matrix.data_ptr()
        want = bovw.transform_csr(pack_descriptions(descs, pin=True), okapi=ok, n_chunks=4).toarray()
        got = bovw.transform_csr(descs, okapi=ok, n_chunks=4).toarray()
        assert np.array_equal(got, want)
    assert np.array_equal(bovw.transform_csr(ints, okapi=ok, n_chunks=4).toarray(),
                          bovw.transform_csr(bytes_, okapi=ok, n_chunks=4).toarray())
    # only an image of the LAST chunk breaks the uint8 narrowing: the chunked packer starts over in float32 after the
    # first chunks were already sent as uint8
    late = [a.copy() for a in ints]
    late[-2][0, 3] += np.float32(0.5)
    want = bovw.transform_csr(pack_descriptions(late, pin=True), okapi=ok, n_chunks=4).toarray()
    assert np.array_equal(bovw.transform_csr(late, okapi=ok, n_chunks=4).toarray(), want)
    assert np.array_equal(bovw.transform_csr(ints, okapi=ok, n_chunks=4).toarray(),        # and uint8 again afterwards
                          bovw.transform_csr(bytes_, okapi=ok, n_chunks=4).toarray())
    # lists the packer does not understand (mixed dtypes, float64) take the generic path and still work
    mixed = [a.astype(np.float64) if i % 2 else a for i, a in enumerate(ints)]
    assert _pack_list_into(mixed, {}) is None
    assert np.array_equal(bovw.transform_csr(mixed, okapi=ok, n_chunks=4).toarray(),
                          bovw.transform_csr(ints, okapi=ok, n_chunks=4).toarray())


def test_pinned_float_matrix_is_narrowed_on_the_wire(monkeypatch):
    """A pinned float32 PackedDescriptions whose values are integers in [0, 255] crosses PCIe as uint8 (narrowed block by
    block on host threads inside transform_csr) and gives exactly the float32-wire result; a single non-integer value
    anywhere makes the call fall back to float32 on the wire."""
    from image_search_engine_b200 import BOVW, FaissKMeans, OkapiTransformer, faiss_compat
    from image_search_engine_b200.bag_of_visual_words import PackedDescriptions
    rng = np.random.default_rng(31)
    k, d, n_img = 512, 128, 700
    gi = faiss_compat.IndexFlatIP(d)
    gi.add(unit_rows(rng, k, d))
    bovw = BOVW(None, n_clusters=k)
    bovw.clusterer = FaissKMeans(k, index=gi)
    ok = OkapiTransformer()
    sizes = rng.integers(150, 260, n_img)
    offsets = np.zeros(n_img + 1, dtype=np.int64)
    np.cumsum(sizes, out=offsets[1:])
    x = sift_like(rng, int(offsets[-1]), d)
    packed = PackedDescriptions(torch.from_numpy(x.copy()), offsets).pin()
    monkeypatch.setenv("ISE_NARROW_PINNED", "0")
    want = bovw.transform_csr(packed, okapi=ok, n_chunks=4).toarray()
    assert bovw._last_transfer["wire"] == "float32"
    monkeypatch.setenv("ISE_NARROW_PINNED", "1")
    got = bovw.transform_csr(packed, okapi=ok, n_chunks=4).toarray()
    # two-ended: host threads narrow chunks from the front while idle PCIe time sends chunks from the back as float32
    assert bovw._last_transfer["wire"].startswith("uint8") and bovw._last_transfer["h2d_bytes"] < 0.9 * x.nbytes
    assert np.array_equal(got, want)
    # a non-integer value in the LAST block: the uint8 attempt is abandoned mid-way, float32 is sent instead
    y = x.copy()
    y[-3, 7] += 0.25
    packed_y = PackedDescriptions(torch.from_numpy(y), offsets).pin()
    got_y = bovw.transform_csr(packed_y, okapi=ok, n_chunks=4).toarray()
    assert "float32" in bovw._last_transfer["wire"]
    monkeypatch.setenv("ISE_NARROW_PINNED", "0")
    assert np.array_equal(got_y, bovw.transform_csr(packed_y, okapi=ok, n_chunks=4).toarray())


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("m,n,d,kind", [(200_000, 4096, 128, "sift"), (150_001, 1000, 64, "sift"), (120_000, 512, 32, "sift"),
                                         (160_000, 2048, 128, "float"), (130_000, 777, 128, "mixed")])
def test_fused_assign_equals_separate_preparation(metric_ip, m, n, d, kind):
    """ise_assign_fused (row preparation inside the contraction kernel) against ise_prepare_rows + ise_gemm_select: same
    ids and scores, and the row operand it leaves behind is the one the stand-alone preparation writes.  "float" rows are
    not exact in one FP16 plane: the device-side flag triggers the follow-up launches with the lo planes; "mixed" has
    both kinds of rows (skipped lo stores completed by the fix-up)."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    dev = ops.require_cuda()
    rng = np.random.default_rng(m + n + d)
    if kind == "sift":
        x = sift_like(rng, m, d)
    else:
        x = (rng.standard_normal((m, d)) * 3).astype(np.float32)
        if kind == "mixed":
            x[::3] = sift_like(rng, len(x[::3]), d)
    c = unit_rows(rng, n, d)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    b = ops.prepare_operand(cd)
    metric = METRIC_IP if metric_ip else METRIC_L2
    got = ops.assign_fused(xd, b, metric, verified=False)
    assert got is not None, "shape should be covered by the fused kernel"
    assert ops.last_search_stats["mode"] == "fused-split"
    val, idx, a_f = got
    a_s = ops.prepare_operand(xd, rows=True)
    val_s, idx_s = ops.gemm_select(a_s, b, metric, 1)
    assert torch.equal(idx, idx_s) and torch.equal(val, val_s)
    assert torch.equal(a_f.hi, a_s.hi) and torch.equal(a_f.norms, a_s.norms) and torch.equal(a_f.row_inv, a_s.row_inv)
    mf, ms = a_f.meta.cpu().numpy(), a_s.meta.cpu().numpy()
    assert mf[2] == ms[2] and (mf[2] == 0.0 if kind == "sift" else 0.0 < mf[2] < 2.0 ** -22)
    assert mf[0] == 1.0 and mf[4] == ms[4] and mf[7] == 0.0
    if kind != "sift":
        assert torch.equal(a_f.lo, a_s.lo)
    # against the oracle on a sample
    from oracle import faiss_shim as fs
    rows = rng.choice(m, 1500, replace=False)
    Dr, Ir = fs.knn(x[rows], c, 1, fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)
    assert_topk_parity(idx.cpu().numpy()[rows], Ir, x[rows], c, metric_ip, max_mismatch_frac=0.01)
    # the public path takes it: FaissKMeans.transform on raw float32 descriptors
    from image_search_engine_b200 import FaissKMeans, faiss_compat
    gi = faiss_compat.IndexFlatIP(d) if metric_ip else faiss_compat.IndexFlatL2(d)
    gi.add(cd)
    words = FaissKMeans(n, index=gi).transform_device(xd)
    assert ops.last_search_stats["mode"] in ("fused-split", "fused-verified") and torch.equal(words, idx.reshape(-1))


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("m,n,d,kind", [(200_000, 4096, 128, "sift"), (150_001, 3000, 64, "sift"), (120_000, 2048, 32, "sift"),
                                         (160_000, 2048, 128, "float"), (130_000, 1777, 128, "mixed"),
                                         (140_000, 2048, 128, "duplicates"), (100_000, 1500, 100, "sift"),
                                         (90_000, 1100, 96, "mixed")])
def test_verified_assign_equals_the_split_products(metric_ip, m, n, d, kind):
    """The verified pipeline (one product per tile with the row tile resident in shared memory, per-row proof, compact
    split-product re-run of the undecided rows, no host round trip) returns exactly the ids of the split products --
    through the fused entry point (raw float32 rows) and through ise_assign_verified (prepared planes); its scores are
    within the coarse bound; "duplicates": every column exists twice, so NO row can be decided and the overflow launch
    must repeat everything."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    dev = ops.require_cuda()
    rng = np.random.default_rng(m + n + d + 1)
    if kind in ("sift", "duplicates"):
        x = sift_like(rng, m, d)
    else:
        x = (rng.standard_normal((m, d)) * 3).astype(np.float32)
        if kind == "mixed":
            x[::3] = sift_like(rng, len(x[::3]), d)
    c = unit_rows(rng, n, d)
    if kind == "duplicates":
        c[n // 2:] = c[:n // 2]
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    b = ops.prepare_operand(cd)
    metric = METRIC_IP if metric_ip else METRIC_L2
    a_s = ops.prepare_operand(xd, rows=True)
    val_s, idx_s = ops.gemm_select(a_s, b, metric, 1)
    # fused entry point
    val, idx, a_f = ops.assign_fused(xd, b, metric)
    st = ops.search_stats()
    assert st["mode"] == "fused-verified", st
    assert torch.equal(idx, idx_s)
    assert torch.equal(a_f.hi, a_s.hi) and torch.equal(a_f.norms, a_s.norms) and torch.equal(a_f.row_inv, a_s.row_inv)
    if kind == "duplicates":
        assert st["fallback_rows"] == m and st["overflow"] == 1, st
    elif kind == "sift":
        assert 0 < st["fallback_rows"] < m // 4 and st["overflow"] == 0, st
    print(f"verified assign {kind} d={d} n={n}: {st['fallback_rows']} of {m} rows re-run")
    xn = torch.linalg.vector_norm(xd, dim=1, keepdim=True)
    tol = (2e-3 if metric_ip else 4e-3) * xn * float(np.linalg.norm(c, axis=1).max()) + 1e-6
    assert bool(((val - val_s).abs() <= tol).all())
    # prepared planes
    got = ops.assign_verified(a_s, b, metric)
    assert got is not None
    st2 = ops.search_stats()
    assert st2["mode"] == "verified-resident" and torch.equal(got[1], idx_s)
    if kind == "sift":
        assert st2["fallback_rows"] == st["fallback_rows"]
    # ids-only public paths: quantisation and one k-means assign
    from image_search_engine_b200 import FaissKMeans, faiss_compat
    gi = faiss_compat.IndexFlatIP(d) if metric_ip else faiss_compat.IndexFlatL2(d)
    gi.add(cd)
    assert torch.equal(FaissKMeans(n, index=gi).transform_device(xd), idx_s.reshape(-1))
    # distances through the search API stay exact FP32 (re-scored)
    D, I = gi._search_device(xd[:50_000], 1)
    De, Ie = ops.flat_search_exact(xd[:64].contiguous(), cd, metric, 1)
    assert torch.equal(I[:64], Ie) or kind == "duplicates"
    assert torch.allclose(D[:64], De, rtol=2e-6, atol=1e-3 if not metric_ip else 1e-4)


def test_verified_assign_with_no_undecided_row():
    """Well separated columns: the one-product pass decides every row, the compact re-run launch finds a row count of zero
    on the device and the overflow launch returns at once -- results still equal the exact search."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    dev = ops.require_cuda()
    d, n, m = 128, 1024, 80_000
    j = np.arange(n)
    c = np.zeros((n, d), dtype=np.float32)
    c[j, j % d] = 1.0
    c[j, (j // d + j % d + 1) % d] += 0.5
    c /= np.linalg.norm(c, axis=1, keepdims=True)
    rng = np.random.default_rng(9)
    pick = rng.integers(0, n, m)
    x = np.zeros((m, d), dtype=np.float32)
    x[np.arange(m), pick % d] = 200.0
    x[np.arange(m), (pick // d + pick % d + 1) % d] += 100.0
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    b = ops.prepare_operand(cd)
    for metric in (METRIC_IP, METRIC_L2):
        val, idx, _ = ops.assign_fused(xd, b, metric)
        st = ops.search_stats()
        assert st["mode"] == "fused-verified" and st["fallback_rows"] == 0 and st["overflow"] == 0, st
        assert np.array_equal(idx.cpu().numpy().reshape(-1), pick)
        got = ops.assign_verified(ops.prepare_operand(xd, rows=True), b, metric)
        assert ops.search_stats()["fallback_rows"] == 0 and np.array_equal(got[1].cpu().numpy().reshape(-1), pick)


def test_verified_assign_takes_uint8_descriptors():
    """ORB / BRISK style uint8 descriptors are widened on the device (per-tensor scale, no per-row scales): the
    verified pipeline over their prepared planes gives the ids of the float32 copy of the same values."""
    from image_search_engine_b200 import FaissKMeans, faiss_compat, ops
    dev = ops.require_cuda()
    rng = np.random.default_rng(21)
    m, n, d = 120_000, 2048, 64
    xb = rng.integers(0, 256, (m, d), dtype=np.uint8)
    c = unit_rows(rng, n, d)
    gi = faiss_compat.IndexFlatIP(d)
    gi.add(c)
    km = FaissKMeans(n, index=gi)
    w8 = km.transform_device(torch.from_numpy(xb).to(dev))
    st = ops.search_stats()
    assert st["mode"] == "verified-resident", st
    wf = km.transform_device(torch.from_numpy(xb.astype(np.float32)).to(dev))
    assert ops.search_stats()["mode"] == "fused-verified" and torch.equal(w8, wf)
    from oracle import faiss_shim as fs
    rows = rng.choice(m, 1000, replace=False)
    _, Ir = fs.knn(xb[rows].astype(np.float32), c, 1, fs.METRIC_INNER_PRODUCT)
    assert_topk_parity(w8.cpu().numpy()[rows].reshape(-1, 1), Ir, xb[rows].astype(np.float32), c, True, max_mismatch_frac=0.01)


def test_fused_assign_declines_shapes_it_does_not_cover():
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP
    dev = ops.require_cuda()
    rng = np.random.default_rng(0)
    b = ops.prepare_operand(torch.from_numpy(unit_rows(rng, 4096, 128)).to(dev))
    few = torch.from_numpy(sift_like(rng, 100, 128)).to(dev)                 # one image: the column range is split
    assert ops.assign_fused(few, b, METRIC_IP) is None
    b2 = ops.prepare_operand(torch.from_numpy(unit_rows(rng, 300, 256)).to(dev))
    wide = torch.from_numpy(rng.standard_normal((200_000, 256)).astype(np.float32)).to(dev)
    assert ops.assign_fused(wide, b2, METRIC_IP) is None                      # d > 128


def test_speculative_kmeans_iterations_equal_the_synchronous_loop(monkeypatch):
    """The Lloyd loop launches the next assign before it has read the previous iteration's statistics back; a wrong
    guess ("no empty clusters") is rolled back.  Same objectives, same split counts, same centroids as the loop that
    synchronises every iteration -- including when EVERY guess after a split is forced (and therefore often wrong)."""
    from image_search_engine_b200 import faiss_compat
    rng = np.random.default_rng(77)
    n, d, k = 60000, 64, 256
    # integer-valued rows (SIFT-like): every FP32 cluster sum is exact whatever the order the rows are added in, so the
    # three runs follow the SAME trajectory and can be compared iteration by iteration (float data would let two
    # otherwise identical runs drift apart through the summation order of the update)
    centers = sift_like(rng, k // 2, d)
    x = np.clip(centers[rng.integers(0, k // 2, n)] + np.rint(4 * rng.standard_normal((n, d))), 0, 255).astype(np.float32)
    x[:6000] = x[0]                                     # duplicates: initial centroids coincide -> empty clusters -> splits
    runs = {}
    for name, env in (("sync", {"ISE_KMEANS_NO_SPECULATION": "1"}), ("spec", {}), ("forced", {"ISE_KMEANS_FORCE_SPECULATION": "1"})):
        for key in ("ISE_KMEANS_NO_SPECULATION", "ISE_KMEANS_FORCE_SPECULATION"):
            monkeypatch.delenv(key, raising=False)
        for key, v in env.items():
            monkeypatch.setenv(key, v)
        km = faiss_compat.Kmeans(d, k, seed=42, niter=12, spherical=True)
        km.train(x)
        runs[name] = km
    ref = runs["sync"]
    nsplit_ref = [s["nsplit"] for s in ref.iteration_stats]
    assert sum(nsplit_ref) > 0, "the data set must exercise the split path"
    assert not any(s.get("speculated") for s in ref.iteration_stats)
    for name in ("spec", "forced"):
        km = runs[name]
        assert [s["nsplit"] for s in km.iteration_stats] == nsplit_ref, name
        np.testing.assert_allclose(km.obj, ref.obj, rtol=1e-6, err_msg=name)
        np.testing.assert_allclose(km.centroids, ref.centroids, rtol=1e-6, atol=1e-7, err_msg=name)
    # the default policy only guesses after an iteration WITHOUT splits; the forced run guesses every time
    can_guess = any(a == 0 for a in nsplit_ref[:-2])
    assert any(s.get("speculated") for s in runs["spec"].iteration_stats) == can_guess
    assert any(s.get("speculated") for s in runs["forced"].iteration_stats)
    assert any(s.get("mis_speculated") for s in runs["forced"].iteration_stats), "the roll-back path was not exercised"
