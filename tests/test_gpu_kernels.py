"""GPU parity tests of the libise kernels against the CPU oracle (through the C ABI via ops.py)."""
import numpy as np
import pytest
import torch

from tests._util import assert_topk_parity, orb_like, sift_like, unit_rows

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from image_search_engine_b200 import ops
    return ops.require_cuda()


def _oracle_knn(x, y, k, metric_ip):
    from oracle import faiss_shim as fs
    return fs.knn(x.astype(np.float32), y.astype(np.float32), k,
                  fs.METRIC_INNER_PRODUCT if metric_ip else fs.METRIC_L2)


def test_prepare_planes_f32(dev):
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(0)
    x = (rng.standard_normal((1000, 100)) * 3.7).astype(np.float32)
    op = ops.prepare_operand(torch.from_numpy(x).to(dev))
    assert op.lo is not None and op.ldp == 104
    meta = op.meta.cpu().numpy()
    scale = meta[0]
    assert scale == 2.0 ** round(np.log2(scale)) and abs(meta[1] * scale - 1) == 0
    assert 8192 <= np.abs(x).max() * scale < 16384
    rec = (op.hi.float() + op.lo.float()).cpu().numpy()[:, :100] / scale
    assert np.abs(rec - x).max() <= np.abs(x).max() * 2.0 ** -21
    assert (op.hi.cpu().numpy()[:, 100:] == 0).all()
    np.testing.assert_allclose(op.norms.cpu().numpy(), (x.astype(np.float64) ** 2).sum(1), rtol=2e-6)


def test_prepare_planes_exact_inputs(dev):
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(1)
    u8 = orb_like(rng, 777, 32)
    op = ops.compact_operand(ops.prepare_operand(torch.from_numpy(u8).to(dev)))
    assert op.lo is None
    assert np.array_equal(op.hi.float().cpu().numpy(), u8.astype(np.float32))
    assert np.array_equal(op.norms.cpu().numpy(), (u8.astype(np.float64) ** 2).sum(1).astype(np.float32))
    s = sift_like(rng, 500, 128)
    op2 = ops.prepare_operand(torch.from_numpy(s).to(dev))
    assert op2.lo is not None and float(op2.meta[2]) == 0.0
    op2 = ops.compact_operand(op2)
    assert op2.lo is None  # integer-valued float32 is exact in one FP16 plane
    scale = float(op2.meta[0])
    assert np.array_equal(op2.hi.float().cpu().numpy() / scale, s)


@pytest.mark.parametrize("m,n,d,kind", [
    (300, 512, 32, "orb"), (1000, 4096, 128, "sift"), (129, 257, 100, "float"), (64, 40, 8, "float"),
    (5000, 1000, 64, "float"), (257, 256, 2048, "unit"),
])
def test_assign_ip_top1(dev, m, n, d, kind):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP
    rng = np.random.default_rng(m + n + d)
    if kind == "orb":
        x = orb_like(rng, m, d)
    elif kind == "sift":
        x = sift_like(rng, m, d)
    elif kind == "unit":
        x = unit_rows(rng, m, d, relu=True)
    else:
        x = rng.standard_normal((m, d)).astype(np.float32)
    c = unit_rows(rng, n, d)
    a = ops.prepare_operand(torch.from_numpy(x).to(dev))
    b = ops.prepare_operand(torch.from_numpy(c).to(dev))
    val, idx = ops.gemm_select(a, b, METRIC_IP, 1)
    D, I = _oracle_knn(x, c, 1, True)
    xf = x.astype(np.float32)
    nm = assert_topk_parity(idx.cpu().numpy(), I, xf, c, True, max_mismatch_frac=0.002)
    np.testing.assert_allclose(val.cpu().numpy(), D, rtol=1e-4, atol=1e-4 * np.abs(D).max())
    print(f"[assign {m}x{n}x{d} {kind}] near-tie mismatches: {nm}")


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("nq,nb,d,k", [(200, 3000, 64, 10), (128, 70000, 32, 20), (333, 1000, 512, 100),
                                        (50, 7, 16, 10)])
def test_flat_search_topk(dev, metric_ip, nq, nb, d, k):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(nq * 7 + nb + d + k)
    db = unit_rows(rng, nb, d, relu=True)
    q = db[rng.integers(0, nb, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    a = ops.prepare_operand(torch.from_numpy(q).to(dev))
    b = ops.prepare_operand(torch.from_numpy(db).to(dev))
    val, idx = ops.gemm_select(a, b, METRIC_IP if metric_ip else METRIC_L2, k)
    D, I = _oracle_knn(q, db, k, metric_ip)
    idx_h, val_h = idx.cpu().numpy(), val.cpu().numpy()
    kk = min(k, nb)
    assert (idx_h[:, kk:] == -1).all() and (I[:, kk:] == -1).all()
    assert_topk_parity(idx_h[:, :kk], I[:, :kk], q, db, metric_ip, max_mismatch_frac=0.05)
    np.testing.assert_allclose(val_h[:, :kk], D[:, :kk], rtol=1e-4, atol=2e-6)
    # sortedness (best first) is size independent
    srt = -val_h[:, :kk] if metric_ip else val_h[:, :kk]
    assert (np.diff(srt, axis=1) >= 0).all()


@pytest.mark.parametrize("metric_ip", [True, False])
def test_exact_small_batch(dev, metric_ip):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(5)
    db = rng.standard_normal((50000, 96)).astype(np.float32)
    q = rng.standard_normal((7, 96)).astype(np.float32)
    val, idx = ops.flat_search_exact(torch.from_numpy(q).to(dev), torch.from_numpy(db).to(dev),
                                     METRIC_IP if metric_ip else METRIC_L2, 20)
    D, I = _oracle_knn(q, db, 20, metric_ip)
    assert_topk_parity(idx.cpu().numpy(), I, q, db, metric_ip, max_mismatch_frac=1.0)
    np.testing.assert_allclose(val.cpu().numpy(), D, rtol=1e-4, atol=1e-4)


def test_ties_lowest_id_wins(dev):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP
    x = np.eye(4, 16, dtype=np.float32)[[0, 1, 2, 3] * 40]          # 160 rows
    c = np.zeros((600, 16), np.float32)
    c[5, 0] = c[300, 0] = c[599, 0] = 1.0      # three identical best columns for e0
    c[7, 1] = c[8, 1] = 2.0
    a = ops.prepare_operand(torch.from_numpy(x).to(dev))
    b = ops.prepare_operand(torch.from_numpy(c).to(dev))
    _, idx = ops.gemm_select(a, b, METRIC_IP, 1)
    idx = idx.cpu().numpy().ravel()
    assert (idx[0::4] == 5).all() and (idx[1::4] == 7).all()
    _, idx3 = ops.gemm_select(a, b, METRIC_IP, 3)
    assert (idx3.cpu().numpy()[0] == [5, 300, 599]).all()
    assert (idx[2::4] == 0).all()  # all-zero scores: first column


def test_topk_merge_matches_unsharded(dev):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(11)
    db = unit_rows(rng, 4000, 64)
    q = unit_rows(rng, 150, 64)
    a = ops.prepare_operand(torch.from_numpy(q).to(dev))
    for metric in (METRIC_IP, METRIC_L2):
        full = ops.gemm_select(a, ops.prepare_operand(torch.from_numpy(db).to(dev)), metric, 10)
        parts_v, parts_i = [], []
        for s in range(4):
            b = ops.prepare_operand(torch.from_numpy(db[s * 1000:(s + 1) * 1000]).to(dev))
            v, i = ops.gemm_select(a, b, metric, 10, id_base=s * 1000)
            parts_v.append(v)
            parts_i.append(i)
        mv, mi = ops.topk_merge(torch.stack(parts_v), torch.stack(parts_i), metric)
        assert_topk_parity(mi.cpu().numpy(), full[1].cpu().numpy(), q, db, metric == METRIC_IP,
                           max_mismatch_frac=0.05)
        np.testing.assert_allclose(mv.cpu().numpy(), full[0].cpu().numpy(), rtol=1e-5, atol=1e-6)


def test_normalize_l2(dev):
    from image_search_engine_b200 import ops
    from oracle import faiss_shim as fs
    rng = np.random.default_rng(3)
    x = rng.standard_normal((1000, 100)).astype(np.float32)
    x[10] = 0
    ref = x.copy()
    fs.normalize_L2(ref)
    t = torch.from_numpy(x.copy()).to(dev)
    ops.normalize_l2_(t)
    np.testing.assert_allclose(t.cpu().numpy(), ref, rtol=1e-6, atol=1e-7)
    assert (t[10] == 0).all()


@pytest.mark.parametrize("k", [200, 512, 4096, 20000])
@pytest.mark.parametrize("mode", ["numpy_compat", "bincount"])
def test_histogram_bit_exact(dev, k, mode):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import HIST_BINCOUNT, HIST_NUMPY_COMPAT
    rng = np.random.default_rng(k)
    sizes = np.concatenate([[0, 1, 3], rng.integers(50, 900, 60)])
    off = np.zeros(len(sizes) + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    words = rng.integers(0, k, off[-1]).astype(np.int64)
    words[off[2]:off[3]] = 7                      # all-equal image -> range [v-.5, v+.5]
    words[off[4]:off[4] + 2] = [0, k - 1]         # image hitting both ends -> identity binning
    H = ops.bovw_histogram(torch.from_numpy(words).to(dev), torch.from_numpy(off).to(dev), k,
                           mode=HIST_NUMPY_COMPAT if mode == "numpy_compat" else HIST_BINCOUNT).cpu().numpy()
    assert H.dtype == np.float64
    for i in range(len(sizes)):
        w = words[off[i]:off[i + 1]]
        ref = np.histogram(w, bins=k)[0] if mode == "numpy_compat" else np.bincount(w, minlength=k)
        assert np.array_equal(H[i], ref), f"image {i} differs"
    assert (H.sum(1) == sizes).all()


def test_okapi_fused_and_dense(dev):
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import HIST_BINCOUNT
    rng = np.random.default_rng(9)
    k, sizes = 300, rng.integers(1, 400, 80)
    off = np.zeros(len(sizes) + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    words = rng.integers(0, k, off[-1]).astype(np.int64)
    wd, od = torch.from_numpy(words).to(dev), torch.from_numpy(off).to(dev)
    H = ops.bovw_histogram(wd, od, k, mode=HIST_BINCOUNT).cpu().numpy()
    dl = H.sum(1, keepdims=True)
    ref = H.copy()
    ref *= 1
    nz = ref != 0
    den = ref + 1 * (1 - 0.75 + 0.75 * (dl / np.mean(dl)))
    ref[nz] = (ref / den)[nz]
    fused = ops.bovw_histogram(wd, od, k, mode=HIST_BINCOUNT, okapi=True).cpu().numpy()
    assert np.array_equal(fused, ref)           # float64, same operation order -> bit exact
    dense = ops.okapi_tf_(torch.from_numpy(H).to(dev)).cpu().numpy()
    assert np.array_equal(dense, ref)
    f32 = ops.bovw_histogram(wd, od, k, mode=HIST_BINCOUNT, okapi=True, out_dtype=torch.float32).cpu().numpy()
    assert np.array_equal(f32, ref.astype(np.float32))


def test_kmeans_update_and_split(dev):
    from image_search_engine_b200 import ops
    from oracle import faiss_shim as fs
    rng = np.random.default_rng(21)
    n, d, k = 20000, 64, 100
    x = rng.standard_normal((n, d)).astype(np.float32)
    assign = rng.integers(0, k - 5, n).astype(np.int64)   # last 5 clusters empty
    dis = rng.random(n).astype(np.float32)
    cent_ref = np.zeros((k, d), np.float32)
    h_ref = np.zeros(k, np.float32)
    fs.compute_centroids(d, k, x, assign, h_ref, cent_ref)
    counts_before = h_ref.copy()
    ns_ref = fs.split_clusters(d, k, n, h_ref, cent_ref)
    fs.normalize_L2(cent_ref)

    xd = torch.from_numpy(x).to(dev)
    accum = torch.zeros(k * d + k, device=dev)
    sums, counts = accum[:k * d].view(k, d), accum[k * d:]
    obj = torch.zeros(1, dtype=torch.float64, device=dev)
    ops.kmeans_accumulate(xd, torch.from_numpy(assign).to(dev), torch.from_numpy(dis).to(dev), sums, counts, obj)
    cent = torch.empty(k, d, device=dev)
    n_empty = torch.zeros(1, dtype=torch.int32, device=dev)
    ops.kmeans_mean(sums, counts, cent, n_empty)
    assert int(n_empty.item()) == 5
    assert np.array_equal(counts.cpu().numpy(), counts_before)
    assert abs(float(obj.item()) - dis.astype(np.float64).sum()) < 1e-6 * n
    pairs, h_new = ops.split_plan(counts.cpu().numpy(), n)
    assert pairs.shape[0] == ns_ref == 5
    assert np.array_equal(h_new, h_ref)
    ops.kmeans_apply_splits(cent, torch.from_numpy(pairs).to(dev))
    ops.normalize_l2_(cent)
    np.testing.assert_allclose(cent.cpu().numpy(), cent_ref, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("nq,nb,d,k", [(300, 20000, 128, 10), (64, 5000, 2048, 10), (500, 70000, 96, 5),
                                        (80000, 1024, 512, 1), (200, 30000, 64, 100), (150, 70000, 128, 40),
                                        (300, 200000, 64, 100),
                                        # d >= 1024 with >= 4 row tiles: CTA pairs for the coarse top-k / collect pass
                                        (600, 20000, 1024, 10), (600, 70000, 1024, 40)])
def test_verified_coarse_search_equals_split(dev, metric_ip, nq, nb, d, k):
    """Default index search = 1-product coarse pass + exact re-score + proof; must agree with the
    3-product split path and with the oracle."""
    from image_search_engine_b200 import faiss_compat, ops
    rng = np.random.default_rng(nq + nb + d + k)
    db = unit_rows(rng, nb, d, relu=True)
    q = db[rng.integers(0, nb, nq)] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    idx = faiss_compat.IndexFlatIP(d) if metric_ip else faiss_compat.IndexFlatL2(d)
    idx.add(db)
    D, I = idx.search(q, k)
    assert ops.last_search_stats["mode"].startswith("verified"), ops.last_search_stats
    n_fallback = ops.last_search_stats["fallback_rows"]
    idx.precision = "split"
    D2, I2 = idx.search(q, k)
    assert ops.last_search_stats["mode"] == "split"
    assert_topk_parity(I, I2, q, db, metric_ip, max_mismatch_frac=0.05)
    np.testing.assert_allclose(D, D2, rtol=1e-5, atol=2e-6)
    Do, Io = _oracle_knn(q, db, k, metric_ip)
    assert_topk_parity(I, Io, q, db, metric_ip, max_mismatch_frac=0.05)
    np.testing.assert_allclose(D, Do, rtol=1e-4, atol=4e-6)
    print(f"[verified {nq}x{nb}x{d} k={k} ip={metric_ip}] fallback rows: {n_fallback}")


def test_verified_search_falls_back_on_unresolvable_rows(dev):
    """Near-duplicate database rows are closer together than the coarse pass can resolve: those queries
    must be flagged and re-run with the split products, and still match the oracle."""
    from image_search_engine_b200 import faiss_compat, ops
    rng = np.random.default_rng(77)
    d, nb = 256, 6000
    base = unit_rows(rng, 60, d)
    db = np.repeat(base, 100, axis=0) + 2e-5 * rng.standard_normal((nb, d)).astype(np.float32)   # 100 near copies each
    db = db.astype(np.float32)
    q = np.concatenate([base[:40] + 1e-5 * rng.standard_normal((40, d)).astype(np.float32),
                        unit_rows(rng, 60, d)]).astype(np.float32)
    idx = faiss_compat.IndexFlatIP(d)
    idx.add(db)
    D, I = idx.search(q, 10)
    assert ops.last_search_stats["fallback_rows"] >= 40, ops.last_search_stats
    Do, Io = _oracle_knn(q, db, 10, True)
    assert_topk_parity(I, Io, q, db, True, max_mismatch_frac=1.0)
    np.testing.assert_allclose(D, Do, rtol=1e-4, atol=2e-6)
    # each near-copy query finds only members of its own cluster
    assert ((I[:40] // 100) == np.arange(40)[:, None]).all()


def test_verified_assign_flags_ties_and_near_ties(dev):
    """Coarse top-1: duplicated / nearly duplicated centroids cannot be separated by the FP16 pass; those
    rows must be flagged and resolved by the split products (exact ties -> lowest id)."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP
    rng = np.random.default_rng(5)
    d, k, n = 512, 512, 80000
    c = unit_rows(rng, k, d)
    c[300] = c[7]                                    # exact duplicate: id 7 must win
    c[301] = c[9] * np.float32(1 + 3e-5)             # near duplicate, slightly better
    x = rng.standard_normal((n, d)).astype(np.float32)
    x[:50] = c[7] * 3 + 0.01 * rng.standard_normal((50, d)).astype(np.float32)
    x[50:100] = c[9] * 2 + 0.01 * rng.standard_normal((50, d)).astype(np.float32)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    a, b = ops.prepare_operand(xd), ops.prepare_operand(cd)
    D, I = ops.search_topk(xd, a, cd, b, METRIC_IP, 1)
    st = ops.search_stats()
    assert st["mode"] == "verified" and 100 <= st["fallback_rows"] < n // 4, st
    Do, Io = _oracle_knn(x, c, 1, True)
    assert (I.cpu().numpy()[:50, 0] == 7).all() and (I.cpu().numpy()[50:100, 0] == 301).all()
    assert_topk_parity(I.cpu().numpy(), Io, x, c, True, max_mismatch_frac=0.002)
    np.testing.assert_allclose(D.cpu().numpy(), Do, rtol=1e-4, atol=1e-5)
    D2, I2 = ops.search_topk(xd, a, cd, b, METRIC_IP, 1, precision="split")
    assert torch.equal(I, I2)


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("d,kind,k", [(32, "orb", 512), (128, "sift", 1000), (100, "float", 300), (256, "float", 257),
                                       (64, "float", 4096)])
def test_assign_many_row_tiles(dev, metric_ip, d, kind, k):
    """Top-1 over >= 2 row tiles per SM (the persistent loop wraps several times, no column splits), with
    ragged tails in rows, columns and d, both metrics, uint8 / integer / general float rows."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(d * 7 + k)
    m = 128 * 148 * 2 + 77
    x = orb_like(rng, m, d) if kind == "orb" else sift_like(rng, m, d) if kind == "sift" else \
        rng.standard_normal((m, d)).astype(np.float32)
    c = unit_rows(rng, k, d) if metric_ip else (rng.standard_normal((k, d)) * 2).astype(np.float32)
    xd = torch.from_numpy(x).to(dev)
    a = ops.prepare_operand(xd)
    b = ops.prepare_operand(torch.from_numpy(c).to(dev))
    val, idx = ops.gemm_select(a, b, METRIC_IP if metric_ip else METRIC_L2, 1)
    D, I = _oracle_knn(x, c, 1, metric_ip)
    xf = x.astype(np.float32)
    assert_topk_parity(idx.cpu().numpy(), I, xf, c, metric_ip, max_mismatch_frac=0.002)
    np.testing.assert_allclose(val.cpu().numpy(), D, rtol=2e-4, atol=2e-4 * np.abs(D).max())


@pytest.mark.parametrize("metric_ip", [True, False])
@pytest.mark.parametrize("n,d,k,kind", [(50000, 128, 4096, "sift"), (30000, 32, 512, "orb"), (20000, 64, 300, "float"),
                                          (9000, 256, 1000, "float"), (6000, 100, 64, "float"), (5000, 2048, 40, "float")])
def test_plain_accumulate_equals_oracle(dev, n, d, k, kind, metric_ip):
    """Global-atomic scatter-add vs the oracle's sequential compute_centroids: counts exact, sums / objective within
    FP32 reassociation."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    from oracle import faiss_shim as fs
    rng = np.random.default_rng(n + d + k)
    x = orb_like(rng, n, d) if kind == "orb" else sift_like(rng, n, d) if kind == "sift" else \
        rng.standard_normal((n, d)).astype(np.float32)
    assign = rng.integers(0, k - 3, n).astype(np.int64)      # last 3 clusters stay empty
    assign[::501] = -1                                       # unassigned rows are skipped
    cent = unit_rows(rng, k, d)
    xf = x.astype(np.float32)
    keep = assign >= 0
    sums_ref = np.zeros((k, d), np.float64)
    np.add.at(sums_ref, assign[keep], xf[keep].astype(np.float64))
    counts_ref = np.bincount(assign[keep], minlength=k).astype(np.float32)
    c64 = cent.astype(np.float64)[assign[keep]]
    obj_ref = float((xf[keep] * c64).sum()) if metric_ip else float(((xf[keep] - c64) ** 2).sum())
    xd, ad, cd = torch.from_numpy(x).to(dev), torch.from_numpy(assign).to(dev), torch.from_numpy(cent).to(dev)
    accum = torch.zeros(k * d + k, device=dev)
    sums, counts = accum[:k * d].view(k, d), accum[k * d:]
    obj = torch.zeros(1, dtype=torch.float64, device=dev)
    ops.kmeans_accumulate(xd, ad, None, sums, counts, obj, centroids=cd, metric=METRIC_IP if metric_ip else METRIC_L2)
    s, c, o = sums.cpu().numpy(), counts.cpu().numpy(), float(obj.item())
    assert np.array_equal(c, counts_ref)
    np.testing.assert_allclose(s, sums_ref, rtol=2e-5, atol=2e-5 * np.abs(sums_ref).max())
    assert abs(o - obj_ref) <= 1e-5 * abs(obj_ref) + 1e-3, (o, obj_ref)


def test_exact_inputs_skip_the_lo_plane_and_nobody_reads_it(dev):
    """Integer-valued float32 descriptors are exact in the FP16 hi plane: prepare does not even write the lo plane
    (META_LO_NONZERO stays 0) and gemm_select must never load it.  The allocator block the lo plane lands in is
    poisoned with NaNs first, so any read of it would surface in the scores."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import METRIC_IP, METRIC_L2
    rng = np.random.default_rng(12)
    x = torch.from_numpy(sift_like(rng, 40000, 128)).to(dev)
    c = torch.from_numpy(unit_rows(rng, 1000, 128)).to(dev)
    b = ops.prepare_operand(c)
    for _ in range(2):
        poison = torch.full((40000, 128), float("nan"), dtype=torch.float16, device=dev)
        poison2 = torch.full((40000, 128), float("nan"), dtype=torch.float16, device=dev)
        del poison, poison2                                    # blocks return to the caching allocator ...
        a = ops.prepare_operand(x)                             # ... and are handed out again for hi / lo
        assert a.lo is not None and float(a.meta[2]) == 0.0
    assert bool(torch.isnan(a.lo.float()).any()), "the lo plane was written although the input is exact"
    assert not bool(torch.isnan(a.hi.float()).any())
    a_hi_only = ops.Operand(a.hi, None, a.norms, a.meta, a.n, a.d, a.ldp)
    for metric in (METRIC_IP, METRIC_L2):
        v2, i2 = ops.gemm_select(a, b, metric, 1)              # PA = 2 plane slots, lo skipped at run time
        v1, i1 = ops.gemm_select(a_hi_only, b, metric, 1)
        assert torch.equal(i1, i2) and torch.equal(v1, v2) and not bool(torch.isnan(v2).any())
    # non-exact data still gets its lo plane
    y = torch.randn((5000, 128), device=dev)
    ay = ops.prepare_operand(y)
    assert float(ay.meta[2]) != 0.0 and not bool(torch.isnan(ay.lo.float()).any())
    # ... and meta[2] carries the largest RELATIVE squared hi-plane residual of a row, which the coarse error bound uses
    sc = float(ay.meta[0])
    res = ((y.double() - ay.hi[:, :128].double() / sc).pow(2).sum(1) / y.double().pow(2).sum(1)).max().item()
    assert res <= float(ay.meta[2]) <= res * 1.001 and float(ay.meta[2]) < 2.0 ** -22
    # the single-pass row preparation publishes the same quantity (per-row scales)
    ar = ops.prepare_operand(y, rows=True)
    hr = ar.hi[:, :128].double() * ar.row_inv.double()[:, None]
    res_r = ((y.double() - hr).pow(2).sum(1) / y.double().pow(2).sum(1)).max().item()
    assert res_r <= float(ar.meta[2]) <= res_r * 1.001 and float(ar.meta[2]) < 2.0 ** -22
    # a value far below the maximum leaves FP16's normal range once scaled: the input no longer counts as exact and
    # the lo plane is written again (zeros here: such a value underflows in both planes, which the coarse error
    # bound accounts for)
    z = x[:4096].clone()
    z[0, 0] = 2.0 ** -40
    poison = torch.full((4096, 128), float("nan"), dtype=torch.float16, device=dev)
    del poison
    az = ops.prepare_operand(z)
    assert not bool(torch.isnan(az.lo.float()).any())


@pytest.mark.parametrize("k,mode_name,out_dtype", [(4096, "numpy", torch.float64), (512, "bincount", torch.float64),
                                                   (1001, "numpy", torch.float32), (4096, "numpy", torch.float32)])
def test_warp_per_image_histogram_equals_cta_kernel(dev, monkeypatch, k, mode_name, out_dtype):
    """Short images with float64 rows go through the warp-per-image kernel; it must equal the CTA-per-image kernel bit
    for bit and np.histogram row by row (empty, one-word and over-long images included; the float32 cases pin the
    CTA kernel the same way)."""
    from image_search_engine_b200 import ops
    from image_search_engine_b200._lib import HIST_BINCOUNT, HIST_NUMPY_COMPAT
    rng = np.random.default_rng(k)
    sizes = rng.integers(0, 220, 2000)
    sizes[:4] = [0, 1, 2500, 130]                      # empty / single / longer than the register window / > 128
    off = np.zeros(len(sizes) + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    words = rng.integers(0, k, int(off[-1]))
    words[off[2]:off[2] + 60] = 5                      # tf beyond the 32-entry Okapi table
    wd, od = torch.from_numpy(words).to(dev), torch.from_numpy(off).to(dev)
    mode = HIST_NUMPY_COMPAT if mode_name == "numpy" else HIST_BINCOUNT
    res = {}
    for which in ("warp", "cta"):
        if which == "cta":
            monkeypatch.setenv("ISE_HIST_CTA", "1")
        else:
            monkeypatch.delenv("ISE_HIST_CTA", raising=False)
        res[which] = (ops.bovw_histogram(wd, od, k, mode=mode, out_dtype=out_dtype),
                      ops.bovw_histogram(wd, od, k, mode=mode, out_dtype=out_dtype, okapi=True, k1=1.3, k2=0.8, b=0.7))
    assert torch.equal(res["warp"][0], res["cta"][0])
    assert torch.equal(res["warp"][1], res["cta"][1])
    H = res["warp"][0].cpu().numpy()
    for i in (0, 1, 2, 3, 17, 1999):
        seg = words[off[i]:off[i + 1]]
        want = np.zeros(k) if seg.size == 0 else (np.histogram(seg, bins=k)[0] if mode_name == "numpy"
                                                   else np.bincount(seg, minlength=k))
        assert np.array_equal(H[i], want.astype(H.dtype)), i
    assert (H.sum(1) == sizes).all()
