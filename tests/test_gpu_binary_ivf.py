"""IndexBinaryIVF on the GPU, bit for bit against the NumPy restatement (tests/_binary_ivf_oracle.py) given the same
quantizer codes: search and range search over code widths, batch sizes (every threads-per-query regime), nprobe and k,
ties, edge cases, training, CUDA tensors, pickling, the workspace bound and a 1 M x 256-bit check."""
import pickle

import numpy as np
import pytest
import torch

from tests._binary_ivf_oracle import IndexBinaryIVF as OracleIVF, binary_to_real, real_to_binary
from tests._binary_oracle import INT32_MAX

pytestmark = pytest.mark.gpu


def _clustered(rng, n, d, ncent=64, flip=0.1):
    """Codes around ncent planted centres with a fraction of their bits flipped."""
    cent = rng.integers(0, 2, (ncent, d), dtype=np.uint8)
    out = np.empty((n, d // 8), np.uint8)
    for r0 in range(0, n, 1 << 16):
        m = min(n - r0, 1 << 16)
        bits = cent[rng.integers(0, ncent, m)] ^ (rng.random((m, d), dtype=np.float32) < flip).astype(np.uint8)
        out[r0:r0 + m] = np.packbits(bits, axis=1, bitorder="little")
    return out


def _pair(quant_codes, d, nlist):
    from image_search_engine_b200 import faiss_compat as fc
    q = fc.IndexBinaryFlat(d)
    q.add(quant_codes)
    return fc.IndexBinaryIVF(q, d, nlist), OracleIVF(quant_codes.copy(), d, nlist)


def _check_range(got, want):
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    assert got[0].dtype == np.uint64 and got[1].dtype == np.int32 and got[2].dtype == np.int64


@pytest.mark.parametrize("nq", [1, 7, 500, 5000])
@pytest.mark.parametrize("d", [8, 64, 256, 520, 2048])
def test_search_and_range_equal_restatement(d, nq):
    rng = np.random.default_rng(d * 7 + nq)
    n, nlist = 6000, 24
    x = _clustered(rng, n, d)
    ix, ref = _pair(x[rng.choice(n, nlist, replace=False)], d, nlist)
    for part in np.array_split(x, 3):                                   # adds in several batches
        ix.add(part)
        ref.add(part)
    assert np.array_equal(np.concatenate([np.full(ix.get_list_size(l), l) for l in range(nlist)]),
                          np.sort(ref.assignment()))
    for l in range(nlist):
        assert np.array_equal(ix.get_list_ids(l), ref.ids[l])
    q = np.concatenate([x[rng.integers(0, n, nq // 2)], _clustered(rng, nq - nq // 2, d)])
    for nprobe in (1, 4, nlist):
        ix.nprobe = ref.nprobe = nprobe
        for k in (1, 10, 128):
            D, I = ix.search(q, k)
            Dr, Ir = ref.search(q, k)
            assert np.array_equal(I, Ir) and np.array_equal(D, Dr), (nprobe, k)
        if nq <= 500:
            for radius in (0, 1, d // 4, d + 1):
                _check_range(ix.range_search(q, radius), ref.range_search(q, radius))


@pytest.mark.parametrize("nlist", [100, 128])
@pytest.mark.parametrize("d", [64, 256])
def test_all_lists_probed_equals_flat(d, nlist):
    """nprobe <= 128 keeps nprobe * S <= 256 chunk lists per query (S <= 256 / nprobe), so one ise_topk_merge joins
    them; nlist 128 fills all 256 inputs of that merge."""
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(d + nlist)
    n, nq = 60000, 50
    x = rng.integers(0, 256, (n, d // 8), dtype=np.uint8)
    ix, _ = _pair(x[:nlist], d, nlist)
    ix.add(x)
    ix.nprobe = nlist
    flat = fc.IndexBinaryFlat(d)
    flat.add(x)
    q = rng.integers(0, 256, (nq, d // 8), dtype=np.uint8)
    for k in (1, 10, 128):
        D, I = ix.search(q, k)
        Df, If = flat.search(q, k)
        assert np.array_equal(D, Df) and np.array_equal(I, If)
    for radius in (d // 4, d // 2):
        lims, RD, RI = ix.range_search(q, radius)
        limf, RDf, RIf = flat.range_search(q, radius)
        assert np.array_equal(lims, limf)
        for i in range(nq):
            o = np.argsort(RI[lims[i]:lims[i + 1]])
            assert np.array_equal(RI[lims[i]:lims[i + 1]][o], RIf[limf[i]:limf[i + 1]])
            assert np.array_equal(RD[lims[i]:lims[i + 1]][o], RDf[limf[i]:limf[i + 1]])
        D, I = ix.search(q, 128)                                        # range distances are search's
        for i in range(nq):
            ids, dis = RI[lims[i]:lims[i + 1]], RD[lims[i]:lims[i + 1]]
            _, a, b = np.intersect1d(ids, I[i], return_indices=True)
            assert np.array_equal(dis[a], D[i, b])


def test_heavy_ties_lowest_ids_win():
    rng = np.random.default_rng(5)
    d, nlist = 64, 8
    base = rng.integers(0, 256, (6, d // 8), dtype=np.uint8)
    x = base[rng.integers(0, 6, 3000)]                                  # duplicated codes over several lists
    lists = rng.integers(0, nlist, x.shape[0])
    ix, ref = _pair(rng.integers(0, 256, (nlist, d // 8), dtype=np.uint8), d, nlist)
    ix.add_preassigned(x, lists)
    ref.add_preassigned(x, lists)
    q = np.concatenate([base, rng.integers(0, 256, (20, d // 8), dtype=np.uint8)])
    for nprobe in (2, 5, 8):
        ix.nprobe = ref.nprobe = nprobe
        for k in (1, 7, 100, 128):
            D, I = ix.search(q, k)
            Dr, Ir = ref.search(q, k)
            assert np.array_equal(I, Ir) and np.array_equal(D, Dr)
        _check_range(ix.range_search(q, 3), ref.range_search(q, 3))


def test_edge_cases():
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(9)
    d, nlist = 256, 10
    quant = rng.integers(0, 256, (nlist, d // 8), dtype=np.uint8)
    q = rng.integers(0, 256, (5, d // 8), dtype=np.uint8)
    un = fc.IndexBinaryIVF(fc.IndexBinaryFlat(d), d, nlist)               # untrained
    D, I = un.search(q, 4)
    assert (I == -1).all() and (D == INT32_MAX).all()
    assert un.range_search(q, 100)[0].tolist() == [0] * 6
    ix, ref = _pair(quant, d, nlist)
    D, I = ix.search(q, 4)                                              # trained, empty
    assert (I == -1).all() and (D == INT32_MAX).all()
    D, I = ix.search(q[:0], 4)
    assert D.shape == (0, 4) and I.shape == (0, 4)
    assert ix.range_search(q[:0], 5)[0].tolist() == [0]
    # lists 0, 3 and a skewed list 7 spanning many chunks; the others empty; ntotal < nlist first
    ix.add_preassigned(q[:3], [0, 3, 3])
    ref.add_preassigned(q[:3], [0, 3, 3])
    ix.nprobe = ref.nprobe = 4
    for k in (1, 5):                                                    # k > ntotal
        assert all(np.array_equal(a, b) for a, b in zip(ix.search(q, k), ref.search(q, k)))
    x = rng.integers(0, 256, (40000, d // 8), dtype=np.uint8)
    lists = np.where(rng.random(40000) < 0.9, 7, rng.choice([0, 3], 40000))
    ix.add_preassigned(x, lists)
    ref.add_preassigned(x, lists)
    for nprobe in (1, 3, 10, 50):                                       # probed-but-empty lists, nprobe > nlist
        ix.nprobe = ref.nprobe = nprobe
        for k in (1, 10, 128):
            D, I = ix.search(q, k)
            Dr, Ir = ref.search(q, k)
            assert np.array_equal(I, Ir) and np.array_equal(D, Dr)
        _check_range(ix.range_search(q, 120), ref.range_search(q, 120))


def test_training_matches_kmeans_on_decoded_sample():
    from image_search_engine_b200 import faiss_compat as fc, ops
    rng = np.random.default_rng(3)
    d, nlist = 64, 16
    for n in (3000, 9000):                                              # below and above 256 * nlist: the sample
        x = _clustered(rng, n, d, ncent=16)
        ix = fc.IndexBinaryIVF(fc.IndexBinaryFlat(d), d, nlist)
        ix.train(x)
        assert ix.is_trained and ix.quantizer.ntotal == nlist
        sample = x[ops.rand_perm_prefix(n, 1234, 256 * nlist)] if n > 256 * nlist else x
        km = fc.Kmeans(d, nlist, niter=10, seed=1234)
        km.train(binary_to_real(sample))
        assert np.array_equal(ix.quantizer.reconstruct_n(), real_to_binary(km.centroids))
        before = ix.quantizer.reconstruct_n()
        ix.train(_clustered(rng, 5000, d))                              # filled quantizer: untouched
        assert np.array_equal(ix.quantizer.reconstruct_n(), before)


def test_conversion_kernels_equal_numpy():
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(4)
    codes = rng.integers(0, 256, (300, 65), dtype=np.uint8)
    x = ops.binary_to_real(torch.from_numpy(codes).cuda(), 65)
    assert np.array_equal(x.cpu().numpy(), binary_to_real(codes))
    r = rng.standard_normal((300, 520)).astype(np.float32)
    r[:, ::7] = 0.0
    assert np.array_equal(ops.real_to_binary(torch.from_numpy(r).cuda(), 65).cpu().numpy(), real_to_binary(r))


def test_training_recall_end_to_end():
    from image_search_engine_b200 import faiss_compat as fc
    rng = np.random.default_rng(8)
    d, n, nlist, nq, k = 256, 20000, 64, 300, 10
    x = _clustered(rng, n, d, ncent=200, flip=0.15)
    q = x[rng.integers(0, n, nq)] ^ (rng.random((nq, d // 8)) < 0.05).astype(np.uint8)
    ix = fc.IndexBinaryIVF(fc.IndexBinaryFlat(d), d, nlist)
    ix.train(x)
    ix.add(x)
    ix.nprobe = 4
    _, I = ix.search(q, k)
    ref = OracleIVF(None, d, nlist)
    ref.train(x)
    ref.add(x)
    ref.nprobe = 4
    _, Ir = ref.search(q, k)
    flat = fc.IndexBinaryFlat(d)
    flat.add(x)
    _, If = flat.search(q, k)
    recall = np.mean([len(set(a) & set(b)) / k for a, b in zip(I, If)])
    recall_ref = np.mean([len(set(a) & set(b)) / k for a, b in zip(Ir, If)])
    assert recall >= recall_ref - 0.05, (recall, recall_ref)


def test_cuda_tensors_pickle_reset():
    rng = np.random.default_rng(6)
    d, nlist = 64, 12
    x = _clustered(rng, 5000, d)
    ix, ref = _pair(x[:nlist], d, nlist)
    ix.add(x)
    ix.nprobe = 3
    q = x[:40]
    D, I = ix.search(q, 10)
    Dt, It = ix.search(torch.from_numpy(q).cuda(), 10)
    assert Dt.is_cuda and It.is_cuda and Dt.dtype == torch.int32
    assert np.array_equal(Dt.cpu().numpy(), D) and np.array_equal(It.cpu().numpy(), I)
    lims, RD, RI = ix.range_search(q, 12)
    lt, RDt, RIt = ix.range_search(torch.from_numpy(q).cuda(), 12)
    assert lt.dtype == torch.int64 and lt.is_cuda and RDt.dtype == torch.int32
    assert np.array_equal(lt.cpu().numpy(), lims.astype(np.int64)) and np.array_equal(RIt.cpu().numpy(), RI)
    ix2 = pickle.loads(pickle.dumps(ix))
    assert ix2.nprobe == 3 and ix2.ntotal == ix.ntotal
    D2, I2 = ix2.search(q, 10)
    assert np.array_equal(D2, D) and np.array_equal(I2, I)
    for l in range(nlist):
        ids = ix2.get_list_ids(l)
        assert np.array_equal(ids, ix.get_list_ids(l)) and (np.diff(ids) > 0).all()
    ix.reset()
    assert ix.ntotal == 0 and ix.is_trained and ix.get_list_size(0) == 0
    assert (ix.search(q, 3)[1] == -1).all()


def test_workspace_bound_and_no_dense_matrix():
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(2)
    d, nlist, n, nq, k, nprobe = 256, 256, 200000, 20000, 10, 8
    x = rng.integers(0, 256, (n, d // 8), dtype=np.uint8)
    ix, _ = _pair(x[:nlist], d, nlist)
    ix.add(x)
    ix.nprobe = nprobe
    q = torch.from_numpy(rng.integers(0, 256, (nq, d // 8), dtype=np.uint8)).cuda()
    ix.search(q, k)                                                     # builds the list storage
    torch.cuda.synchronize()
    ws = ops.binary_ivf_search_workspace_bytes(nq, nprobe, nlist, int(ix._sizes.max()), d // 8, k)
    assert ws < nq * n                                                  # far below an [nq, ntotal] int8 matrix
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    ix.search(q, k)
    torch.cuda.synchronize()
    probe_ws = ops.binary_knn_workspace_bytes(nq, nlist, d // 8, nprobe)
    outputs = nq * k * 12 + nq * nprobe * 12 + nq * 64                  # D, I, probes (+ their distances), padded q
    assert torch.cuda.max_memory_allocated() - base <= max(ws, probe_ws) + outputs + (4 << 20)


def test_benchmark_size_sampled_exact():
    rng = np.random.default_rng(11)
    d, n, nlist, nq, k, nprobe = 256, 1_000_000, 4096, 10_000, 10, 16
    x = _clustered(rng, n, d, ncent=4096, flip=0.1)
    from image_search_engine_b200 import faiss_compat as fc
    quant = fc.IndexBinaryFlat(d)
    quant.add(x[rng.choice(n, nlist, replace=False)])
    ix = fc.IndexBinaryIVF(quant, d, nlist)
    ix.add(x)
    ix.nprobe = nprobe
    q = x[rng.integers(0, n, nq)] ^ (rng.random((nq, d // 8)) < 0.02).astype(np.uint8)
    D, I = ix.search(q, k)
    sample = rng.choice(nq, 200, replace=False)
    probes = ix._probes(ix.quantizer._device_rows(q[sample])[0]).cpu().numpy()
    ref = OracleIVF(quant.reconstruct_n(), d, nlist)
    ref.nprobe = nprobe
    for l in range(nlist):                                              # the GPU's lists
        ref.ids[l] = ix.get_list_ids(l)
        ref.codes[l] = x[ref.ids[l]]
    ref.ntotal = n
    Dr, Ir = ref.search(q[sample], k, probes=probes)
    assert np.array_equal(D[sample], Dr) and np.array_equal(I[sample], Ir)
