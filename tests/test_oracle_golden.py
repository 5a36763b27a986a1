"""CPU: the oracle (oracle/faiss_shim.py) against the committed golden fixtures, which were produced by
the reference's own Python running on the shim (oracle/make_golden.py), plus the SURVEY known answers."""
from pathlib import Path

import numpy as np
import pytest

from oracle import cpu_baseline, faiss_shim as fs

GOLD = Path(__file__).parent / "golden"


@pytest.fixture(scope="module")
def g():
    return np.load(GOLD / "bovw_c1mini.npz")


@pytest.fixture(scope="module")
def kats():
    return np.load(GOLD / "kats.npz")


def test_kmeans_reproduces_fixture(g):
    km = fs.Kmeans(d=32, k=int(g["k"]), seed=42, niter=4, nredo=2, spherical=True, verbose=False)
    km.train(g["X"].astype(np.float32))
    assert np.array_equal(km.centroids, g["centroids"])
    assert np.array_equal(km.obj, g["obj"])
    assert km.obj[-1] == g["inertia"]
    np.testing.assert_allclose(np.linalg.norm(km.centroids, axis=1), 1.0, rtol=1e-6)  # spherical
    _, I = km.index.search(g["X"].astype(np.float32), 1)
    assert I.dtype == np.int64 and I.shape == g["words"].shape and np.array_equal(I, g["words"])


def test_histogram_and_okapi_loop(g):
    idx = cpu_baseline.codebook_index(g["centroids"])
    off = g["offsets"]
    descs = [g["X"][off[i]:off[i + 1]] for i in range(len(off) - 1)]
    H = cpu_baseline.visual_word_histograms(idx, descs, int(g["k"]))
    assert np.array_equal(H, g["hist"])
    assert (H.sum(1) == np.diff(off)).all()
    T = cpu_baseline.okapi_transform(H)
    assert np.array_equal(np.asarray(T.todense()), g["okapi"])


def test_flat_search_fixture(g):
    ip = fs.IndexFlatIP(32)
    ip.add(g["cos_db"])
    D, I = ip.search(g["q"], 10)
    assert np.array_equal(I, g["I_cos"]) and np.array_equal(D, g["D_cos"])
    assert (np.diff(D, axis=1) <= 0).all()                      # IP: descending
    l2 = fs.IndexFlatL2(32)
    l2.add(g["feats"])
    D, I = l2.search(g["q"], 10)
    assert np.array_equal(I, g["I_l2"]) and np.array_equal(D, g["D_l2"])
    assert (np.diff(D, axis=1) >= 0).all() and (D >= 0).all()   # L2: ascending, squared, clamped
    assert (I[:, 0] == np.arange(25)).all()
    D1, I1 = l2.search(g["q"][:1], 10)                          # nq < 20: direct path
    assert np.array_equal(I1, g["I_l2_1"]) and np.array_equal(D1, g["D_l2_1"])
    Dp, Ip = ip.search(g["q"][:1], 50)                          # k > ntotal
    assert np.array_equal(Ip, g["I_cos_1"]) and (Ip[0, 40:] == -1).all()
    assert (Dp[0, 40:] == -np.finfo(np.float32).max).all()


def test_index_file_format(g, tmp_path):
    idx = fs.IndexFlatIP(32)
    idx.add(g["centroids"])
    p = tmp_path / "c.faiss"
    fs.write_index(idx, str(p))
    raw = np.frombuffer(p.read_bytes(), dtype=np.uint8)
    assert np.array_equal(raw, g["codebook_file"])
    assert raw[:4].tobytes() == b"IxFI" and raw.size == 4 + 4 + 8 + 16 + 1 + 4 + 8 + 32 * 32 * 4
    back = fs.read_index(str(p))
    assert back.metric_type == fs.METRIC_INNER_PRODUCT and back.ntotal == 32
    assert np.array_equal(back.reconstruct_n(), g["centroids"])


def test_known_answers(kats):
    # SURVEY Q1: np.histogram bins over [min, max], bincount over [0, k)
    assert list(np.nonzero(kats["hist_q1_numpy"])[0]) == [0, 4, 103, 199]
    assert list(np.nonzero(kats["hist_q1_bincount"])[0]) == [3, 7, 100, 190]
    ip = fs.IndexFlatIP(2)
    ip.add(kats["tie_c"])
    D, I = ip.search(kats["tie_x"], 1)
    assert np.array_equal(I, kats["tie_I"]) and list(I[:4].ravel()) == [0, 2, 0, 0]   # tie -> lowest id
    D3, I3 = ip.search(kats["tie_x"], 3)
    assert np.array_equal(I3, kats["tie_I3"]) and list(I3[0]) == [0, 1, 2]
    D5, I5 = ip.search(kats["tie_x"], 5)
    assert np.array_equal(I5, kats["tie_I5"]) and (I5[:, 3:] == -1).all()
    T = cpu_baseline.okapi_transform(kats["okapi_in"])
    assert np.array_equal(np.asarray(T.todense()), kats["okapi_out"])
    one = np.asarray(cpu_baseline.okapi_transform(kats["okapi_in"][:1]).todense())
    assert np.array_equal(one, kats["okapi_single_row"])
    np.testing.assert_allclose(one[0, 0], 2 / (2 + 1.0))       # single row: dl/avgdl == 1 (quirk Q3)
    n = np.array([[3, 4], [0, 0], [1, 0]], dtype=np.float32)
    fs.normalize_L2(n)
    assert np.array_equal(n, kats["normalize_out"]) and (n[1] == 0).all()


def test_rand_perm_is_mt19937():
    # first outputs of std::mt19937(5489 default seed is 3499211612); seed 42 -> 1608637542
    assert int(fs.RandomGenerator(5489).raw(1)[0]) == 3499211612
    assert int(fs.RandomGenerator(42).raw(1)[0]) == 1608637542
    p = fs.rand_perm(1000, 7)
    assert sorted(p.tolist()) == list(range(1000))
    assert np.array_equal(fs.rand_perm(100000, 7, prefix=300), fs.rand_perm(100000, 7)[:300])


def test_clustering_edge_cases():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((50, 8)).astype(np.float32)
    with pytest.raises(RuntimeError):
        fs.Kmeans(8, 64).train(x)                       # fewer points than clusters
    bad = x.copy()
    bad[3, 2] = np.nan
    with pytest.raises(RuntimeError):
        fs.Kmeans(8, 4).train(bad)
    km = fs.Kmeans(8, 50, niter=3)
    km.train(x)                                         # nx == k: points copied, one fake stat
    assert np.array_equal(km.centroids, x) and len(km.obj) == 1
    # duplicate points force empty clusters -> split path with a deterministic RNG
    xd = np.repeat(x[:6], 40, axis=0)
    km = fs.Kmeans(8, 12, niter=4, seed=3)
    km.train(xd)
    assert sum(s["nsplit"] for s in km.iteration_stats) > 0
    km2 = fs.Kmeans(8, 12, niter=4, seed=3)
    km2.train(xd)
    assert np.array_equal(km.centroids, km2.centroids)


def test_cluster_score_fixture_is_davies_bouldin(g):
    """The committed cluster_score fixture (reference calc_sampled_cluster_score) restated on the CPU: minus the
    mean of 10 sklearn Davies-Bouldin scores over RandomState(42) samples of 2000 descriptors, labels from the
    oracle's flat-IP search against the fixture codebook."""
    from sklearn.metrics import davies_bouldin_score
    gold = np.load(GOLD / "cluster_score.npz")
    assert np.array_equal(gold["centroids"], g["centroids"])
    X = g["X"]
    idx = fs.IndexFlatIP(32)
    idx.add(g["centroids"])
    labels = idx.search(X.astype(np.float32), 1)[1].ravel()
    rs = np.random.RandomState(42)
    for key in ("score_first_call", "score_second_call"):
        scores = []
        for _ in range(10):
            s = rs.choice(X.shape[0], size=2000, replace=False)
            scores.append(davies_bouldin_score(X[s], labels[s]))
        assert -np.mean(scores) == pytest.approx(float(gold[key]), rel=1e-12)


def test_ivfpq_restatement_sanity():
    """The oracle's IndexIVFPQ (the reference's 'cell-probe' configuration, utils.py:311-325): stored vectors find
    themselves, results are sorted, all probed lists together return every id once, short results are padded."""
    rng = np.random.default_rng(5)
    cent = rng.standard_normal((12, 32)).astype(np.float32) * 3
    x = (cent[rng.integers(0, 12, 900)] + rng.standard_normal((900, 32))).astype(np.float32)
    ix = fs.IndexIVFPQ(fs.IndexFlatL2(32), 32, 8, 16, 8)
    ix.nprobe = 5
    with pytest.raises(RuntimeError):
        ix.add(x)                                   # not trained yet
    ix.train(x)
    ix.add(x)
    assert ix.ntotal == 900 and sum(len(i) for i in ix.ids) == 900
    D, I = ix.search(x[:40], 5)
    assert (I[:, 0] == np.arange(40)).mean() >= 0.9 and (np.diff(D, axis=1) >= 0).all()
    ix.nprobe = 8                                   # every list probed: each id appears exactly once
    D, I = ix.search(x[:2], 900)
    assert np.array_equal(np.sort(I[0]), np.arange(900))
    ix.nprobe = 1
    D, I = ix.search(x[:2], 900)
    assert (I[0] == -1).any() and (D[0][I[0] == -1] == np.finfo(np.float32).max).all()
    with pytest.raises(RuntimeError):
        fs.IndexIVFPQ(fs.IndexFlatL2(30), 30, 8, 16, 8)    # d must be a multiple of M
