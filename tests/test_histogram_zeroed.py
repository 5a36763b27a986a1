"""GPU: the zeroed-output histogram (only the non-zero bins written into a matrix cleared beforehand) equals the dense
write-out bit for bit in every kernel, and BOVW.histograms_device (matrix cleared on a side stream while the assign
runs) equals assign + dense histogram on the benchmark's C2 inputs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from image_search_engine_b200 import ops
    return ops.require_cuda()


def _edge_batch(rng, k, n_img):
    sizes = rng.integers(0, 220, n_img)
    # empty, one descriptor, past the warp kernel's 128 ids held in registers, past the CTA kernel's 512, all equal
    sizes[:5] = [0, 1, 130, 700, 40]
    off = np.zeros(n_img + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    words = rng.integers(0, k, int(off[-1]))
    words[off[2]:off[2] + 60] = 5          # tf beyond the 32-entry Okapi table
    words[off[3]] = k + 5                  # bincount: outside [0, k), not counted
    words[off[4]:off[5]] = k // 3          # numpy-compat: min == max, bins over [v - 0.5, v + 0.5]
    return words, off


def _dense_and_zeroed(words, off, k, dev, monkeypatch, cta, **kw):
    """(dense histogram, zeroed histogram written into a NaN-filled buffer that clear_ zeroed)"""
    from image_search_engine_b200 import ops
    if cta:
        monkeypatch.setenv("ISE_HIST_CTA", "1")
    else:
        monkeypatch.delenv("ISE_HIST_CTA", raising=False)
    wd, od = torch.from_numpy(words).to(dev), torch.from_numpy(off).to(dev)
    dense = ops.bovw_histogram(wd, od, k, **kw)
    buf = torch.full_like(dense, float("nan"))
    ops.clear_(buf)
    zeroed = ops.bovw_histogram(wd, od, k, out=buf, zeroed=True, **kw)
    return dense, zeroed


@pytest.mark.parametrize("out_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("okapi", [False, True])
@pytest.mark.parametrize("mode_name", ["numpy", "bincount"])
@pytest.mark.parametrize("k", [4096, 1001])
def test_zeroed_equals_dense_edge_cases(dev, monkeypatch, k, mode_name, okapi, out_dtype):
    """2001 images (enough for the warp-per-image kernel; float32 rows and ISE_HIST_CTA take the CTA kernel); k = 1001
    is not a multiple of 4 and makes the matrix's byte count leave a tail after the 16-byte clear stores."""
    from image_search_engine_b200._lib import HIST_BINCOUNT, HIST_NUMPY_COMPAT
    rng = np.random.default_rng(k + 7 * okapi)
    words, off = _edge_batch(rng, k, 2001)
    kw = dict(mode=HIST_NUMPY_COMPAT if mode_name == "numpy" else HIST_BINCOUNT, out_dtype=out_dtype)
    if okapi:
        kw.update(okapi=True, k1=1.3, k2=0.8, b=0.7)
    for cta in ((False, True) if out_dtype == torch.float64 else (False,)):
        dense, zeroed = _dense_and_zeroed(words, off, k, dev, monkeypatch, cta, **kw)
        assert torch.equal(zeroed, dense), f"cta={cta}"
    H = dense.cpu().numpy()
    for i in range(6):
        seg = words[off[i]:off[i + 1]]
        if mode_name == "bincount":
            seg = seg[seg < k]
        want = np.zeros(k) if seg.size == 0 else (np.histogram(seg, bins=k)[0] if mode_name == "numpy"
                                                   else np.bincount(seg, minlength=k))
        assert np.array_equal(H[i] != 0, want != 0), i


def test_zeroed_without_shared_memory_counters(dev, monkeypatch):
    """k beyond the shared-memory counter budget: counts are added into the cleared row itself (no memset)."""
    from image_search_engine_b200 import ops
    rng = np.random.default_rng(3)
    k = ops.CSR_MAX_BINS + 700
    words, off = _edge_batch(rng, k, 300)
    dense, zeroed = _dense_and_zeroed(words, off, k, dev, monkeypatch, False, okapi=True)
    assert torch.equal(zeroed, dense)


@pytest.mark.parametrize("out_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("okapi", [False, True])
@pytest.mark.parametrize("mode_name", ["numpy", "bincount"])
def test_zeroed_equals_dense_c2_shape(dev, monkeypatch, mode_name, okapi, out_dtype):
    """10 000 images x 100 random words, k = 4096."""
    from image_search_engine_b200._lib import HIST_BINCOUNT, HIST_NUMPY_COMPAT
    rng = np.random.default_rng(11)
    k, n_img, per = 4096, 10_000, 100
    off = np.arange(0, n_img * per + 1, per, dtype=np.int64)
    words = rng.integers(0, k, n_img * per)
    kw = dict(mode=HIST_NUMPY_COMPAT if mode_name == "numpy" else HIST_BINCOUNT, out_dtype=out_dtype)
    if okapi:
        kw.update(okapi=True)
    dense, zeroed = _dense_and_zeroed(words, off, k, dev, monkeypatch, False, **kw)
    assert torch.equal(zeroed, dense)
    assert float((dense != 0).sum(1).max()) <= per


def test_histograms_device_equals_dense_on_bench_inputs(dev):
    """The benchmark's seeded C2 step (rank 0 inputs, codebook from 2 Lloyd iterations): histograms_device, which
    clears the matrix beside the assign and writes the non-zero bins, equals assign followed by the dense histogram."""
    from bench import C2, sift_like
    from image_search_engine_b200 import BOVW, FaissKMeans, ops
    from image_search_engine_b200.bag_of_visual_words import PackedDescriptions
    from image_search_engine_b200.utils import OkapiTransformer
    rng = np.random.default_rng(2)
    X = torch.from_numpy(sift_like(rng, C2["n_desc"], C2["d"])).to(dev)
    offsets = np.arange(0, C2["n_desc"] + 1, C2["per_img"], dtype=np.int64)
    km = FaissKMeans(C2["k"], n_init=1, max_iter=2)
    km.fit(X)
    bovw = BOVW(None, n_clusters=C2["k"])
    bovw.clusterer = km
    okapi = OkapiTransformer()
    for _ in range(2):                     # the second call reuses the side stream
        got = bovw.histograms_device(PackedDescriptions(X, offsets), okapi=okapi)
    want = ops.bovw_histogram(km.transform_device(X), torch.from_numpy(offsets).to(dev), C2["k"], okapi=True,
                              k1=okapi.k1, k2=okapi.k2, b=okapi.b)
    assert torch.equal(got, want)
    plain = bovw.histograms_device(PackedDescriptions(X, offsets), out_dtype=torch.float32)
    assert float(plain.sum()) == C2["n_desc"] and bool((plain.sum(1) == C2["per_img"]).all())
