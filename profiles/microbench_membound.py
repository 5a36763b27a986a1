"""HBM-bound kernels of the path at C2 size (1M x 128 descriptors, k = 4096, 10k images): device time
(CUDA events, 10 launches after 3 warm-ups; every launch touches > 126 MB so nothing survives in L2 except the
8 MB id array) and achieved algorithmic GB/s against MEASURED_PEAKS.json."""
import json
import sys
import numpy as np, torch
sys.path.insert(0, ".")
from bench import sift_like, C2, peaks
from image_search_engine_b200 import ops
from image_search_engine_b200._lib import METRIC_IP, HIST_NUMPY_COMPAT, HIST_BINCOUNT
dev = ops.require_cuda()
P = peaks()["hbm"]


def t(fn, n=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


rng = np.random.default_rng(2)
n, d, k, n_img = C2["n_desc"], C2["d"], C2["k"], C2["n_img"]
X = torch.from_numpy(sift_like(rng, n, d)).to(dev)
Xu8 = X.to(torch.uint8)
cent = X[torch.randperm(n, device=dev)[:k]].clone()
ops.normalize_l2_(cent)
a = ops.compact_operand(ops.prepare_operand(X)); b = ops.prepare_operand(cent)
_, words = ops.gemm_select(a, b, METRIC_IP, 1)
off = torch.arange(0, n + 1, C2["per_img"], dtype=torch.int64, device=dev)
out64 = torch.empty((n_img, k), dtype=torch.float64, device=dev)
out32 = torch.empty((n_img, k), dtype=torch.float32, device=dev)
accum = torch.zeros((k * d + k,), dtype=torch.float32, device=dev)
sums, counts = accum[: k * d].view(k, d), accum[k * d:]
obj = torch.zeros((1,), dtype=torch.float64, device=dev)
rows = []


def rec(name, ms, nbytes):
    gbs = nbytes / (ms * 1e-3) / 1e9
    rows.append(dict(kernel=name, ms=ms, algorithmic_bytes=nbytes, gbs=gbs, frac_of_hbm_peak=gbs / P))
    print(f"{name:58s} {ms*1e3:8.1f} us  {gbs:7.0f} GB/s  {gbs/P:5.2f} of {P:.0f}")


rec("prepare f32, integer-valued (absmax + hi plane + norms; 10 B/element moved)", t(lambda: ops.prepare_operand(X)), n * d * 10)
Xf = X + 0.37
rec("prepare f32, general (absmax + hi/lo planes + norms; 12 B/element moved)", t(lambda: ops.prepare_operand(Xf)), n * d * 12)
rec("prepare ROWS f32, integer-valued (single pass: 4 B read + hi plane + norms; 6 B/element)", t(lambda: ops.prepare_operand(X, rows=True)), n * d * 6)
rec("prepare ROWS f32, general (single pass: 4 B read + hi/lo planes + norms; 8 B/element)", t(lambda: ops.prepare_operand(Xf, rows=True)), n * d * 8)
rec("prepare u8 (one plane + norms)", t(lambda: ops.prepare_operand(Xu8)), n * d * (1 + 2))
rec("histogram f64 numpy-compat + okapi", t(lambda: ops.bovw_histogram(words, off, k, mode=HIST_NUMPY_COMPAT, okapi=True, out=out64)), n * 8 + n_img * k * 8)
rec("histogram f64 bincount", t(lambda: ops.bovw_histogram(words, off, k, mode=HIST_BINCOUNT, out=out64)), n * 8 + n_img * k * 8)
rec("histogram f32 numpy-compat + okapi", t(lambda: ops.bovw_histogram(words, off, k, mode=HIST_NUMPY_COMPAT, okapi=True, out_dtype=torch.float32, out=out32)), n * 8 + n_img * k * 4)
rec("okapi_tf_ dense f64 in place (row sums + weights)", t(lambda: ops.okapi_tf_(out64)), n_img * k * 8 * 2)
ws = [None]
def _sorted(x):
    ws[0] = ops.kmeans_accumulate_sorted(x, words, sums, counts, obj, centroids=cent, workspace=ws[0])
rec("kmeans_accumulate_sorted f32 (counting sort + gather-reduce, + exact objective)", t(lambda: _sorted(X)), n * (4 * d + 8))
rec("kmeans_accumulate_sorted u8", t(lambda: _sorted(Xu8)), n * (d + 8))
a_rows = ops.compact_operand(ops.prepare_operand(X, rows=True))
def _sorted_h():
    ws[0] = ops.kmeans_accumulate_sorted(X, words, sums, counts, obj, centroids=cent, workspace=ws[0], exact_op=a_rows)
rec("kmeans_accumulate_sorted, rows gathered from the exact FP16 hi plane (2 d + 12 B/row)", t(_sorted_h), n * (2 * d + 12))
val = torch.empty((n, 1), dtype=torch.float32, device=dev)
rec("rescore top-1 (exact distances of the winners)", t(lambda: ops.rescore_topk_(X, cent, a, b, METRIC_IP, val, words)), n * (4 * d + 12))
Y = X.clone()
rec("normalize_L2 in place", t(lambda: ops.normalize_l2_(Y)), n * d * 8)
big = torch.empty((256 << 20,), dtype=torch.float32, device=dev)
big2 = torch.empty_like(big)
rec("(reference) torch copy 1 GiB -> 1 GiB", t(lambda: big2.copy_(big)), big.numel() * 8)
rec("(reference) cudaMemset 1 GiB", t(lambda: big.zero_()), big.numel() * 4)
# write-only stream of REAL data (not a constant the memory system can compress): the source is a 1 MiB tile that stays in L2
tile = torch.randn((1 << 18,), device=dev)
bigv = big.view(-1, 1 << 18)
rec("(reference) write-only 1 GiB of random data (L2-resident 1 MiB tile broadcast)", t(lambda: bigv.copy_(tile.expand_as(bigv))), big.numel() * 4)
rec("(reference) read-only 1 GiB (sum)", t(lambda: big.sum()), big.numel() * 4)
half = torch.empty((big.numel() // 2,), dtype=torch.float16, device=dev)
rec("(reference) float32 -> float16 cast of 1 GiB (read 4 B, write 2 B per element)", t(lambda: half.copy_(big[: half.numel()])), half.numel() * 6)
u8big = torch.empty((big.numel() // 2,), dtype=torch.uint8, device=dev)
rec("(reference) uint8 -> float16 cast (read 1 B, write 2 B per element)", t(lambda: half.copy_(u8big)), half.numel() * 3)
json.dump(rows, open("gpurun_out/r02_membound.json", "w"), indent=1)
