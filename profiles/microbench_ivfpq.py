"""IndexIVFPQ search and range search on one GPU: the grouped path (ise_ivfpq_search, ise_ivfpq_range_count / _fill)
against the dense path it replaces for k <= 128 (ise_ivfpq_scan into a [min(nq, 4096), ntotal] matrix, then the top-k
selection), per-phase kernel time (look-up tables, grouping, scan, merge) and recall@10 against IndexFlatL2, for:

  the reference's "cell-probe" configuration IndexIVFPQ(IndexFlatL2(512), 512, 8, 16, 8), nprobe 5, over 100 000
  BoVW-like rows (non-negative, L2-normalised);  1 M and 10 M x 128 SIFT-like rows, nlist 1024, M 16, nprobe in
  {1, 8, 32};  nq in {1, 10 000}, k = 10;  range search at the radii that give about 10 and 100 results per query.

The indexes are trained on the GPU (IndexIVFPQ.train on at most 100 000 rows) and filled with IndexIVFPQ.add.  Times
are CUDA events around whole calls (median of --reps after --warmup, queries already probed for the kernel split);
the split comes from a separate torch.profiler pass.  The dense path is not run where one chunk's matrix
(min(nq, 4096) * ntotal * 4 bytes) exceeds --dense-budget; the row then records the bytes it would need.  Writes JSON
to --out (default profiles/r05_microbench_ivfpq.json)."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from image_search_engine_b200 import faiss_compat as fc  # noqa: E402
from image_search_engine_b200 import ops  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def kernel_split(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"lut": 0.0, "group": 0.0, "scan": 0.0, "merge": 0.0}
    for ev in prof.key_averages():
        name = ev.key
        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        if "ivfpq_lut_kernel" in name:
            out["lut"] += us / 1e3
        elif "ivfpq_grouped_scan" in name or "ivfpq_range" in name:
            out["scan"] += us / 1e3
        elif "topk_merge" in name or "range_lims" in name or "range_offsets" in name:
            out["merge"] += us / 1e3
        elif "ivf_" in name or "Radix" in name or "DeviceScan" in name or "emset" in name:
            out["group"] += us / 1e3
    return out


def dataset(kind, n, d, g):
    if kind == "bovw":
        x = torch.rand((n, d), generator=g, device="cuda") ** 8
        return x / x.norm(dim=1, keepdim=True)
    x = torch.randn((n, d), generator=g, device="cuda") ** 2
    x *= 512.0 / x.norm(dim=1, keepdim=True)
    return torch.clamp(torch.round(x), max=255.0)


def build(x, d, nlist, M, g):
    ix = fc.IndexIVFPQ(fc.IndexFlatL2(d), d, nlist, M, 8)
    ix.train(x[torch.randperm(x.shape[0], generator=g, device="cuda")[:100_000]])
    for i0 in range(0, x.shape[0], 1_000_000):
        ix.add(x[i0:i0 + 1_000_000])
    return ix


def dense_search(ix, q, k):
    """IndexIVFPQ.search through the dense path (the one k > 128 takes)."""
    ix._grouped = lambda k: False
    try:
        return ix.search(q, k)
    finally:
        del ix._grouped


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dense-budget", type=float, default=24e9, help="bytes of one dense chunk matrix")
    ap.add_argument("--sizes", default="ref,1m,10m")
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent / "r05_microbench_ivfpq.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    k = 10
    res = {"card (name, power limit, max SM clock)": card(), "k": k, "dense_budget_bytes": args.dense_budget,
           "lut_budget_bytes": ops.IVFPQ_LUT_BUDGET, "runs": []}
    configs = {"ref": ("bovw", 100_000, 512, 8, 16, (5,)), "1m": ("sift", 1_000_000, 128, 1024, 16, (1, 8, 32)),
               "10m": ("sift", 10_000_000, 128, 1024, 16, (1, 8, 32))}
    for name in args.sizes.split(","):
        kind, n, d, nlist, M, nprobes = configs[name]
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = dataset(kind, n, d, g)
        qall = (x[torch.randint(0, n, (10_000,), generator=g, device="cuda")] +
                0.05 * x.abs().mean() * torch.randn((10_000, d), generator=g, device="cuda"))
        ix = build(x, d, nlist, M, g)
        flat = fc.IndexFlatL2(d)
        flat.add(x)
        _, If_all = flat.search(qall, k)
        If_all = If_all.cpu().numpy()
        del flat
        torch.cuda.empty_cache()
        codes, ids, off, sizes = ix._lists()
        max_len = int(sizes.max())
        coarse = ix.quantizer._database()
        for nq in (1, 10_000):
            q = qall[:nq].contiguous()
            for nprobe in nprobes:
                ix.nprobe = nprobe
                probes = ix._probes(q)
                search_ms = timed(lambda: ix.search(q, k), args.warmup, args.reps)
                call = lambda: ops.ivfpq_search(q, coarse, ix.pq_centroids, codes, ids, off, max_len, probes, k)
                split = kernel_split(call)
                D, I = ix.search(q, k)
                dense_bytes = min(nq, 4096) * ix.ntotal * 4
                if dense_bytes <= args.dense_budget:
                    dense_ms = timed(lambda: dense_search(ix, q, k), args.warmup, args.reps)
                    Dd, _ = dense_search(ix, q, k)
                    same_d = bool(torch.equal(D, Dd))
                else:
                    dense_ms, same_d = f"not run: needs {dense_bytes} bytes", None
                recall = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(I.cpu().numpy(), If_all[:nq])]))
                p = probes.cpu().numpy()
                run = dict(index=name, data=kind, n=n, d=d, nlist=nlist, M=M, nq=nq, nprobe=nprobe,
                           max_list_len=max_len, scanned_codes=int(sizes[p[p >= 0]].sum()),
                           search_ms=search_ms, dense_search_ms=dense_ms,
                           speedup=dense_ms / search_ms if isinstance(dense_ms, float) else None,
                           dense_equal_distances=same_d, kernel_ms=split, recall_at_10=recall)
                # range search at the radii of the 10th and 100th neighbour (median over the queries)
                D100, _ = ix.search(q, 100)
                for target, col in ((10, 9), (100, 99)):
                    radius = float(D100[:, col].median())
                    range_ms = timed(lambda: ix.range_search(q, radius), args.warmup, args.reps)
                    rsplit = kernel_split(lambda: ops.ivfpq_range_search(q, coarse, ix.pq_centroids, codes, ids, off,
                                                                         max_len, probes, radius))
                    lims, _, _ = ix.range_search(q, radius)
                    run[f"range_{target}"] = dict(radius=radius, results_per_query=int(lims[-1]) / nq,
                                                  range_ms=range_ms, kernel_ms=rsplit)
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
        del ix, x, codes, ids, off, coarse
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
