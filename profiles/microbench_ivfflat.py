"""IndexIVFFlat search on one GPU: time per phase (probe, group, scan, merge), scanned pairs, algorithmic FLOP/s and the
scan's bytes/s, recall@10 against IndexFlat.search and the time ratio to it, for the shapes of DESIGN section 7:

  1 M x 2048 unit rows (CNN embeddings), IP, nlist 4096;  1 M x 128 SIFT-like rows, L2, nlist 1024;
  nprobe in {1, 8, 32, 128}, nq in {1, 10 000}, k = 10.

The coarse centroids are nlist database rows drawn with a fixed seed (training is not what is measured here).  Times are
CUDA events around whole calls (median of --reps after --warmup); the split of one call into grouping / scan / merge
kernels comes from a separate torch.profiler pass.  The vectors (1 GB or 8 GB) exceed the 126 MB L2, so a list is read
from HBM the first time a call touches it.  Writes JSON to --out (default profiles/r03_microbench_ivfflat.json)."""
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
    out = {"group": 0.0, "scan": 0.0, "merge": 0.0}
    for ev in prof.key_averages():
        name = ev.key
        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        if "ivfflat_scan_kernel" in name:
            out["scan"] += us / 1e3
        elif "topk_merge" in name:
            out["merge"] += us / 1e3
        elif "ivf_" in name or "Radix" in name or "DeviceScan" in name or "Memset" in name or "memset" in name:
            out["group"] += us / 1e3
    return out


def data(shape, n, d, g):
    if shape == "cnn":
        x = torch.randn((n, d), generator=g, device="cuda")
        x = torch.relu(x)
        x /= x.norm(dim=1, keepdim=True)
        return x
    x = torch.randn((n, d), generator=g, device="cuda") ** 2
    x *= 512.0 / x.norm(dim=1, keepdim=True)
    return torch.clamp(torch.round(x), max=255.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent / "r03_microbench_ivfflat.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "n": args.n, "k": 10, "runs": []}
    k = 10
    for shape, d, metric, nlist in (("cnn", 2048, fc.METRIC_INNER_PRODUCT, 4096), ("sift", 128, fc.METRIC_L2, 1024)):
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = data(shape, args.n, d, g)
        qall = x[torch.randint(0, args.n, (10_000,), generator=g, device="cuda")] + 0.01 * torch.randn(
            (10_000, d), generator=g, device="cuda")
        cent = x[torch.randint(0, args.n, (nlist,), generator=g, device="cuda")].clone()
        quant = fc.IndexFlatIP(d) if metric == fc.METRIC_INNER_PRODUCT else fc.IndexFlatL2(d)
        quant.add(cent)
        ix = fc.IndexIVFFlat(quant, d, nlist, metric)
        ix.add(x)
        flat = fc.IndexFlatIP(d) if metric == fc.METRIC_INNER_PRODUCT else fc.IndexFlatL2(d)
        flat.add(x)
        xs, ids, off = ix._lists()
        sizes = ix._sizes
        max_len = int(sizes.max())
        for nq in (1, 10_000):
            q = qall[:nq].contiguous()
            flat_ms = timed(lambda: flat.search(q, k), args.warmup, args.reps)
            _, If = flat.search(q, k)
            for nprobe in (1, 8, 32, 128):
                ix.nprobe = nprobe
                _, probes = quant._search_device(q, nprobe, need_distances=False)
                probe_ms = timed(lambda: quant._search_device(q, nprobe, need_distances=False), args.warmup, args.reps)
                scan_call_ms = timed(lambda: ops.ivfflat_search(q, xs, ids, off, max_len, probes, metric, k),
                                     args.warmup, args.reps)
                total_ms = timed(lambda: ix.search(q, k), args.warmup, args.reps)
                split = kernel_split(lambda: ops.ivfflat_search(q, xs, ids, off, max_len, probes, metric, k))
                _, I = ix.search(q, k)
                p = probes.cpu().numpy()
                pairs = int(sizes[p].sum())
                # bytes the scan must read: every probed list once per block of <= 32 of its queries, plus the queries
                per_list = np.bincount(p.ravel(), minlength=nlist)
                vec_bytes = int((np.ceil(per_list / 32) * sizes).sum()) * d * 4 + nq * nprobe * d * 4
                flop = pairs * d * (2 if metric == fc.METRIC_INNER_PRODUCT else 3)
                If_np, I_np = If.cpu().numpy(), I.cpu().numpy()
                recall = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(I_np, If_np)]))
                run = dict(shape=shape, d=d, metric="IP" if metric == fc.METRIC_INNER_PRODUCT else "L2", nlist=nlist,
                           nq=nq, nprobe=nprobe, max_list_len=max_len, scanned_pairs=pairs,
                           scanned_fraction=pairs / (nq * args.n), probe_ms=probe_ms, ivfflat_call_ms=scan_call_ms,
                           search_ms=total_ms, kernel_ms=split,
                           scan_tflops=flop / (split["scan"] * 1e-3) / 1e12 if split["scan"] else None,
                           scan_gbps=vec_bytes / (split["scan"] * 1e-3) / 1e9 if split["scan"] else None,
                           recall_at_10=recall, flat_search_ms=flat_ms, time_ratio_to_flat=total_ms / flat_ms)
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
        del ix, flat, x, xs, ids, off, quant
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
