"""IndexBinaryIVF on one GPU against IndexBinaryFlat on the same codes and queries:

  ORB     1 M x 256-bit codes, nlist in {1024, 4096};
  dHash   10 M x 64-bit codes, nlist 16384;
  nq in {1, 500, 10 000}, nprobe in {1, 8, 32}, k in {2, 10}, and one range search per shape (radius 40 for ORB, 8 for
  dHash) at nq 10 000, nprobe 8.

Two code distributions: "clustered" (codes around planted centres with 10 % of their bits flipped, queries are stored
codes with 2 % more flips, so recall means something) and "uniform" (random codes and queries: the lists are balanced
but the nearest neighbours are spread over all lists, the worst case for recall).  Each index is trained with its own
train() (k-means on the decoded sample) and filled with add().

Per case: `ivf_ms`, the median over --reps of CUDA events around IndexBinaryIVF.search / range_search with CUDA tensors
(probe + scan, after --warmup); `flat_ms`, the same for IndexBinaryFlat; their ratio; `scanned_pairs` = sum over the
queries of the sizes of their probed lists, and its share of nq * ntotal; `recall_at_k` = |IVF ids & flat ids| / k
averaged over the queries.  `phases_ms` comes from a separate torch.profiler pass of one call: probe (the quantizer
binary_knn), group (ivf_* kernels and CUB sort / scan), scan (binary_ivf_* kernels), merge (topk merge, int32
distances, range offsets; the probe's own merge and distance kernels count here too, so "probe" is its scan kernel
only).  The card's name, power limit and max SM clock are read in the same run.  JSON to --out.
"""
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


def phases(fn):
    """Kernel time per phase of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = dict(probe=0.0, group=0.0, scan=0.0, merge=0.0, other=0.0)
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name, us = e.name, e.device_time
        if "binary_ivf" in name:
            out["scan"] += us
        elif "binary_knn" in name:
            out["probe"] += us
        elif "ivf_" in name or "Radix" in name or "Scan" in name and "lims" not in name:
            out["group"] += us
        elif "merge" in name or "binary_dis" in name or "lims" in name or "range" in name:
            out["merge"] += us
        else:
            out["other"] += us
    return {k: v / 1e3 for k, v in out.items()}


def clustered(g, n, cs, ncent, flip):
    """Codes around ncent planted centres, each bit flipped with probability flip (device, in slices)."""
    cent = torch.randint(0, 2, (ncent, 8 * cs), generator=g, device="cuda", dtype=torch.uint8)
    w = (2 ** torch.arange(8, device="cuda", dtype=torch.int32)).repeat(cs)
    out = torch.empty((n, cs), dtype=torch.uint8, device="cuda")
    for r0 in range(0, n, 1 << 20):
        m = min(n - r0, 1 << 20)
        bits = cent[torch.randint(0, ncent, (m,), generator=g, device="cuda")]
        bits = bits ^ (torch.rand((m, 8 * cs), generator=g, device="cuda") < flip).to(torch.uint8)
        out[r0:r0 + m] = (bits.to(torch.int32) * w).reshape(m, cs, 8).sum(-1).to(torch.uint8)
    return out


def flip_bits(g, x, p):
    cs = x.shape[1]
    w = (2 ** torch.arange(8, device="cuda", dtype=torch.int32)).repeat(cs)
    mask = (torch.rand((x.shape[0], 8 * cs), generator=g, device="cuda") < p).to(torch.int32) * w
    return x ^ mask.reshape(x.shape[0], cs, 8).sum(-1).to(torch.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent / "r03_microbench_binary_ivf.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "runs": []}
    g = torch.Generator(device="cuda").manual_seed(1234)
    shapes = (("orb", 256, 1_000_000, (1024, 4096), 40), ("dhash", 64, 10_000_000, (16384,), 8))
    for name, d, ntotal, nlists, radius in shapes:
        cs = d // 8
        for dist in ("clustered", "uniform"):
            if dist == "clustered":
                x = clustered(g, ntotal, cs, ncent=max(nlists), flip=0.1)
                qall = flip_bits(g, x[torch.randint(0, ntotal, (10_000,), generator=g, device="cuda")], 0.02)
            else:
                x = torch.randint(0, 256, (ntotal, cs), generator=g, device="cuda", dtype=torch.uint8)
                qall = torch.randint(0, 256, (10_000, cs), generator=g, device="cuda", dtype=torch.uint8)
            flat = fc.IndexBinaryFlat(d)
            flat.add(x)
            flat_ref = {}
            for nlist in nlists:
                ix = fc.IndexBinaryIVF(fc.IndexBinaryFlat(d), d, nlist)
                ix.train(x)
                ix.add(x)
                sizes = torch.from_numpy(ix._sizes).cuda()
                for nq in (1, 500, 10_000):
                    q = qall[:nq].contiguous()
                    for k in (2, 10):
                        if (nq, k) not in flat_ref:
                            flat_ref[(nq, k)] = (timed(lambda: flat.search(q, k), args.warmup, args.reps),
                                                 flat.search(q, k)[1])
                        flat_ms, If = flat_ref[(nq, k)]
                        for nprobe in (1, 8, 32):
                            ix.nprobe = nprobe
                            ms = timed(lambda: ix.search(q, k), args.warmup, args.reps)
                            _, I = ix.search(q, k)
                            pairs = int(sizes[ix._probes(ix.quantizer._device_rows(q)[0])].sum())
                            hit = (I[:, :, None] == If[:, None, :]) & (I[:, :, None] >= 0)
                            run = dict(shape=name, data=dist, op="search", d=d, ntotal=ntotal, nlist=nlist, nq=nq, k=k,
                                       nprobe=nprobe, ivf_ms=ms, flat_ms=flat_ms, flat_over_ivf=flat_ms / ms,
                                       scanned_pairs=pairs, scanned_share=pairs / (nq * ntotal),
                                       recall_at_k=float(hit.any(2).sum(1).float().mean() / k),
                                       phases_ms=phases(lambda: ix.search(q, k)))
                            res["runs"].append(run)
                            print(json.dumps(run), flush=True)
                q = qall.contiguous()
                ix.nprobe = 8
                ms = timed(lambda: ix.range_search(q, radius), args.warmup, args.reps)
                fms = timed(lambda: flat.range_search(q, radius), args.warmup, args.reps)
                lims, _, _ = ix.range_search(q, radius)
                limf, _, _ = flat.range_search(q, radius)
                run = dict(shape=name, data=dist, op="range_search", d=d, ntotal=ntotal, nlist=nlist, nq=q.shape[0],
                           nprobe=8, radius=radius, ivf_ms=ms, flat_ms=fms, flat_over_ivf=fms / ms,
                           results=int(lims[-1]), flat_results=int(limf[-1]),
                           recall=int(lims[-1]) / max(1, int(limf[-1])),
                           phases_ms=phases(lambda: ix.range_search(q, radius)))
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
                del ix
                torch.cuda.empty_cache()
            del flat, x, qall
            torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
