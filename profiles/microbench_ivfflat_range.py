"""IndexIVFFlat.range_search on one GPU: time per phase (probe, group, count, lims, fill), results per query, and the time
ratios to IndexIVFFlat.search(x, k) at the same nprobe (k = results per query, capped at 128) and to
IndexFlat.range_search at the same radius, for the shapes of microbench_ivfflat.py:

  1 M x 2048 unit rows (CNN embeddings), IP, nlist 4096;  1 M x 128 SIFT-like rows, L2, nlist 1024;
  nq in {1, 10 000}, nprobe in {8, 32}, radii aimed at about 10, 100 and 1000 results per query.

A radius is the median, over 100 sampled queries, of the score of each query's n-th best vector among its probed lists.
The coarse centroids are nlist database rows drawn with a fixed seed.  Times are CUDA events around whole calls (median of
--reps after --warmup).  The split of one call into kernels comes from a separate torch.profiler pass: group = pair keys,
radix sort and list items; count / fill = the two range kernels; lims = the CUB scans and the lims gather (the grouping's
(nlist + 1)-entry item scan is counted here too); probe = the quantizer's search, timed on its own.  The card's name, power
limit and max SM clock are read in the same run.  Writes JSON to --out (default profiles/r04_microbench_ivfflat_range.json).
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
    out = {"group": 0.0, "count": 0.0, "lims": 0.0, "fill": 0.0}
    for ev in prof.key_averages():
        name = ev.key
        ms = (getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)) / 1e3
        if "ivfflat_range_count_kernel" in name:
            out["count"] += ms
        elif "ivfflat_range_fill_kernel" in name:
            out["fill"] += ms
        elif "DeviceScan" in name or "ivf_range_lims" in name:
            out["lims"] += ms
        elif "ivf_" in name or "Radix" in name or "Memset" in name or "memset" in name:
            out["group"] += ms
    return out


def data(shape, n, d, g):
    if shape == "cnn":
        x = torch.relu(torch.randn((n, d), generator=g, device="cuda"))
        x /= x.norm(dim=1, keepdim=True)
        return x
    x = torch.randn((n, d), generator=g, device="cuda") ** 2
    x *= 512.0 / x.norm(dim=1, keepdim=True)
    return torch.clamp(torch.round(x), max=255.0)


def radii(q, xs, off, probes, ip, targets):
    """Median over the sampled queries of the targets[i]-th best score among each query's probed vectors."""
    nlist = off.shape[0] - 1
    row_list = torch.repeat_interleave(torch.arange(nlist, device=xs.device), torch.diff(off))
    s = q @ xs.T
    if not ip:
        s = (q * q).sum(1, keepdim=True) + (xs * xs).sum(1)[None, :] - 2 * s
    out = {t: [] for t in targets}
    for i in range(q.shape[0]):
        v = s[i][torch.isin(row_list, probes[i])]
        v = torch.sort(v, descending=ip).values
        for t in targets:
            out[t].append(float(v[min(t, v.numel()) - 1]))
    return {t: float(np.median(v)) for t, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent / "r04_microbench_ivfflat_range.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "n": args.n, "runs": []}
    for shape, d, metric, nlist in (("cnn", 2048, fc.METRIC_INNER_PRODUCT, 4096), ("sift", 128, fc.METRIC_L2, 1024)):
        ip = metric == fc.METRIC_INNER_PRODUCT
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = data(shape, args.n, d, g)
        qall = x[torch.randint(0, args.n, (10_000,), generator=g, device="cuda")] + 0.01 * torch.randn(
            (10_000, d), generator=g, device="cuda")
        cent = x[torch.randint(0, args.n, (nlist,), generator=g, device="cuda")].clone()
        quant = fc.IndexFlatIP(d) if ip else fc.IndexFlatL2(d)
        quant.add(cent)
        ix = fc.IndexIVFFlat(quant, d, nlist, metric)
        ix.add(x)
        flat = fc.IndexFlatIP(d) if ip else fc.IndexFlatL2(d)
        flat.add(x)
        xs, ids, off = ix._lists()
        max_len = int(ix._sizes.max())
        for nprobe in (8, 32):
            ix.nprobe = nprobe
            _, sample_probes = quant._search_device(qall[:100].contiguous(), nprobe, need_distances=False)
            rad = radii(qall[:100], xs, off, sample_probes, ip, (10, 100, 1000))
            for nq in (1, 10_000):
                q = qall[:nq].contiguous()
                _, probes = quant._search_device(q, nprobe, need_distances=False)
                probe_ms = timed(lambda: quant._search_device(q, nprobe, need_distances=False), args.warmup, args.reps)
                for target, radius in rad.items():
                    range_ms = timed(lambda: ix.range_search(q, radius), args.warmup, args.reps)
                    call_ms = timed(lambda: ops.ivfflat_range_search(q, xs, ids, off, max_len, probes, metric, radius),
                                    args.warmup, args.reps)
                    split = kernel_split(lambda: ops.ivfflat_range_search(q, xs, ids, off, max_len, probes, metric,
                                                                          radius))
                    lims, _, _ = ix.range_search(q, radius)
                    per_query = int(lims[-1]) / nq
                    k = int(min(128, max(1, round(per_query))))
                    search_ms = timed(lambda: ix.search(q, k), args.warmup, args.reps)
                    flat_ms = timed(lambda: flat.range_search(q, radius), args.warmup, args.reps)
                    lf, _, _ = flat.range_search(q, radius)
                    run = dict(shape=shape, d=d, metric="IP" if ip else "L2", nlist=nlist, nq=nq, nprobe=nprobe,
                               target_per_query=target, radius=radius, results_per_query=per_query,
                               flat_results_per_query=int(lf[-1]) / nq, probe_ms=probe_ms, range_call_ms=call_ms,
                               range_search_ms=range_ms, kernel_ms=split, search_k=k, ivf_search_ms=search_ms,
                               ratio_to_ivf_search=range_ms / search_ms, flat_range_search_ms=flat_ms,
                               ratio_to_flat_range=range_ms / flat_ms)
                    res["runs"].append(run)
                    print(json.dumps(run), flush=True)
        del ix, flat, x, xs, ids, off, quant
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
