"""Range search on the flat index: phase times, throughput, ratio to top-k search and a sampled oracle parity check.

Shapes: C3 (1 M x 2048 IP, 10 k queries) and one C5 shard (1.25 M x 512 IP, 10 k queries); radii from score quantiles of
a query sample so that the mean result count per query is about 10, 100 and 1000.  Phases (CUDA events): seed, first
collect, exact filter (count), overflow re-run (collect + count of the rows beyond the first cap), lims + fill + sort.

    python profiles/microbench_range.py [--out profiles/r03_microbench_range.json] [--shapes c3,c5]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

SHAPES = {"c3": (1_000_000, 2048), "c5": (1_250_000, 512)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the name from torch still identifies the card
        return dict(gpu=torch.cuda.get_device_name(), power_limit=f"unknown ({e})")


def phases(q, a, db, b, radius):
    """ops.range_search's steps one by one, each between CUDA events (same calls, same order)."""
    from image_search_engine_b200 import _lib, ops
    from image_search_engine_b200.ops import _ptr, _stream
    lib, ctx = _lib.load(), _lib.ctx(q.device.index or 0)
    nq, cap = a.n, ops.RANGE_CAP
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    ev[0].record()
    seed = torch.empty((nq,), dtype=torch.float32, device=q.device)
    _lib.check(lib.ise_range_seed(ctx, _ptr(a.meta), _ptr(a.norms), _ptr(a.row_inv), _ptr(b.meta), nq, a.d, 0,
                                  float(radius), _ptr(seed), _stream()))
    ev[1].record()
    cv, ci, rc = ops.gemm_collect(a.hi_only(), b.hi_only(), 0, seed, cap)
    ev[2].record()
    kept = torch.empty((nq + 1,), dtype=torch.int64, device=q.device)
    _lib.check(lib.ise_range_count(ctx, _ptr(q), 0, q.stride(0), _ptr(db), db.stride(0), nq, db.shape[0], a.d, 0,
                                   float(radius), 0, _ptr(a.norms), _ptr(b.norms), cap, _ptr(rc), _ptr(cv), _ptr(ci),
                                   _ptr(kept), _stream()))
    ev[3].record()
    rc_h = rc.cpu().numpy().astype(np.int64)
    over = np.nonzero(rc_h > cap)[0]
    reruns = []
    t_over = 0.0
    if over.size:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sel = torch.from_numpy(over).to(q.device)
        cap2 = int(rc_h[over].max())
        cv2, ci2, rc2, kept2 = ops._range_candidates(q.index_select(0, sel), db, a.rows(sel), b, 0, float(radius),
                                                     seed.index_select(0, sel), cap2, 0)
        kept.index_copy_(0, sel, kept2[:-1])
        reruns.append((sel, cap2, rc2, cv2, ci2))
        e1.record()
        e1.synchronize()
        t_over = e0.elapsed_time(e1)
    ev[4].record()
    lims = ops._range_lims(kept, nq)
    total = int(lims[nq].item())
    D = torch.empty((total,), dtype=torch.float32, device=q.device)
    I = torch.empty((total,), dtype=torch.int64, device=q.device)
    ops._range_fill(nq, cap, rc, cv, ci, None, lims, D, I)
    for sel, c2, r2, v2, i2 in reruns:
        ops._range_fill(sel.numel(), c2, r2, v2, i2, sel, lims, D, I)
    ws = torch.empty((int(lib.ise_range_sort_workspace_bytes(ctx, nq, total)),), dtype=torch.uint8, device=q.device)
    _lib.check(lib.ise_range_sort(ctx, nq, _ptr(lims), total, _ptr(D), _ptr(I), _ptr(ws), ws.numel(), _stream()))
    ev[5].record()
    ev[5].synchronize()
    return dict(ms_seed=ev[0].elapsed_time(ev[1]), ms_collect=ev[1].elapsed_time(ev[2]),
                ms_count=ev[2].elapsed_time(ev[3]), ms_overflow_rerun=t_over,
                ms_lims_fill_sort=ev[4].elapsed_time(ev[5]),
                candidates_per_query=float(np.minimum(rc_h, cap).sum() + rc_h[over].sum()) / nq,
                overflow_rows=int(over.size), results=total)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps, out


def run_shape(name, nq, reps, sample):
    from image_search_engine_b200 import faiss_compat, ops
    from oracle import faiss_shim as fs
    from tests._range_oracle import range_search
    n, d = SHAPES[name]
    dev = ops.require_cuda()
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    db = torch.randn((n, d), generator=gen, device=dev)
    db /= db.norm(dim=1, keepdim=True)
    # queries near database rows (so that near neighbours exist, like an image-search workload)
    q = db[torch.randint(0, n, (nq,), generator=gen, device=dev)] + 0.7 * torch.randn((nq, d), generator=gen,
                                                                                         device=dev) / d ** 0.5
    q /= q.norm(dim=1, keepdim=True)
    index = faiss_compat.IndexFlatIP(d)
    index.add(db)
    b = index._operand()
    a = ops.prepare_operand(q, rows=True)
    # radii: quantiles of the scores of 64 queries against the whole database
    s = torch.empty((64, n), dtype=torch.float32, device=dev)
    ops._lib.check(ops._lib.load().ise_pair_scores(ops._lib.ctx(dev.index or 0), ops._ptr(q[:64].contiguous()), 64,
                                                   ops._ptr(db), n, d, 0, ops._ptr(s), ops._stream()))
    s_sorted = torch.sort(s, dim=1, descending=True).values
    dbh = db.cpu().numpy()
    out = []
    for per_query in (10, 100, 1000):
        radius = float(s_sorted[:, per_query - 1].mean())
        ms_total, (lims, D, I) = timed(lambda: index.range_search(q, radius), reps)
        st = ops.search_stats()
        ph = phases(q, a, db, b, radius)
        k = min(100, max(1, int(round(float(lims[-1]) / nq))))
        ms_search, _ = timed(lambda: index.search(q, k), reps)
        # sampled oracle parity: `sample` queries against the full database (FP32 BLAS regime of the oracle)
        rows = np.random.default_rng(0).choice(nq, sample, replace=False)
        qh = q[torch.from_numpy(rows).to(dev)].cpu().numpy()
        lr, Dr, Ir = range_search(qh, dbh, radius, fs.METRIC_INNER_PRODUCT)
        lims_h, I_h = lims.cpu().numpy(), I.cpu().numpy()
        mism = 0
        for j, i in enumerate(rows):
            got = set(I_h[lims_h[i]:lims_h[i + 1]].tolist())
            want = set(Ir[int(lr[j]):int(lr[j + 1])].tolist())
            mism += len(got ^ want)
        res = dict(shape=name, n=n, d=d, nq=nq, radius=radius, target_per_query=per_query,
                   results_per_query=float(lims[-1]) / nq, ms_total=ms_total, queries_per_s=nq / ms_total * 1e3,
                   results_per_s=float(lims[-1]) / ms_total * 1e3, stats=st, phases=ph,
                   search_k=k, ms_search_k=ms_search, ratio_to_search=ms_total / ms_search,
                   oracle_sample_queries=sample, oracle_id_differences=mism)
        print(json.dumps(res), flush=True)
        out.append(res)
    del index, db, q, a, b
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r03_microbench_range.json")
    ap.add_argument("--shapes", default="c3,c5")
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sample", type=int, default=100)
    args = ap.parse_args()
    t0 = time.time()
    res = dict(**gpu_info(), rows=[])
    for name in args.shapes.split(","):
        res["rows"] += run_shape(name, args.nq, args.reps, args.sample)
    res["wall_s"] = time.time() - t0
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
