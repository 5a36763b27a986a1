"""IndexBinaryFlat on one GPU: Hamming kNN and range search over random packed codes, at the shapes its users run:

  ORB matching   1 M x 256-bit codes, nq in {500, 10 000}, k in {2, 10};
  BRISK          1 M x 512-bit codes, nq 10 000, k = 2;
  dHash          10 M x 64-bit codes, nq in {1, 10 000}, k = 10, and range search with radius 10.

As context, one row times what users do today: the same ORB codes as 32-D uint8 rows in IndexFlatL2 (a different metric,
not a like-for-like comparison).

Times are CUDA events around whole calls, median of --reps after --warmup: `call_ms` is ops.binary_knn /
ops.binary_range_search on padded device rows (the kernels plus their workspace), `index_ms` is the faiss_compat call
with a CUDA tensor (adds the query padding copy).  Rates come from the shapes: query pairs per second = nq * ntotal /
call time; compared code bytes per second = nq * ntotal * code_size / call time; database bytes per second = one pass
over the stored rows (ntotal * pitch) / call time.  The stored rows of the ORB (32 MB) and BRISK (64 MB) databases fit in
the 126 MB L2 and are read from there after the first pass; the dHash rows (160 MB with the 16-byte pitch) do not.
The card's name, power limit and max SM clock are read in the same run.  Writes JSON to --out.
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


def codes(n, code_size, g):
    return torch.randint(0, 256, (n, code_size), generator=g, device="cuda", dtype=torch.uint8)


def rates(nq, ntotal, code_size, ms):
    s = ms / 1e3
    return dict(pairs_per_s=nq * ntotal / s, compared_code_bytes_per_s=nq * ntotal * code_size / s,
                db_bytes_per_s=ntotal * ops.binary_pitch(code_size) / s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=str(Path(__file__).resolve().parent / "r03_microbench_binary.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "runs": []}
    g = torch.Generator(device="cuda").manual_seed(1234)
    shapes = (("orb", 256, 1_000_000, ((500, 2), (500, 10), (10_000, 2), (10_000, 10)), None),
              ("brisk", 512, 1_000_000, ((10_000, 2),), None),
              ("dhash", 64, 10_000_000, ((1, 10), (10_000, 10)), 10))
    for name, d, ntotal, searches, radius in shapes:
        cs = d // 8
        ix = fc.IndexBinaryFlat(d)
        ix.add(codes(ntotal, cs, g))
        db = ix._database()
        qall = codes(10_000, cs, g)
        for nq, k in searches:
            q = qall[:nq].contiguous()
            qp = torch.zeros((nq, ops.binary_pitch(cs)), dtype=torch.uint8, device="cuda")
            qp[:, :cs] = q
            call_ms = timed(lambda: ops.binary_knn(qp, db, cs, k), args.warmup, args.reps)
            index_ms = timed(lambda: ix.search(q, k), args.warmup, args.reps)
            run = dict(shape=name, op="search", d=d, ntotal=ntotal, nq=nq, k=k, call_ms=call_ms, index_ms=index_ms,
                       **rates(nq, ntotal, cs, call_ms))
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
            if radius is not None:
                call_ms = timed(lambda: ops.binary_range_search(qp, db, cs, radius), args.warmup, args.reps)
                index_ms = timed(lambda: ix.range_search(q, radius), args.warmup, args.reps)
                lims, _, _ = ops.binary_range_search(qp, db, cs, radius)
                run = dict(shape=name, op="range_search", d=d, ntotal=ntotal, nq=nq, radius=radius,
                           results_per_query=int(lims[-1]) / nq, call_ms=call_ms, index_ms=index_ms,
                           **rates(nq, ntotal, cs, call_ms))
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
        if name == "orb":
            # context: the same codes as 32-D uint8 rows in the float L2 index (not Hamming distances)
            flat = fc.IndexFlatL2(cs)
            flat.add(db[:, :cs].contiguous())
            for nq, k in ((500, 2), (10_000, 2)):
                q = qall[:nq].contiguous()
                ms = timed(lambda: flat.search(q, k), args.warmup, args.reps)
                run = dict(shape="orb_as_uint8_rows_in_IndexFlatL2", op="search", metric="L2 over 32-D uint8 rows "
                           "(different metric, context only)", d=cs, ntotal=ntotal, nq=nq, k=k, index_ms=ms,
                           pairs_per_s=nq * ntotal / (ms / 1e3))
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
            del flat
        del ix, db, qall
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
