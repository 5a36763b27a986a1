"""The C2 step with the histogram matrix cleared beside the assign (BOVW.histograms_device: clear kernel on a side
stream while the assign runs, then the histogram writes only the non-zero bins) against the step it replaced (assign,
then the dense histogram writing all 328 MB).  Inputs are bench.py's seeded C2 inputs (rank 0).

Timing: the two steps alternate, --rounds rounds of --steps steps each (the first arm swaps every round), CUDA events
around each round; median, min, max and spread (max - min) of ms per step for each, and of the per-round difference.
Then, each on its own: the assign, the clear, the dense histogram and the zeroed histogram (the matrix cleared
outside the timed window before every launch), float64 and float32 rows; these include the host's launch latency,
since the device is idle before each launch.  --trace DIR instead makes one torch.profiler run of a few new steps
(CUDA activities), writes the trace under DIR and reports whether each clear kernel ran inside the fused assign's
span.  The card's name, power limit and max SM clock are read in the same run.

usage: python profiles/microbench_hist_zeroed.py [--rounds 9] [--steps 10] [--out FILE.json] [--trace DIR]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from bench import C2, sift_like  # noqa: E402
from image_search_engine_b200 import BOVW, FaissKMeans, ops  # noqa: E402
from image_search_engine_b200 import bag_of_visual_words as bv  # noqa: E402
from image_search_engine_b200.bag_of_visual_words import PackedDescriptions  # noqa: E402
from image_search_engine_b200.utils import OkapiTransformer  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name(0)


def stats(v):
    return dict(median=statistics.median(v), min=min(v), max=max(v), spread=max(v) - min(v), n=len(v))


def events_ms(fn, reps, before=None):
    """ms per call of fn from CUDA events around each call; `before` runs outside the timed window"""
    out = []
    for _ in range(reps):
        if before is not None:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        out.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out")
    ap.add_argument("--trace", metavar="DIR")
    args = ap.parse_args()

    dev = ops.require_cuda()
    rng = np.random.default_rng(2)
    X = torch.from_numpy(sift_like(rng, C2["n_desc"], C2["d"])).to(dev)
    offsets = np.arange(0, C2["n_desc"] + 1, C2["per_img"], dtype=np.int64)
    off = torch.from_numpy(offsets).to(dev)
    km = FaissKMeans(C2["k"], n_init=1, max_iter=2)
    km.fit(X)
    bovw = BOVW(None, n_clusters=C2["k"])
    bovw.clusterer = km
    okapi = OkapiTransformer()
    packed = PackedDescriptions(X, offsets)
    hist_kw = dict(okapi=True, k1=okapi.k1, k2=okapi.k2, b=okapi.b)

    def old_step():
        # the parent's histograms_device: offsets to the device, assign, dense histogram into a fresh matrix
        o = torch.from_numpy(offsets).to(dev, non_blocking=True)
        return ops.bovw_histogram(km.transform_device(X), o, C2["k"], **hist_kw)

    def new_step():
        return bovw.histograms_device(packed, okapi=okapi)

    same = bool(torch.equal(old_step(), new_step()))
    for _ in range(3):
        old_step()
        new_step()
    torch.cuda.synchronize()

    if args.trace:
        from torch.profiler import ProfilerActivity, profile
        Path(args.trace).mkdir(parents=True, exist_ok=True)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                new_step()
            torch.cuda.synchronize()
        path = Path(args.trace) / "hist_zeroed_c2.pt.trace.json"
        prof.export_chrome_trace(str(path))
        kern = [e for e in json.loads(path.read_text())["traceEvents"] if e.get("cat") == "kernel"]
        assign = sorted((e for e in kern if "gemm_select_kernel" in e["name"]),   # the longest launch of each step
                        key=lambda e: -e["dur"])[:3]
        assign.sort(key=lambda e: e["ts"])
        clears = sorted((e for e in kern if "clear_kernel" in e["name"]), key=lambda e: e["ts"])
        hists = sorted((e for e in kern if "histogram_warp_kernel" in e["name"]), key=lambda e: e["ts"])
        rows = []
        for a, c, h in zip(assign, clears, hists):
            rows.append(dict(assign_us=a["dur"], clear_us=c["dur"], hist_us=h["dur"],
                             clear_starts_after_assign_us=c["ts"] - a["ts"],
                             clear_ends_before_assign_end_us=(a["ts"] + a["dur"]) - (c["ts"] + c["dur"]),
                             clear_inside_assign=bool(c["ts"] >= a["ts"] and c["ts"] + c["dur"] <= a["ts"] + a["dur"])))
        res = dict(card=card(), trace=str(path), outputs_equal=same, steps=rows)
        print(json.dumps(res, indent=1))
        return

    rounds = {"old": [], "new": []}
    for r in range(args.rounds):
        for name in (("old", "new") if r % 2 == 0 else ("new", "old")):
            fn = old_step if name == "old" else new_step
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            rounds[name].append(e0.elapsed_time(e1) / args.steps)
    diff = [o - n for o, n in zip(rounds["old"], rounds["new"])]

    words = km.transform_device(X)
    buf = torch.empty((C2["n_img"], C2["k"]), dtype=torch.float64, device=dev)
    buf32 = torch.empty((C2["n_img"], C2["k"]), dtype=torch.float32, device=dev)
    alone = dict(
        assign=stats(events_ms(lambda: km.transform_device(X), 20)),
        clear_unpaced=stats(events_ms(lambda: ops.clear_(buf), 20)),
        clear_paced=stats(events_ms(lambda: ops.clear_(buf, bv._CLEAR_GB_PER_S), 20)),
        hist_dense=stats(events_ms(lambda: ops.bovw_histogram(words, off, C2["k"], out=buf, **hist_kw), 20)),
        hist_zeroed=stats(events_ms(lambda: ops.bovw_histogram(words, off, C2["k"], out=buf, zeroed=True, **hist_kw), 20,
                                    before=lambda: ops.clear_(buf))),
        hist_dense_f32=stats(events_ms(lambda: ops.bovw_histogram(words, off, C2["k"], out=buf32, out_dtype=torch.float32,
                                                                  **hist_kw), 20)),
        hist_zeroed_f32=stats(events_ms(lambda: ops.bovw_histogram(words, off, C2["k"], out=buf32, out_dtype=torch.float32,
                                                                   zeroed=True, **hist_kw), 20,
                                        before=lambda: ops.clear_(buf32))))
    res = dict(card=card(), outputs_equal=same, rounds=args.rounds, steps_per_round=args.steps,
               ms_per_step=dict(old_assign_then_dense=stats(rounds["old"]), new_clear_beside_assign=stats(rounds["new"]),
                                old_minus_new=stats(diff)),
               per_round_ms=rounds, alone_ms=alone,
               mdesc_per_s=dict(old=C2["n_desc"] / statistics.median(rounds["old"]) / 1e3,
                                new=C2["n_desc"] / statistics.median(rounds["new"]) / 1e3))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
