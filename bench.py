#!/usr/bin/env python
"""Headline benchmark of the B200 retrieval core (contract: see the task statement / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-knn] [--no-c4] [--no-c5]
                  [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input at BASELINE.json configs[1]
(C2): quantise 1,000,000 SIFT-like 128-D descriptors against a k=4096 codebook (fused tcgen05
assign), per-image BoVW histogram over 10,000 images and Okapi tf weighting.  The second half of the
metric (kNN QPS at 1M x 2048, top-10 = configs[2], C3) is measured in the same run and reported under
"knn".  N > 1: one process per GPU (torchrun), every rank quantises its own C2-sized shard of images
(no data-path collective, weak scaling) and holds its own 1M-row shard of the flat index.

The two configurations north_star shards across the box are on the same clock, at EVERY N, fixed global size
(strong scaling), each with a result check against the CPU oracle:
  "c4"  configs[3]: k-means over 10 M x 128 descriptors, k = 65 536: rows split over the ranks, one NCCL all-reduce of
        the [k*d | k] sums/counts buffer per iteration; per-iteration ms split into assign / update / all-reduce /
        finalize, all-reduce GB/s; parity = sampled rows re-assigned by oracle.faiss_shim.knn on the host + identical
        centroids on every rank.
  "c5"  configs[4]: flat IP index of 10 M x 512 vectors split over the ranks, 10 k queries, top-100: per-shard search,
        all-to-all + on-device merge; QPS; parity = sampled queries searched by the oracle over EVERY shard on the host
        cores and merged (= the unsharded search).
"""
from __future__ import annotations

import os
import sys

if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must use every host core (read before NumPy loads)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(_v, None)

import argparse
import json
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

C2 = dict(n_desc=1_000_000, d=128, k=4096, n_img=10_000, per_img=100)
C3 = dict(nb=1_000_000, d=2048, nq=10_000, topk=10)
C4 = dict(n=10_000_000, d=128, k=65_536, centres=100_000, sigma=8.0, block=250_000)
C5 = dict(nb=10_000_000, d=512, nq=10_000, topk=100, block=250_000)
METRIC = "Mdescriptors/s for k-means assign+histogram"
WORKLOAD = ("C2: 1M SIFT-like 128-D float32 descriptors per GPU, k=4096 codebook, 10k images: quantise (assign) + "
            "BoVW histogram (numpy-compat) + Okapi tf")


def sift_like(rng, n, d):
    g = rng.standard_normal((n, d), dtype=np.float32)
    g *= g
    g *= (512.0 / np.linalg.norm(g, axis=1, keepdims=True)).astype(np.float32)
    np.rint(g, out=g)
    np.minimum(g, 255, out=g)
    return g


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j.get("bf16_tflops_sustained"),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def ncu_traffic(key):
    """Per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernels, from the committed
    ncu summary of the CURRENT code (profiles/r02_ncu_traffic.json, written by profiles/summarize_ncu.py); None when
    there is no capture for that kernel -- nothing is hard-coded here."""
    p = ROOT / "profiles" / "r02_ncu_traffic.json"
    if not p.exists():
        return None, "no ncu capture committed (profiles/r02_ncu_traffic.json missing)"
    j = json.loads(p.read_text())
    e = j.get(key)
    if not e:
        return None, f"profiles/r02_ncu_traffic.json has no entry '{key}'"
    return float(e["dram_bytes"]), f"profiles/r02_ncu_traffic.json['{key}']: {e.get('note', '')}"


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed regions, read through NVML from a thread of
    this process (pynvml).  Spawning `nvidia-smi -lms` instead was measured to slow host-side CUDA calls
    enough to distort millisecond-scale steps (profiles/r01_findings.md); pause() stops sampling for the
    host/PCIe-bound e2e legs."""

    def __init__(self, gpu_index, period_s=0.02):
        import threading
        self.mode = os.environ.get("ISE_BENCH_SAMPLER", "on")   # debugging aid: on | idle | off
        self.period = period_s
        self.rows = []
        self.active = threading.Event()
        self.quit = threading.Event()
        self.h = None
        self.err = None
        try:
            if self.mode == "off":
                raise RuntimeError("sampler disabled by ISE_BENCH_SAMPLER=off")
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ent = vis.split(",")[gpu_index].strip()
                phys = int(ent) if ent.isdigit() else None
            self.h = (pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None
                      else pynvml.nvmlDeviceGetHandleByUUID(ent))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover - depends on the box
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.quit.is_set():
            if self.active.is_set():
                try:
                    sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.rows.append((float(sm), float(pw), int(rs)))
                except Exception as e:  # pragma: no cover
                    self.err = repr(e)
            time.sleep(self.period)

    def start(self):
        if self.mode == "on":
            self.active.set()

    def pause(self):
        self.active.clear()

    def stop(self):
        self.pause()
        self.quit.set()
        if self.h is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        reasons = sorted(n for n, bit in names.items() if any(r[2] & bit for r in self.rows))
        pmax = max(r[1] for r in self.rows)
        load = [r[0] for r in self.rows if r[1] >= 0.5 * pmax] or [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": self.sm_max, "reasons": reasons,
                "samples": len(self.rows), "power_w_max": pmax, "source": "NVML, 20 ms period, device-timed regions"}


# ----------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference loops; also the cpu_baseline leg of the GPU arm)
# ----------------------------------------------------------------------------------------------
def use_all_host_cores():
    """BLAS threads = every core this process may run on, whatever OMP_NUM_THREADS said when NumPy loaded (torchrun
    sets it to 1).  Returns the thread count actually in force."""
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        ncpu = os.cpu_count() or 1
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=ncpu)        # stays in force for the rest of the process
        n = max([p.get("num_threads", 1) for p in threadpoolctl.threadpool_info()] or [1])
    except Exception:  # pragma: no cover
        n = ncpu
    return int(n)


def cpu_assign_histogram(n_img_sample, seed=2, reps=1):
    """Times the reference's per-image quantise + np.histogram + Okapi loop on `n_img_sample` images."""
    from oracle import cpu_baseline, faiss_shim
    rng = np.random.default_rng(seed)
    X = sift_like(rng, n_img_sample * C2["per_img"], C2["d"])
    cent = X[rng.choice(X.shape[0], C2["k"], replace=X.shape[0] < C2["k"])].copy()
    faiss_shim.normalize_L2(cent)
    index = cpu_baseline.codebook_index(cent)
    descs = [X[i * C2["per_img"]:(i + 1) * C2["per_img"]] for i in range(n_img_sample)]
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_baseline.assign_histogram_step(index, descs, C2["k"])
        best = min(best, time.perf_counter() - t0)
    return X.shape[0] / best / 1e6, best


def cpu_knn(nb_sample, nq_sample, seed=3):
    from oracle import cpu_baseline
    rng = np.random.default_rng(seed)
    db = np.maximum(rng.standard_normal((nb_sample, C3["d"]), dtype=np.float32), 0)
    db /= np.linalg.norm(db, axis=1, keepdims=True)
    q = db[rng.integers(0, nb_sample, nq_sample)] + 0.05 * rng.standard_normal((nq_sample, C3["d"]), dtype=np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    t0 = time.perf_counter()
    cpu_baseline.flat_search(db, q.astype(np.float32), C3["topk"], "ip")
    dt = time.perf_counter() - t0
    # flat search cost is linear in nb: QPS at the full 1M-row index = sample QPS * nb_sample / nb
    return nq_sample / dt * (nb_sample / C3["nb"]), dt


def run_reference(args):
    """The reference's CPU implementation of the step (oracle port: no faiss wheel exists here) on ALL host cores, on
    the SAME configuration as our arm: every step is the full C2 batch (10,000 images x 100 descriptors, ~3 s)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = use_all_host_cores()
    n_img = C2["n_img"]
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt = cpu_assign_histogram(n_img)
        if i >= args.warmup:
            vals.append((v, dt))
        if sum(d for _, d in vals) > 150:      # bounded: the run must end within a few minutes whatever K says
            break
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([d for _, d in vals]) * 1e3)
    sample = (f"all {n_img} images x {C2['per_img']} descriptors per step (the full C2 batch), "
              f"per-image Faiss-shim search + np.histogram + Okapi, NumPy/OpenBLAS on {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mdescriptors/s", "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mdescriptors/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mdescriptors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_knn:
        q, dt = cpu_knn(200_000, 1000)
        line["knn"] = {"metric": "kNN QPS at 1M x 2048 top-10", "value": q, "unit": "queries/s",
                       "sample": "200k of 1M DB rows x 1000 of 10k queries (%.1f s), scaled linearly in nb" % dt}
    emit(line)


# ----------------------------------------------------------------------------------------------
# C4 / C5 data: a deterministic function of the GLOBAL row index (fixed 250k-row blocks, one seed per block), so the
# matrix is the same whatever the number of ranks it is split over
# ----------------------------------------------------------------------------------------------
def _block_range(n, block, rank, world):
    nblk = n // block
    assert nblk % world == 0, "global size must split into whole blocks per rank"
    per = nblk // world
    return rank * per, (rank + 1) * per


def c4_rows(torch, dev, rank, world):
    g = torch.Generator(device=dev)
    g.manual_seed(4)                                   # the same centre table on every rank
    centres = torch.randn((C4["centres"], C4["d"]), generator=g, device=dev).square_()
    centres *= 512.0 / centres.norm(dim=1, keepdim=True)
    b0, b1 = _block_range(C4["n"], C4["block"], rank, world)
    x = torch.empty(((b1 - b0) * C4["block"], C4["d"]), dtype=torch.float32, device=dev)
    for b in range(b0, b1):
        g.manual_seed(4000 + b)
        blk = x[(b - b0) * C4["block"]:(b - b0 + 1) * C4["block"]]
        pick = torch.randint(0, C4["centres"], (C4["block"],), generator=g, device=dev)
        torch.index_select(centres, 0, pick, out=blk)
        blk.add_(torch.randn((C4["block"], C4["d"]), generator=g, device=dev), alpha=C4["sigma"])
        blk.round_().clamp_(0, 255)
    return x


def c5_rows(torch, dev, rank, world, ops):
    b0, b1 = _block_range(C5["nb"], C5["block"], rank, world)
    db = torch.empty(((b1 - b0) * C5["block"], C5["d"]), dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev)
    for b in range(b0, b1):
        g.manual_seed(5000 + b)
        db[(b - b0) * C5["block"]:(b - b0 + 1) * C5["block"]].normal_(generator=g)
    ops.normalize_l2_(db)
    return db, b0 * C5["block"]


def run_c4(args, torch, dist, dev, rank, world, barrier, max_over_ranks, ops, P):
    from image_search_engine_b200._lib import METRIC_IP
    from image_search_engine_b200.parallel import ShardedKmeans
    x = c4_rows(torch, dev, rank, world)
    n_local = int(x.shape[0])
    iters = args.c4_iters
    km = ShardedKmeans(C4["d"], C4["k"], seed=42, niter=iters, spherical=True)
    if world > 1:
        warm = torch.ones(1 << 20, device=dev)
        for _ in range(3):
            dist.all_reduce(warm)                      # communicator set-up is not part of the k-means time
    barrier()
    t0 = time.perf_counter()
    km.train(x)
    torch.cuda.synchronize()
    s_total = max_over_ranks((time.perf_counter() - t0) * 1e3) / 1e3
    st = km.iteration_stats
    phases = {p_: [s[p_] for s in st] for p_ in ("ms_assign", "ms_accumulate", "ms_allreduce", "ms_finalize_host")}
    # per-iteration time = the four phases of the slowest rank; steady = iterations after the first two (their
    # empty-cluster split plans are a start-up effect of the random initialisation)
    it_ms = [max_over_ranks(sum(phases[p_][i] for p_ in phases)) for i in range(iters)]
    steady = it_ms[2:] or it_ms
    ar_bytes = 4 * (C4["k"] * C4["d"] + C4["k"]) + 8
    ar_ms = [max_over_ranks(v) for v in phases["ms_allreduce"]]
    ar_steady = float(np.median(ar_ms[1:] or ar_ms))
    as_ms = [max_over_ranks(v) for v in phases["ms_assign"]]            # collectives: every rank takes part
    a_ms = float(np.median(as_ms[1:] or as_ms))
    # the collective on its own: the per-iteration figure above (event after the update -> event after the all-reduce)
    # also contains the time this rank WAITS for the slowest rank's assign to finish (rank skew), which is what made the
    # round-1 numbers look erratic (0.3 - 3.6 ms for the same 33.8 MB); here: same buffer size, ranks aligned by a barrier
    ar_pure = None
    if world > 1:
        buf = torch.zeros((C4["k"] * C4["d"] + C4["k"],), dtype=torch.float32, device=dev)
        for _ in range(2):
            dist.all_reduce(buf)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            dist.all_reduce(buf)
        e1.record()
        torch.cuda.synchronize()
        ar_pure = max_over_ranks(e0.elapsed_time(e1) / 5)
        del buf
    # ---- parity: (1) every rank ends with bit-identical centroids (the finalize is deterministic, no broadcast);
    #      (2) >= 256 sampled rows of this rank re-assigned by the oracle against the trained 65 536-centroid codebook
    cent = torch.from_numpy(km.centroids).to(dev)
    spread = 0.0
    if world > 1:
        ref = cent.clone()
        dist.broadcast(ref, src=0)
        dmax = (cent - ref).abs().max().reshape(1)
        dist.all_reduce(dmax, op=dist.ReduceOp.MAX)
        spread = float(dmax.item())
    parity = None
    if rank == 0:
        from oracle import faiss_shim as fs
        from tests._util import assert_topk_parity
        g = torch.Generator(device=dev)
        g.manual_seed(44)
        rows = torch.randperm(n_local, generator=g, device=dev)[:256]
        xs = x[rows].contiguous()
        _, got = km.index._search_device(xs, 1)          # nq >= 20: the tensor-core assign at k = 65 536
        xs_h = xs.cpu().numpy()
        _, want = fs.knn(xs_h, km.centroids, 1, fs.METRIC_INNER_PRODUCT)
        try:
            near = assert_topk_parity(got.cpu().numpy(), want, xs_h, km.centroids, True, max_mismatch_frac=0.02)
            ok, why = True, ""
        except AssertionError as e:  # pragma: no cover - a parity failure must show up in the line, not kill the bench
            near, ok, why = -1, False, str(e)[:300]
        obj = [float(o) for o in km.obj]
        parity = {"ok": bool(ok and spread == 0.0 and all(b >= a * (1 - 1e-6) for a, b in zip(obj, obj[1:]))),
                  "rows_checked_vs_oracle": 256, "near_tie_rows": near, "error": why,
                  "centroid_max_abs_diff_across_ranks": spread, "objective_non_decreasing": obj,
                  "check": "oracle.faiss_shim.knn (host) on 256 sampled rows vs the trained codebook; centroids "
                           "bit-identical on every rank; spherical objective non-decreasing"}
    out = None
    if rank == 0:
        flops = 2.0 * C4["n"] * C4["k"] * C4["d"]
        out = {"config": "C4: k-means, 10M x 128 SIFT-like descriptors (100k-component mixture), k = 65536, spherical, "
                         f"{iters} iterations, rows split over {world} rank(s)", "scaling": "strong",
               "n": C4["n"], "d": C4["d"], "k": C4["k"], "iters": iters, "s_total_incl_setup": s_total,
               "ms_per_iter": it_ms, "ms_per_iter_steady": float(np.median(steady)),
               "phases_ms_rank0": {p_: [round(v, 3) for v in phases[p_]] for p_ in phases},
               "nsplit": [s["nsplit"] for s in st],
               "allreduce": {"bytes_per_iter": ar_bytes, "ms_in_loop_incl_rank_skew": ar_ms,
                             "ms_in_loop_steady": ar_steady, "ms_collective_alone": ar_pure,
                             "algbw_gbs": (ar_bytes / (ar_pure * 1e-3) / 1e9) if ar_pure else None,
                             "busbw_gbs": (ar_bytes * 2 * (world - 1) / world / (ar_pure * 1e-3) / 1e9) if ar_pure else None},
               "Mdescriptors_per_s_steady": C4["n"] / (float(np.median(steady)) * 1e-3) / 1e6,
               "assign_roofline": {"bound": "tensor", "achieved": flops / world / (a_ms * 1e-3) / 1e12, "peak": P["tf_burst"],
                                   "unit": "TFLOP/s per GPU", "frac": flops / world / (a_ms * 1e-3) / 1e12 / P["tf_burst"],
                                   "ms_assign_steady": a_ms},
               "parity": parity}
    del x, km
    torch.cuda.empty_cache()
    return out


def run_c5(args, torch, dist, dev, rank, world, barrier, max_over_ranks, ops, P):
    from image_search_engine_b200._lib import METRIC_IP
    from image_search_engine_b200.parallel import ShardedIndexFlat
    db, base = c5_rows(torch, dev, rank, world, ops)
    nb_local = int(db.shape[0])
    nq, d, topk = C5["nq"], C5["d"], C5["topk"]
    g = torch.Generator(device=dev)
    g.manual_seed(55)                                   # same picks / noise on every rank
    pick = torch.randint(0, C5["nb"], (nq,), generator=g, device=dev)
    q = torch.zeros((nq, d), dtype=torch.float32, device=dev)
    mine = (pick >= base) & (pick < base + nb_local)
    q[mine] = db[pick[mine] - base]
    if world > 1:
        dist.all_reduce(q)                              # every picked row is owned by exactly one rank
    q += 0.05 * torch.randn((nq, d), generator=g, device=dev)
    ops.normalize_l2_(q)
    idx = ShardedIndexFlat(d, METRIC_IP)
    idx.add_local(db)                                   # planes + norms + samples built once (index build, untimed)
    for _ in range(2):
        D, I = idx.search(q, topk)
    barrier()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        D, I = idx.search(q, topk)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / reps)
    stats = ops.search_stats()
    # ---- parity: 128 sampled queries, oracle search of EVERY shard on the host cores of its rank, merged on rank 0 with
    #      the canonical (score, id) order = the unsharded oracle search of the 10 M-row index
    from oracle import faiss_shim as fs
    cores = use_all_host_cores()
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=max(1, cores // world))   # the ranks share the host
    except Exception:  # pragma: no cover
        pass
    ns = 128
    gs = torch.Generator(device=dev)
    gs.manual_seed(56)
    rows = torch.randperm(nq, generator=gs, device=dev)[:ns]
    qs = q[rows].cpu().numpy()
    t_or = time.perf_counter()
    Dl = np.empty((ns, topk), np.float32)
    Il = np.empty((ns, topk), np.int64)
    run_s = run_i = None
    for s0 in range(0, nb_local, 1_250_000):             # slabs bound the host copy of the shard
        slab = db[s0:s0 + 1_250_000].cpu().numpy()
        ds, is_ = fs.knn(qs, slab, topk, fs.METRIC_INNER_PRODUCT, db_block=65536)
        is_ = is_ + (base + s0)
        if run_s is None:
            run_s, run_i = ds, is_
        else:
            cs, ci = np.concatenate([run_s, ds], 1), np.concatenate([run_i, is_], 1)
            order = np.lexsort((ci, -cs), axis=1)[:, :topk]
            run_s, run_i = np.take_along_axis(cs, order, 1), np.take_along_axis(ci, order, 1)
        del slab
    Dl[:], Il[:] = run_s, run_i
    if world > 1:
        Dg = [torch.empty((ns, topk), dtype=torch.float32, device=dev) for _ in range(world)]
        Ig = [torch.empty((ns, topk), dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(Dg, torch.from_numpy(Dl).to(dev))
        dist.all_gather(Ig, torch.from_numpy(Il).to(dev))
        cs = torch.cat(Dg, 1).cpu().numpy()
        ci = torch.cat(Ig, 1).cpu().numpy()
        order = np.lexsort((ci, -cs), axis=1)[:, :topk]
        Dl, Il = np.take_along_axis(cs, order, 1), np.take_along_axis(ci, order, 1)
    t_or = time.perf_counter() - t_or
    out = None
    if rank == 0:
        got_I, got_D = I[rows].cpu().numpy(), D[rows].cpu().numpy()
        diff_rows = int((got_I != Il).any(axis=1).sum())
        # near ties: positions where the ids differ must carry (FP32-)equal scores
        gap = np.abs(got_D - Dl)
        tol = 16 * float(np.finfo(np.float32).eps)      # unit vectors: |q||y| = 1
        ok = bool((gap[got_I != Il] <= tol).all()) and bool(np.allclose(got_D, Dl, rtol=1e-4, atol=1e-6))
        flops = 2.0 * nq * C5["nb"] * d
        out = {"config": f"C5: flat IP index, 10M x 512 unit vectors over {world} shard(s) of {nb_local} rows, 10k queries, "
                         "top-100: per-shard verified search (collect mode) + all-to-all + on-device merge",
               "scaling": "strong", "nb": C5["nb"], "d": d, "nq": nq, "topk": topk, "ms_per_batch": ms,
               "qps": nq / (ms * 1e-3), "search_stats_rank0": stats,
               "exchange_bytes_per_rank": getattr(idx, "last_exchange_bytes", 0),
               "roofline": {"bound": "tensor", "achieved": flops / world / (ms * 1e-3) / 1e12, "peak": P["tf_burst"],
                            "unit": "TFLOP/s per GPU (whole search incl. seed pre-pass, re-score, exchange, merge)",
                            "frac": flops / world / (ms * 1e-3) / 1e12 / P["tf_burst"]},
               "parity": {"ok": ok, "queries_checked_vs_oracle": ns, "rows_with_any_id_difference": diff_rows,
                          "max_abs_distance_diff": float(gap.max()), "oracle_s": t_or,
                          "check": "oracle.faiss_shim.knn over every shard on the host (each rank its own shard), merged "
                                   "with the canonical (score, id) order = unsharded oracle search of all 10M rows; id "
                                   "differences only where the scores are FP32-equal (tau = 16 eps), distances <= 1e-4"}}
    del db, idx
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
DUMP_ROWS = 1024         # image rows of the step's [10k x 4096] float64 result that --dump-outputs keeps: 32 MiB


def dump_outputs(out_dir, tf, codebook):
    """Writes what the last timed step returned, for comparing two builds output for output: the same DUMP_ROWS image
    rows (fixed seed, ascending) of the Okapi tf matrix, whose 328 MB are too many to keep whole, and the codebook the
    step quantised against.  The codebook is trained on the device during set-up, so a difference there explains a
    difference in the rows."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.default_rng(7).choice(tf.shape[0], DUMP_ROWS, replace=False))
    sample = tf.index_select(0, torch.from_numpy(rows).to(tf.device)).cpu().numpy()
    np.save(os.path.join(out_dir, "okapi_tf_rows.npy"), sample)
    np.save(os.path.join(out_dir, "codebook.npy"), np.asarray(codebook, dtype=np.float32))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from image_search_engine_b200 import BOVW, FaissKMeans, faiss_compat, ops
    from image_search_engine_b200._lib import METRIC_IP
    from image_search_engine_b200.bag_of_visual_words import PackedDescriptions

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = None
    if world > 1 and not os.environ.get("ISE_BENCH_NO_BIND"):
        from image_search_engine_b200.parallel import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local_rank)     # before any pinned allocation (first touch)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    P = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return float(ms)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- C2 inputs (per rank: its own shard of 10k images) ----------------
    rng = np.random.default_rng(2 + rank)
    X_host = sift_like(rng, C2["n_desc"], C2["d"])
    offsets = np.arange(0, C2["n_desc"] + 1, C2["per_img"], dtype=np.int64)
    packed = PackedDescriptions(X_host, offsets).pin()
    X_dev = packed.matrix.to(dev)
    off_dev = torch.from_numpy(offsets).to(dev)

    # codebook: 2 Lloyd iterations from the Faiss-style random init (untimed set-up)
    km = FaissKMeans(C2["k"], n_init=1, max_iter=2)
    km.fit(X_dev)
    bovw = BOVW(None, n_clusters=C2["k"])
    bovw.clusterer = km

    from image_search_engine_b200.utils import OkapiTransformer
    okapi = OkapiTransformer()

    # CUDA events around every gemm_select launch made inside the timed regions (roofline numerator)
    kernel_events = []
    _orig_gemm_select = ops.gemm_select

    def _timed_gemm_select(*a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = _orig_gemm_select(*a, **kw)
        e1.record()
        kernel_events.append((e0, e1))
        return r

    ops.gemm_select = _timed_gemm_select
    # the quantisation of raw float32 descriptors goes through the fused assign (row preparation inside the kernel)
    _orig_assign_fused = ops.assign_fused

    def _timed_assign_fused(*a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = _orig_assign_fused(*a, **kw)
        e1.record()
        if r is not None:
            kernel_events.append((e0, e1))
        return r

    ops.assign_fused = _timed_assign_fused
    packed_dev = PackedDescriptions(X_dev, offsets)

    def device_step():
        # the public device-resident path: prepare row planes (one pass) -> fused assign -> histogram + Okapi tf
        return bovw.histograms_device(packed_dev, okapi=okapi)

    for _ in range(args.warmup):
        device_step()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    l0 = ops.launches()
    kernel_events.clear()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for _ in range(args.steps - 1):
        device_step()
    last = device_step()
    t_end.record()
    barrier()
    launches = ops.launches() - l0
    ms_step = max_over_ranks(t_start.elapsed_time(t_end) / args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, km.cluster_centers_)
    del last
    # all gemm_select launches of a step (main launch + any fallback re-run) count towards the kernel time
    kern_ms = float(np.sum([a.elapsed_time(b) for a, b in kernel_events]) / args.steps)
    assign_stats = ops.search_stats()
    if assign_stats.get("mode") == "fused-verified":
        kernel_name = ("gemm_select_kernel<PA=1,PB=1,IP,top-1,VERIFY,CG=2,CONV,ARES>: one tcgen05 product per tile + per-row "
                       "proof of the winner (float32 -> FP16 plane conversion by converter warps inside the launch, row tile "
                       "resident in shared memory), then gather + split-product re-run of the flagged rows (all launches timed)")
        mma_products = 1.0 + 2.0 * assign_stats.get("fallback_rows", 0) / max(1, assign_stats.get("rows", 1))
    elif assign_stats.get("mode") == "fused-split":
        kernel_name = ("gemm_select_kernel<PA=1,PB=2,IP,top-1,CG=2,CONV> (fused assign: float32 -> FP16 plane conversion by "
                       "converter warps inside the launch)")
        mma_products = 2.0
    else:
        kernel_name, mma_products = "gemm_select_kernel<2,2,IP,1>", 2.0
    value = world * C2["n_desc"] / (ms_step * 1e-3) / 1e6

    # ---- parity of THIS step's result at full size: 2 000 sampled descriptors re-assigned by the oracle (host) ----
    step_parity = None
    if rank == 0:
        from oracle import faiss_shim as fs
        from tests._util import assert_topk_parity
        words_all = km.transform_device(X_dev)
        gp = torch.Generator(device=dev)
        gp.manual_seed(22)
        rows = torch.randperm(C2["n_desc"], generator=gp, device=dev)[:2000]
        xs = X_dev[rows].cpu().numpy()
        cent_h = km.cluster_centers_
        _, want = fs.knn(xs, cent_h, 1, fs.METRIC_INNER_PRODUCT)
        try:
            near = assert_topk_parity(words_all[rows].cpu().numpy().reshape(-1, 1), want, xs, cent_h, True,
                                      max_mismatch_frac=0.002)
            step_parity = {"ok": True, "rows_checked_vs_oracle": 2000, "near_tie_rows": near}
        except AssertionError as e:  # pragma: no cover
            step_parity = {"ok": False, "rows_checked_vs_oracle": 2000, "error": str(e)[:300]}
        del words_all

    # ---------------- the step's HBM-bound kernels, timed alone (explains the non-tensor share of the step) ----
    def _time(fn, reps=5):
        fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    words_dev = km.transform_device(X_dev)
    hist_out = torch.empty((C2["n_img"], C2["k"]), dtype=torch.float64, device=dev)
    accum = torch.zeros((C2["k"] * C2["d"] + C2["k"],), dtype=torch.float32, device=dev)
    a_sums, a_counts = accum[: C2["k"] * C2["d"]].view(C2["k"], C2["d"]), accum[C2["k"] * C2["d"]:]
    a_obj = torch.zeros((1,), dtype=torch.float64, device=dev)
    cent_dev = torch.from_numpy(km.cluster_centers_).to(dev)
    acc_ws = [None]

    def _acc():
        acc_ws[0] = ops.kmeans_accumulate_sorted(X_dev, words_dev, a_sums, a_counts, a_obj, centroids=cent_dev,
                                                 workspace=acc_ws[0])

    hbm_kernels = []
    for name, fn, nbytes in (
            # algorithmic = actual traffic now: every float read once, the one FP16 plane integer-valued descriptors
            # need written once, + norms and per-row scales
            ("prepare_rows_f32_kernel (single pass, per-row scales)", lambda: ops.prepare_operand(X_dev, rows=True),
             C2["n_desc"] * (C2["d"] * 6 + 8)),
            ("histogram_warp_kernel<double> (numpy-compat + Okapi)",
             lambda: ops.bovw_histogram(words_dev, off_dev, C2["k"], okapi=True, out=hist_out),
             C2["n_desc"] * 8 + C2["n_img"] * C2["k"] * 8),
            ("k-means update: count + scan + scatter + gather_reduce_kernel (training loop, not part of the step)", _acc,
             C2["n_desc"] * (4 * C2["d"] + 8))):
        ms = _time(fn)
        hbm_kernels.append({"kernel": name, "ms": ms, "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s",
                            "peak": P["hbm"], "frac": nbytes / (ms * 1e-3) / 1e9 / P["hbm"], "algorithmic_bytes": nbytes})
    del hist_out, words_dev, accum, cent_dev

    # ---------------- e2e: host descriptors -> host histogram matrix ----------------
    sampler.pause()   # clocks are sampled during the device-timed regions only (see ClockSampler.pause)
    bovw.descriptions = None

    def timed_host(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)

    # (1) the Pipeline-level call: pinned host descriptors -> scipy CSR float64 (histogram + Okapi tf), which is what
    #     the reference's pipeline.transform() returns (utils.py:153-202).  H2D chunks overlap the quantisation; the
    #     CSR arrays are built in HBM and come back in one small copy.
    csr_holder = {}

    def e2e_step_csr():
        csr_holder["m"] = bovw.transform_csr(packed, okapi=okapi, n_chunks=16, copy=False)

    # float32 on the wire (the copy the input format implies), then the library's own policy: with host cores to spare
    # it narrows integer-valued descriptors to uint8 block by block on host threads INSIDE the call (a quarter of the
    # PCIe bytes; same result); with many ranks sharing the host it keeps float32
    os.environ["ISE_NARROW_PINNED"] = "0"
    e2e_f32_ms = timed_host(e2e_step_csr)
    csr_f32 = csr_holder["m"].copy()
    os.environ.pop("ISE_NARROW_PINNED")
    e2e_ms = timed_host(e2e_step_csr)
    e2e_same = bool((csr_holder["m"] != csr_f32).nnz == 0)
    del csr_f32
    e2e_val = world * C2["n_desc"] / (e2e_ms * 1e-3) / 1e6
    e2e_transfer = dict(bovw.__dict__.get("_last_transfer", {}))
    h2d = int(e2e_transfer.get("h2d_bytes", X_host.nbytes + offsets.nbytes))     # what actually crossed PCIe
    h2d_f32 = int(X_host.nbytes + offsets.nbytes)
    d2h = int((C2["n_img"] + 1) * 4 + C2["n_desc"] * 12)       # indptr + (int32 index, float64 value) per descriptor slot
    csr_nnz = int(csr_holder["m"].nnz)
    assert csr_holder["m"].shape == (C2["n_img"], C2["k"]) and float(csr_holder["m"].sum()) > 0
    csr_ref = csr_holder["m"].copy()

    # the node's host -> device ceiling for this step's input, measured the same way: every rank copies its pinned
    # 512 MB at the same time, nothing else running (N >= 4 is bound by this, not by any kernel)
    h2d_buf = torch.empty(packed.matrix.shape, dtype=packed.matrix.dtype, device=dev)
    for _ in range(2):
        h2d_buf.copy_(packed.matrix, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        h2d_buf.copy_(packed.matrix, non_blocking=True)
    torch.cuda.synchronize()
    h2d_alone_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / 5)
    del h2d_buf

    # (2) the reference's OWN input contract: a Python LIST of 10,000 per-image arrays (descriptors.py:104-139) ->
    #     scipy CSR.  Packing (C list walk + multi-threaded copy into a persistent pinned buffer, uint8 on the wire
    #     because these SIFT values are integers <= 255) is INSIDE the timed region.
    desc_list = [X_host[i * C2["per_img"]:(i + 1) * C2["per_img"]] for i in range(C2["n_img"])]

    def e2e_step_list():
        csr_holder["l"] = bovw.transform_csr(desc_list, okapi=okapi, n_chunks=16, copy=False)

    e2e_list_ms = timed_host(e2e_step_list)
    same_as_packed = bool((csr_holder["l"] != csr_ref).nnz == 0)
    list_transfer = dict(bovw.__dict__.get("_last_transfer", {}))
    list_h2d = int(list_transfer.get("h2d_bytes", 0))
    del desc_list, csr_ref

    # (3) the same step with the reference's DENSE float64 matrix as the result (BOVW.transform's own format):
    #     H2D | kernels | D2H of 328 MB chunk-pipelined on three streams
    out_pin = torch.empty((C2["n_img"], C2["k"]), dtype=torch.float64, pin_memory=True)

    def e2e_step_dense():
        return bovw.histograms_host(packed, out_pin, okapi=okapi, n_chunks=16)

    e2e_dense_ms = timed_host(e2e_step_dense)
    d2h_dense = int(out_pin.numel() * 8)
    del out_pin

    # ---------------- k-means training (C2: k = 4096, 20 iterations) ----------------
    barrier()
    t0 = time.perf_counter()
    km2 = FaissKMeans(C2["k"], n_init=1, max_iter=20)
    km2.fit(X_dev)
    torch.cuda.synchronize()
    kmeans_fit_ms = (time.perf_counter() - t0) * 1e3
    kst = km2.kmeans.iteration_stats
    # whole fit / 20 (incl. the one-off row preparation, initialisation, final index build) and the steady iteration
    # (first and last iteration end with a synchronisation, so their time stamps are exact)
    kmeans_iter_ms = kmeans_fit_ms / 20
    kmeans_iter_steady_ms = (kst[-1]["time"] - kst[0]["time"]) * 1e3 / (len(kst) - 1)
    km_phases = {p_: float(np.median([s_[p_] for s_ in kst[1:]])) for p_ in ("ms_assign", "ms_accumulate")}
    km_phases["speculated_iterations"] = int(sum(1 for s_ in kst if s_.get("speculated")))
    km_phases["mis_speculated"] = int(sum(1 for s_ in kst if s_.get("mis_speculated")))
    km_phases["nsplit"] = [int(s_["nsplit"]) for s_ in kst]
    del km2

    # ---------------- C3: flat IP search, 1M x 2048 per rank, 10k queries, top-10 ----------------
    knn = None
    if not args.no_knn:
        g = torch.Generator(device=dev)
        g.manual_seed(3 + rank)
        db = torch.empty((C3["nb"], C3["d"]), dtype=torch.float32, device=dev)
        for i in range(0, C3["nb"], 100_000):
            blk = db[i:i + 100_000]
            blk.normal_(generator=g)
            blk.clamp_(min=0)
        ops.normalize_l2_(db)
        gq = torch.Generator(device=dev)
        gq.manual_seed(1003)  # same queries on every rank
        pick = torch.randint(0, C3["nb"], (C3["nq"],), generator=gq, device=dev)
        q = db[pick] + 0.05 * torch.randn((C3["nq"], C3["d"]), generator=gq, device=dev)
        if world > 1:
            dist.broadcast(q, src=0)
        ops.normalize_l2_(q)
        from image_search_engine_b200.parallel import ShardedIndexFlat
        sidx = ShardedIndexFlat(C3["d"], METRIC_IP)
        sidx.add_local(db)                      # planes + norms built once (index build, untimed)
        torch.cuda.synchronize()

        def knn_step(qd):
            # public sharded-index search: prepare(q) -> gemm_select top-10 -> exact re-score ->
            # [all-to-all + on-device merge of this rank's query slice + all-gather when world > 1]
            return sidx.search(qd, C3["topk"])

        ksteps = max(2, min(args.steps, 5))
        for _ in range(2):
            knn_step(q)
        barrier()
        sampler.start()
        kernel_events.clear()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(ksteps):
            D, I = knn_step(q)
        e.record()
        barrier()
        knn_ms = max_over_ranks(s.elapsed_time(e) / ksteps)
        # sample pre-pass + coarse main launch + split re-run of unproven rows, all tcgen05 gemm_select launches
        knn_kern_ms = float(np.sum([a.elapsed_time(b) for a, b in kernel_events]) / ksteps)
        knn_stats = ops.search_stats()
        sampler.pause()
        # self-check (size independent): every query's best hit is the row it was derived from (rank 0's shard)
        hit = float((I[:, 0] == pick).float().mean().item())
        # parity at full size (N = 1: the index IS the 1M x 2048 database): 200 sampled queries searched by the oracle
        # over the whole database on the host
        knn_parity = None
        if world == 1:
            from oracle import faiss_shim as fs
            from tests._util import assert_topk_parity
            gs = torch.Generator(device=dev)
            gs.manual_seed(33)
            rows = torch.randperm(C3["nq"], generator=gs, device=dev)[:200]
            qs = q[rows].cpu().numpy()
            run_s = run_i = None
            for s0 in range(0, C3["nb"], 250_000):
                slab = db[s0:s0 + 250_000].cpu().numpy()
                ds, is_ = fs.knn(qs, slab, C3["topk"], fs.METRIC_INNER_PRODUCT, db_block=65536)
                is_ = is_ + s0
                if run_s is None:
                    run_s, run_i = ds, is_
                else:
                    cs, ci = np.concatenate([run_s, ds], 1), np.concatenate([run_i, is_], 1)
                    order = np.lexsort((ci, -cs), axis=1)[:, :C3["topk"]]
                    run_s, run_i = np.take_along_axis(cs, order, 1), np.take_along_axis(ci, order, 1)
            gI, gD = I[rows].cpu().numpy(), D[rows].cpu().numpy()
            gap = np.abs(gD - run_s)
            okk = bool((gap[gI != run_i] <= 16 * float(np.finfo(np.float32).eps)).all()) and \
                bool(np.allclose(gD, run_s, rtol=1e-4, atol=1e-6))
            knn_parity = {"ok": okk, "queries_checked_vs_oracle": 200,
                          "rows_with_any_id_difference": int((gI != run_i).any(axis=1).sum()),
                          "max_abs_distance_diff": float(gap.max()),
                          "check": "oracle.faiss_shim.knn over the full 1M x 2048 database on the host"}
        # e2e: pinned host queries in, host (D, I) out
        q_pin = q.cpu().pin_memory()
        barrier()
        t0 = time.perf_counter()
        for _ in range(ksteps):
            qd = q_pin.to(dev, non_blocking=True)
            D, I = knn_step(qd)
            Dh, Ih = D.cpu(), I.cpu()
        torch.cuda.synchronize()
        knn_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / ksteps)
        flops = 2.0 * C3["nq"] * C3["nb"] * C3["d"]
        traffic, traffic_src = ncu_traffic("knn_coarse")
        knn = {
            "metric": "kNN QPS at 1M x 2048 top-10", "value": C3["nq"] / (knn_ms * 1e-3), "unit": "queries/s",
            "ms_per_step": knn_ms, "steps": ksteps, "nb_per_gpu": C3["nb"], "nb_total": C3["nb"] * world,
            "e2e": {"value": C3["nq"] / (knn_e2e_ms * 1e-3), "unit": "queries/s",
                    "h2d_bytes_per_step": int(q.numel() * 4), "d2h_bytes_per_step": int(C3["nq"] * C3["topk"] * 12)},
            "roofline": {"bound": "tensor", "achieved": flops / (knn_kern_ms * 1e-3) / 1e12, "peak": P["tf_burst"],
                         "unit": "TFLOP/s", "frac": flops / (knn_kern_ms * 1e-3) / 1e12 / P["tf_burst"],
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "gemm_select_kernel<1,1,IP,32> coarse (+ sample pre-pass, split re-run of unproven "
                                   "rows, topk_merge_kernel)", "kernel_ms": knn_kern_ms, "search": knn_stats,
                         "peak_source": P["src"] + ", bf16 burst"},
            "top1_self_hit": hit, "parity": knn_parity,
        }
        del db, sidx, q
        torch.cuda.empty_cache()

    clocks = sampler.stop()
    ops.gemm_select = _orig_gemm_select
    ops.assign_fused = _orig_assign_fused
    del X_dev, packed_dev
    torch.cuda.empty_cache()

    # ---------------- C4 / C5: the two sharded configurations, fixed global size, every N ----------------
    c4 = None if args.no_c4 else run_c4(args, torch, dist, dev, rank, world, barrier, max_over_ranks, ops, P)
    c5 = None if args.no_c5 else run_c5(args, torch, dist, dev, rank, world, barrier, max_over_ranks, ops, P)

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = use_all_host_cores()
        v1, dt1 = cpu_assign_histogram(300)
        n_img = int(min(C2["n_img"], max(300, 300 * 15.0 / max(dt1, 1e-3))))
        v, dt = cpu_assign_histogram(n_img)
        cpu = {"value": v, "unit": "Mdescriptors/s", "cores": cores, "kind": "port",
               "sample": f"{n_img} of {C2['n_img']} images x {C2['per_img']} descriptors ({dt:.1f} s): per-image "
                         f"Faiss-shim IndexFlatIP.search + np.histogram + Okapi on NumPy/OpenBLAS"}
        if knn is not None:
            qv, qdt = cpu_knn(200_000, 1000)
            cpu["knn_qps"] = qv
            cpu["knn_sample"] = f"200k of 1M DB rows x 1000 of 10k queries ({qdt:.1f} s), scaled linearly in nb"

    if rank == 0:
        flops = 2.0 * C2["k"] * C2["d"] * C2["n_desc"]
        ach = flops / (kern_ms * 1e-3) / 1e12
        traffic, traffic_src = ncu_traffic("assign")
        line = {
            "metric": METRIC, "value": value, "unit": "Mdescriptors/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16x2-split (fp32 accumulate)", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "l2": "inputs larger than L2 (512 MB descriptors + 328 MB histogram per step)",
                       "step": "fused assign (row-plane conversion inside gemm_select, top-1) + bovw_histogram(okapi)"},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "Mdescriptors/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "api": "BOVW.transform_csr(pinned PackedDescriptions, okapi=OkapiTransformer()) "
                    "-> scipy CSR float64 [10k x 4096]", "result_nnz": csr_nnz,
                    "input_bytes_per_step": h2d_f32, "wire": e2e_transfer.get("wire"),
                    "wire_note": "the pinned float32 input is narrowed to uint8 by host threads inside the timed call when "
                                 "every value is an integer in [0, 255] and this rank has >= 8 host cores; h2d_bytes_per_step "
                                 "is what crossed PCIe",
                    "float32_wire": {"ms_per_step": e2e_f32_ms, "value": world * C2["n_desc"] / (e2e_f32_ms * 1e-3) / 1e6,
                                     "h2d_bytes_per_step": h2d_f32, "same_result": e2e_same},
                    "aggregate_h2d_gbs": world * h2d / (e2e_ms * 1e-3) / 1e9,
                    "h2d_copy_alone": {"ms": h2d_alone_ms, "aggregate_gbs": world * X_host.nbytes / (h2d_alone_ms * 1e-3) / 1e9,
                                       "note": "all ranks copying their pinned 512 MB input at once, no kernels: the node's "
                                               "host->device ceiling; ms_per_step / this = how close the pipelined step is"}},
            "e2e_from_list": {"value": world * C2["n_desc"] / (e2e_list_ms * 1e-3) / 1e6, "unit": "Mdescriptors/s",
                              "ms_per_step": e2e_list_ms, "h2d_bytes_per_step": list_h2d, "d2h_bytes_per_step": d2h,
                              "api": "BOVW.transform_csr(list of 10,000 float32 (100, 128) arrays, okapi=...) -> scipy CSR: the "
                                     "reference's input contract; list walk + multi-threaded, chunk-ordered pack into a "
                                     "persistent pinned buffer (uint8 on the wire when the values allow it) inside the timed "
                                     "region, chunk i + 1 packed while chunk i is copied and quantised",
                              "equals_packed_path": same_as_packed},
            "e2e_dense": {"value": world * C2["n_desc"] / (e2e_dense_ms * 1e-3) / 1e6, "unit": "Mdescriptors/s",
                          "h2d_bytes_per_step": h2d_f32, "d2h_bytes_per_step": d2h_dense, "ms_per_step": e2e_dense_ms,
                          "api": "BOVW.histograms_host(...) -> dense float64 [10k x 4096] (BOVW.transform's format)"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": P["tf_burst"], "unit": "TFLOP/s",
                         "frac": ach / P["tf_burst"], "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": kernel_name,
                         "kernel_ms": kern_ms, "search": assign_stats, "kernel_share_of_step": kern_ms / ms_step,
                         "peak_source": P["src"] + ", bf16 burst",
                         # tcgen05 products issued per algorithmic FLOP: FP32-grade scores need hi*hi + hi*lo(centroids)
                         # = 2; the verified pipeline issues 1 for every row + 2 more for the rows it re-runs
                         "mma_products": mma_products, "achieved_mma_tflops": mma_products * ach,
                         "frac_mma": mma_products * ach / P["tf_burst"]},
            "parity": step_parity,
            "hbm_kernels": hbm_kernels,
            "cpu_baseline": cpu,
            "host_binding": None if numa_cpus is None else f"rank 0 bound to {len(numa_cpus)} CPUs local to its GPU (NVML)",
            "kmeans_fit_20iter_ms": kmeans_fit_ms, "kmeans_iter_ms": kmeans_iter_ms,
            "kmeans_iter_steady_ms": kmeans_iter_steady_ms, "kmeans_iter_phases_ms": km_phases,
            "knn": knn, "c4": c4, "c5": c5,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _protect_stdout():
    """Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is ONE JSON line
    on stdout, so everything else is routed to stderr and the JSON goes to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-knn", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--c4-iters", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
