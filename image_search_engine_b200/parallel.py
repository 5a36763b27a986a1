"""Multi-GPU data parallelism for the two parts of the hot path that shard (SURVEY section 8e).

One process per GPU, ``torch.distributed`` for the plumbing (NCCL over NVLink on the B200 box).

* ShardedKmeans   descriptor rows are split contiguously over the ranks; every Lloyd iteration
                  all-reduces ONE contiguous float32 buffer [k*d sums | k counts] plus the float64
                  objective, then every rank runs the identical deterministic finalize (mean ->
                  split-empty with mt19937(1234) -> renorm), so no broadcast is needed.
                  33.8 MB per iteration at k = 65536, d = 128.
* ShardedIndexFlat database rows are split contiguously (ids = local + id_base), queries are
                  replicated, per-rank sorted top-k lists are all-gathered and merged on the device
                  with the canonical (score, id) rule, so the result equals the unsharded search.

The reference has no distributed code at all; the contract here is "same result as the single-GPU
drop-in".  The collective-free part (quantise + histogram) shards by image with no exchange.

``local_ops`` is the seam that lets the CPU test-suite drive this exact control flow over gloo with
the oracle standing in for the kernels (tests/test_parallel_gloo.py); the product default is
DeviceOps, which calls libise and has no fallback.
"""
from __future__ import annotations

import time

import numpy as np
import torch
import torch.distributed as dist

from . import ops
from ._lib import METRIC_IP, METRIC_L2, IseError
from .faiss_compat import ClusteringParameters, IndexFlat, IndexFlatIP, IndexFlatL2


def bind_to_gpu_numa(device_index: int) -> list[int] | None:
    """Pins this process to the CPUs NVML reports as local to ``device_index`` (physical index, after
    CUDA_VISIBLE_DEVICES).  One process per GPU means eight processes pin host staging buffers and drive
    eight PCIe links at once; with first-touch allocation the pinned buffers then live on the GPU's own NUMA
    node instead of wherever torchrun happened to start the rank.  Returns the CPU list, or None when NVML
    has no answer (single-socket VMs): never an error."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = device_index
        if vis:
            ent = vis.split(",")[device_index].strip()
            if not ent.isdigit():
                return None
            phys = int(ent)
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus or len(cpus) == len(allowed):
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


class DeviceOps:
    """libise-backed local compute (the product path)."""

    def __init__(self):
        self._acc_ws = None       # persistent workspace of the sorted-gather update
        self._stat = None         # 16 device bytes: float64 objective | int32 number of empty clusters
        self._stat_slots = None   # two pinned mirrors + events: ONE 16-byte readback per iteration, possibly one iteration late
        self._slot = 0

    def device(self):
        return ops.require_cuda()

    def to_local(self, x):
        dev = self.device()
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        if t.dtype not in (torch.float32, torch.uint8):
            t = t.to(torch.float32)
        return t.to(dev, non_blocking=True)

    def prepare(self, x, reuse=False, rows=False, reject_nonfinite=False):
        """rows=True: the row side of a contraction (descriptors / queries): single-pass, per-row scales.
        reuse=True: one 32-byte readback drops an all-zero lo plane (and can reject NaN / Inf input)."""
        op = ops.prepare_operand(x, rows=rows)
        return ops.compact_operand(op, reject_nonfinite=reject_nonfinite) if reuse else op

    def new_buffers(self, k, d, dev):
        """(accum [k*d + k] float32 = the all-reduce payload, sums view, counts view, obj float64[1])."""
        accum = torch.empty((k * d + k,), dtype=torch.float32, device=dev)
        self._stat = torch.zeros((16,), dtype=torch.uint8, device=dev)
        return accum, accum[:k * d].view(k, d), accum[k * d:], self._stat[:8].view(torch.float64)

    def assign(self, x, a_op, cent, metric, precision="verified"):
        return ops.search_topk(x, a_op, cent, ops.prepare_operand(cent), metric, 1, precision=precision,
                               need_distances=False)

    def accumulate(self, x, assign, dis, sums, counts, obj, cent=None, metric=METRIC_IP, a_op=None):
        # ids from the tensor cores; the objective terms are recomputed in exact FP32 inside the update; descriptors
        # that are exact in their FP16 hi plane (integer-valued SIFT, ORB as float) are gathered from that plane
        self._acc_ws = ops.kmeans_accumulate_sorted(x, assign, sums, counts, obj, centroids=cent, metric=metric,
                                                    workspace=self._acc_ws, exact_op=a_op)

    def finalize_begin(self, sums, counts, cent, obj):
        """mean -> cent, then the 16 statistics bytes (objective, number of empty clusters) start their way to a pinned
        host slot.  Returns a handle for finalize_read; nothing here waits for the device."""
        n_empty = self._stat[8:12].view(torch.int32)
        ops.kmeans_mean(sums, counts, cent, n_empty)
        if self._stat_slots is None:
            self._stat_slots = [(torch.zeros((16,), dtype=torch.uint8, pin_memory=True), torch.cuda.Event()) for _ in range(2)]
        self._slot ^= 1
        host, ev = self._stat_slots[self._slot]
        host.copy_(self._stat, non_blocking=True)
        ev.record()
        return self._slot

    def finalize_read(self, handle):
        """(objective, number of empty clusters) of the iteration behind ``handle``; waits for its copy only."""
        host, ev = self._stat_slots[handle]
        ev.synchronize()
        return float(host[:8].view(torch.float64)[0]), int(host[8:12].view(torch.int32)[0])

    def apply_splits(self, counts, cent, n_global):
        """Faiss's split_clusters: sequential-RNG plan on the host (sparse stream index), applied on the device."""
        pairs, _ = ops.split_plan(counts.cpu().numpy(), n_global)
        ops.kmeans_apply_splits(cent, torch.from_numpy(pairs).to(cent.device))
        return int(pairs.shape[0])

    def finalize(self, sums, counts, cent, n_global, spherical, obj):
        """mean -> split empties (host plan, sequential Faiss RNG) -> renorm.  Returns (nsplit, objective): the
        objective and the number of empty clusters come back in ONE 16-byte copy, the only host synchronisation
        of an iteration."""
        o, n_empty = self.finalize_read(self.finalize_begin(sums, counts, cent, obj))
        nsplit = self.apply_splits(counts, cent, n_global) if n_empty > 0 else 0
        if spherical:
            ops.normalize_l2_(cent)
        return nsplit, o

    def normalize(self, cent):
        ops.normalize_l2_(cent)

    def search(self, q, db, b_op, metric, k, id_base):
        """local top-k with exact FP32 scores, so the cross-rank merge compares exact scores; the unsharded IndexFlat's
        own dispatch, so near-tied neighbours cannot differ between the two"""
        return ops.flat_search(q, db, metric, k, operand=lambda: b_op, id_base=id_base)

    def merge(self, D_parts, I_parts, metric):
        return ops.topk_merge(D_parts, I_parts, metric)

    def range_search(self, q, db, b_op, metric, radius, id_base):
        """local range search -> (lims int64 [nq + 1], D, I) with global ids, ascending within a query; the unsharded
        IndexFlat's own dispatch"""
        return ops.flat_range_search(q, db, metric, radius, operand=lambda: b_op, id_base=id_base)


def _world(group):
    if not dist.is_available() or not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def shard_bounds(n: int, world: int) -> np.ndarray:
    """Contiguous row partition: rank r owns [b[r], b[r+1])."""
    base, rem = divmod(int(n), int(world))
    sizes = np.full(world, base, dtype=np.int64)
    sizes[:rem] += 1
    b = np.zeros(world + 1, dtype=np.int64)
    np.cumsum(sizes, out=b[1:])
    return b


SPECULATE_MAX_ASSIGN_MS = 10.0      # see lloyd_train: iterations whose assign is longer than this always synchronise


def lloyd_train(cp, d, k, x_train, n_train, a_op, lops, *, init_rows, init_centroids=None, allreduce=None,
                trace=None, precision="verified"):
    """The Lloyd iterations of faiss Clustering::train (SURVEY appendix A.2, steps 4a-4g) over this process's rows;
    shared by faiss_compat.Kmeans (one GPU, ``allreduce=None``) and ShardedKmeans (rows split over ranks: ``allreduce``
    sums the [k*d | k] buffer and the objective across ranks, after which every rank runs the identical finalize).

    ``init_rows(seed)`` -> [k - n_input, d] float32: rows perm[n_input:k] of rand_perm(n_train, seed) (A.2 step 4).
    Returns (centroids [k, d] on the device, iteration stats)."""
    dev = x_train.device
    metric = METRIC_IP if cp.spherical else METRIC_L2
    if init_centroids is not None:
        ic = np.ascontiguousarray(init_centroids, dtype=np.float32)[:k]
        assert ic.shape[1] == d
    else:
        ic = np.zeros((0, d), np.float32)
    n_input = ic.shape[0]
    accum, sums, counts, obj = lops.new_buffers(k, d, dev)
    cent = torch.empty((k, d), dtype=torch.float32, device=dev)
    lower_is_better = not cp.spherical
    best_obj = float("inf") if lower_is_better else float("-inf")
    best_cent, best_stats, stats = None, [], []
    timed = x_train.is_cuda
    t_start = time.time()
    # Speculation (device path, no lock-step trace): an iteration's readback decides only whether empty clusters must be
    # split before the next assign -- rare once the first iterations are over.  When the previous iteration had no
    # split, the next assign is launched on the assumption that this one has none either; the 16 bytes are read while
    # that assign runs, so the host never stalls the device.  A wrong guess restores the saved means, splits,
    # renormalises and repeats the assign: same results either way (tests/test_gpu_round2.py), one wasted assign at most
    # per change of regime.
    import os
    spec_ok = hasattr(lops, "finalize_begin") and trace is None and timed and not os.environ.get("ISE_KMEANS_NO_SPECULATION")
    spec_force = bool(os.environ.get("ISE_KMEANS_FORCE_SPECULATION"))      # tests: guess "no split" even after a split
    cent_bak = torch.empty_like(cent) if spec_ok else None

    def phase_ms(ev):
        return dict(ms_assign=ev[0].elapsed_time(ev[1]), ms_accumulate=ev[1].elapsed_time(ev[2]),
                    ms_allreduce=ev[2].elapsed_time(ev[3]))

    for redo in range(cp.nredo):
        if n_input:
            cent[:n_input] = torch.from_numpy(ic).to(dev)
        if n_input < k:
            cent[n_input:] = init_rows(cp.seed + 1 + redo * 15486557, n_input)
        if cp.spherical:
            lops.normalize(cent)
        o = 0.0
        pending, prev_nsplit, last_assign_ms = None, None, None
        for it in range(cp.niter):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed else None
            if timed:
                ev[0].record()
            dis, assign = lops.assign(x_train, a_op, cent, metric, precision)
            if pending is not None:
                # the previous iteration's statistics (its copy finished long ago: the device is busy with the assign above)
                t_fin = time.time()
                o_prev, n_empty_prev = lops.finalize_read(pending["handle"])
                nsplit_prev = 0
                if n_empty_prev > 0:
                    cent.copy_(cent_bak)                   # the means, before the renormalisation
                    nsplit_prev = lops.apply_splits(counts, cent, n_train)      # counts still hold the previous iteration's
                    if cp.spherical:
                        lops.normalize(cent)
                    if timed:
                        ev[0].record()
                    dis, assign = lops.assign(x_train, a_op, cent, metric, precision)
                st = stats[pending["index"]]
                st.update(obj=o_prev, nsplit=nsplit_prev, speculated=True, mis_speculated=n_empty_prev > 0,
                          ms_finalize_host=pending["host_ms"] + (time.time() - t_fin) * 1e3, **phase_ms(pending["ev"]))
                prev_nsplit, pending, last_assign_ms = nsplit_prev, None, st["ms_assign"]
            if timed:
                ev[1].record()
            accum.zero_()
            obj.zero_()
            lops.accumulate(x_train, assign, dis, sums, counts, obj, cent, metric, a_op)
            if trace is not None:
                trace.append(dict(redo=redo, it=it, centroids_in=cent.clone(), assign=assign.clone(), dis=dis.clone()))
            if timed:
                ev[2].record()
            if allreduce is not None:
                allreduce(accum)     # [k*d sums | k counts] in one NCCL all-reduce
                allreduce(obj)
            if timed:
                ev[3].record()
            st = dict(obj=float("nan"), nsplit=0, time=time.time() - t_start, time_search=0.0, imbalance_factor=float("nan"))
            if cp.verbose:
                cs = counts.double()
                st["imbalance_factor"] = float((cs * cs).sum() * k / (cs.sum() ** 2))
            # worth guessing only where the host latency it hides is a visible share of an iteration: a wrong guess costs
            # one assign, so long assigns (large codebooks: 28 - 230 ms at C4) always synchronise
            cheap = last_assign_ms is not None and last_assign_ms < SPECULATE_MAX_ASSIGN_MS
            if spec_ok and ((prev_nsplit == 0 and cheap) or (spec_force and prev_nsplit is not None)) and it < cp.niter - 1:
                t_fin = time.time()
                handle = lops.finalize_begin(sums, counts, cent, obj)
                cent_bak.copy_(cent)
                if cp.spherical:
                    lops.normalize(cent)
                stats.append(st)
                pending = dict(handle=handle, index=len(stats) - 1, ev=ev, host_ms=(time.time() - t_fin) * 1e3)
                continue
            if timed:
                torch.cuda.current_stream().synchronize()     # finalize reads the statistics back anyway; this keeps the
            t_fin = time.time()                               # device phases out of its host wall time
            nsplit, o = lops.finalize(sums, counts, cent, n_train, cp.spherical, obj)
            st.update(obj=o, nsplit=nsplit, time=time.time() - t_start)
            if timed:
                # device time of the three phases of this rank + host wall time of the finalize (mean, 16-byte readback,
                # Faiss's sequential split_clusters plan when clusters came out empty, renorm)
                st.update(ms_finalize_host=(time.time() - t_fin) * 1e3, speculated=False, **phase_ms(ev))
            stats.append(st)
            prev_nsplit = nsplit
            if timed:
                last_assign_ms = st["ms_assign"]
            if trace is not None:
                trace[-1]["centroids_out"] = cent.clone()
                trace[-1]["nsplit"] = nsplit
        if cp.nredo > 1:
            if (lower_is_better and o < best_obj) or (not lower_is_better and o > best_obj):
                best_cent, best_stats, best_obj = cent.clone(), list(stats), o
    if cp.nredo > 1:
        cent, stats = best_cent, best_stats
    return cent, stats


class ShardedKmeans:
    """faiss.Kmeans semantics (Clustering.cpp) over rows sharded across ranks."""

    def __init__(self, d, k, group=None, local_ops=None, **kwargs):
        self.d, self.k = int(d), int(k)
        self.cp = ClusteringParameters()
        for key, v in kwargs.items():
            getattr(self.cp, key)
            setattr(self.cp, key, v)
        self.group = group
        self.lops = local_ops or DeviceOps()
        self.centroids = None
        self.obj = None
        self.iteration_stats = None
        self.index = None

    # -- collectives --
    def _allreduce(self, t):
        if _world(self.group)[1] > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def _gather_rows(self, x_local, start, global_ids):
        """Rows of the global matrix by global id: each rank contributes the rows it owns (exactly one
        rank owns each id), summed across ranks."""
        ids = torch.as_tensor(global_ids, dtype=torch.int64, device=x_local.device)
        n_local = x_local.shape[0]
        mine = (ids >= start) & (ids < start + n_local)
        rows = torch.zeros((ids.shape[0], self.d), dtype=torch.float32, device=x_local.device)
        if bool(mine.any()):
            rows[mine] = x_local.index_select(0, ids[mine] - start).to(torch.float32)
        return self._allreduce(rows)

    def train(self, x_local, init_centroids=None):
        """x_local: this rank's contiguous slice of the descriptor matrix (rank order = row order)."""
        cp, d, k = self.cp, self.d, self.k
        rank, world = _world(self.group)
        lops = self.lops
        x = lops.to_local(x_local)
        n_local = int(x.shape[0])
        sizes = torch.zeros((world,), dtype=torch.float64, device=x.device)
        sizes[rank] = n_local
        self._allreduce(sizes)
        sizes = sizes.cpu().numpy().astype(np.int64)
        start = int(sizes[:rank].sum())
        n_glob = int(sizes.sum())
        if n_glob < k:
            raise RuntimeError("Number of training points (%d) should be at least as large as number of "
                               "clusters (%d)" % (n_glob, k))
        # Faiss sub-samples to k*256 rows with rand_perm(n, seed): every rank derives the same global
        # permutation and keeps the sampled rows it owns; sub_ids maps "row of the sub-sampled matrix"
        # to global id so the centroid initialisation picks the same vectors as a single process.
        sub_ids = None
        if n_glob > k * cp.max_points_per_centroid:
            nsub = k * cp.max_points_per_centroid
            sub_ids = ops.rand_perm_prefix(n_glob, cp.seed, nsub)
            mine = sub_ids[(sub_ids >= start) & (sub_ids < start + n_local)] - start
            x_train = x.index_select(0, torch.from_numpy(mine).to(x.device))
            n_train = nsub
        else:
            x_train, n_train = x, n_glob
        if n_train == k:
            # Clustering::train: as many points as centroids -> the points ARE the centroids, one fake iteration
            cent = self._gather_rows(x, start, np.arange(n_glob, dtype=np.int64))
            self.centroids = cent.cpu().numpy()
            self.iteration_stats = [dict(obj=0.0, nsplit=0, time=0.0)]
            self.obj = np.array([0.0])
            if isinstance(lops, DeviceOps):
                self.index = IndexFlatIP(d) if cp.spherical else IndexFlatL2(d)
                self.index.add(cent)
            return 0.0
        if isinstance(lops, DeviceOps) and k >= 1024:
            ops.split_plan_warm(min(k * 2048, 1 << 28))
        a_op = lops.prepare(x_train, reuse=True, rows=True, reject_nonfinite=True)

        def init_rows(seed, n_input):
            perm = ops.rand_perm_prefix(n_train, seed, k)[n_input:k]
            gids = sub_ids[perm] if sub_ids is not None else perm
            return self._gather_rows(x, start, gids)

        cent, stats = lloyd_train(cp, d, k, x_train, n_train, a_op, lops, init_rows=init_rows,
                                  init_centroids=init_centroids, allreduce=self._allreduce if world > 1 else None)
        self.centroids = cent.cpu().numpy()
        self.iteration_stats = stats
        self.obj = np.array([s["obj"] for s in stats])
        if isinstance(lops, DeviceOps):
            self.index = IndexFlatIP(d) if cp.spherical else IndexFlatL2(d)
            self.index.add(cent)
        return self.obj[-1] if self.obj.size else 0.0


class ShardedIndexFlat:
    """Flat index whose rows are split contiguously across ranks; search results equal the unsharded ones."""

    def __init__(self, d, metric=METRIC_IP, group=None, local_ops=None):
        self.d, self.metric_type = int(d), int(metric)
        self.group = group
        self.lops = local_ops or DeviceOps()
        self._local = None
        self._b_op = None
        self.id_base = 0
        self.ntotal = 0

    def add_local(self, x_local):
        """x_local: this rank's slice; global ids follow rank order."""
        rank, world = _world(self.group)
        x = self.lops.to_local(x_local)
        if x.dtype != torch.float32:
            x = x.to(torch.float32)
        sizes = torch.zeros((world,), dtype=torch.float64, device=x.device)
        sizes[rank] = x.shape[0]
        if world > 1:
            dist.all_reduce(sizes, group=self.group)
        sizes = sizes.cpu().numpy().astype(np.int64)
        self.id_base = int(sizes[:rank].sum())
        self.ntotal = int(sizes.sum())
        self._local = x
        self._b_op = self.lops.prepare(x, reuse=True, rows=False)
        if isinstance(self.lops, DeviceOps):
            ops.attach_sample(self._b_op)

    def search(self, q, k):
        """q replicated on every rank.  Returns (D [nq, k], I [nq, k]) identical on every rank.

        Exchange: ONE all-to-all of the packed (id, score) lists hands rank j the lists of query slice j from every
        shard, rank j merges only its 1/world of the queries on the device (canonical (score, id) order), and one
        all-gather of the merged slices gives every rank the full answer -- (2 - 1/world) * nq * k * 12 bytes per rank
        instead of world * nq * k * 12, and no redundant merging."""
        rank, world = _world(self.group)
        k = int(k)
        if not 1 <= k <= ops.MAX_TOPK:            # on every rank, before any of them enters the exchange
            raise IseError(f"topk must be in [1, {ops.MAX_TOPK}]")
        qd = self.lops.to_local(q)
        nq = int(qd.shape[0])
        if self._local is None or self._local.shape[0] == 0 or nq == 0:
            # a rank that owns no rows still takes part in the exchange with empty (padded) lists
            D, I = ops.topk_padding(nq, k, self.metric_type, qd.device)
        else:
            D, I = self.lops.search(qd, self._local, self._b_op, self.metric_type, k, self.id_base)
        if world == 1:
            return D, I
        per = -(-nq // world)                       # queries per merging rank (last slices padded)
        send = torch.zeros((world * per, k, 3), dtype=torch.int32, device=D.device)
        send[:nq, :, :2] = I.contiguous().view(torch.int32).view(nq, k, 2)
        send[:nq, :, 2] = D.contiguous().view(torch.int32)
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send, group=self.group)        # recv[r] = shard r's lists of MY query slice
        recv = recv.view(world, per, k, 3)
        Ig = recv[..., :2].contiguous().view(torch.int64).view(world, per, k)
        Dg = recv[..., 2].contiguous().view(torch.float32)
        Dm, Im = self.lops.merge(Dg, Ig, self.metric_type)
        mine = torch.empty((per, k, 3), dtype=torch.int32, device=D.device)
        mine[..., :2] = Im.contiguous().view(torch.int32).view(per, k, 2)
        mine[..., 2] = Dm.contiguous().view(torch.int32)
        full = torch.empty((world * per, k, 3), dtype=torch.int32, device=D.device)
        dist.all_gather_into_tensor(full, mine, group=self.group)
        I_out = full[:nq, :, :2].contiguous().view(torch.int64).view(nq, k)
        D_out = full[:nq, :, 2].contiguous().view(torch.float32)
        self.last_exchange_bytes = int(send.numel() * 4 * (world - 1) // world + full.numel() * 4 * (world - 1) // world)
        return D_out, I_out

    def range_search(self, q, radius):
        """q replicated on every rank.  Returns (lims int64 [nq + 1], D, I) identical on every rank and equal to the
        unsharded IndexFlat.range_search: each query's results are rank 0's, then rank 1's, ... -- shards are contiguous
        and ascending, so ids stay ascending.

        Exchange: one all-gather of the per-query result counts ([world, nq] int64), then one all-gather of every
        rank's packed (id, dis) results, padded to the largest rank's total."""
        rank, world = _world(self.group)
        qd = self.lops.to_local(q)
        nq = int(qd.shape[0])
        dev = qd.device
        if self._local is None or self._local.shape[0] == 0 or nq == 0:
            # a rank that owns no rows still takes part in the exchange, with no results
            lims, D, I = ops.range_empty(nq, dev)
        else:
            lims, D, I = self.lops.range_search(qd, self._local, self._b_op, self.metric_type, radius, self.id_base)
        if world == 1:
            return lims, D, I
        counts = torch.empty((world * nq,), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(counts, (lims[1:] - lims[:-1]).contiguous(), group=self.group)
        C = counts.cpu().numpy().reshape(world, nq)
        totals = C.sum(axis=1)
        pad = max(int(totals.max()), 1)
        send = torch.zeros((pad, 3), dtype=torch.int32, device=dev)
        n_mine = int(D.shape[0])
        send[:n_mine, :2] = I.contiguous().view(torch.int32).view(n_mine, 2)
        send[:n_mine, 2] = D.contiguous().view(torch.int32)
        full = torch.empty((world * pad, 3), dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(full, send, group=self.group)
        # payload order is (rank, query, id); a stable sort by query gives (query, rank, id)
        query_of = np.concatenate([np.repeat(np.arange(nq, dtype=np.int64), C[r]) for r in range(world)])
        src = np.concatenate([r * pad + np.arange(totals[r], dtype=np.int64) for r in range(world)])
        src = torch.from_numpy(src[np.argsort(query_of, kind="stable")]).to(dev)
        out = full.index_select(0, src)
        lims_h = np.zeros(nq + 1, dtype=np.int64)
        np.cumsum(C.sum(axis=0), out=lims_h[1:])
        I_out = out[:, :2].contiguous().view(torch.int64).view(-1)
        D_out = out[:, 2].contiguous().view(torch.float32)
        self.last_exchange_bytes = int(counts.numel() * 8 * (world - 1) // world + full.numel() * 4 * (world - 1) // world)
        return torch.from_numpy(lims_h).to(dev), D_out, I_out
