"""Tensor-level wrappers over the C ABI (include/ise.h).

PyTorch is plumbing here: it owns device memory and streams; every arithmetic step
of the hot path is a libise kernel.  All functions take CUDA tensors and launch on
``torch.cuda.current_stream()``.  Nothing falls back to torch math or the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import (DTYPE_F32, DTYPE_U8, HIST_BINCOUNT, HIST_NUMPY_COMPAT, METRIC_IP, METRIC_L2, OUT_F32,
                   OUT_F64, IseError)

MAX_TOPK = 128
CSR_MAX_BINS = 12 * 1024     # ise_bovw_histogram_csr keeps one int32 counter per bin in shared memory

# kernel-launch counter (bench.py reports it as gpu_launches)
_launches = 0
_launch_lock = threading.Lock()


def _count(n: int = 1):
    global _launches
    with _launch_lock:
        _launches += n


def launches() -> int:
    return _launches


def _ptr(t: torch.Tensor | None):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(t: torch.Tensor) -> int:
    if not t.is_cuda:
        raise IseError("libise operates on CUDA tensors only (no CPU fallback)")
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise IseError("no CUDA device: image_search_engine_b200 needs a B200 (sm_100a); there is no CPU fallback")
    _lib.ctx(torch.cuda.current_device())
    return torch.device("cuda", torch.cuda.current_device())


# ------------------------------------------------------------------------------------------
# host helpers (sequential Faiss RNG semantics)
# ------------------------------------------------------------------------------------------
def rand_perm_prefix(n: int, seed: int, m: int) -> np.ndarray:
    out = np.empty(int(m), dtype=np.int64)
    _lib.check(_lib.load().ise_rand_perm_prefix(int(n), int(seed), int(m), out.ctypes.data_as(C.c_void_p)))
    return out


def split_plan(hassign: np.ndarray, n: int) -> tuple[np.ndarray, np.ndarray]:
    """Returns (pairs int32 [nsplit, 2], updated hassign)."""
    h = np.ascontiguousarray(hassign, dtype=np.float32).copy()
    k = h.shape[0]
    pairs = np.empty(2 * k, dtype=np.int32)
    ns = C.c_int32(0)
    _lib.check(_lib.load().ise_split_plan(h.ctypes.data_as(C.c_void_p), k, int(n),
                                          pairs.ctypes.data_as(C.c_void_p), C.byref(ns)))
    return pairs[: 2 * ns.value].reshape(-1, 2).copy(), h


def split_plan_warm(n_draws: int) -> None:
    """Starts generating the sparse index of split_clusters' mt19937(1234) stream in a background thread (no-op
    when it already covers n_draws); k-means training on a large codebook calls this up front."""
    _lib.check(_lib.load().ise_split_plan_warm(int(n_draws)))


# ------------------------------------------------------------------------------------------
# operands
# ------------------------------------------------------------------------------------------
@dataclass
class Operand:
    """FP16 hi/lo planes + FP32 norms of a row-major matrix, ready for gemm_select."""
    hi: torch.Tensor          # [n, ldp] float16
    lo: torch.Tensor | None   # [n, ldp] float16 (None when the source is exactly representable)
    norms: torch.Tensor       # [n] float32 sum of squares
    meta: torch.Tensor        # [8] float32: scale, 1/scale, lo_nonzero, absmax, max row norm^2, pad
    n: int
    d: int
    ldp: int
    sample: "Operand | None" = None        # strided 1/64 row sample (hi plane only): seeds for k <= 16
    sample_dense: "Operand | None" = None  # strided 1/16 row sample: seeds for the collect mode (k > 16)
    row_inv: torch.Tensor | None = None    # [n] float32, ROW operands only: 1 / (power-of-two scale of the row's planes)

    def rows(self, sel: torch.Tensor) -> "Operand":
        """Sub-operand of the selected rows (planes gathered, not re-prepared)."""
        return Operand(self.hi.index_select(0, sel), None if self.lo is None else self.lo.index_select(0, sel),
                       self.norms.index_select(0, sel), self.meta, int(sel.numel()), self.d, self.ldp,
                       row_inv=None if self.row_inv is None else self.row_inv.index_select(0, sel))

    def hi_only(self) -> "Operand":
        return Operand(self.hi, None, self.norms, self.meta, self.n, self.d, self.ldp, row_inv=self.row_inv)


def prepare_operand(x: torch.Tensor, *, keep_lo: bool | None = None, rows: bool = False) -> Operand:
    """x: [n, d] float32 or uint8 CUDA tensor (row-major, last dim contiguous).

    ``rows=True`` marks a ROW operand (the descriptors of an assign, the queries of a search -- never the codebook /
    database side): float32 rows are then converted in ONE pass with a power-of-two scale per row
    (``Operand.row_inv``), which halves the HBM traffic of the preparation (no absmax pre-pass, no lo store for rows
    that are exact in one FP16 plane) and also reports NaN / Inf through ``meta[7]``.

    No host synchronisation: float32 inputs always get a lo plane and the device-side
    ``meta[lo_nonzero]`` flag tells gemm_select at run time whether to load / multiply it (integer
    valued descriptors are exact in the hi plane).  uint8 inputs never need one.  ``keep_lo=False``
    skips the lo plane when the caller knows the data is exact; ``compact_operand`` drops it after
    one flag readback (worth it for operands reused across many launches, e.g. k-means training).
    """
    if x.dim() != 2:
        raise IseError("prepare_operand expects a 2-D tensor")
    if x.dtype == torch.float32:
        dt = DTYPE_F32
    elif x.dtype == torch.uint8:
        dt = DTYPE_U8
    else:
        raise IseError(f"unsupported descriptor dtype {x.dtype}; use float32 or uint8")
    if x.stride(1) != 1:
        x = x.contiguous()
    dev = _dev(x)
    n, d = x.shape
    ldp = (d + 7) // 8 * 8
    hi = torch.empty((n, ldp), dtype=torch.float16, device=x.device)
    want_lo = dt == DTYPE_F32 and keep_lo is not False
    lo = torch.empty((n, ldp), dtype=torch.float16, device=x.device) if want_lo else None
    norms = torch.empty((n,), dtype=torch.float32, device=x.device)
    meta = torch.empty((8,), dtype=torch.float32, device=x.device)
    if n == 0:                  # an empty operand (e.g. a rank that owns no rows): nothing to convert
        _lib.ctx(dev)
        meta.zero_()
        return Operand(hi, None, norms, meta, 0, d, ldp)
    if rows and dt == DTYPE_F32:
        row_inv = torch.empty((n,), dtype=torch.float32, device=x.device)
        skipped = torch.empty((n,), dtype=torch.uint8, device=x.device) if want_lo else None
        _lib.check(_lib.load().ise_prepare_rows(
            _lib.ctx(dev), _ptr(x), dt, n, d, x.stride(0), _ptr(hi), _ptr(lo), ldp, _ptr(norms), _ptr(row_inv),
            _ptr(skipped), _ptr(meta), _stream()))
        _count(2 if want_lo else 1)
        return Operand(hi, lo, norms, meta, n, d, ldp, row_inv=row_inv)
    _lib.check(_lib.load().ise_prepare_planes(
        _lib.ctx(dev), _ptr(x), dt, n, d, x.stride(0) if n > 0 else d, _ptr(hi), _ptr(lo), ldp, _ptr(norms),
        _ptr(meta), _stream()))
    _count(3 if dt == DTYPE_F32 else 1)   # absmax + the exact / general conversion kernels (one of them returns at once)
    return Operand(hi, lo, norms, meta, n, d, ldp)


SAMPLE_FRACTION = 64       # one row in 64 ...
SAMPLE_MIN_ROWS = 1024     # ... but never fewer than this, and only for operands at least 64x larger
SAMPLE_MAX_ROWS = 16384
DENSE_SAMPLE_FRACTION = 16   # collect mode (k > 16) needs a tighter handle on how many columns beat the seed
DENSE_SAMPLE_MIN_ROWS = 4096


def attach_sample(op: Operand) -> Operand:
    """Adds a strided sample of the rows to a (database) operand.  search_topk runs a cheap pre-pass
    over it; each query's 2nd-best sample score seeds the selection threshold of the full pass."""
    def strided(ns):
        rows = torch.arange(ns, device=op.hi.device, dtype=torch.int64) * (op.n // ns)
        return Operand(op.hi.index_select(0, rows), None, op.norms.index_select(0, rows), op.meta, ns, op.d, op.ldp)

    if op.n >= SAMPLE_FRACTION * SAMPLE_MIN_ROWS and op.sample is None:
        op.sample = strided(min(max(op.n // SAMPLE_FRACTION, SAMPLE_MIN_ROWS), SAMPLE_MAX_ROWS))
    if op.n >= DENSE_SAMPLE_FRACTION * DENSE_SAMPLE_MIN_ROWS and op.sample_dense is None:
        op.sample_dense = strided(op.n // DENSE_SAMPLE_FRACTION)
    return op


def compact_operand(op: Operand, *, reject_nonfinite: bool = False) -> Operand:
    """Drops an all-zero lo plane (one 32-byte D2H readback of ``meta``): smaller smem stages, deeper pipeline.
    The same readback carries the NaN / Inf flag of the conversion pass (``reject_nonfinite``: raise like
    faiss.Kmeans.train does -- no separate validation pass over the data)."""
    if op.n > 0:
        meta = op.meta.cpu()
        if reject_nonfinite and float(meta[7]) != 0.0:
            raise RuntimeError("input contains NaN's or Inf's")
        if op.lo is not None and float(meta[2]) == 0.0:
            op.lo = None
    return op


def has_nonfinite(x: torch.Tensor) -> bool:
    """True when a float32 matrix holds a NaN or an Inf (one read-only pass, one 4-byte readback)."""
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise IseError("has_nonfinite: row-major float32 matrix")
    if x.shape[0] == 0:
        return False
    meta = torch.empty((8,), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().ise_scan_f32(_lib.ctx(_dev(x)), _ptr(x), x.shape[0], x.shape[1], x.stride(0), _ptr(meta), _stream()))
    _count()
    return float(meta[7].item()) != 0.0


def normalize_l2_(x: torch.Tensor) -> torch.Tensor:
    if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous():
        raise IseError("normalize_L2 needs a contiguous float32 2-D tensor")
    _lib.check(_lib.load().ise_normalize_l2(_lib.ctx(_dev(x)), _ptr(x), x.shape[0], x.shape[1], _stream()))
    _count()
    return x


# ------------------------------------------------------------------------------------------
# fused contraction + selection
# ------------------------------------------------------------------------------------------
def gemm_select(a: Operand, b: Operand, metric: int, topk: int, id_base: int = 0,
                row_seed: torch.Tensor | None = None, flags: tuple | None = None):
    """Top-k columns of b for every row of a.  Returns (val float32 [m, k], idx int64 [m, k]).
    row_seed [m] (optional, topk > 1): only columns scoring strictly better than it are kept."""
    if a.d != b.d:
        raise IseError(f"dimension mismatch {a.d} vs {b.d}")
    if not 1 <= topk <= MAX_TOPK:
        raise IseError(f"topk must be in [1, {MAX_TOPK}]")
    if b.n == 0:
        raise IseError("empty column operand")
    if b.row_inv is not None:
        raise IseError("the column operand (codebook / database) must be prepared with rows=False")
    dev = _dev(a.hi)
    lib, ctx = _lib.load(), _lib.ctx(dev)
    val = torch.empty((a.n, topk), dtype=torch.float32, device=a.hi.device)
    idx = torch.empty((a.n, topk), dtype=torch.int64, device=a.hi.device)
    if a.n == 0:
        return val, idx
    a_lo, b_lo = a.lo, b.lo
    if a_lo is not None and b_lo is None:  # kernel has no (2,1) variant: give b an all-zero lo plane
        b_lo = torch.zeros_like(b.hi)
    ws_bytes = lib.ise_gemm_select_workspace_bytes(ctx, a.n, b.n, a.d, topk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=a.hi.device) if ws_bytes else None
    _lib.check(lib.ise_gemm_select(
        ctx, _ptr(a.hi), _ptr(a_lo), a.ldp, _ptr(a.meta), _ptr(a.norms), _ptr(a.row_inv),
        _ptr(b.hi), _ptr(b_lo), b.ldp, _ptr(b.meta), _ptr(b.norms),
        a.n, b.n, a.d, int(metric), int(topk), int(id_base), _ptr(row_seed),
        _ptr(flags[0] if flags else None), _ptr(flags[1] if flags else None), _ptr(val), _ptr(idx), _ptr(ws),
        ws_bytes, _stream()))
    _count(2 if ws_bytes else 1)
    return val, idx


def _assign_workspace(n: int, d: int, device) -> torch.Tensor:
    lib, ctx = _lib.load(), _lib.ctx(device.index if device.index is not None else torch.cuda.current_device())
    return torch.empty((int(lib.ise_assign_workspace_bytes(ctx, n, d)),), dtype=torch.uint8, device=device)


def assign_fused(x: torch.Tensor, b: Operand, metric: int, id_base: int = 0, verified: bool = True):
    """Top-1 of every raw float32 row of ``x`` against the column operand ``b`` with the row preparation fused into
    the contraction kernel (include/ise.h: ise_assign_fused).  Returns (val [n, 1], idx [n, 1], row operand of x), or
    None when the shape is not covered by the fused kernel (the caller then prepares the rows separately).

    verified=True (default): where the shape allows it (d <= 128, enough rows) the ids come from ONE tensor-core product
    per tile plus a per-row proof, with a compact split-product re-run of the undecided rows (no host round trip); the
    ids are the split products', ``val`` then holds one-product scores (re-score for distances).
    ``last_search_stats`` tells which mode ran."""
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1 or x.shape[1] != b.d or b.n == 0:
        return None
    n, d = x.shape
    if n == 0 or d % 4 != 0 or d > 128:
        return None
    dev = _dev(x)
    lib, ctx = _lib.load(), _lib.ctx(dev)
    ldp = (d + 7) // 8 * 8
    hi = torch.empty((n, ldp), dtype=torch.float16, device=x.device)
    lo = torch.empty((n, ldp), dtype=torch.float16, device=x.device) if b.lo is not None else None
    norms = torch.empty((n,), dtype=torch.float32, device=x.device)
    row_inv = torch.empty((n,), dtype=torch.float32, device=x.device)
    skipped = torch.empty((n,), dtype=torch.uint8, device=x.device) if lo is not None else None
    meta = torch.empty((8,), dtype=torch.float32, device=x.device)
    val = torch.empty((n, 1), dtype=torch.float32, device=x.device)
    idx = torch.empty((n, 1), dtype=torch.int64, device=x.device)
    ws = None
    if verified and b.lo is not None and lib.ise_assign_verified_covers(ctx, n, b.n, d):
        ws = _assign_workspace(n, d, x.device)
    rc = lib.ise_assign_fused(ctx, _ptr(x), x.stride(0), n, d, _ptr(hi), _ptr(lo), ldp, _ptr(norms), _ptr(row_inv),
                              _ptr(skipped), _ptr(meta), _ptr(b.hi), _ptr(b.lo), b.ldp, _ptr(b.meta), _ptr(b.norms), b.n,
                              int(metric), int(id_base), _ptr(val), _ptr(idx), _ptr(ws), 0 if ws is None else ws.numel(),
                              _stream())
    if rc == 2:
        return None
    _lib.check(rc)
    if ws is not None:
        ctrl = ws[:16].view(torch.int32)
        last_search_stats.update(mode="fused-verified", fallback_rows=ctrl[0], rows=n, overflow=ctrl[2])
        _count(6 if lo is not None else 4)
    else:
        last_search_stats.update(mode="fused-split", fallback_rows=0, rows=n)
        _count(3 if lo is not None else 1)
    return val, idx, Operand(hi, lo, norms, meta, n, d, ldp, row_inv=row_inv)


def assign_verified(a: Operand, b: Operand, metric: int, id_base: int = 0):
    """Verified top-1 over PREPARED row planes (include/ise.h: ise_assign_verified): one product per tile + proof +
    compact split re-run, no host round trip.  Returns (val [n, 1] one-product scores, idx [n, 1]) or None when the shape
    is not covered."""
    if b.lo is None or a.d > 128 or a.n == 0 or b.n < 2:
        return None
    dev = _dev(a.hi)
    lib, ctx = _lib.load(), _lib.ctx(dev)
    if not lib.ise_assign_verified_covers(ctx, a.n, b.n, a.d):
        return None
    val = torch.empty((a.n, 1), dtype=torch.float32, device=a.hi.device)
    idx = torch.empty((a.n, 1), dtype=torch.int64, device=a.hi.device)
    ws = _assign_workspace(a.n, a.d, a.hi.device)
    rc = lib.ise_assign_verified(ctx, _ptr(a.hi), _ptr(a.lo), a.ldp, _ptr(a.meta), _ptr(a.norms), _ptr(a.row_inv),
                                 _ptr(b.hi), _ptr(b.lo), b.ldp, _ptr(b.meta), _ptr(b.norms), a.n, b.n, a.d, int(metric),
                                 int(id_base), _ptr(val), _ptr(idx), _ptr(ws), ws.numel(), _stream())
    if rc == 2:
        return None
    _lib.check(rc)
    ctrl = ws[:16].view(torch.int32)
    last_search_stats.update(mode="verified-resident", fallback_rows=ctrl[0], rows=a.n, overflow=ctrl[2])
    _count(4)
    return val, idx


def rescore_topk_(a_raw: torch.Tensor, b_raw: torch.Tensor, a_op: Operand, b_op: Operand, metric: int,
                  val: torch.Tensor, idx: torch.Tensor, id_base: int = 0):
    """Exact FP32 re-score + re-rank (in place) of candidates picked by gemm_select."""
    if b_raw.dtype != torch.float32 or b_raw.stride(1) != 1:
        raise IseError("rescore: column rows must be float32, row-major")
    if a_raw.dtype not in (torch.float32, torch.uint8) or a_raw.stride(1) != 1:
        raise IseError("rescore: rows must be float32 or uint8, row-major")
    m, k = val.shape
    if m == 0:
        return val, idx
    _lib.check(_lib.load().ise_rescore_topk(
        _lib.ctx(_dev(val)), _ptr(a_raw), DTYPE_F32 if a_raw.dtype == torch.float32 else DTYPE_U8, a_raw.stride(0),
        _ptr(b_raw), b_raw.stride(0), m, b_raw.shape[0], a_raw.shape[1], int(metric), k, int(id_base),
        _ptr(a_op.norms), _ptr(b_op.norms), _ptr(val), _ptr(idx), _stream()))
    _count()
    return val, idx


def gemm_collect(a: Operand, b: Operand, metric: int, row_seed: torch.Tensor, cap: int, id_base: int = 0):
    """Collect mode: every column of b whose score beats row_seed[row] is appended (unsorted) to the row's
    buffer.  Returns (cand_val [m, cap], cand_idx [m, cap] (-1 = empty), row_count int32 [m])."""
    dev = a.hi.device
    cv = torch.empty((a.n, cap), dtype=torch.float32, device=dev)
    ci = torch.empty((a.n, cap), dtype=torch.int64, device=dev)
    cnt = torch.empty((max(a.n, 1),), dtype=torch.int32, device=dev)
    a_lo, b_lo = a.lo, b.lo
    if a_lo is not None and b_lo is None:
        b_lo = torch.zeros_like(b.hi)
    _lib.check(_lib.load().ise_gemm_collect(
        _lib.ctx(_dev(a.hi)), _ptr(a.hi), _ptr(a_lo), a.ldp, _ptr(a.meta), _ptr(a.norms), _ptr(a.row_inv),
        _ptr(b.hi), _ptr(b_lo), b.ldp, _ptr(b.meta), _ptr(b.norms), a.n, b.n, a.d, int(metric), int(id_base),
        _ptr(row_seed), int(cap), _ptr(cv), _ptr(ci), _ptr(cnt), _stream()))
    _count()
    return cv, ci, cnt


def rescore_select(a_raw: torch.Tensor, b_raw: torch.Tensor, a_op: Operand, b_op: Operand, metric: int,
                   cand_val: torch.Tensor, cand_idx: torch.Tensor, topk: int, id_base: int = 0,
                   row_seed: torch.Tensor | None = None, row_count: torch.Tensor | None = None):
    """Exact FP32 re-score of kc coarse candidates -> exact top-k + the rows whose candidate list could
    not be proven complete.  Returns (val [m,k], idx [m,k], flag_rows int32 [m], flag_count int32 [1])."""
    m, kc = cand_idx.shape
    dev = cand_idx.device
    val = torch.empty((m, topk), dtype=torch.float32, device=dev)
    idx = torch.empty((m, topk), dtype=torch.int64, device=dev)
    flag_rows = torch.empty((max(m, 1),), dtype=torch.int32, device=dev)
    flag_count = torch.zeros((1,), dtype=torch.int32, device=dev)
    if m == 0:
        return val, idx, flag_rows, flag_count
    _lib.check(_lib.load().ise_rescore_select(
        _lib.ctx(_dev(cand_idx)), _ptr(a_raw), DTYPE_F32 if a_raw.dtype == torch.float32 else DTYPE_U8,
        a_raw.stride(0), _ptr(a_op.meta), _ptr(a_op.norms), _ptr(a_op.row_inv), _ptr(b_raw), b_raw.stride(0), _ptr(b_op.meta),
        _ptr(b_op.norms), m, b_raw.shape[0], a_raw.shape[1], int(metric), kc, int(topk), int(id_base),
        _ptr(row_seed), _ptr(row_count), _ptr(cand_val.contiguous()), _ptr(cand_idx.contiguous()), _ptr(val), _ptr(idx), _ptr(flag_rows),
        _ptr(flag_count), _stream()))
    _count()
    return val, idx, flag_rows, flag_count


# Below this dimension a top-1 tile is bound by reading the 128 x 256 FP32 accumulator out of TMEM
# (~2.4k cycles, measured) rather than by its MMAs (d/64 * 512 cycles per product), so dropping the lo
# product buys nothing and the split products are used directly (profiles/r01_findings.md).
COARSE_TOP1_MIN_D = int(os.environ.get("ISE_COARSE_TOP1_MIN_D", "512"))
VERIFIED_MAX_K = 100   # coarse candidates: 32 per query for k <= 16, 128 for k <= 100

# statistics of the last search_topk call on this process (bench.py / tests read them)
class _SearchStats(dict):
    """Counters of the sync-free pipelines stay on the device until somebody asks for them."""

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if isinstance(v, torch.Tensor):
            v = int(v.item())
            dict.__setitem__(self, key, v)
        return v

    def resolved(self) -> dict:
        return {k: self[k] for k in list(self.keys())}


last_search_stats = _SearchStats(mode=None, fallback_rows=0, rows=0)


def search_stats() -> dict:
    """last_search_stats with device-side counters read back (one small synchronising copy each)."""
    return last_search_stats.resolved()


def search_topk(q_raw: torch.Tensor, a_op: Operand, db_raw: torch.Tensor, b_op: Operand, metric: int, k: int,
                id_base: int = 0, precision: str = "verified", need_distances: bool = True):
    """Flat top-k of every query row against the database operand (the tensor-core path, nq >= 20).

    precision="verified" (default): ONE tcgen05 product per tile (FP16 hi planes only).
      k == 1 (quantisation / k-means assign): the kernel tracks the exact runner-up of every row and flags
        the rows whose winner is not separated from it by more than the rigorous coarse error bound;
      2 <= k <= 100: up to 32 (k <= 16) or 128 candidates per query are kept, ise_rescore_select re-scores
        them exactly in FP32 and proves from the same bound that the list contains the true top-k.
      Flagged rows (rare) are re-run with the split products, so results equal the split path's at
      roughly a third (k > 1) or half (k == 1, exact rows) of the tensor-core work.
    precision="split": hi*hi + hi*lo + lo*hi products for every tile (FP32-grade scores throughout),
      then exact re-score of the k winners.
    """
    nb = b_op.n
    kc = 32 if k <= 16 else MAX_TOPK
    a_hi, b_hi = a_op.hi_only(), b_op.hi_only()

    def rerun_rows(rows, cnt, D, I):
        """Re-runs the flagged rows with the split products (planes gathered, not re-prepared)."""
        nflag = int(cnt.item())                       # 4-byte readback: how many rows need the split path
        if nflag:
            sel = rows[:nflag].to(torch.int64)
            sub = a_op.rows(sel)
            D2, I2 = gemm_select(sub, b_op, metric, k, id_base)
            if need_distances:
                rescore_topk_(q_raw.index_select(0, sel), db_raw, sub, b_op, metric, D2, I2, id_base)
            D.index_copy_(0, sel, D2)
            I.index_copy_(0, sel, I2)
        return nflag

    if precision == "verified" and k == 1 and nb > 1 and a_op.d <= 128:
        # resident-row-tile pipeline: one product + proof + compact re-run, nothing read back
        got = assign_verified(a_op, b_op, metric, id_base)
        if got is not None:
            D, I = got
            if need_distances:
                rescore_topk_(q_raw, db_raw, a_op, b_op, metric, D, I, id_base)
            return D, I
    if precision == "verified" and k == 1 and nb > 1 and a_op.d >= COARSE_TOP1_MIN_D:
        # the verifying kernel keeps one runner-up per row, i.e. does not split the column range over
        # CTAs: only worth it when the rows alone give every SM a few 128-row tiles
        if a_op.n >= 4 * 128 * _lib.load().ise_ctx_sm_count(_lib.ctx(_dev(a_op.hi))):
            rows = torch.empty((a_op.n,), dtype=torch.int32, device=a_op.hi.device)
            cnt = torch.zeros((1,), dtype=torch.int32, device=a_op.hi.device)
            # coarse top-1 + exact runner-up; rows whose winner is not provably unique are flagged
            D, I = gemm_select(a_hi, b_hi, metric, 1, id_base, flags=(rows, cnt))
            nflag = rerun_rows(rows, cnt, D, I)
            if need_distances:
                rescore_topk_(q_raw, db_raw, a_op, b_op, metric, D, I, id_base)
            last_search_stats.update(mode="verified", fallback_rows=nflag, rows=a_op.n)
            return D, I
    if (precision == "verified" and 16 < k <= VERIFIED_MAX_K and need_distances and b_op.sample_dense is not None
            and nb >= 64 * k):
        # large k: seed = r-th best of a 1/16 column sample (about 16 r +- 16 sqrt(r) columns beat it, with
        # r chosen for ~3.75 k), COLLECT every column beating the seed, then sort / prove on the exact scores
        r = min(32, -(-15 * k // (4 * DENSE_SAMPLE_FRACTION)))
        cap = 256 if k <= 32 else 1024
        sv, _ = gemm_select(a_hi, b_op.sample_dense, metric, r)
        seed = sv[:, r - 1].contiguous()
        cv, ci, rc = gemm_collect(a_hi, b_hi, metric, seed, cap, id_base)
        D, I, rows, cnt = rescore_select(q_raw, db_raw, a_op, b_op, metric, cv, ci, k, id_base, row_seed=seed,
                                         row_count=rc)
        nflag = rerun_rows(rows, cnt, D, I)
        last_search_stats.update(mode="verified-collect", fallback_rows=nflag, rows=a_op.n)
        return D, I
    if precision == "verified" and 2 <= k <= VERIFIED_MAX_K and nb > kc and need_distances:
        seed = None
        if b_op.sample is not None:
            # pre-pass over 1/64 of the columns: the r-th best sample score of each query is a score real
            # columns reach, and about 64*r columns of the full set beat it (r grows with k so that at
            # least ~2k do); nothing at or below it needs to be tracked by the main pass
            r = max(2, -(-2 * k // SAMPLE_FRACTION) + 1)
            sv, _ = gemm_select(a_hi, b_op.sample, metric, r)
            seed = sv[:, r - 1].contiguous()
        cv, ci = gemm_select(a_hi, b_hi, metric, kc, id_base, row_seed=seed)
        D, I, rows, cnt = rescore_select(q_raw, db_raw, a_op, b_op, metric, cv, ci, k, id_base, row_seed=seed)
        nflag = rerun_rows(rows, cnt, D, I)
        last_search_stats.update(mode="verified", fallback_rows=nflag, rows=a_op.n)
        return D, I
    D, I = gemm_select(a_op, b_op, metric, k, id_base)
    if need_distances:
        rescore_topk_(q_raw, db_raw, a_op, b_op, metric, D, I, id_base)
    last_search_stats.update(mode="split", fallback_rows=0, rows=a_op.n)
    return D, I


# ------------------------------------------------------------------------------------------
# range search (Faiss IndexFlat::range_search)
# ------------------------------------------------------------------------------------------
RANGE_CAP = 256                   # candidate slots per query of the first collect; rows beyond it are re-run
RANGE_BUDGET_BYTES = 1 << 30      # candidate buffers (m x cap x 12 B) of one query chunk / one overflow batch


def _rows_slice(op: Operand, r0: int, r1: int) -> Operand:
    """Rows [r0, r1) of an operand as views (no copy)."""
    return Operand(op.hi[r0:r1], None if op.lo is None else op.lo[r0:r1], op.norms[r0:r1], op.meta, r1 - r0, op.d,
                   op.ldp, row_inv=None if op.row_inv is None else op.row_inv[r0:r1])


def _range_lims(kept: torch.Tensor, m: int, base: int = 0) -> torch.Tensor:
    """lims [m + 1] int64 = base + exclusive scan of kept [m + 1] (kept[m] == 0)."""
    lib, ctx = _lib.load(), _lib.ctx(_dev(kept))
    lims = torch.empty((m + 1,), dtype=torch.int64, device=kept.device)
    ws = torch.empty((int(lib.ise_range_lims_workspace_bytes(ctx, m)),), dtype=torch.uint8, device=kept.device)
    _lib.check(lib.ise_range_lims(ctx, _ptr(kept), m, int(base), _ptr(lims), _ptr(ws), ws.numel(), _stream()))
    _count()
    return lims


def _range_candidates(q_raw, db_raw, a: Operand, b: Operand, metric: int, radius: float, seed, cap: int, id_base: int):
    """Collect over the hi planes + exact filter.  Returns (cand_val, cand_idx, row_count, kept [m + 1])."""
    cv, ci, rc = gemm_collect(a.hi_only(), b.hi_only(), metric, seed, cap, id_base)
    kept = torch.empty((a.n + 1,), dtype=torch.int64, device=cv.device)
    _lib.check(_lib.load().ise_range_count(
        _lib.ctx(_dev(cv)), _ptr(q_raw), DTYPE_F32 if q_raw.dtype == torch.float32 else DTYPE_U8, q_raw.stride(0),
        _ptr(db_raw), db_raw.stride(0), a.n, db_raw.shape[0], a.d, int(metric), radius, int(id_base), _ptr(a.norms),
        _ptr(b.norms), int(cap), _ptr(rc), _ptr(cv), _ptr(ci), _ptr(kept), _stream()))
    _count()
    return cv, ci, rc, kept


def _range_fill(m, cap, rc, cv, ci, row_map, lims, D, I):
    _lib.check(_lib.load().ise_range_fill(_lib.ctx(_dev(cv)), m, int(cap), _ptr(rc), _ptr(cv), _ptr(ci), _ptr(row_map),
                                          _ptr(lims), _ptr(D), _ptr(I), _stream()))
    _count()


def _range_concat(parts, nq: int, device):
    """Joins per-chunk (kept [m + 1], lims [m + 1], D, I) results (chunks in query order)."""
    if len(parts) == 1:
        _, lims, D, I = parts[0]
        return lims, D, I
    kept = torch.cat([p[0][:-1] for p in parts] + [torch.zeros((1,), dtype=torch.int64, device=device)])
    return _range_lims(kept, nq), torch.cat([p[2] for p in parts]), torch.cat([p[3] for p in parts])


def _range_empty(nq: int, device):
    return (torch.zeros((nq + 1,), dtype=torch.int64, device=device), torch.empty((0,), dtype=torch.float32, device=device),
            torch.empty((0,), dtype=torch.int64, device=device))


def range_search(q_raw: torch.Tensor, a_op: Operand, db_raw: torch.Tensor, b_op: Operand, metric: int, radius: float,
                 id_base: int = 0, _cap: int = RANGE_CAP):
    """Every database row whose exact FP32 score beats ``radius`` (IP: > radius, L2: squared distance < radius), for
    every query row (the tensor-core path, nq >= 20).  Returns (lims int64 [nq + 1], D float32 [lims[nq]],
    I int64 [lims[nq]]) on the device; the results of query i are D / I[lims[i]:lims[i+1]], in ascending id.

    One coarse product over the FP16 hi planes collects every column that beats the radius loosened by the rigorous
    coarse error bound (ise_range_seed), so the candidate set is complete by construction; the candidates are
    re-scored exactly in FP32 and filtered with the strict test.  The per-query candidate counts are read back once;
    queries with more than ``_cap`` candidates are collected again with a buffer sized to their count."""
    nq = a_op.n
    dev = q_raw.device
    radius = float(np.float32(radius))
    if q_raw.dtype not in (torch.float32, torch.uint8) or q_raw.stride(1) != 1:
        raise IseError("range_search: query rows must be float32 or uint8, row-major")
    if db_raw.dtype != torch.float32 or db_raw.stride(1) != 1:
        raise IseError("range_search: database rows must be float32, row-major")
    if a_op.d != b_op.d:
        raise IseError(f"dimension mismatch {a_op.d} vs {b_op.d}")
    if nq == 0 or b_op.n == 0:
        last_search_stats.update(mode="range", rows=nq, candidates=0, overflow_rows=0, results=0, fallback_rows=0)
        return _range_empty(nq, dev)
    lib, ctx = _lib.load(), _lib.ctx(_dev(q_raw))
    seed = torch.empty((nq,), dtype=torch.float32, device=dev)
    _lib.check(lib.ise_range_seed(ctx, _ptr(a_op.meta), _ptr(a_op.norms), _ptr(a_op.row_inv), _ptr(b_op.meta), nq,
                                  a_op.d, int(metric), radius, _ptr(seed), _stream()))
    _count()
    chunk = max(1, RANGE_BUDGET_BYTES // (12 * _cap))
    parts, n_cand, n_over = [], 0, 0
    for q0 in range(0, nq, chunk):
        q1 = min(nq, q0 + chunk)
        m = q1 - q0
        cv, ci, rc, kept = _range_candidates(q_raw[q0:q1], db_raw, _rows_slice(a_op, q0, q1), b_op, metric, radius,
                                             seed[q0:q1], _cap, id_base)
        rc_h = rc[:m].cpu().numpy().astype(np.int64)          # the one readback of the candidate counts
        over = np.nonzero(rc_h > _cap)[0]
        n_cand += int(np.minimum(rc_h, _cap).sum())
        n_over += int(over.size)
        reruns = []
        if over.size:
            # overflowing queries again, largest first, in batches whose buffers fit the budget (cap = largest count)
            over = over[np.argsort(-rc_h[over], kind="stable")]
            i0 = 0
            while i0 < over.size:
                cap2 = int(rc_h[over[i0]])
                i1 = min(over.size, i0 + max(1, RANGE_BUDGET_BYTES // (12 * cap2)))
                sel = torch.from_numpy(over[i0:i1]).to(dev)
                gsel = sel + q0
                cv2, ci2, rc2, kept2 = _range_candidates(q_raw.index_select(0, gsel), db_raw, a_op.rows(gsel), b_op,
                                                         metric, radius, seed.index_select(0, gsel), cap2, id_base)
                got = int(rc2.max().item())
                if got > cap2:
                    raise IseError(f"range_search: a re-run query found {got} candidates, more than the {cap2} its "
                                   "first pass counted")
                kept.index_copy_(0, sel, kept2[:-1])
                n_cand += int(rc_h[over[i0:i1]].sum())
                reruns.append((sel, cap2, rc2, cv2, ci2))
                i0 = i1
        lims = _range_lims(kept, m)
        total = int(lims[m].item())
        D = torch.empty((total,), dtype=torch.float32, device=dev)
        I = torch.empty((total,), dtype=torch.int64, device=dev)
        if total:
            _range_fill(m, _cap, rc, cv, ci, None, lims, D, I)
            for sel, cap2, rc2, cv2, ci2 in reruns:
                _range_fill(sel.numel(), cap2, rc2, cv2, ci2, sel, lims, D, I)
            ws = torch.empty((int(lib.ise_range_sort_workspace_bytes(ctx, m, total)),), dtype=torch.uint8, device=dev)
            _lib.check(lib.ise_range_sort(ctx, m, _ptr(lims), total, _ptr(D), _ptr(I), _ptr(ws), ws.numel(), _stream()))
            _count(2)
        parts.append((kept, lims, D, I))
    lims, D, I = _range_concat(parts, nq, dev)
    last_search_stats.update(mode="range", rows=nq, candidates=n_cand, overflow_rows=n_over, results=int(D.numel()),
                             fallback_rows=0)
    return lims, D, I


def range_search_exact(q: torch.Tensor, db: torch.Tensor, metric: int, radius: float, id_base: int = 0,
                       max_score_bytes: int = 1 << 30):
    """Range search with Faiss's direct per-pair formulas (its nq < 20 regime): exact FP32 pair scores of a query chunk
    (ise_pair_scores), then counts, offsets and the results in column order (ise_scores_range).  Same return as
    range_search."""
    if q.dtype != torch.float32 or db.dtype != torch.float32 or not q.is_contiguous() or not db.is_contiguous():
        raise IseError("range_search_exact needs contiguous float32 tensors")
    nq, d = q.shape
    nb = db.shape[0]
    radius = float(np.float32(radius))
    if nq == 0 or nb == 0:
        last_search_stats.update(mode="range-exact", rows=nq, results=0, fallback_rows=0)
        return _range_empty(nq, q.device)
    lib, ctx = _lib.load(), _lib.ctx(_dev(q))
    chunk = int(max(1, min(nq, 65535, max_score_bytes // (4 * nb))))
    parts, base = [], 0
    for q0 in range(0, nq, chunk):
        qs = q[q0:q0 + chunk]
        n = qs.shape[0]
        scores = torch.empty((n, nb), dtype=torch.float32, device=q.device)
        _lib.check(lib.ise_pair_scores(ctx, _ptr(qs), n, _ptr(db), nb, d, int(metric), _ptr(scores), _stream()))
        ws = torch.empty((int(lib.ise_scores_range_workspace_bytes(ctx, n, nb)),), dtype=torch.uint8, device=q.device)
        lims = torch.empty((n + 1,), dtype=torch.int64, device=q.device)
        _lib.check(lib.ise_scores_range(ctx, _ptr(scores), n, nb, int(metric), radius, int(id_base), base, _ptr(lims),
                                        None, None, _ptr(ws), ws.numel(), _stream()))
        total = int(lims[n].item()) - base
        D = torch.empty((total,), dtype=torch.float32, device=q.device)
        I = torch.empty((total,), dtype=torch.int64, device=q.device)
        if total:
            _lib.check(lib.ise_scores_range(ctx, _ptr(scores), n, nb, int(metric), radius, int(id_base), base,
                                            _ptr(lims), _ptr(D), _ptr(I), _ptr(ws), ws.numel(), _stream()))
        _count(6 if total else 4)
        parts.append((lims, D, I))
        base += total
    lims = parts[0][0] if len(parts) == 1 else torch.cat([p[0][:-1] for p in parts] + [parts[-1][0][-1:]])
    D = parts[0][1] if len(parts) == 1 else torch.cat([p[1] for p in parts])
    I = parts[0][2] if len(parts) == 1 else torch.cat([p[2] for p in parts])
    last_search_stats.update(mode="range-exact", rows=nq, results=int(D.numel()), fallback_rows=0)
    return lims, D, I


def flat_search_exact(q: torch.Tensor, db: torch.Tensor, metric: int, topk: int, id_base: int = 0):
    """Exact FP32 CUDA-core search (Faiss's n < 20 path)."""
    if q.dtype != torch.float32 or db.dtype != torch.float32 or not q.is_contiguous() or not db.is_contiguous():
        raise IseError("flat_search_exact needs contiguous float32 tensors")
    if not 1 <= topk <= MAX_TOPK:
        raise IseError(f"topk must be in [1, {MAX_TOPK}]")
    dev = _dev(q)
    lib, ctx = _lib.load(), _lib.ctx(dev)
    nq, d = q.shape
    nb = db.shape[0]
    val = torch.empty((nq, topk), dtype=torch.float32, device=q.device)
    idx = torch.empty((nq, topk), dtype=torch.int64, device=q.device)
    if nq == 0:
        return val, idx
    ws_bytes = lib.ise_flat_search_exact_workspace_bytes(ctx, nq, nb, topk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=q.device)
    _lib.check(lib.ise_flat_search_exact(ctx, _ptr(q), nq, _ptr(db), nb, d, int(metric), int(topk), int(id_base),
                                         _ptr(val), _ptr(idx), _ptr(ws), ws_bytes, _stream()))
    _count(3)
    return val, idx


def search_exact_any_k(q: torch.Tensor, db: torch.Tensor, metric: int, k: int, id_base: int = 0,
                       max_score_bytes: int = 1 << 30):
    """Flat search for k beyond the fused-selection limit (Faiss's IndexFlat.search takes any k): the exact FP32
    pair scores of a query chunk are materialised once, then ceil(k / 128) selection passes each return the next
    best 128 -- the entries already returned are masked -- in the canonical (score, id) order.  CUDA cores only;
    an edge path (the reference asks for k = 20, engine.py:55)."""
    if q.dtype != torch.float32 or db.dtype != torch.float32 or not q.is_contiguous() or not db.is_contiguous():
        raise IseError("search_exact_any_k needs contiguous float32 tensors")
    dev = _dev(q)
    lib, ctx = _lib.load(), _lib.ctx(dev)
    nq, d = q.shape
    nb = db.shape[0]
    k_eff = min(int(k), nb)
    pad = -3.4028234663852886e38 if metric == METRIC_IP else 3.4028234663852886e38
    val = torch.full((nq, k), pad, dtype=torch.float32, device=q.device)
    idx = torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
    if nq == 0 or nb == 0:
        return val, idx
    chunk = int(max(1, min(nq, 65535, max_score_bytes // (4 * nb))))
    for q0 in range(0, nq, chunk):
        qs = q[q0:q0 + chunk]
        n = qs.shape[0]
        scores = torch.empty((n, nb), dtype=torch.float32, device=q.device)
        _lib.check(lib.ise_pair_scores(ctx, _ptr(qs), n, _ptr(db), nb, d, int(metric), _ptr(scores), _stream()))
        _count()
        val[q0:q0 + n], idx[q0:q0 + n] = scores_topk_any_k_(scores, metric, k, id_base)
    return val, idx


def scores_topk_any_k_(scores: torch.Tensor, metric: int, k: int, id_base: int = 0):
    """Per-row top-k of a score matrix for any k: ceil(k / 128) selection passes, masking what a pass returned
    (``scores`` is consumed).  Rows shorter than k are padded with id -1 / -+FLT_MAX like Faiss."""
    nq, nb = scores.shape
    pad = -3.4028234663852886e38 if metric == METRIC_IP else 3.4028234663852886e38
    if k <= MAX_TOPK:
        return scores_topk(scores, metric, k, id_base)
    val = torch.full((nq, k), pad, dtype=torch.float32, device=scores.device)
    idx = torch.full((nq, k), -1, dtype=torch.int64, device=scores.device)
    k_eff = min(int(k), nb)
    lib, ctx = _lib.load(), _lib.ctx(_dev(scores))
    for k0 in range(0, k_eff, MAX_TOPK):
        kk = min(MAX_TOPK, k_eff - k0)
        v, i = scores_topk(scores, metric, kk, id_base)
        val[:, k0:k0 + kk] = v
        idx[:, k0:k0 + kk] = i
        if k0 + kk < k_eff:
            _lib.check(lib.ise_scores_mask(ctx, _ptr(scores), nq, nb, _ptr(i), kk, int(id_base), int(metric), _stream()))
            _count()
    return val, idx


def topk_merge(val_parts: torch.Tensor, idx_parts: torch.Tensor, metric: int):
    """[g, m, k] sorted partial lists -> ([m, k], [m, k])."""
    g, m, k = val_parts.shape
    val_parts = val_parts.contiguous()
    idx_parts = idx_parts.contiguous()
    val = torch.empty((m, k), dtype=torch.float32, device=val_parts.device)
    idx = torch.empty((m, k), dtype=torch.int64, device=val_parts.device)
    _lib.check(_lib.load().ise_topk_merge(_lib.ctx(_dev(val_parts)), _ptr(val_parts), _ptr(idx_parts), g, m, k,
                                          int(metric), _ptr(val), _ptr(idx), _stream()))
    _count()
    return val, idx


# ------------------------------------------------------------------------------------------
# IVFPQ ("cell-probe") building blocks
# ------------------------------------------------------------------------------------------
def scores_topk(scores: torch.Tensor, metric: int, topk: int, id_base: int = 0):
    """Per-row top-k of a [nq, nb] float32 score matrix (IP: largest, L2: smallest; +-inf never selected)."""
    if scores.dtype != torch.float32 or scores.dim() != 2 or not scores.is_contiguous():
        raise IseError("scores_topk needs a contiguous float32 matrix")
    if not 1 <= topk <= MAX_TOPK:
        raise IseError(f"topk must be in [1, {MAX_TOPK}]")
    nq, nb = scores.shape
    lib, ctx = _lib.load(), _lib.ctx(_dev(scores))
    val = torch.empty((nq, topk), dtype=torch.float32, device=scores.device)
    idx = torch.empty((nq, topk), dtype=torch.int64, device=scores.device)
    if nq == 0:
        return val, idx
    ws_bytes = lib.ise_scores_topk_workspace_bytes(ctx, nq, nb, topk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=scores.device)
    _lib.check(lib.ise_scores_topk(ctx, _ptr(scores), nq, nb, int(metric), int(topk), int(id_base), _ptr(val), _ptr(idx),
                                   _ptr(ws), ws_bytes, _stream()))
    _count(2)
    return val, idx


def ivfpq_residual(x: torch.Tensor, centroids: torch.Tensor, assign: torch.Tensor) -> torch.Tensor:
    """x[i] - centroids[assign[i]] (float32)."""
    if x.dtype != torch.float32 or x.stride(1) != 1 or centroids.dtype != torch.float32 or not centroids.is_contiguous():
        raise IseError("ivfpq_residual: float32 rows")
    n, d = x.shape
    out = torch.empty((n, d), dtype=torch.float32, device=x.device)
    assign = assign.reshape(-1).contiguous()
    _lib.check(_lib.load().ise_ivfpq_residual(_lib.ctx(_dev(x)), _ptr(x), x.stride(0) if n > 0 else d, n, d,
                                              _ptr(centroids), _ptr(assign), _ptr(out), _stream()))
    _count()
    return out


def ivfpq_scan(q: torch.Tensor, coarse: torch.Tensor, probes: torch.Tensor, pq_centroids: torch.Tensor,
               codes: torch.Tensor, list_offsets: torch.Tensor) -> torch.Tensor:
    """Asymmetric distances of every query to the codes of its probed lists: [nq, ntotal] (list-sorted order,
    +inf where a list is not probed)."""
    nq, d = q.shape
    M, ksub, dsub = pq_centroids.shape
    ntotal = codes.shape[0]
    if M * dsub != d or codes.dtype != torch.uint8 or codes.shape[1] != M or probes.dtype != torch.int64:
        raise IseError("ivfpq_scan: inconsistent shapes / dtypes")
    dist = torch.full((nq, max(ntotal, 1)), float("inf"), dtype=torch.float32, device=q.device)
    if nq == 0 or ntotal == 0:
        return dist
    _lib.check(_lib.load().ise_ivfpq_scan(
        _lib.ctx(_dev(q)), _ptr(q.contiguous()), nq, d, _ptr(coarse.contiguous()), coarse.shape[0],
        _ptr(probes.contiguous()), probes.shape[1], _ptr(pq_centroids.contiguous()), M, ksub, _ptr(codes.contiguous()),
        _ptr(list_offsets.contiguous()), ntotal, _ptr(dist), _stream()))
    _count()
    return dist


# ------------------------------------------------------------------------------------------
# k-means update
# ------------------------------------------------------------------------------------------
def kmeans_accumulate(x: torch.Tensor, assign: torch.Tensor, dis: torch.Tensor | None, sums: torch.Tensor,
                      counts: torch.Tensor, obj: torch.Tensor | None, centroids: torch.Tensor | None = None,
                      metric: int = METRIC_IP):
    """centroids given: the objective is recomputed in exact FP32 inside the kernel (dis is ignored)."""
    dt = DTYPE_F32 if x.dtype == torch.float32 else DTYPE_U8
    if x.dtype not in (torch.float32, torch.uint8):
        raise IseError("kmeans_accumulate: float32 or uint8 rows")
    n, d = x.shape
    assign = assign.reshape(-1)
    if dis is not None:
        dis = dis.reshape(-1)
    _lib.check(_lib.load().ise_kmeans_accumulate(
        _lib.ctx(_dev(x)), _ptr(x), dt, n, d, x.stride(0) if n > 0 else d, _ptr(assign), _ptr(dis),
        _ptr(centroids), int(sums.shape[0]), int(metric), _ptr(sums), _ptr(counts), _ptr(obj), _stream()))
    _count()


def kmeans_accumulate_sorted(x: torch.Tensor, assign: torch.Tensor, sums: torch.Tensor, counts: torch.Tensor,
                             obj: torch.Tensor | None, centroids: torch.Tensor | None = None, metric: int = METRIC_IP,
                             workspace: torch.Tensor | None = None, exact_op: "Operand | None" = None):
    """Atomics-free update: counting sort of the rows by centroid + chunked gather-reduce (see include/ise.h).
    ``workspace``: optional persistent uint8 tensor (grown by the caller across iterations).
    ``exact_op``: the row operand of ``x`` when it is EXACT in its FP16 hi plane (``lo is None`` after
    ``compact_operand``, per-row scales): the rows are then gathered from that plane -- the same values at half the
    bytes of the float32 rows."""
    if x.dtype not in (torch.float32, torch.uint8):
        raise IseError("kmeans_accumulate_sorted: float32 or uint8 rows")
    n, d = x.shape
    k = int(sums.shape[0])
    assign = assign.reshape(-1)
    src, dt, ld, row_inv = x, (DTYPE_F32 if x.dtype == torch.float32 else DTYPE_U8), (x.stride(0) if n > 0 else d), None
    if (exact_op is not None and x.dtype == torch.float32 and exact_op.lo is None and exact_op.row_inv is not None
            and exact_op.n == n and d % 4 == 0):
        src, dt, ld, row_inv = exact_op.hi, _lib.DTYPE_F16, exact_op.ldp, exact_op.row_inv
    lib, ctx = _lib.load(), _lib.ctx(_dev(x))
    need = lib.ise_kmeans_accumulate_workspace_bytes(ctx, n, k)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((max(need, 1),), dtype=torch.uint8, device=x.device)
    _lib.check(lib.ise_kmeans_accumulate_sorted(
        ctx, _ptr(src), dt, n, d, ld, _ptr(row_inv), _ptr(assign), _ptr(centroids), k, int(metric), _ptr(sums),
        _ptr(counts), _ptr(obj), _ptr(workspace), workspace.numel(), _stream()))
    _count(4)
    return workspace


def kmeans_mean(sums: torch.Tensor, counts: torch.Tensor, centroids: torch.Tensor, n_empty: torch.Tensor):
    k, d = centroids.shape
    _lib.check(_lib.load().ise_kmeans_mean(_lib.ctx(_dev(sums)), _ptr(sums), _ptr(counts), k, d, _ptr(centroids),
                                           _ptr(n_empty), _stream()))
    _count()


def kmeans_apply_splits(centroids: torch.Tensor, pairs: torch.Tensor):
    k, d = centroids.shape
    ns = pairs.shape[0]
    _lib.check(_lib.load().ise_kmeans_apply_splits(_lib.ctx(_dev(centroids)), _ptr(centroids), k, d, _ptr(pairs),
                                                   ns, _stream()))
    _count()


# ------------------------------------------------------------------------------------------
# BoVW histogram / Okapi
# ------------------------------------------------------------------------------------------
def bovw_histogram(words: torch.Tensor, img_offsets: torch.Tensor, k: int, *, mode: int = HIST_NUMPY_COMPAT,
                   out_dtype: torch.dtype = torch.float64, okapi: bool = False, k1: float = 1.0, k2: float = 1.0,
                   b: float = 0.75, avgdl: float = -1.0, out: torch.Tensor | None = None) -> torch.Tensor:
    if words.dtype != torch.int64 or img_offsets.dtype != torch.int64:
        raise IseError("bovw_histogram: words and img_offsets must be int64")
    words = words.reshape(-1).contiguous()
    n_img = img_offsets.numel() - 1
    od = OUT_F64 if out_dtype == torch.float64 else OUT_F32
    if out_dtype not in (torch.float32, torch.float64):
        raise IseError("bovw_histogram: float32 or float64 output")
    if out is None:
        out = torch.empty((n_img, k), dtype=out_dtype, device=words.device)
    elif tuple(out.shape) != (n_img, k) or out.dtype != out_dtype or not out.is_contiguous():
        raise IseError("bovw_histogram: out must be a contiguous [n_img, k] tensor of out_dtype")
    _lib.check(_lib.load().ise_bovw_histogram(
        _lib.ctx(_dev(img_offsets)), _ptr(words), int(words.numel()), _ptr(img_offsets), n_img, int(k), int(mode), od,
        _ptr(out), 1 if okapi else 0, float(k1), float(k2), float(b), float(avgdl), _stream()))
    _count()
    return out


def bovw_histogram_csr(words: torch.Tensor, img_offsets: torch.Tensor, k: int, *, mode: int = HIST_NUMPY_COMPAT,
                       out_dtype: torch.dtype = torch.float64, okapi: bool = False, k1: float = 1.0, k2: float = 1.0,
                       b: float = 0.75, avgdl: float = -1.0, out: tuple | None = None):
    """Histogram (+ fused Okapi) as CSR: returns (indptr int32 [n_img+1], indices int32 [cap], data [cap]) on the
    device; the used length is indptr[-1] <= cap = number of words.  ``out`` = preallocated (indptr, indices, data)."""
    if words.dtype != torch.int64 or img_offsets.dtype != torch.int64:
        raise IseError("bovw_histogram_csr: words and img_offsets must be int64")
    if out_dtype not in (torch.float32, torch.float64):
        raise IseError("bovw_histogram_csr: float32 or float64 data")
    words = words.reshape(-1).contiguous()
    n_img = img_offsets.numel() - 1
    cap = max(int(words.numel()), 1)
    dev = words.device
    if out is None:
        out = (torch.empty((n_img + 1,), dtype=torch.int32, device=dev), torch.empty((cap,), dtype=torch.int32, device=dev),
               torch.empty((cap,), dtype=out_dtype, device=dev))
    indptr, indices, data = out
    if indptr.numel() < n_img + 1 or indices.numel() < words.numel() or data.numel() < words.numel() or \
            indptr.dtype != torch.int32 or indices.dtype != torch.int32 or data.dtype != out_dtype:
        raise IseError("bovw_histogram_csr: out buffers too small or of the wrong dtype")
    row_nnz = torch.empty((max(n_img, 1),), dtype=torch.int32, device=dev)
    _lib.check(_lib.load().ise_bovw_histogram_csr(
        _lib.ctx(_dev(img_offsets)), _ptr(words), _ptr(img_offsets), n_img, int(k), int(mode),
        OUT_F64 if out_dtype == torch.float64 else OUT_F32, _ptr(row_nnz), _ptr(indptr), _ptr(indices), _ptr(data),
        1 if okapi else 0, float(k1), float(k2), float(b), float(avgdl), _stream()))
    _count(3)
    return indptr, indices, data


def okapi_tf_(h: torch.Tensor, k1: float = 1.0, k2: float = 1.0, b: float = 0.75, avgdl: float = -1.0):
    if h.dtype not in (torch.float32, torch.float64) or h.dim() != 2 or not h.is_contiguous():
        raise IseError("okapi_tf_: contiguous float32/float64 matrix")
    n_img, k = h.shape
    od = OUT_F64 if h.dtype == torch.float64 else OUT_F32
    ws = torch.empty((n_img + 1,), dtype=torch.float64, device=h.device)
    _lib.check(_lib.load().ise_okapi_tf(_lib.ctx(_dev(h)), _ptr(h), od, n_img, k, float(k1), float(k2), float(b),
                                        float(avgdl), _ptr(ws), _stream()))
    _count(2)
    return h


def okapi_csr_(indptr: torch.Tensor, indices: torch.Tensor | None, data: torch.Tensor, k1: float = 1.0, k2: float = 1.0,
               b: float = 0.75, avgdl: float = -1.0, idf: torch.Tensor | None = None, norm: int = 0):
    """OkapiTransformer.transform on the data array of a CSR matrix, in place (O(nnz)).  idf / norm: the opt-in
    corrected tf-idf mode (see include/ise.h)."""
    if indptr.dtype != torch.int64 or data.dtype != torch.float64 or not data.is_contiguous():
        raise IseError("okapi_csr_: int64 indptr, contiguous float64 data")
    if indices is not None and indices.dtype != torch.int32:
        raise IseError("okapi_csr_: int32 indices")
    if idf is not None and (idf.dtype != torch.float64 or indices is None):
        raise IseError("okapi_csr_: idf must be float64 and needs the column indices")
    n_rows = indptr.numel() - 1
    ws = torch.empty((n_rows + 1,), dtype=torch.float64, device=data.device)
    _lib.check(_lib.load().ise_okapi_csr(_lib.ctx(_dev(data)), _ptr(indptr), _ptr(indices), _ptr(data), n_rows, float(k1),
                                         float(k2), float(b), float(avgdl), _ptr(idf), int(norm), _ptr(ws), _stream()))
    _count(2)
    return data


def tfidf_finish_(h: torch.Tensor, idf: torch.Tensor | None, norm: int):
    """h[i, j] *= idf[j], then l1 / l2 row normalisation, in place (dense half of the opt-in tf-idf mode)."""
    if h.dtype not in (torch.float32, torch.float64) or h.dim() != 2 or not h.is_contiguous():
        raise IseError("tfidf_finish_: contiguous float32/float64 matrix")
    if idf is not None and (idf.dtype != torch.float64 or idf.numel() != h.shape[1]):
        raise IseError("tfidf_finish_: idf must be float64 [k]")
    od = OUT_F64 if h.dtype == torch.float64 else OUT_F32
    _lib.check(_lib.load().ise_tfidf_finish(_lib.ctx(_dev(h)), _ptr(h), od, h.shape[0], h.shape[1], _ptr(idf), int(norm),
                                            _stream()))
    _count()
    return h
