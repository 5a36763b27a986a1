"""Every gemm_select_kernel instantiation against an FP64 reference, value by value, at the edge shapes of its launch plan.

The kernel is one template <PA, PB, L2, KSEL, VERIFY, CG, MT, CONV, CL, ARES>; which instantiation runs depends on the
shape (pick_cg / pick_mt / pick_cl / make_plan / setup_sync in csrc/gemm_select.cu) and on the entry point.  The cases
below call the C entry points directly (no FP32 re-score in between), check every returned slot against FP64 scores with
the error bounds the kernel claims, and record -- through torch.profiler -- which instantiation each call ran.  The last
test asserts that every instantiation the library contains was reached.

Shape arithmetic in the comments assumes the B200 (148 SMs): 128-row x 256-column tiles, slots = 148 single CTAs,
74 CTA pairs, ~33 clusters of two pairs.
"""
import math
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

IP, L2 = 0, 1
FLT_MAX = float(np.finfo(np.float32).max)
BIG_ID = 2 ** 33 + 5


# ------------------------------------------------------------------------------------------------------------------
# the instantiations, as the dispatch code builds them (tuple order = template parameter order)
# ------------------------------------------------------------------------------------------------------------------
def V(pa, pb, l2, ksel, verify=0, cg=1, mt=1, conv=0, cl=1, ares=0):
    return (pa, pb, int(l2), ksel, verify, cg, mt, conv, cl, ares)


def _instantiation_table():
    t = set()
    for l2 in (0, 1):
        for verify in (0, 1):                      # dispatch_k -> launch: coarse top-1, single CTAs, MT 1 / 2
            for mt in (1, 2):
                t.add(V(1, 1, l2, 1, verify, 1, mt))
        for ksel in (1, 32, 128, 0):               # split top-1 / top-k (dispatch_k) and collect (ise_gemm_collect)
            for pa, pb in ((1, 2), (2, 2)):
                for cg in (1, 2):
                    t.add(V(pa, pb, l2, ksel, 0, cg))
        for ksel in (32, 128, 0):                  # coarse top-k / collect: CTA pairs, multicast clusters of two pairs
            for cg, cl in ((1, 1), (2, 1), (2, 2)):
                t.add(V(1, 1, l2, ksel, 0, cg, 1, 0, cl))
        for conv in (0, 1):                        # verified_launches: resident row tile (ise_assign_verified / _fused)
            t.add(V(1, 1, l2, 1, 1, 2, 1, conv, 1, 1))
        t.add(V(1, 1, l2, 1, 0, 1, 1, 1))          # ise_assign_fused without a B lo plane
        for cg in (1, 2):                          # ise_assign_fused with a B lo plane
            t.add(V(1, 2, l2, 1, 0, cg, 1, 1))
    return t


INSTANTIATIONS = _instantiation_table()
assert len(INSTANTIATIONS) == 68

_REACHED: dict = {}          # instantiation -> names of the cases that ran it
_NAME = re.compile(r"gemm_select_kernel<([^>]*)>")


def _parse(name):
    m = _NAME.search(name)
    if m is None:
        return None
    out = []
    for tok in m.group(1).split(","):
        tok = re.sub(r"^\((?:bool|int)\)", "", tok.strip())
        out.append(1 if tok == "true" else 0 if tok == "false" else int(tok))
    return tuple(out)


def _capture(case, fn):
    """Runs fn() under torch.profiler; returns (fn's result, set of gemm_select_kernel instantiations it launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not names:
        pytest.fail("torch.profiler recorded no CUDA kernel at all: the launch variants of this case cannot be checked")
    ran = {v for v in map(_parse, names) if v is not None}
    for v in ran:
        _REACHED.setdefault(v, set()).add(case)
    return out, ran


# ------------------------------------------------------------------------------------------------------------------
# operands and raw entry points
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    from image_search_engine_b200 import ops
    return ops.require_cuda()


def _lib():
    from image_search_engine_b200 import _lib as L
    return L.load(), L.ctx(torch.cuda.current_device())


def _p(t):
    from image_search_engine_b200.ops import _ptr
    return _ptr(t)


def _stream():
    from image_search_engine_b200.ops import _stream as s
    return s()


def _check(rc):
    from image_search_engine_b200 import _lib as L
    L.check(rc)


def _prep(x, rows=False, compact=False):
    from image_search_engine_b200 import ops
    op = ops.prepare_operand(x, rows=rows)
    return ops.compact_operand(op) if compact else op


def _widen(op, extra):
    """Same operand with `extra` more columns of row pitch; every column from d on holds FP16 NaN (never read)."""
    from image_search_engine_b200.ops import Operand

    def w(t):
        if t is None:
            return None
        out = torch.full((t.shape[0], op.ldp + extra), float("nan"), dtype=torch.float16, device=t.device)
        out[:, :op.d] = t[:, :op.d]
        return out
    return Operand(w(op.hi), w(op.lo), op.norms, op.meta, op.n, op.d, op.ldp + extra, row_inv=op.row_inv)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _unit(n, d, g):
    x = torch.randn((n, d), generator=g, device="cuda")
    return x / torch.linalg.vector_norm(x, dim=1, keepdim=True)


def _sift(n, d, g):
    """Integer-valued float32 rows (SIFT-like): exact in one FP16 plane."""
    x = torch.randn((n, d), generator=g, device="cuda").abs() ** 2
    x *= 512.0 / torch.linalg.vector_norm(x, dim=1, keepdim=True).clamp_min(1e-30)
    return x.round().clamp(0, 255)


def _u8(n, d, g, hi=256):
    return torch.randint(0, hi, (n, d), generator=g, device="cuda", dtype=torch.uint8)


def _select(a, b, metric, topk, *, a_lo=True, b_lo=True, id_base=0, seed=None, flags=False):
    lib, ctx = _lib()
    m = a.n
    val = torch.empty((m, topk), dtype=torch.float32, device="cuda")
    idx = torch.empty((m, topk), dtype=torch.int64, device="cuda")
    wsb = int(lib.ise_gemm_select_workspace_bytes(ctx, m, b.n, a.d, topk))
    ws = torch.empty((wsb,), dtype=torch.uint8, device="cuda") if wsb else None
    fr = torch.full((m,), -7, dtype=torch.int32, device="cuda") if flags else None
    fc = torch.zeros((1,), dtype=torch.int32, device="cuda") if flags else None
    _check(lib.ise_gemm_select(ctx, _p(a.hi), _p(a.lo if a_lo else None), a.ldp, _p(a.meta), _p(a.norms), _p(a.row_inv),
                               _p(b.hi), _p(b.lo if b_lo else None), b.ldp, _p(b.meta), _p(b.norms), m, b.n, a.d, metric,
                               topk, id_base, _p(seed), _p(fr), _p(fc), _p(val), _p(idx), _p(ws), wsb, _stream()))
    return val, idx, fr, fc


def _collect(a, b, metric, seed, cap, *, a_lo=True, b_lo=True, id_base=0):
    lib, ctx = _lib()
    cv = torch.empty((a.n, cap), dtype=torch.float32, device="cuda")
    ci = torch.empty((a.n, cap), dtype=torch.int64, device="cuda")
    cnt = torch.empty((a.n,), dtype=torch.int32, device="cuda")
    _check(lib.ise_gemm_collect(ctx, _p(a.hi), _p(a.lo if a_lo else None), a.ldp, _p(a.meta), _p(a.norms), _p(a.row_inv),
                                _p(b.hi), _p(b.lo if b_lo else None), b.ldp, _p(b.meta), _p(b.norms), a.n, b.n, a.d,
                                metric, id_base, _p(seed), cap, _p(cv), _p(ci), _p(cnt), _stream()))
    return cv, ci, cnt


def _fused(x, b, metric, *, a_lo, b_lo, workspace):
    """ise_assign_fused; returns (rc, val, idx, row operand written by the kernel, workspace)."""
    from image_search_engine_b200.ops import Operand
    lib, ctx = _lib()
    n, d = x.shape
    ldp = (d + 7) // 8 * 8
    e = dict(device="cuda")
    hi = torch.empty((n, ldp), dtype=torch.float16, **e)
    lo = torch.empty((n, ldp), dtype=torch.float16, **e) if a_lo else None
    skipped = torch.empty((n,), dtype=torch.uint8, **e) if a_lo else None
    norms, row_inv = torch.empty((n,), **e), torch.empty((n,), **e)
    meta = torch.empty((8,), **e)
    val = torch.empty((n, 1), **e)
    idx = torch.empty((n, 1), dtype=torch.int64, **e)
    wsb = int(lib.ise_assign_workspace_bytes(ctx, n, d)) if workspace else 0
    ws = torch.empty((wsb,), dtype=torch.uint8, **e) if workspace else None
    rc = lib.ise_assign_fused(ctx, _p(x), x.stride(0), n, d, _p(hi), _p(lo), ldp, _p(norms), _p(row_inv), _p(skipped),
                              _p(meta), _p(b.hi), _p(b.lo if b_lo else None), b.ldp, _p(b.meta), _p(b.norms), b.n, metric,
                              0, _p(val), _p(idx), _p(ws), wsb, _stream())
    return rc, val, idx, Operand(hi, lo, norms, meta, n, d, ldp, row_inv=row_inv), ws


def _verified(a, b, metric, *, a_lo=True):
    lib, ctx = _lib()
    val = torch.empty((a.n, 1), device="cuda")
    idx = torch.empty((a.n, 1), dtype=torch.int64, device="cuda")
    wsb = int(lib.ise_assign_workspace_bytes(ctx, a.n, a.d))
    ws = torch.empty((wsb,), dtype=torch.uint8, device="cuda")
    rc = lib.ise_assign_verified(ctx, _p(a.hi), _p(a.lo if a_lo else None), a.ldp, _p(a.meta), _p(a.norms),
                                 _p(a.row_inv), _p(b.hi), _p(b.lo), b.ldp, _p(b.meta), _p(b.norms), a.n, b.n, a.d, metric,
                                 0, _p(val), _p(idx), _p(ws), wsb, _stream())
    _check(rc)
    return val, idx, ws


# ------------------------------------------------------------------------------------------------------------------
# FP64 reference and the error bounds the kernel claims
# ------------------------------------------------------------------------------------------------------------------
def _ref(xa, xb, metric, rows):
    """FP64 scores (IP: <a,b>; L2: |a|^2 + |b|^2 - 2<a,b>) of the selected rows of xa against every row of xb, from the
    same float32 / uint8 inputs the kernel was given (cuBLAS DGEMM, row chunks)."""
    yb = xb.double()
    bn = (yb * yb).sum(1)
    out, an = [], []
    for r0 in range(0, rows.numel(), 512):
        ya = xa.index_select(0, rows[r0:r0 + 512]).double()
        ip = ya @ yb.T
        a2 = (ya * ya).sum(1)
        an.append(a2)
        out.append(ip if metric == IP else a2[:, None] + bn[None, :] - 2 * ip)
    return torch.cat(out), torch.cat(an), bn


def _rel_residual(flag):
    """CoarseBound::rel_residual (common.cuh)."""
    if flag == 0.0:
        return 0.0
    return 2.0 ** -11 if flag == 1.0 else min(1.0001 * math.sqrt(flag), 2.0 ** -11)


def _a_inv(a, rows):
    return a.row_inv.index_select(0, rows).double() if a.row_inv is not None else float(a.meta[1])


def _eps_coarse(a, b, rows):
    """CoarseBound (common.cuh) in FP64 from the operands' meta: |one-product <a,b> - exact <a,b>| <= eps per row."""
    ma, mb = a.meta.double().cpu().tolist(), b.meta.double().cpu().tolist()
    d = a.d
    ca, cb = _rel_residual(ma[2]), _rel_residual(mb[2])
    kappa = 1.02 * (ca + cb) + 2.4e-7 + (d // 16 + 4) * 2.0 ** -23
    sq = math.sqrt(d) * 2.0 ** -24
    uf_a = sq * _a_inv(a, rows) if ca != 0 else 0.0
    uf_b = sq * mb[1] if cb != 0 else 0.0
    nb = math.sqrt(mb[4])
    na = a.norms.index_select(0, rows).double().sqrt()
    return kappa * nb * na + uf_a * nb + uf_b * na


def _eps_split(a, b, rows, an64, bn64, a_lo, b_lo):
    """Bound on |split-product <a,b> - exact <a,b>|, derived from the kernel.

    An operand row x with power-of-two scale s has hi = fp16(s x) and, when its lo plane is in use, lo = fp16(s x - hi),
    so |lo_i| <= 2^-11 |s x_i| and the residual r = s x - hi - lo has |r_i| <= 2^-22 |s x_i| + 2^-24 (the two roundings
    of values below the FP16 normal range, 2^-25 each).  With A' = hi_a + lo_a (= s_a a - r_a) and B' likewise, the MMAs
    compute P = hi_a hi_b + hi_a lo_b + lo_a hi_b = A'.B' - lo_a.lo_b, hence
        s_a s_b <a,b> - P = lo_a.lo_b + r_a.B' + A'.r_b + r_a.r_b
    and by Cauchy-Schwarz |.| <= (c_a + c_b + c_a c_b + l_a l_b)(1 + 2^-10) |s_a a||s_b b| + the underflow terms
    2^-24 sqrt(d) (|s_b b| + |s_a a|), with c = 2^-22, l = 2^-11 for an operand whose lo plane is multiplied, c = l = 0 for
    an operand that is exact in its hi plane (meta[LO_NONZERO] == 0: the kernel skips its lo plane then) and c = the
    CoarseBound residual for an inexact operand passed without lo.  The lo.lo product is the one the kernel neglects.
    The tensor core accumulates in FP32 with truncation: every tcgen05.mma (K = 16) adds a relative error <= 2^-23 of the
    running sum, which never exceeds sum |a_i b_i| <= |a||b|; there are ceil(d/16) MMAs per product in use (1 + one per
    lo plane in use), plus the 4 units CoarseBound allows for the alignment inside one MMA: (n_mma + 4) 2^-23 |a||b|.
    The rescale by 1 / (s_a s_b) is exact (powers of two)."""
    ma, mb = a.meta.double().cpu().tolist(), b.meta.double().cpu().tolist()
    d = a.d

    def plane(flag, lo_used):
        if flag == 0.0:
            return 0.0, 0.0, 0
        if lo_used:
            return 2.0 ** -22, 2.0 ** -11, 1
        return _rel_residual(flag), 0.0, 0

    ca, la, ua = plane(ma[2], a_lo and a.lo is not None)
    cb, lb, ub = plane(mb[2], b_lo and b.lo is not None)
    n_mma = -(-d // 16) * (1 + ua + ub)
    rel = (ca + cb + ca * cb + la * lb) * (1 + 2.0 ** -10) + (n_mma + 4) * 2.0 ** -23
    na, nb = an64.sqrt(), float(bn64.max().sqrt())
    uf = 2.0 ** -24 * math.sqrt(d) * ((_a_inv(a, rows) * nb if ca != 0 else 0.0) + (mb[1] * na if cb != 0 else 0.0))
    return rel * (1 + 2.0 ** -20) * na * nb + uf


def _bound(eps, metric, a, b, rows, an64, bn64):
    """Per-row bound on |returned value - FP64 score|.  L2 returns max(0, |a|^2 - (2<a,b> - |b|^2)) from the FP32 norms:
    twice the inner-product bound, the norms' own rounding (measured against FP64), and the rounding of the fmaf and the
    subtraction (2^-24 of |2<a,b> - |b|^2| and of the result)."""
    if metric == IP:
        return eps
    an32, bn32 = a.norms.index_select(0, rows).double(), b.norms.double()
    na, nb = an64.sqrt(), float(bn64.max().sqrt())
    rnd = 2.0 ** -24 * (an32 + 4 * na * nb + 2 * float(bn32.max())) * 1.01
    return 2 * eps + (an32 - an64).abs() + float((bn32 - bn64).abs().max()) + rnd


# ------------------------------------------------------------------------------------------------------------------
# checks
# ------------------------------------------------------------------------------------------------------------------
def _fail_rows(ok, what, extra=None):
    if bool(ok.all()):
        return
    bad = torch.nonzero(~ok).flatten()[:5].tolist()
    pytest.fail(f"{what}: {int((~ok).sum())} violations, first rows {bad}" + (f" ({extra})" if extra else ""))


def _check_topk(val, idx, s, bnd, metric, k, *, id_base=0, seed=None, exact=False):
    """val / idx [m, k] from the kernel for the rows of s [m, n] (FP64 scores), bnd [m] the value bound."""
    m, n = s.shape
    sg = 1.0 if metric == IP else -1.0           # compare as "larger is better"
    S = sg * s
    valid = idx >= 0
    nv = valid.sum(1)
    assert bool((valid[:, 1:] <= valid[:, :-1]).all()), "a valid slot after padding"
    assert bool((val[~valid] == (-FLT_MAX if metric == IP else FLT_MAX)).all()), "padding value is not -+FLT_MAX"
    if seed is None:
        assert bool((nv == min(k, n)).all()), "list shorter than min(topk, n) without a seed"
    col = torch.where(valid, idx - id_base, torch.zeros_like(idx))
    assert bool(((col >= 0) & (col < n))[valid].all()), "id outside [id_base, id_base + n)"
    uniq = torch.where(valid, col, -1 - torch.arange(k, device=col.device)[None, :]).sort(1).values
    assert bool((uniq[:, 1:] != uniq[:, :-1]).all()), "duplicate id in a list"
    Vv = sg * val.double()
    pair = valid[:, 1:]
    # IP values are the selection scores times a power of two, so equal values are equal scores and go by id.  L2
    # values are max(0, |a|^2 - s) of the selection score s = 2<a,b> - |b|^2: that last FP32 rounding can make two
    # different scores return the same distance, in score order (not id order), so only the value order is checked
    order_ok = (Vv[:, :-1] > Vv[:, 1:]) | ((Vv[:, :-1] == Vv[:, 1:]) & ((idx[:, :-1] < idx[:, 1:]) | (metric == L2)))
    _fail_rows((order_ok | ~pair).all(1), "list not sorted by (value, id)")
    sc = S.gather(1, col)
    has = nv > 0
    Ss = S.sort(dim=1, descending=True, stable=True)
    kth_ref = Ss.values.gather(1, (nv - 1).clamp_min(0)[:, None]).squeeze(1)
    low = torch.where(valid, sc, torch.full_like(sc, float("inf"))).min(1).values
    _fail_rows(~has | (low >= kth_ref - 2 * bnd), "a returned id's FP64 score is not within the bound of the FP64 k-th best")
    inside = torch.zeros((m, n), dtype=torch.int32, device=s.device).scatter_add_(1, col, valid.int()) > 0
    out_best = S.masked_fill(inside, float("-inf")).max(1).values
    full = nv == k
    _fail_rows(~(full & has) | (out_best <= low + 2 * bnd), "a column outside the list beats the returned k-th")
    err = (Vv - sc).abs()
    if exact:
        _fail_rows(((err == 0) | ~valid).all(1), "value differs from the exact score")
    else:
        ratio = torch.where(valid, err / bnd[:, None], torch.zeros_like(err))
        _fail_rows((ratio <= 1).all(1), "|value - FP64 score| above the bound", f"worst {float(ratio.max()):.3g} x bound")
    if seed is not None:
        sd = sg * seed.double()
        beats = (Vv > sd[:, None]) if metric == IP else (Vv >= sd[:, None])
        _fail_rows((beats | ~valid).all(1), "a returned value does not beat the row seed")
        _fail_rows(full | (out_best <= sd + bnd), "a column beating the seed is missing from a short list")
    if exact:   # exact arithmetic: the list is the stable (score, id) order itself
        ref = Ss.indices[:, :k]
        _fail_rows(((ref == col) | ~valid).all(1), "ids differ from the exact stable order")


def _check_collect(cv, ci, cnt, s, bnd, metric, cap, seed, *, id_base=0):
    m, n = s.shape
    sg = 1.0 if metric == IP else -1.0
    S, sd = sg * s, sg * seed.double()
    cnt = cnt.long()
    valid = ci >= 0
    filled = torch.arange(cap, device=ci.device)[None, :] < cnt.clamp(max=cap)[:, None]
    _fail_rows((valid == filled).all(1), "valid slots are not exactly the first min(row_count, cap)")
    col = torch.where(valid, ci - id_base, torch.zeros_like(ci))
    assert bool(((col >= 0) & (col < n))[valid].all()), "id outside [id_base, id_base + n)"
    uniq = torch.where(valid, col, -1 - torch.arange(cap, device=ci.device)[None, :]).sort(1).values
    _fail_rows((uniq[:, 1:] != uniq[:, :-1]).all(1), "duplicate id in a collect buffer")
    Vv = sg * cv.double()
    sc = S.gather(1, col)
    ratio = torch.where(valid, (Vv - sc).abs() / bnd[:, None], torch.zeros_like(Vv))
    _fail_rows((ratio <= 1).all(1), "|value - FP64 score| above the bound", f"worst {float(ratio.max()):.3g} x bound")
    beats = (Vv > sd[:, None]) if metric == IP else (Vv >= sd[:, None])
    _fail_rows((beats | ~valid).all(1), "a collected value does not beat the seed")
    _fail_rows(((sc > sd[:, None] - bnd[:, None]) | ~valid).all(1), "a collected column is worse than the seed beyond the bound")
    sure = S > (sd + bnd)[:, None]
    maybe = S > (sd - bnd)[:, None]
    _fail_rows((cnt >= sure.sum(1)) & (cnt <= maybe.sum(1)), "row_count outside the FP64 count band")
    inside = torch.zeros((m, n), dtype=torch.int32, device=s.device).scatter_add_(1, col, valid.int()) > 0
    _fail_rows((cnt > cap) | ~(sure & ~inside).any(1), "a column beating the seed beyond the bound is missing")


def _check_flags(a, b, metric, idx, fr, fc, s, bn64, rows):
    """Coarse top-1 with flags: rows must be listed exactly when the one-product gap does not exceed the proof's margin.

    The kernel's scores are the hi-plane products, which are computed here exactly in FP64 (h); they differ from the
    kernel's FP32 values only by the accumulation error (ceil(d/16) + 4) 2^-23 |hi_a||hi_b| (and, for L2, the fmaf
    rounding).  So every row whose gap over h (winner minus best other column) is below the margin by more than that
    must be listed, and every row above it by more must not be."""
    d, m = a.d, a.n
    fc = int(fc.item())
    flagged = fr[:fc].long()
    assert 0 <= fc <= m and bool(((flagged >= 0) & (flagged < m)).all()), "flag list out of range"
    assert flagged.unique().numel() == fc, "a row is flagged twice"
    is_f = torch.zeros(m, dtype=torch.bool, device="cuda")
    is_f[flagged] = True
    is_f = is_f[rows]
    inv_a = _a_inv(a, rows)
    inv_b = float(b.meta[1])
    ha, hb = a.hi.index_select(0, rows)[:, :d].double(), b.hi[:, :d].double()
    h = (ha @ hb.T) * (inv_a[:, None] if torch.is_tensor(inv_a) else inv_a) * inv_b
    nha = (ha * ha).sum(1).sqrt() * inv_a
    nhb = float((hb * hb).sum(1).sqrt().max()) * inv_b
    acc = (-(-d // 16) + 4) * 2.0 ** -23 * nha * nhb * 1.01
    bn32 = b.norms.double()
    v = h if metric == IP else 2 * h - bn32[None, :]
    tol = 2 * acc if metric == IP else 2 * (2 * acc + 2.0 ** -24 * (2 * nha * nhb + float(bn32.max())))
    best = idx[rows, :1]
    vb = v.gather(1, best).squeeze(1)
    g = vb - v.scatter(1, best, float("-inf")).max(1).values
    eps = _eps_coarse(a, b, rows)
    need = (2.0 if metric == IP else 4.0) * eps
    must = g + tol < need * (1 - 1e-5)
    must_not = g - tol > need * (1 + 1e-5)
    _fail_rows(is_f | ~must, "row inside the proof's margin is not flagged")
    _fail_rows(~is_f | ~must_not, "row outside the proof's margin is flagged")
    # unflagged rows carry the FP64 winner
    sg = 1.0 if metric == IP else -1.0
    top2 = (sg * s).topk(2, dim=1)
    win = (sg * s).sort(dim=1, descending=True, stable=True).indices[:, 0]
    _fail_rows(is_f | (best.squeeze(1) == win), "an unflagged row does not carry the FP64 winner")
    # the proof is not vacuous: a row whose FP64 top-2 gap exceeds twice the margin (plus, for L2, the FP32 rounding
    # of the column norms the kernel subtracts) is never flagged
    gap64 = top2.values[:, 0] - top2.values[:, 1]
    slack = 2 * tol + (2 * float((bn32 - bn64).abs().max()) if metric == L2 else 0.0)
    _fail_rows(~is_f | ~(gap64 > 2 * need + slack), "a clearly decided row is flagged")
    # the data must exercise the margin itself (rows a proof with a quarter of the margin would wrongly accept)
    assert bool((must & (g > need / 4 + tol)).any()), "no row near the margin: the data does not test the bound"




# ------------------------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------------------------
def _run_topk_case(case, metric, xa, xb, a, b, topks, expect, *, a_lo=True, b_lo=True, id_base=0, rows=None,
                   mode="split", exact=False, seed_fn=None):
    rows = torch.arange(a.n, device="cuda") if rows is None else rows
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    eps = _eps_coarse(a, b, rows) if mode == "coarse" else _eps_split(a, b, rows, an64, bn64, a_lo, b_lo)
    bnd = _bound(eps, metric, a, b, rows, an64, bn64)
    for k in topks:
        seed = seed_fn(s, k) if seed_fn else None
        seed_full = None
        if seed is not None:
            seed_full = torch.zeros(a.n, dtype=torch.float32, device="cuda")
            seed_full[rows] = seed
        (val, idx, _, _), ran = _capture(f"{case}/k{k}", lambda: _select(a, b, metric, k, a_lo=a_lo, b_lo=b_lo,
                                                                            id_base=id_base, seed=seed_full))
        _check_topk(val[rows], idx[rows], s, bnd, metric, k, id_base=id_base, seed=seed, exact=exact)
        ks = 1 if k == 1 else 32 if k <= 32 else 128
        want = {v for v in expect if v[3] == ks}
        assert ran == want, f"{case} k={k}: ran {sorted(ran)}, expected {sorted(want)}"


def _ksel_set(pa, pb, l2, ksels, **kw):
    return {V(pa, pb, l2, ks, **kw) for ks in ksels}


SPLIT_TOPKS = (1, 2, 16, 17, 32, 33, 100, 128)


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("case", ["pa2_cg1", "pa2_cg2_odd", "pa2_one_tile_merge", "pa2_small_n", "pa2_d1024",
                                  "pa1_u8_cg1", "pa1_u8_cg2_odd", "pa1_sift_d2048", "exact_ties_merge"])
def test_split_products_select(dev, metric, case):
    """ise_gemm_select with lo planes (split products), plane combinations (2, 2) and (1, 2)."""
    g = _gen(sum(map(ord, case)) + metric)
    l2 = metric == L2
    if case == "pa2_cg1":
        # 300 rows = 3 row tiles < 4: single CTAs; 5000 columns = 20 tiles, 2 column splits (<= 20 / 8) + merge
        xa, xb = _unit(300, 100, g) * 3.7, _unit(5000, 100, g)
        a, b = _prep(xa), _prep(xb)
        _run_topk_case(case, metric, xa, xb, a, b, SPLIT_TOPKS, _ksel_set(2, 2, l2, (1, 32, 128)))
    elif case == "pa2_cg2_odd":
        # 637 rows = 5 row tiles (last one 125 rows): CTA pairs, 3 pairs, the third pair's second CTA has no rows;
        # 3000 columns = 12 tiles: one split; pitch 16 columns wider than the planes, slack = NaN; ids above 2^31
        xa, xb = _unit(637, 192, g), _unit(3000, 192, g)
        a, b = _widen(_prep(xa, rows=True), 16), _widen(_prep(xb), 24)
        _run_topk_case(case, metric, xa, xb, a, b, (1, 17, 33, 128), _ksel_set(2, 2, l2, (1, 32, 128), cg=2),
                       id_base=BIG_ID)
    elif case == "pa2_one_tile_merge":
        # one row tile against 70000 columns = 274 tiles (last one 112 columns): up to 274 / 8 = 34 splits; the
        # makespan minimum is 9 tiles per split -> 31 splits, the last one 4 tiles long; topk_merge with ids above 2^31
        xa, xb = _unit(100, 16, g), _unit(70000, 16, g)
        a, b = _prep(xa), _prep(xb)
        _run_topk_case(case, metric, xa, xb, a, b, (1, 2, 32, 128), _ksel_set(2, 2, l2, (1, 32, 128)), id_base=BIG_ID)
    elif case == "pa2_small_n":
        # 70 columns < one tile and < topk: the tail is id -1 / -+FLT_MAX
        xa, xb = torch.randn((300, 8), generator=g, device="cuda"), torch.randn((70, 8), generator=g, device="cuda")
        a, b = _prep(xa), _prep(xb)
        _run_topk_case(case, metric, xa, xb, a, b, (1, 2, 70, 100, 128), _ksel_set(2, 2, l2, (1, 32, 128)))
    elif case == "pa2_d1024":
        # 520 rows = 5 tiles: CTA pairs; d = 1024 = 16 k-blocks
        xa, xb = _unit(520, 1024, g), _unit(600, 1024, g)
        a, b = _prep(xa), _prep(xb)
        _run_topk_case(case, metric, xa, xb, a, b, (1, 32, 128), _ksel_set(2, 2, l2, (1, 32, 128), cg=2))
    elif case == "pa1_u8_cg1":
        # uint8 rows (no lo plane) x float32 columns: (1, 2); 200 rows = 2 tiles: single CTAs
        xa, xb = _u8(200, 128, g), _unit(4000, 128, g)
        a, b = _prep(xa), _prep(xb)
        _run_topk_case(case, metric, xa, xb, a, b, SPLIT_TOPKS, _ksel_set(1, 2, l2, (1, 32, 128)))
    elif case == "pa1_u8_cg2_odd":
        # 637 rows = 5 tiles: CTA pairs, the last pair half empty; wider pitches with NaN slack
        xa, xb = _u8(637, 96, g), _unit(2500, 96, g)
        a, b = _widen(_prep(xa), 8), _widen(_prep(xb), 32)
        _run_topk_case(case, metric, xa, xb, a, b, (1, 17, 100), _ksel_set(1, 2, l2, (1, 32, 128), cg=2))
    elif case == "pa1_sift_d2048":
        # integer-valued float32 rows compacted to their hi plane: (1, 2); 300 rows: single CTAs
        xa, xb = _sift(300, 2048, g), _unit(1000, 2048, g)
        a, b = _prep(xa, rows=True, compact=True), _prep(xb)
        assert a.lo is None
        _run_topk_case(case, metric, xa, xb, a, b, (1, 32, 128), _ksel_set(1, 2, l2, (1, 32, 128)))
    else:
        # exact arithmetic (small integers) with every column duplicated 20000 columns further on: equal scores in
        # different column splits (one row tile x 157 tiles -> ~20 splits); the merge must order them by id
        xa = _u8(100, 32, g, hi=4)
        half = torch.randint(0, 4, (20000, 32), generator=g, device="cuda").float()
        xb = torch.cat([half, half])
        a, b = _prep(xa), _prep(xb)
        assert float(b.meta[2]) == 0.0
        _run_topk_case(case, metric, xa, xb, a, b, (1, 2, 32, 33, 128), _ksel_set(1, 2, l2, (1, 32, 128)), exact=True)


def _near_tie_data(m, n, d, g):
    """Unit columns, the last 64 of which are perturbed copies of the first 64 (perturbation norms log-spaced over
    1e-3 .. 0.3), and rows of which half lie close to one of those pairs: top-2 gaps (~1.5 |a| delta^2) spread across
    the proof's margin."""
    xb = _unit(n, d, g)
    delta = torch.logspace(-3, -0.5, 64, device="cuda")[:, None]
    xb[n - 64:] = xb[:64] + delta * torch.randn((64, d), generator=g, device="cuda") / math.sqrt(d)
    xb[n - 64:] /= torch.linalg.vector_norm(xb[n - 64:], dim=1, keepdim=True)
    xa = torch.randn((m, d), generator=g, device="cuda") / math.sqrt(d)
    pick = torch.arange(m // 2, device="cuda") % 64
    xa[: m // 2] = xb[pick] + 1e-2 * xa[: m // 2]
    return 3.0 * xa, xb


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("case", ["mt1", "mt2_odd", "mt2_d2048"])
@pytest.mark.parametrize("flags", [False, True], ids=["plain", "flags"])
def test_coarse_top1(dev, metric, case, flags):
    """One product (hi planes only), top-1: single CTAs with one or two row tiles (MT); the flags variant lists every row
    the CoarseBound proof cannot decide, and no other."""
    g = _gen(len(case) * 31 + metric + 2 * flags)
    l2 = metric == L2
    if case == "mt1":
        xa, xb = _near_tie_data(300, 3000, 128, g)          # d < 1024: one row tile per CTA
        a, b, mt = _prep(xa), _prep(xb), 1
    elif case == "mt2_odd":
        # d = 1024, 637 rows = 5 tiles: two row tiles per CTA, 3 work items per split, the last CTA's second tile empty
        xa, xb = _near_tie_data(637, 3000, 1024, g)
        a, b, mt = _widen(_prep(xa, rows=True), 8), _widen(_prep(xb), 8), 2
    else:
        xa, xb = _near_tie_data(300, 600, 2048, g)          # 3 tiles: MT = 2, the second item has one tile
        a, b, mt = _prep(xa), _prep(xb), 2
    rows = torch.arange(a.n, device="cuda")
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    eps = _eps_coarse(a, b, rows)
    bnd = _bound(eps, metric, a, b, rows, an64, bn64)
    (val, idx, fr, fc), ran = _capture(f"coarse_top1/{case}/{'flags' if flags else 'plain'}",
                                       lambda: _select(a, b, metric, 1, a_lo=False, b_lo=False, flags=flags))
    _check_topk(val, idx, s, bnd, metric, 1)
    if flags:
        _check_flags(a, b, metric, idx, fr, fc, s, bn64, rows)
    assert ran == {V(1, 1, l2, 1, int(flags), 1, mt)}, sorted(ran)


@pytest.fixture(scope="module")
def big_columns(dev):
    """131072 x 1024 float32 columns: a B hi plane of exactly 256 MB, the multicast-cluster threshold."""
    g = _gen(4242)
    xb = _unit(131072, 1024, g)
    return xb, _prep(xb)


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("case", ["cg1", "cg2_odd", "cl2_9tiles", "cl2_10tiles", "lockstep", "seeds_exact"])
def test_coarse_topk(dev, metric, case, request):
    """One product (hi planes only), KSEL 32 / 128: single CTAs, CTA pairs, multicast clusters of two pairs, the soft
    lock-step, and row seeds."""
    g = _gen(len(case) * 17 + metric)
    l2 = metric == L2
    ks = (2, 32, 33, 128)
    if case == "cg1":
        xa, xb = torch.randn((300, 128), generator=g, device="cuda"), _unit(5000, 128, g)     # d < 1024: single CTAs
        _run_topk_case(case, metric, xa, xb, _prep(xa), _prep(xb), ks, _ksel_set(1, 1, l2, (32, 128)),
                       a_lo=False, b_lo=False, mode="coarse")
    elif case == "cg2_odd":
        # d = 1024 and 1147 rows = 9 tiles: CTA pairs (5 pairs, the last CTA without rows); B plane 8 MB: no multicast
        xa, xb = torch.randn((1147, 1024), generator=g, device="cuda"), _unit(4096, 1024, g)
        _run_topk_case(case, metric, xa, xb, _widen(_prep(xa), 8), _prep(xb), ks, _ksel_set(1, 1, l2, (32, 128), cg=2),
                       a_lo=False, b_lo=False, mode="coarse")
    elif case.startswith("cl2"):
        # B plane 256 MB and >= 8 row tiles: clusters of two CTA pairs (4 row tiles per work item); 9 tiles -> the
        # third cluster has one real row tile of four, 10 tiles -> two of four
        xb, b = request.getfixturevalue("big_columns")
        m = 1147 if case == "cl2_9tiles" else 1270
        xa = torch.randn((m, 1024), generator=g, device="cuda")
        last = torch.arange((m - 1) // 128 * 128, m, device="cuda")
        rows = torch.cat([torch.randperm(m - last.numel(), generator=g, device="cuda")[:200], last])
        _run_topk_case(case, metric, xa, xb, _prep(xa), b, (32, 128), _ksel_set(1, 1, l2, (32, 128), cg=2, cl=2),
                       a_lo=False, b_lo=False, mode="coarse", rows=rows)
    elif case == "lockstep":
        # 37885 rows = 296 tiles = 148 CTA-pair groups (2 rounds of 74 pairs): the split search of make_plan keeps
        # one split (cost 2 waves x 128 tiles either way), so one work item streams 128 tiles x 512 KB = 64 MB of B,
        # above setup_sync's 24 MB: check-ins every 16 MB / 512 KB = 32 tiles, 4 counters per (round, split)
        xa, xb = torch.randn((37885, 1024), generator=g, device="cuda"), _unit(32768, 1024, g)
        last = torch.arange(295 * 128, 37885, device="cuda")
        rows = torch.cat([torch.randperm(295 * 128, generator=g, device="cuda")[:300], last])
        _run_topk_case(case, metric, xa, xb, _prep(xa), _prep(xb), (32,), _ksel_set(1, 1, l2, (32,), cg=2),
                       a_lo=False, b_lo=False, mode="coarse", rows=rows)
    else:
        # exact integer scores; per row a seed that excludes every column, one equal to the 5th best exact score (only
        # strictly better columns may come back: a list shorter than topk), or one that leaves the list full
        xa, xb = _u8(300, 64, g, hi=8), torch.randint(0, 8, (5000, 64), generator=g, device="cuda").float()

        def seed_fn(s, k):
            sg = 1.0 if metric == IP else -1.0
            srt = (sg * s).sort(1, descending=True).values
            r = torch.arange(s.shape[0], device="cuda") % 3
            sd = torch.where(r == 0, srt[:, 0] + 1, torch.where(r == 1, srt[:, 4], srt[:, k + 10]))
            return (sg * sd).float()
        _run_topk_case(case, metric, xa, xb, _prep(xa), _prep(xb), (2, 32, 100), _ksel_set(1, 1, l2, (32, 128)),
                       a_lo=False, b_lo=False, mode="coarse", exact=True, seed_fn=seed_fn)


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("case", ["p11_cg1", "p11_cg2", "p11_cl2", "p12_cg1", "p12_cg2", "p22_cg1", "p22_cg2"])
def test_collect(dev, metric, case, request):
    """ise_gemm_collect (KSEL = 0): every column beating the row's seed, unsorted, with overflowing rows."""
    g = _gen(len(case) * 7 + metric)
    l2 = metric == L2
    a_lo = b_lo = not case.startswith("p11")
    id_base, rows = 0, None
    if case == "p11_cg1":      # 300 rows, d = 64: single CTAs; wider pitch, ids above 2^31
        xa, xb = torch.randn((300, 64), generator=g, device="cuda"), _unit(20000, 64, g)
        a, b, want = _widen(_prep(xa), 8), _widen(_prep(xb), 8), V(1, 1, l2, 0)
        id_base = BIG_ID
    elif case == "p11_cg2":    # d = 1024, 637 rows = 5 tiles: CTA pairs, the last pair half empty
        xa, xb = torch.randn((637, 1024), generator=g, device="cuda"), _unit(8192, 1024, g)
        a, b, want = _prep(xa), _prep(xb), V(1, 1, l2, 0, cg=2)
    elif case == "p11_cl2":    # B plane 256 MB, 1147 rows = 9 tiles: clusters of two pairs, the last one 1 tile of 4
        xb, b = request.getfixturevalue("big_columns")
        xa = torch.randn((1147, 1024), generator=g, device="cuda")
        a, want = _prep(xa), V(1, 1, l2, 0, cg=2, cl=2)
        rows = torch.cat([torch.arange(0, 1147, 9, device="cuda"), torch.arange(1024, 1147, device="cuda")]).unique()
    elif case.startswith("p12"):   # uint8 rows x float32 columns
        m = 300 if case.endswith("cg1") else 637
        xa, xb = _u8(m, 128, g), _unit(6000, 128, g)
        a, b, want = _prep(xa), _prep(xb), V(1, 2, l2, 0, cg=1 if m == 300 else 2)
    else:
        m = 300 if case.endswith("cg1") else 637
        xa, xb = torch.randn((m, 100), generator=g, device="cuda"), _unit(6000, 100, g)
        a, b, want = _prep(xa, rows=True), _prep(xb), V(2, 2, l2, 0, cg=1 if m == 300 else 2)
    rows = torch.arange(a.n, device="cuda") if rows is None else rows
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    eps = _eps_split(a, b, rows, an64, bn64, a_lo, b_lo) if a_lo else _eps_coarse(a, b, rows)
    bnd = _bound(eps, metric, a, b, rows, an64, bn64)
    cap = 64
    sg = 1.0 if metric == IP else -1.0
    srt = (sg * s).sort(1, descending=True).values
    over = torch.arange(rows.numel(), device="cuda") % 5 == 0          # these rows get ~200 columns: overflow
    sd = sg * torch.where(over, srt[:, 200], srt[:, 40])
    seed = torch.zeros(a.n, device="cuda")
    seed[rows] = sd.float()
    (cv, ci, cnt), ran = _capture(f"collect/{case}", lambda: _collect(a, b, metric, seed, cap, a_lo=a_lo, b_lo=b_lo,
                                                                      id_base=id_base))
    _check_collect(cv[rows], ci[rows], cnt[rows], s, bnd, metric, cap, seed[rows], id_base=id_base)
    assert bool((cnt[rows][over] > cap).all()) and bool((cnt[rows][~over] <= cap).all()), "overflow rows not as planned"
    assert ran == {want}, sorted(ran)


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("case", ["no_b_lo_exact_rows", "b_lo_cg1", "b_lo_cg2", "b_lo_cg1_exact_rows", "b_lo_d8"])
def test_fused_assign(dev, metric, case):
    """ise_assign_fused without workspace: the converter warps prepare the rows inside the contraction kernel; inexact
    rows are repeated with the split products.  Column ranges of <= 15 tiles are never split."""
    g = _gen(len(case) * 13 + metric)
    l2 = metric == L2
    if case == "no_b_lo_exact_rows":
        # integer rows and an integer codebook passed without lo planes (the caller knows both are exact)
        xa, xb = _sift(300, 128, g), _sift(1000, 128, g)
        b = _prep(xb, compact=True)
        assert b.lo is None
        a_lo, want = False, {V(1, 1, l2, 1, conv=1)}
    else:
        m = 637 if case == "b_lo_cg2" else 300      # 5 tiles: CTA pairs; 3 tiles: single CTAs
        d = 8 if case == "b_lo_d8" else 64
        xa = _sift(m, d, g) if "exact_rows" in case else torch.randn((m, d), generator=g, device="cuda") * 3
        xb = _unit(2000, d, g)
        b, a_lo = _prep(xb), True
        cg = 2 if m == 637 else 1
        want = {V(1, 2, l2, 1, cg=cg, conv=1), V(2, 2, l2, 1, cg=cg)}   # + the repeat pass (returns at once if exact)
    (rc, val, idx, a, _), ran = _capture(f"fused/{case}", lambda: _fused(xa, b, metric, a_lo=a_lo, b_lo=b.lo is not None,
                                                                        workspace=False))
    _check(rc)
    rows = torch.arange(xa.shape[0], device="cuda")
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    eps = _eps_split(a, b, rows, an64, bn64, a_lo, True)
    _check_topk(val, idx, s, _bound(eps, metric, a, b, rows, an64, bn64), metric, 1)
    assert ran == want, sorted(ran)
    if case == "no_b_lo_exact_rows":
        # rows that may be inexact need the split products: a_lo without b_lo is refused, not answered from hi alone
        rc, *_ = _fused(xa, b, metric, a_lo=True, b_lo=False, workspace=False)
        assert rc != 0


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
def test_ops_assign_fused_with_an_exact_codebook(dev, metric):
    """ops.assign_fused over float32 rows that are NOT exact in one FP16 plane, against a codebook without a lo plane
    (integer-valued, compacted): the ids must be the split products', not those of the rows' hi plane alone."""
    from image_search_engine_b200 import ops
    g = _gen(99 + metric)
    l2 = metric == L2
    xa, xb = torch.randn((20000, 64), generator=g, device="cuda"), _sift(1000, 64, g)
    b = _prep(xb, compact=True)
    assert b.lo is None
    (val, idx, a), ran = _capture("ops.assign_fused/exact_codebook", lambda: ops.assign_fused(xa, b, metric, verified=False))
    rows = torch.arange(xa.shape[0], device="cuda")
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    a_ref = _prep(xa, rows=True)             # what the fused kernel writes, lo plane included: the split bound applies
    eps = _eps_split(a_ref, b, rows, an64, bn64, True, True)
    _check_topk(val, idx, s, _bound(eps, metric, a_ref, b, rows, an64, bn64), metric, 1)
    # 20000 rows = 157 tiles: CTA pairs; the fused launch over the hi plane, then the split products over all rows
    assert ran == {V(1, 2, l2, 1, cg=2, conv=1), V(2, 2, l2, 1, cg=2)}, sorted(ran)


def _verified_data(m, n, d, flagged, g):
    """Well separated columns e_{j % d} + 0.5 e_{(j // d + j % d + 1) % d} (normalised), except that the last 16 are
    copies of the first 16: a row pointing at one of those has an exact tie and must be listed; `flagged` rows do."""
    j = torch.arange(n, device="cuda")
    xb = torch.zeros((n, d), device="cuda")
    xb[j, j % d] = 1.0
    xb[j, (j // d + j % d + 1) % d] += 0.5
    xb /= torch.linalg.vector_norm(xb, dim=1, keepdim=True)
    xb[n - 16:] = xb[:16]
    pick = torch.randint(16, n - 16, (m,), generator=g, device="cuda")
    pick[:flagged] = torch.arange(flagged, device="cuda") % 16
    pick = pick[torch.randperm(m, generator=g, device="cuda")]
    xa = torch.zeros((m, d), device="cuda")
    r = torch.arange(m, device="cuda")
    xa[r, pick % d] = 200.0
    xa[r, (pick // d + pick % d + 1) % d] += 100.0
    return xa, xb, pick


@pytest.mark.parametrize("metric", [IP, L2], ids=["ip", "l2"])
@pytest.mark.parametrize("flagged", ["none", "capacity", "capacity_plus_one"])
def test_verified_pipeline(dev, metric, flagged):
    """The verified top-1 pipeline (resident row tile, proof, compact split re-run, overflow repeat) through
    ise_assign_fused (raw rows, workspace) and ise_assign_verified (prepared rows, with and without their lo plane)."""
    lib, ctx = _lib()
    l2 = metric == L2
    m, n, d = 2 * 128 * int(lib.ise_ctx_sm_count(ctx)) + 1000, 1024, 128      # 1024 columns x 2 k-blocks = 8 stages
    assert lib.ise_assign_verified_covers(ctx, m, n, d) == 1
    cap = min(-(-m // 128) * 128, -(-max(m // 4, 1024) // 128) * 128)        # verified_ws
    f = {"none": 0, "capacity": cap, "capacity_plus_one": cap + 1}[flagged]
    g = _gen(f + metric)
    xa, xb, pick = _verified_data(m, n, d, f, g)
    b = _prep(xb)
    rows = torch.arange(m, device="cuda")
    s, an64, bn64 = _ref(xa, xb, metric, rows)
    sg = 1.0 if metric == IP else -1.0
    win = (sg * s).sort(dim=1, descending=True, stable=True).indices[:, 0]
    assert bool((win == torch.where(pick >= n - 16, pick - (n - 16), pick)).all())
    runs = [
        ("fused", lambda: _fused(xa, b, metric, a_lo=True, b_lo=True, workspace=True),
         {V(1, 1, l2, 1, 1, 2, 1, 1, 1, 1), V(1, 2, l2, 1, cg=2), V(2, 2, l2, 1, cg=2)}),
        ("verified", lambda: _verified(_prep(xa, rows=True), b, metric),
         {V(1, 1, l2, 1, 1, 2, 1, 0, 1, 1), V(2, 2, l2, 1, cg=2)}),
        ("verified_hi_only", lambda: _verified(_prep(xa, rows=True, compact=True), b, metric, a_lo=False),
         {V(1, 1, l2, 1, 1, 2, 1, 0, 1, 1), V(1, 2, l2, 1, cg=2)}),
    ]
    for name, fn, want in runs:
        out, ran = _capture(f"verified/{name}/{flagged}", fn)
        if name == "fused":
            rc, val, idx, a, ws = out
            _check(rc)
        else:
            val, idx, ws = out
            a = _prep(xa, rows=True)
        assert torch.equal(idx.squeeze(1), win), f"{name}: ids differ from the FP64 winner"
        eps = _eps_coarse(a, b, rows)         # decided rows carry one-product scores, re-run rows split-product ones
        ratio = ((sg * val.squeeze(1).double() - (sg * s).gather(1, win[:, None]).squeeze(1)).abs()
                 / _bound(eps, metric, a, b, rows, an64, bn64))
        assert float(ratio.max()) <= 1, f"{name}: value {float(ratio.max()):.3g} x the coarse bound"
        ctrl = ws[:16].view(torch.int32)[:3].tolist()
        assert ctrl == [f, min(f, cap), int(f > cap)], f"{name}: workspace[0..2] = {ctrl}"
        assert ran == want, f"{name}: {sorted(ran)}"


# ------------------------------------------------------------------------------------------------------------------
# coverage
# ------------------------------------------------------------------------------------------------------------------
def _nm_table():
    from image_search_engine_b200 import _lib as L
    nm = shutil.which("nm")
    if nm is None:
        return None
    out = subprocess.run([nm, "-C", str(L.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    return {v for v in map(_parse, out.splitlines()) if v is not None}


def test_zz_every_instantiation_reached(request):
    """Runs last: every instantiation in the table ran in some case above, and the table is what the library holds."""
    mine = [i for i in request.session.items if i.module is request.module and i is not request.node]
    if len(mine) < 74 or request.config.option.keyword:      # 74 cases above
        pytest.skip("instantiation coverage is only meaningful when the whole module runs")
    built = _nm_table()
    if built is not None:
        assert built == INSTANTIATIONS, (f"libise.so holds {len(built)} instantiations; not in the table: "
                                         f"{sorted(built - INSTANTIATIONS)}, table entries not built: "
                                         f"{sorted(INSTANTIATIONS - built)}")
    print(f"\n{'instantiation <PA,PB,L2,KSEL,VERIFY,CG,MT,CONV,CL,ARES>':58s} reached by")
    for v in sorted(INSTANTIATIONS):
        cases = sorted(_REACHED.get(v, ()))
        print(f"  {str(v):56s} {cases[0] + (f' (+{len(cases) - 1})' if len(cases) > 1 else '') if cases else '-- NOT REACHED'}")
    unknown = set(_REACHED) - INSTANTIATIONS
    assert not unknown, f"kernels outside the table ran: {sorted(unknown)}"
    missing = INSTANTIATIONS - set(_REACHED)
    print(f"{len(INSTANTIATIONS) - len(missing)} of {len(INSTANTIATIONS)} instantiations reached")
    assert not missing, f"{len(missing)} instantiations never ran: {sorted(missing)}"
