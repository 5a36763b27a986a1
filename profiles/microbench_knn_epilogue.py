"""Where does the seeded coarse top-32 pass (C3 shape) spend its time beyond the coarse top-1 pass?  Same launch with a
seed nothing can beat (pure scan, no insert ever), with the real seed, and the top-1 kernels for reference."""
import sys
import torch
sys.path.insert(0, ".")
from image_search_engine_b200 import ops
from image_search_engine_b200._lib import METRIC_IP
nb, d, nq = 1_000_000, 2048, 10_000
dev = ops.require_cuda()
g = torch.Generator(device=dev); g.manual_seed(3)
db = torch.empty((nb, d), device=dev)
for i in range(0, nb, 100_000):
    db[i:i + 100_000].normal_(generator=g).clamp_(min=0)
ops.normalize_l2_(db)
q = db[torch.randint(0, nb, (nq,), generator=g, device=dev)] + 0.05 * torch.randn((nq, d), generator=g, device=dev)
ops.normalize_l2_(q)
b = ops.attach_sample(ops.prepare_operand(db)); a = ops.prepare_operand(q, rows=True)
seed = ops.gemm_select(a.hi_only(), b.sample, METRIC_IP, 2)[0][:, 1].contiguous()
never = torch.full_like(seed, 1e30)
def t(fn, n=4):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
for rep in range(2):
    for name, fn in (
        ("top-32, real seed          ", lambda: ops.gemm_select(a.hi_only(), b.hi_only(), METRIC_IP, 32, row_seed=seed)),
        ("top-32, seed nothing beats ", lambda: ops.gemm_select(a.hi_only(), b.hi_only(), METRIC_IP, 32, row_seed=never)),
        ("top-1                      ", lambda: ops.gemm_select(a.hi_only(), b.hi_only(), METRIC_IP, 1)),
    ):
        print(f"{name}: {t(fn):7.2f} ms", flush=True)
