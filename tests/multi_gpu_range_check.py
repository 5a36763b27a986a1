"""torchrun target (one rank per GPU, NCCL): ShardedIndexFlat.range_search on real devices must equal the single-GPU
IndexFlat.range_search.  Launched by tests/test_gpu_range_search.py; exit code 0 = parity."""
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    from image_search_engine_b200 import faiss_compat
    from image_search_engine_b200._lib import METRIC_IP
    from image_search_engine_b200.parallel import ShardedIndexFlat, shard_bounds

    rng = np.random.default_rng(41)
    nb, d = 50001, 96
    db = rng.standard_normal((nb, d)).astype(np.float32)
    db /= np.linalg.norm(db, axis=1, keepdims=True)
    db[40000] = db[7]                                       # exact cross-shard duplicate
    cut = int(shard_bounds(nb, world)[1])
    db[cut - 6:cut + 6] = db[cut] + 0.01 * rng.standard_normal((12, d)).astype(np.float32)   # cluster across the cut
    q = (db[rng.integers(0, nb, 400)] + 0.02 * rng.standard_normal((400, d))).astype(np.float32)
    q[0], q[1] = db[7], db[cut]
    bd = shard_bounds(nb, world)
    for metric, radius in ((METRIC_IP, 0.3), (faiss_compat.METRIC_L2, 1.4)):
        six = ShardedIndexFlat(d, metric)
        six.add_local(db[bd[rank]:bd[rank + 1]])
        full = faiss_compat.IndexFlatIP(d) if metric == METRIC_IP else faiss_compat.IndexFlatL2(d)
        full.add(db)
        for nq in (400, 33, 7):
            lims, D, I = six.range_search(q[:nq], radius)
            lr, Dr, Ir = full.range_search(q[:nq], radius)
            lims, D, I = lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
            assert np.array_equal(lims, lr.astype(np.int64)), f"metric {metric}, nq {nq}: lims differ"
            assert np.array_equal(I, Ir), f"metric {metric}, nq {nq}: ids differ"
            assert np.array_equal(D, Dr), f"metric {metric}, nq {nq}: distances differ"
            ids0, ids1 = I[lims[0]:lims[1]], I[lims[1]:lims[2]]
            assert 7 in ids0 and 40000 in ids0
            assert ids1.min() < cut <= ids1.max()
            got = [torch.empty(3, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(got, torch.tensor([lims[-1], int(I.sum()), int(D.view(np.int32).astype(np.int64).sum())],
                                              device="cuda"))
            assert all(torch.equal(g, got[0]) for g in got), "ranks returned different results"
    dist.barrier()
    if rank == 0:
        print("MULTI_GPU_RANGE_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
