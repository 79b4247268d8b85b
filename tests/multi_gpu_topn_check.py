"""Run under torchrun on >= 2 GPUs: recsim.top_n with the users sharded over the ranks (each rank runs its block on the
replicated profile and tables, one all-gather of the lists) must be bit-identical to one GPU, with and without decay,
and with the item axis tiled.  (Not collected by pytest.)

  python -m torch.distributed.run --nproc-per-node 2 tests/multi_gpu_topn_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from tests.test_gpu_topn import _dup, _zipf
    from xmap_b200 import recsim
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for p, stride in ((_zipf(), 1), (_dup(), 2400)):                 # stride 2400: 1.2 M items, a tiled item axis
        item, nI = p["item"] * stride, p["n_items"] * stride
        knn = recsim.item_knn(p["user"], item, p["rating"], nI, 50, k=10)
        for decay in (False, True):
            args = (p["user"], item, p["rating"], p["ts"], p["n_users"] + 2, knn, knn.nb, 64)
            one = recsim.top_n(*args, decay=decay)
            got = recsim.top_n(*args, decay=decay, shard=True)
            ok = ok and torch.equal(one.idx, got.idx) and torch.equal(one.len, got.len)
            ok = ok and torch.equal(one.score.view(torch.int64), got.score.view(torch.int64))
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("multi-GPU (world=%d) top_n lists bit-identical to single GPU: %s" % (world, bool(flag.item())))
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
