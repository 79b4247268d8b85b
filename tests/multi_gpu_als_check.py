"""Run under torchrun on >= 2 GPUs: als.train with the rows of every half-step sharded over the ranks (each rank solves
a block of rows of equal record count on the replicated records, one all-gather per half-step) and als.top_n with
the users sharded must be bit-identical to one GPU.  (Not collected by pytest.)

  python -m torch.distributed.run --nproc-per-node 2 tests/multi_gpu_als_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from tests.test_gpu_als import _case, _init
    from xmap_b200 import als
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for r, lam in ((10, 0.01), (64, 1.0)):
        user, item, rating, nU, nI = _case(r)
        args = (torch.from_numpy(user), torch.from_numpy(item), torch.from_numpy(rating), nU, nI, r, 3, lam)
        init = torch.from_numpy(_init(r, nU, r))
        one = als.train(*args, init=init)
        got = als.train(*args, init=init, shard=True)
        ok = ok and torch.equal(one.user_factors, got.user_factors) and torch.equal(one.item_factors, got.item_factors)
        for users in (None, torch.arange(nU - 1, -1, -3)):
            a = als.top_n(one, 64, args[0], args[1], users=users)
            b = als.top_n(one, 64, args[0], args[1], users=users, shard=True)
            ok = ok and torch.equal(a.idx, b.idx) and torch.equal(a.len, b.len)
            ok = ok and torch.equal(a.score.view(torch.int64), b.score.view(torch.int64))
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("multi-GPU (world=%d) ALS factors and top-N lists bit-identical to single GPU: %s" % (world, bool(flag.item())))
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
