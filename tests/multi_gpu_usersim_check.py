"""Run under torchrun on >= 2 GPUs: usersim.user_knn with the query users sharded over the ranks (blocks of equal
co-rating products, one all-gather of the tables) must be bit-identical to one GPU, in select and in emit (private)
mode, for every user and for a `users=` subset.  (Not collected by pytest.)

  python -m torch.distributed.run --nproc-per-node 2 tests/multi_gpu_usersim_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from tests.test_gpu_usersim import _profile, _tables_equal
    from xmap_b200 import usersim
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    user, item, rating, _, nU, nI = _profile(81, nU=3000, nI=500, n=60000)
    sel = torch.randperm(nU, generator=torch.Generator().manual_seed(3))[:700]
    ok = True
    for private in (None, dict(privacy_epsilon=0.6, rpo=0.1, seed=4)):
        for users in (None, sel):
            one = usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=private, users=users)
            got = usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=private, users=users, shard=True)
            ok = ok and _tables_equal(one.nb, got.nb)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("multi-GPU (world=%d) user_knn tables bit-identical to single GPU: %s" % (world, bool(flag.item())))
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
