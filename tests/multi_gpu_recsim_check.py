"""Run under torchrun on >= 2 GPUs: item_knn with the item rows sharded over the ranks (each rank runs its own passes
on the replicated profile, one all-gather of the tables) must be bit-identical to one GPU, non-private and private.
(Not collected by pytest.)

  python -m torch.distributed.run --nproc-per-node 2 tests/multi_gpu_recsim_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from tests.test_gpu_recsim_passes import _zipf_profile
    from xmap_b200 import recsim
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    p = _zipf_profile()
    args = (p["user"], p["item"], p["rating"], p["n_items"], 50)
    small = int(recsim.row_entries(p["user"], p["item"], p["n_items"]).max()) * recsim.ENTRY_BYTES
    ok = True
    for private in (None, dict(seed=5)):
        one = recsim.item_knn(*args, k=10, private=private)
        for budget in (None, small):
            got = recsim.item_knn(*args, k=10, private=private, budget=budget, shard=True)
            ok = ok and all(torch.equal(getattr(one.nb, f).view(torch.int64) if f == "sim" else getattr(one.nb, f),
                                        getattr(got.nb, f).view(torch.int64) if f == "sim" else getattr(got.nb, f))
                            for f in ("idx", "sim", "len"))
            ok = ok and torch.equal(one.info, got.info)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("multi-GPU (world=%d) item_knn tables bit-identical to single GPU: %s" % (world, bool(flag.item())))
    dist.destroy_process_group()
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
