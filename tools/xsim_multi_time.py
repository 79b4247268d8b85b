"""Under torchrun: where the time of a sharded X-SIM run goes on every rank (kernel, unit-result all-reduce, merge)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, torch.distributed as dist, bench
from xmap_b200 import engine as E, extend as X, _native as N, multi as MG

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)
wl = bench.make_workload(sys.argv[1] if len(sys.argv) > 1 else "cfg2")
meta = E.to_device_meta(wl["meta"], dev)
lay = E.build_layout(wl["user"], wl["item"], wl["rating"], wl["n_users"], wl["n_items"], device=dev)
tabs = E.SimEngine(lay, meta, "adjust_cosine", 50, wl["k"]).run()
plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
for rep in range(3):
    xe = X.XsimEngine(plan, 10)
    order = xe.unit_order[rank::world]
    work = (plan.ub[xe.unit_start].double() / xe.n_units_x[xe.unit_start].double())[order.long()]
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    res = xe.run(rank, world)
    ev[1].record()
    torch.cuda.synchronize(); t1 = time.perf_counter()
    dist.barrier(); torch.cuda.synchronize(); t2 = time.perf_counter()
    print("rep %d rank %d: run %.1f ms (device %.1f ms), with barrier %.1f ms; units %d, est. paths %.4g, heaviest unit %.3g"
          % (rep, rank, (t1 - t0) * 1e3, ev[0].elapsed_time(ev[1]), (t2 - t0) * 1e3, order.numel(), float(work.sum()),
             float(work.max())), flush=True)
# the kernel alone on this rank's share (no collective)
xe = X.XsimEngine(plan, 10)
keep = []
a = xe._args(keep)
nu, m, n = xe.n_units, xe.top_m, int(plan.start_item.numel())
z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
bufs = [z(nu, torch.int32), z(nu, torch.int64), z((nu, m), torch.int32), z((nu, m), torch.float64), z(nu, torch.int32)]
a.unit_count, a.unit_combos, a.unit_top_end, a.unit_top_xsim, a.unit_top_len = [N.ptr(t) for t in bufs]
order = xe.unit_order[rank::world].contiguous()
a.unit_order, a.n_units = N.ptr(order), int(order.numel())
for rep in range(2):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    N.check(N.lib().xmap_xsim_extend(a, torch.cuda.current_stream().cuda_stream), "x")
    torch.cuda.synchronize()
    print("rank %d kernel alone %.1f ms, paths %d" % (rank, (time.perf_counter() - t0) * 1e3, int(bufs[1].sum())), flush=True)
dist.destroy_process_group()
