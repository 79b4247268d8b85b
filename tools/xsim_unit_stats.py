"""Per-unit descriptor work of the X-SIM plan (pairs of the start x passes of the unit) next to its paths."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench
from xmap_b200 import engine as E, extend as X
wl = bench.make_workload(sys.argv[1] if len(sys.argv) > 1 else "cfg2")
dev = torch.device("cuda"); meta = E.to_device_meta(wl["meta"], dev)
lay = E.build_layout(wl["user"], wl["item"], wl["rating"], wl["n_users"], wl["n_items"], device=dev)
tabs = E.SimEngine(lay, meta, "adjust_cosine", 50, wl["k"]).run()
plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
xe = X.XsimEngine(plan, 10)
pairs_x = xe.lp_ptr[plan.leg_ptr[1:]] - xe.lp_ptr[plan.leg_ptr[:-1]]          # (leg, partner) pairs per start
us = xe.unit_start
desc = pairs_x[us] * xe.unit_npass.long()
paths = plan.ub[us].double() / xe.n_units_x[us].double()
cost = paths + 8.0 * desc.double()
print("starts %d units %d; pairs per start: max %d, mean %.1f; total descriptor look-ups %.4g vs paths %.4g" % (
    pairs_x.numel(), us.numel(), int(pairs_x.max()), float(pairs_x.double().mean()), float(desc.sum()), float(plan.ub.sum())))
o = torch.argsort(desc, descending=True)[:12]
for u in o.tolist():
    x = int(us[u])
    print("unit %d start %d: pairs %d x passes %d = %d look-ups, paths/unit %.4g (start: ub %d, T %d, units %d)" % (
        u, x, int(pairs_x[x]), int(xe.unit_npass[u]), int(desc[u]), float(paths[u]), int(plan.ub[x]), int(xe.T[x]), int(xe.n_units_x[x])))
q = torch.tensor([0.5, 0.9, 0.99, 0.999, 1.0], dtype=torch.float64, device=dev)
print("per-unit look-ups quantiles", torch.quantile(desc.double(), q).tolist())
print("per-unit paths quantiles", torch.quantile(paths, q).tolist())

# measured: SM cycles per unit (one full run with the per-unit clock on)
from xmap_b200 import _native as N
keep = []
a = xe._args(keep)
nu, m = xe.n_units, xe.top_m
z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
bufs = [z(nu, torch.int32), z(nu, torch.int64), z((nu, m), torch.int32), z((nu, m), torch.float64), z(nu, torch.int32)]
a.unit_count, a.unit_combos, a.unit_top_end, a.unit_top_xsim, a.unit_top_len = [N.ptr(t) for t in bufs]
cyc = z(nu, torch.int64)
a.unit_cycles = N.ptr(cyc)
a.unit_order, a.n_units = N.ptr(xe.unit_order), nu
N.check(N.lib().xmap_xsim_extend(a, torch.cuda.current_stream().cuda_stream), "x")
torch.cuda.synchronize()
ms = cyc.double() / 1.965e6
print("per-unit ms quantiles", torch.quantile(ms, q).tolist(), "sum %.1f warp-ms" % float(ms.sum()))
o = torch.argsort(cyc, descending=True)[:10]
for u in o.tolist():
    x = int(us[u])
    print("unit %d start %d: %.1f ms; pairs %d x passes %d, paths %d, ends %d, g [%d, %d) (start: ub %d, T %d, units %d)" % (
        u, x, float(ms[u]), int(pairs_x[x]), int(xe.unit_npass[u]), int(bufs[1][u]), int(bufs[0][u]), int(xe.unit_g0[u]),
        int(xe.unit_g1[u]), int(plan.ub[x]), int(xe.T[x]), int(xe.n_units_x[x])))
