"""BASELINE.json configs[2]: two-domain pipeline with differentially private AlterEgo generation (exponential
mechanism, Philox draws) followed by item-kNN prediction on the AlterEgo profile (RecommenderSim cosine_item ->
non-private neighbour selection -> item-based prediction + MAE).  Array-level calls (the C ABI through the Python
drivers), device-timed per stage.  One JSON line.

  python tools/cfg3_leg.py [workload=cfg2] [test_pairs=200000] [out_dir]

With out_dir the line is also written to out_dir/cfg3_leg_<workload>.json.  The GPU name and power limit are read
in the same run.

The RecommenderSim stage and the neighbour selection run as recsim.item_knn: the co-rating entries of one block of
item rows at a time are filled, radix-sorted and reduced (csrc/recsim.cu), so the whole profile's pairs never exist
at once.  The line gives the entry count, the number of passes and the largest row's entries.
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    import numpy as np
    import torch
    import bench
    from ingest_time import gpu_info
    from xmap_b200 import engine as E, extend as X, generate as G, recsim as RS
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    n_test = int(sys.argv[2]) if len(sys.argv) > 2 else 200000
    wl = bench.make_workload(name)
    dev = torch.device("cuda")
    meta = E.to_device_meta(wl["meta"], dev)
    T = {}

    def timed(key, fn):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize(); T[key] = (time.perf_counter() - t0) * 1e3
        return r
    for rep in range(2):                                   # second pass warm
        lay = timed("layout_ms", lambda: E.build_layout(wl["user"], wl["item"], wl["rating"], wl["n_users"], wl["n_items"], device=dev))
        eng = E.SimEngine(lay, meta, "adjust_cosine", 50, wl["k"])
        tabs = timed("similarity_ms", eng.run)
        plan = timed("extend_plan_ms", lambda: X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T))
        res = timed("extend_ms", lambda: X.XsimEngine(plan, 10).run())
        # private generation: exponential mechanism, eps = 0.6, mapping_range = 1 (parameters.yaml:22-25), Philox draws
        ch = timed("choose_exp_mech_ms", lambda: G.choose_mapping(res, "exp_mech", epsilon=0.6, mapping_range=1,
                                                                 sim_method="adjust_cosine", seed=20261018))
        mp = G.invert_mapping(res.start_item, ch, wl["n_items"])
        ou, oi, orr, ot = timed("alterego_ms", lambda: G.build_alterego(lay, wl["ts"], mp))
        # the AlterEgo profile: untouched target ratings + the synthetic records (generator.py:156-157)
        item_all = torch.as_tensor(wl["item"], device=dev).long()
        keep = meta.has_T[item_all]
        pu = torch.cat([torch.as_tensor(wl["user"], device=dev).long()[keep], ou.long()])
        pi = torch.cat([item_all[keep], oi.long()])
        pr = torch.cat([torch.as_tensor(wl["rating"], device=dev).double()[keep], orr])
        pt = torch.cat([torch.as_tensor(wl["ts"], device=dev)[keep], ot])
        o = torch.argsort(pu * wl["n_items"] + pi, stable=True)
        pu, pi, pr, pt = pu[o], pi[o], pr[o], pt[o]
        knn = timed("item_knn_ms", lambda: RS.item_knn(pu, pi, pr, wl["n_items"], 50, 10))
        # hidden test ratings: random (profile user, target item) pairs with integer ratings
        g = torch.Generator(device="cpu").manual_seed(7)
        t_items = torch.unique(pi).cpu()
        tu = pu[torch.randint(0, pu.numel(), (n_test,), generator=g).to(dev)].to(torch.int32)
        ti = t_items[torch.randint(0, t_items.numel(), (n_test,), generator=g)].to(dev).to(torch.int32)
        tr = torch.randint(1, 6, (n_test,), generator=g).double().to(dev)
        p0, p1, m0, m1 = timed("prediction_ms", lambda: RS.predict(pu, pi, pr, pt, wl["n_users"], knn, knn.nb, tu, ti, tr, 0.03))
        out = dict(T)
    line = {"workload": "cfg3 @ %s" % bench.workload_label(wl, "adjust_cosine"), **gpu_info(),
            "generation": "exponential mechanism, eps=0.6, mapping_range=1, Philox4x32-10(seed, row)",
            "stage_ms": {k: round(v, 3) for k, v in out.items()},
            "profile_records": int(pu.numel()), "synthetic_records": int(ou.numel()),
            "recsim_entries": knn.n_entries, "recsim_passes": knn.passes, "recsim_max_row_entries": knn.max_row_entries,
            "recsim_ms_per_pass": round(out["item_knn_ms"] / max(knn.passes, 1), 3),
            "recsim_entries_per_s": knn.n_entries / (out["item_knn_ms"] * 1e-3),
            "items_with_neighbours": int((knn.nb.len > 0).sum().item()),
            "test_pairs": n_test, "predicted": int((p0 >= 0).sum().item()),
            "mae_nodecay": m0, "mae_decay": m1,
            "note": "test ratings are random (no signal): the MAE only shows the stage runs end to end; parity of every stage "
                    "is pinned by tests/golden/*_recsim.npz and *_recpred.npz"}
    print(json.dumps(line))
    if len(sys.argv) > 3:
        os.makedirs(sys.argv[3], exist_ok=True)
        with open(os.path.join(sys.argv[3], "cfg3_leg_%s.json" % name), "w") as f:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
