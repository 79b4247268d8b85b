"""User-based kNN (usersim.py, DESIGN.md 3.9) on the BASELINE.json configs[2] AlterEgo profile, built as
tools/cfg3_leg.py builds it, k = 10, non-private.  Device-timed after a warm-up call.  One JSON line:

- the profile's sum over items of c_i (c_i - 1): the co-rating entries the item-based path on the transposed profile
  would materialise (64 B each);
- per row: co-rating products, distinct neighbours and passes (quantiles), and the rows per launch shape;
- the time of user_knn for 6 215 users (the size of the cfg2 evaluation's test-user set) and for 2 000 users, both
  fixed random samples, and for every user when the 6 215-user rate predicts under `all_limit_s` seconds;
- the time of the prediction (200 000 random pairs of the 6 215 users) and of the top-10 of those users;
- products/s, the GPU name and power limit;
- a check of sampled rows (the 5 heaviest by products included) against a host restatement: numpy sums of the
  products per (u, v) with np.bincount, the same cosine and significance weighting, the first 10 by |sim| then the
  smaller user.  Sims agree to 1e-12 relative and lists are equal except where |sim| ties within 1e-12.

  python tools/usersim_time.py [workload=cfg2] [all_limit_s=120] [out_dir]
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def host_rows(users, t_user, t_item, t_rating, item_ptr, u_recs, norm, n_users, num_atleast, k):
    """user -> (neighbours, sims) by the restatement described above."""
    import numpy as np
    out = {}
    for u in users:
        acc = np.zeros(n_users)
        cnt = np.zeros(n_users, np.int64)
        for r in u_recs[u]:
            i = t_item[r]
            lo, hi = item_ptr[i], item_ptr[i + 1]
            b = np.arange(lo, hi)
            b = b[b != r]
            acc += np.bincount(t_user[b], weights=t_rating[r] * t_rating[b], minlength=n_users)
            cnt += np.bincount(t_user[b], minlength=n_users)
        v = np.flatnonzero(cnt)
        nn = norm[u] * norm[v]
        sim = np.where(nn != 0, acc[v] / np.where(nn != 0, nn, 1.0), 0.0) * np.minimum(cnt[v], num_atleast) / num_atleast
        o = np.lexsort((v, -np.abs(sim)))[:k]
        out[u] = (v[o], sim[o])
    return out


def main():
    import numpy as np
    import torch
    import bench
    from cfg3_leg import alterego_profile
    from ingest_time import gpu_info
    from xmap_b200 import usersim as US
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    all_limit = float(sys.argv[2]) if len(sys.argv) > 2 else 120.0
    wl = bench.make_workload(name)
    dev = torch.device("cuda")
    pu, pi, pr, pt, n_syn = alterego_profile(wl, dev)
    n_users, n_items = wl["n_users"], wl["n_items"]
    c = torch.bincount(pi, minlength=n_items)
    entries = int((c * (c - 1)).sum())
    rng = np.random.default_rng(2026)
    present = torch.unique(pu).cpu().numpy()
    test_users = torch.from_numpy(np.sort(rng.choice(present, 6215, replace=False))).to(dev)
    sample = torch.from_numpy(np.sort(rng.choice(present, 2000, replace=False))).to(dev)

    def timed(fn, reps=3, warm=True):
        if warm:
            fn()                                              # warm-up: module load, sort and allocator paths
        ms, res = [], None
        for _ in range(reps):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize(); ms.append((time.perf_counter() - t0) * 1e3)
        return min(ms), ms, res

    ms_test, runs_test, knn = timed(lambda: US.user_knn(pu, pi, pr, n_users, n_items, 50, 10, users=test_users))
    ms_sample, _, knn_s = timed(lambda: US.user_knn(pu, pi, pr, n_users, n_items, 50, 10, users=sample))
    ms_all = knn_all = None
    if ms_test * 1e-3 * len(present) / 6215 <= all_limit:
        ms_all, _, knn_all = timed(lambda: US.user_knn(pu, pi, pr, n_users, n_items, 50, 10), reps=1, warm=False)
    # prediction and top-10 of the test users on their rows
    g = torch.Generator().manual_seed(7)
    tu = test_users[torch.randint(0, 6215, (200000,), generator=g).to(dev)]
    ti = torch.randint(0, n_items, (200000,), generator=g).to(dev)
    ms_pred, _, pred = timed(lambda: US.predict(pu, pi, pr, pt, n_items, knn, knn.nb, tu, ti))
    ms_top, _, top = timed(lambda: US.top_n(pu, pi, pr, pt, n_users, n_items, knn, knn.nb, 10, users=test_users))
    # per row statistics over the test users
    prof = US.UserProfile(pu, pi, pr, n_users, n_items, dev)
    rp = prof.row_products[test_users].double().cpu().numpy()
    q = lambda a: {p: float(np.quantile(a, p / 100)) for p in (50, 90, 99, 100)}
    # the sampled check
    heavy = test_users[torch.argsort(prof.row_products[test_users], descending=True)[:5]].cpu().numpy()
    check = np.unique(np.r_[heavy, rng.choice(test_users.cpu().numpy(), 45, replace=False)])
    t_user, t_item = prof.t_user.cpu().numpy(), prof.t_item.cpu().numpy()
    t_rating, item_ptr = prof.t_rating.cpu().numpy(), prof.item_ptr.cpu().numpy()
    u_rec, u_ptr = prof.u_rec.cpu().numpy(), prof.u_ptr.cpu().numpy()
    u_recs = {u: u_rec[u_ptr[u]:u_ptr[u + 1]] for u in check}
    t0 = time.perf_counter()
    host = host_rows(check, t_user, t_item, t_rating, item_ptr, u_recs, knn.info[:, 1].cpu().numpy(), n_users, 50, 10)
    host_s = time.perf_counter() - t0
    idx, sim, ln = knn.nb.idx.cpu().numpy(), knn.nb.sim.cpu().numpy(), knn.nb.len.cpu().numpy()
    ok, near, max_rel = True, 0, 0.0
    for u in check:
        hv, hs = host[u]
        L = len(hv)
        if ln[u] != L:
            ok = False
            continue
        rel = np.abs(np.abs(sim[u, :L]) - np.abs(hs)) / np.maximum(np.abs(hs), 1e-300)
        max_rel = max(max_rel, float(rel.max()) if L else 0.0)
        ok = ok and bool((rel <= 1e-12).all())
        d = np.flatnonzero(idx[u, :L] != hv)
        if len(d):                                            # allowed only inside a run of |sim| equal to 1e-12
            near += len(d)
            ok = ok and bool(np.all(np.abs(np.abs(sim[u, d]) - np.abs(hs[d])) <= 1e-12 * np.abs(hs[d])))
    line = {"workload": "cfg3 @ %s" % bench.workload_label(wl, "adjust_cosine"), **gpu_info(),
            "tables": "non-private user-kNN, k=10, num_atleast=50",
            "users": n_users, "profile_users": int(len(present)), "items": n_items,
            "profile_records": int(pu.numel()), "synthetic_records": n_syn,
            "item_entries_sum_c_i_c_i_minus_1": entries,
            "item_entries_bytes_at_64B": entries * 64,
            "test_users": 6215, "test_row_products": q(rp),
            "test_row_distinct_neighbours_total": knn.pairs, "test_passes_total": knn.passes,
            "test_products_total": knn.products, "test_warp_rows": knn.warp_rows, "test_cta_rows": knn.cta_rows,
            "user_knn_test_ms": round(ms_test, 3), "user_knn_test_ms_runs": [round(x, 3) for x in runs_test],
            "user_knn_test_products_per_s": knn.products / (ms_test * 1e-3),
            "user_knn_sample2000_ms": round(ms_sample, 3), "sample2000_products": knn_s.products,
            "user_knn_all_ms": None if ms_all is None else round(ms_all, 3),
            "all_products": None if knn_all is None else knn_all.products,
            "all_passes": None if knn_all is None else knn_all.passes,
            "all_products_per_s": None if knn_all is None else knn_all.products / (ms_all * 1e-3),
            "predict_200k_pairs_ms": round(ms_pred, 3), "predicted": int((pred[0] >= 0).sum()),
            "top10_test_users_ms": round(ms_top, 3), "top10_visits": top.visits, "top10_candidates": top.candidates,
            "top10_warp_users": top.warp_users, "top10_cta_users": top.cta_users,
            "check_rows": int(len(check)), "check_heaviest_products": int(prof.row_products[test_users].max()),
            "check_host_s": round(host_s, 1), "check_max_rel": max_rel, "check_near_ties": near,
            "sample_check": bool(ok)}
    print(json.dumps(line))
    if len(sys.argv) > 3:
        os.makedirs(sys.argv[3], exist_ok=True)
        with open(os.path.join(sys.argv[3], "usersim_time_%s.json" % name), "w") as f:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
