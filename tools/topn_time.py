"""Top-N recommendation (recsim.top_n) for every user of the BASELINE.json configs[2] AlterEgo profile, built as
tools/cfg3_leg.py builds it, on the non-private item-kNN tables (k = 10).  Device-timed after a warm-up call.  One
JSON line: users, reverse-index visits, distinct overlap candidates, users per launch shape, ms and users/s, the GPU
name and power limit, and a check of sampled users against a host path that shares nothing with the kernels.

  python tools/topn_time.py [workload=cfg2] [n=10] [sample=2000] [out_dir]

The host path, per sampled user (the heaviest 20 by reverse-index bound included): the overlap candidates by numpy
from a reverse index built with numpy, scored by oracle/restate.recommender_predict(raw=True) (no decay), merged with
the items that score their average, in (average desc, index asc) order, and cut at n.  With out_dir the line is also
written to out_dir/topn_time_<workload>.json.
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def host_top_n(prof, ln, nb_idx, nb_sim, avg, users, n):
    """user -> (items, scores) by the host path described above.  prof: (user, item, rating, ts) numpy, list order."""
    import numpy as np
    from oracle import restate as RE
    pu, pi, pr, pt = prof
    n_items, k = nb_idx.shape
    m = np.arange(k)[None, :] < ln[:, None]
    rows = np.repeat(np.arange(n_items), ln)
    nbr = nb_idx[m]
    o = np.argsort(nbr.astype(np.int64) * n_items + rows, kind="stable")
    rev_ptr = np.zeros(n_items + 1, np.int64)
    rev_ptr[1:] = np.cumsum(np.bincount(nbr, minlength=n_items))
    rev = rows[o]
    ptr = np.zeros(n_items + 1, np.int64)
    ptr[1:] = np.cumsum(ln)
    fb = np.flatnonzero((ln > 0) & ~np.isnan(avg))
    fb = fb[np.lexsort((fb, -avg[fb]))]
    sel = np.isin(pu, users)
    su, si, sr, st = pu[sel], pi[sel], pr[sel], pt[sel]
    rated, cand = {}, {}
    for u in users:
        P = np.unique(si[su == u])
        C = np.unique(np.concatenate([rev[rev_ptr[j]:rev_ptr[j + 1]] for j in P])) if len(P) else np.zeros(0, np.int64)
        rated[u], cand[u] = P, C[~np.isin(C, P)]
    tu = np.concatenate([np.full(len(cand[u]), u) for u in users])
    ti = np.concatenate([cand[u] for u in users])
    raw0 = RE.recommender_predict(su, si, sr, st, ptr, nb_idx[m], nb_sim[m], avg, tu, ti, np.zeros(len(tu)),
                                  raw=True)[4]
    out, q = {}, 0
    for u in users:
        C = cand[u]
        s = raw0[q:q + len(C)]
        q += len(C)
        head = fb[:n + len(rated[u]) + len(C)]             # enough of the average order to fill n
        rest = head[~np.isin(head, rated[u]) & ~np.isin(head, C)][:n]
        items = np.r_[C[~np.isnan(s)], rest]
        scores = np.r_[s[~np.isnan(s)], avg[rest]]
        o = np.lexsort((items, -scores))[:n]
        out[u] = (items[o], scores[o])
    return out, len(ti)


def main():
    import numpy as np
    import torch
    import bench
    from cfg3_leg import alterego_profile
    from ingest_time import gpu_info
    from xmap_b200 import recsim as RS
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    n_sample = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
    wl = bench.make_workload(name)
    dev = torch.device("cuda")
    pu, pi, pr, pt, n_syn = alterego_profile(wl, dev)
    n_users, n_items = wl["n_users"], wl["n_items"]
    knn = RS.item_knn(pu, pi, pr, n_items, 50, 10)
    args = (pu, pi, pr, pt, n_users, knn, knn.nb, n)
    RS.top_n(*args)                                         # warm-up: module load, sort and allocator paths
    ms = []
    for _ in range(3):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        res = RS.top_n(*args)
        torch.cuda.synchronize(); ms.append((time.perf_counter() - t0) * 1e3)
    best = min(ms)
    # sampled check: the heaviest 20 users by reverse-index bound and random others
    rev_ptr, _ = RS.reverse_index(knn.nb)
    bound = torch.zeros(n_users, dtype=torch.int64, device=dev).index_add_(0, pu.long(), (rev_ptr[1:] - rev_ptr[:-1])[pi.long()])
    heavy = torch.argsort(bound, descending=True)[:20].cpu().numpy()
    rng = np.random.default_rng(2026)
    users = np.unique(np.r_[heavy, rng.choice(n_users, max(n_sample - 20, 0), replace=False)])[:n_sample]
    t0 = time.perf_counter()
    prof = tuple(x.cpu().numpy() for x in (pu, pi, pr, pt))
    host, host_pairs = host_top_n(prof, knn.nb.len.cpu().numpy(), knn.nb.idx.cpu().numpy(), knn.nb.sim.cpu().numpy(),
                                  knn.info[:, 0].cpu().numpy(), users, n)
    host_s = time.perf_counter() - t0
    idx, score, ln = res.idx.cpu().numpy(), res.score.cpu().numpy(), res.len.cpu().numpy()
    same, near = True, 0
    for u in users:
        hi, hs = host[u]
        L = len(hi)
        if ln[u] != L or not np.array_equal(score[u, :L].view(np.int64), hs.view(np.int64)):
            same = False
            continue
        diff = np.flatnonzero(idx[u, :L] != hi)
        near += len(diff)                                  # equal scores listed in another order would show here
        same = same and len(diff) == 0
    line = {"workload": "cfg3 @ %s" % bench.workload_label(wl, "adjust_cosine"), **gpu_info(),
            "tables": "non-private item-kNN, k=10, num_atleast=50", "n": n, "decay": False,
            "users": n_users, "profile_records": int(pu.numel()), "synthetic_records": n_syn,
            "reverse_index_visits": res.visits, "overlap_candidates": res.candidates,
            "warp_shape_users": res.warp_users, "cta_shape_users": res.cta_users,
            "top_n_ms": round(best, 3), "top_n_ms_runs": [round(x, 3) for x in ms],
            "users_per_s": n_users / (best * 1e-3),
            "sample_users": int(len(users)), "sample_heaviest_bound": int(bound.max().item()),
            "sample_host_pairs": host_pairs, "sample_host_s": round(host_s, 1),
            "sample_matches_host": bool(same), "sample_near_ties": near}
    print(json.dumps(line))
    if len(sys.argv) > 4:
        os.makedirs(sys.argv[4], exist_ok=True)
        with open(os.path.join(sys.argv[4], "topn_time_%s.json" % name), "w") as f:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
