"""RecommenderSim on the AlterEgo profile (C ABI section 5).

Reference: RecommenderSim.get_info / produce_pairwise / cosine_sim / calculate_sim with method
"cosine_item" (recommenderSim.py:29-62, 64-75, 90-132, 186-195), driven by
assist.recommender_calculate_sim_pipeline (assist.py:153-175).
"""
from dataclasses import dataclass

import torch

from . import _native as N


def _st():
    return torch.cuda.current_stream().cuda_stream


@dataclass
class RecSim:
    """Every directed item pair with at least one co-rating entry, sorted by (i, j) (self pairs included)."""
    i: torch.Tensor          # int32
    j: torch.Tensor          # int32
    n: torch.Tensor          # int64  co-rating entries
    sim: torch.Tensor        # f64    cosine * min(n, N) / N          (recommenderSim.py:121-122)
    ls: torch.Tensor         # f64    local sensitivity              (:98-116)
    info: torch.Tensor       # f64 [n_items, 3] = (average, norm2, count) over the records of the item (:29-62)
    n_entries: int


def cosine_item(user, item, rating, n_items, num_atleast=50, device="cuda"):
    """user / item / rating: the flat profile records in the order the reference receives them
    (only the order of a user's records matters: it fixes the arrival order of a pair's entries)."""
    L = N.lib()
    dev = torch.device(device)
    user = torch.as_tensor(user, dtype=torch.int64).to(dev)
    item = torch.as_tensor(item, dtype=torch.int32).to(dev).contiguous()
    rating = torch.as_tensor(rating, dtype=torch.float64).to(dev).contiguous()
    n_rec = int(user.numel())
    i64 = dict(dtype=torch.int64, device=dev)
    # ---- item info: records grouped by item ---------------------------------------------------------
    oi = torch.argsort(item.long(), stable=True)
    item_ptr = torch.zeros(n_items + 1, **i64)
    item_ptr[1:] = torch.cumsum(torch.bincount(item.long(), minlength=n_items), 0)
    info = torch.zeros((n_items, 3), dtype=torch.float64, device=dev)
    N.check(L.xmap_recsim_item_info(N.ptr(item_ptr), N.ptr(rating[oi].contiguous()), n_items, N.ptr(info), _st()),
            "xmap_recsim_item_info")
    # ---- co-rating entries: records grouped by user, list order kept ---------------------------------
    ou = torch.argsort(user, stable=True)
    u_s, it_s, r_s = user[ou], item[ou].contiguous(), rating[ou].contiguous()
    uniq, d = torch.unique_consecutive(u_s, return_counts=True)
    n_users = int(uniq.numel())
    user_ptr = torch.zeros(n_users + 1, **i64)
    user_ptr[1:] = torch.cumsum(d, 0)
    ent_off = torch.zeros(n_users + 1, **i64)
    ent_off[1:] = torch.cumsum(d * (d - 1), 0)
    total = int(ent_off[-1].item()) if n_users else 0
    key = torch.empty(total, **i64)
    src = torch.empty(total, **i64)
    N.check(L.xmap_recsim_fill_entries(N.ptr(user_ptr), N.ptr(ent_off), n_users, N.ptr(it_s), n_items, total,
                                       N.ptr(key), N.ptr(src), _st()), "xmap_recsim_fill_entries")
    key_s, perm = torch.sort(key, stable=True)          # CUB radix sort (library plumbing); stable: arrival order kept
    src_s = src[perm].contiguous()
    seg_key, cnt = torch.unique_consecutive(key_s, return_counts=True)
    n_pairs = int(seg_key.numel())
    seg_ptr = torch.zeros(n_pairs + 1, **i64)
    seg_ptr[1:] = torch.cumsum(cnt, 0)
    out_i = torch.empty(n_pairs, dtype=torch.int32, device=dev)
    out_j = torch.empty(n_pairs, dtype=torch.int32, device=dev)
    out_n = torch.empty(n_pairs, **i64)
    out_sim = torch.empty(n_pairs, dtype=torch.float64, device=dev)
    out_ls = torch.empty(n_pairs, dtype=torch.float64, device=dev)
    N.check(L.xmap_recsim_pairs(N.ptr(seg_ptr), N.ptr(seg_key.contiguous()), N.ptr(src_s), N.ptr(r_s), N.ptr(info),
                                n_items, n_pairs, int(num_atleast), N.ptr(out_i), N.ptr(out_j), N.ptr(out_n),
                                N.ptr(out_sim), N.ptr(out_ls), _st()), "xmap_recsim_pairs")
    return RecSim(out_i, out_j, out_n, out_sim, out_ls, info, total)


@dataclass
class Neighbors:
    idx: torch.Tensor        # int32 [n_items, k]
    sim: torch.Tensor        # f64   [n_items, k]
    len: torch.Tensor        # int32 [n_items]


def neighbors(rs, n_items, k=10):
    """RecommenderPrivacy.nonprivate_neighbor_selection + nonnoise_perturbation (recommenderPrivacy.py:141-189):
    {item: [(neighbour, sim)] first k by |sim|} as fixed-width tables."""
    L = N.lib()
    dev = rs.i.device
    row_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
    row_ptr[1:] = torch.cumsum(torch.bincount(rs.i.long(), minlength=n_items), 0)
    nb_idx = torch.full((n_items, k), -1, dtype=torch.int32, device=dev)
    nb_sim = torch.zeros((n_items, k), dtype=torch.float64, device=dev)
    nb_len = torch.zeros(n_items, dtype=torch.int32, device=dev)
    N.check(L.xmap_recsim_neighbors(N.ptr(row_ptr), N.ptr(rs.j.contiguous()), N.ptr(rs.sim.contiguous()), n_items, int(k),
                                    N.ptr(nb_idx), N.ptr(nb_sim), N.ptr(nb_len), _st()), "xmap_recsim_neighbors")
    return Neighbors(nb_idx, nb_sim, nb_len)


def private_neighbors(rs, n_items, mapping_range=10, privacy_epsilon=0.6, rpo=0.1, u_pick=None, u_noise=None, seed=0):
    """RecommenderPrivacy.private_neighbor_selection + noise_perturbation (recommenderPrivacy.py:35-139, 152-171) as the
    reference behaves under Python 3: ONE neighbour per item, drawn by the exponential mechanism over all its neighbours,
    its similarity plus Laplace noise.  u_pick / u_noise: one injected uniform per item THAT HAS NEIGHBOURS, in item
    order (the reference's np.random draws replayed), or None -> Philox4x32-10(seed, item).  Returns Neighbors with k = 1."""
    L = N.lib()
    dev = rs.i.device
    cnt = torch.bincount(rs.i.long(), minlength=n_items)
    row_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
    row_ptr[1:] = torch.cumsum(cnt, 0)
    # |sim| descending, stable (ties keep the (i, j) order), inside every item (recommenderPrivacy.py:123)
    o1 = torch.sort(rs.sim.abs(), descending=True, stable=True).indices
    o = o1[torch.sort(rs.i.long()[o1], stable=True).indices]
    nbr, sim, ls = rs.j[o].contiguous(), rs.sim[o].contiguous(), rs.ls[o].contiguous()

    def per_item(u):
        if u is None:
            return None
        u = torch.as_tensor(u, dtype=torch.float64).to(dev)
        have = torch.nonzero(cnt > 0).flatten()
        if u.numel() != have.numel():
            raise ValueError("need one uniform per item that has neighbours (%d), got %d" % (have.numel(), u.numel()))
        full = torch.zeros(n_items, dtype=torch.float64, device=dev)
        full[have] = u
        return full
    up, un = per_item(u_pick), per_item(u_noise)
    scratch = torch.empty(max(int(sim.numel()), 1), dtype=torch.float64, device=dev)
    nb_idx = torch.full((n_items, 1), -1, dtype=torch.int32, device=dev)
    nb_sim = torch.zeros((n_items, 1), dtype=torch.float64, device=dev)
    nb_len = torch.zeros(n_items, dtype=torch.int32, device=dev)
    N.check(L.xmap_recsim_private_neighbor(N.ptr(row_ptr), N.ptr(nbr), N.ptr(sim), N.ptr(ls), n_items, int(mapping_range),
                                           float(privacy_epsilon) / 2.0, float(rpo), N.ptr(up), N.ptr(un),
                                           int(seed) & (2 ** 64 - 1), N.ptr(scratch), N.ptr(nb_idx), N.ptr(nb_sim),
                                           N.ptr(nb_len), _st()), "xmap_recsim_private_neighbor")
    return Neighbors(nb_idx, nb_sim, nb_len)


def predict(user, item, rating, ts, n_users, rs, nb, test_user, test_item, test_rating=None, alpha=0.03):
    """RecommenderPrediction.item_based_recommendation + calculate_mae (recommenderPrediction.py:26-139) on the
    profile records (list order).  Returns (pred_nodecay, pred_decay, mae_nodecay, mae_decay); predictions are -1
    where the test item has no neighbour list, the MAEs are None without test ratings."""
    L = N.lib()
    dev = rs.i.device
    user = torch.as_tensor(user, dtype=torch.int64).to(dev)
    ou = torch.argsort(user, stable=True)
    prof_ptr = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
    prof_ptr[1:] = torch.cumsum(torch.bincount(user, minlength=n_users), 0)
    p_item = torch.as_tensor(item, dtype=torch.int32).to(dev)[ou].contiguous()
    p_rating = torch.as_tensor(rating, dtype=torch.float64).to(dev)[ou].contiguous()
    p_ts = torch.as_tensor(ts, dtype=torch.int64).to(dev)[ou].contiguous()
    # checked in int64 before the narrowing copy: the kernel indexes the profile by user and the neighbour
    # tables by item without a bound check
    tu = torch.as_tensor(test_user, dtype=torch.int64).flatten()
    ti = torch.as_tensor(test_item, dtype=torch.int64).flatten()
    n_test = int(tu.numel())
    if int(ti.numel()) != n_test:
        raise ValueError("test_user and test_item differ in length (%d, %d)" % (n_test, int(ti.numel())))
    n_tab = int(nb.idx.shape[0])
    if n_test and (int(tu.min()) < 0 or int(tu.max()) >= n_users):
        raise ValueError("test_user outside [0, %d)" % n_users)
    if n_test and (int(ti.min()) < 0 or int(ti.max()) >= n_tab):
        raise ValueError("test_item outside [0, %d)" % n_tab)
    tu = tu.to(device=dev, dtype=torch.int32).contiguous()
    ti = ti.to(device=dev, dtype=torch.int32).contiguous()
    p0 = torch.empty(n_test, dtype=torch.float64, device=dev)
    p1 = torch.empty(n_test, dtype=torch.float64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    k = int(nb.idx.shape[1])
    N.check(L.xmap_recsim_predict(N.ptr(prof_ptr), N.ptr(p_item), N.ptr(p_rating), N.ptr(p_ts), N.ptr(rs.info),
                                  N.ptr(nb.idx), N.ptr(nb.sim), N.ptr(nb.len), k, N.ptr(tu), N.ptr(ti), n_test,
                                  float(alpha), N.ptr(p0), N.ptr(p1), N.ptr(err), _st()), "xmap_recsim_predict")
    if int(err.item()):
        raise N.NativeError("prediction kernel error %d (4: more than 128 matching profile records)" % int(err.item()))
    mae0 = mae1 = None
    if test_rating is not None:
        tr = torch.as_tensor(test_rating, dtype=torch.float64).to(dev)
        ok = p0 >= 0
        cnt = int(ok.sum().item())
        if cnt:
            mae0 = float((tr[ok] - p0[ok]).abs().sum().item()) / cnt          # recommenderPrediction.py:116-139
            mae1 = float((tr[ok] - p1[ok]).abs().sum().item()) / cnt
    return p0, p1, mae0, mae1
