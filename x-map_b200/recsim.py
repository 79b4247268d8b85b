"""RecommenderSim on the AlterEgo profile (C ABI section 5).

Reference: RecommenderSim.get_info / produce_pairwise / cosine_sim / calculate_sim with method
"cosine_item" (recommenderSim.py:29-62, 64-75, 90-132, 186-195), driven by
assist.recommender_calculate_sim_pipeline (assist.py:153-175).
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import _native as N
from . import multi as M

# Peak device bytes per co-rating entry while a pass runs: key and record positions (16), the stable sort's keys,
# permutation and scratch (~32), the permuted positions (8), rounded up for the pair outputs.
ENTRY_BYTES = 64
INT32_MAX = (1 << 31) - 1


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


def row_entries(user, item, n_items):
    """Co-rating entries whose first record lies on each item: sum over the item's records of (d_u - 1), d_u the
    record count of the record's user.  One scatter-add; works on any device."""
    user = torch.as_tensor(user, dtype=torch.int64)
    item = torch.as_tensor(item, dtype=torch.int64).to(user.device)
    _, inv, d = torch.unique(user, return_inverse=True, return_counts=True)
    out = torch.zeros(n_items, dtype=torch.int64, device=user.device)
    return out.index_add_(0, item, d[inv] - 1)


def pass_plan(row_ent, budget, lo=0, hi=None):
    """Cut the item rows [lo, hi) into contiguous blocks of at most `budget` bytes (ENTRY_BYTES per entry), each as
    long as the budget allows.  Returns the block bounds [lo, ..., hi].  A row over the budget raises ValueError."""
    ent = torch.as_tensor(row_ent, dtype=torch.int64).cpu()
    hi = int(ent.numel()) if hi is None else hi
    if int(ent.numel()):
        big = int(torch.argmax(ent))
        if int(ent[big]) * ENTRY_BYTES > budget:
            raise ValueError("item row %d has %d co-rating entries (%d bytes), more than the pass budget of %d bytes"
                             % (big, int(ent[big]), int(ent[big]) * ENTRY_BYTES, budget))
    csum = torch.zeros(hi - lo + 1, dtype=torch.int64)
    csum[1:] = torch.cumsum(ent[lo:hi] * ENTRY_BYTES, 0)
    bounds = [lo]
    while len(bounds) == 1 or bounds[-1] < hi:          # an empty range is one empty block
        a = bounds[-1] - lo
        b = int(torch.searchsorted(csum, csum[a] + int(budget), right=True)) - 1      # largest b: csum[b] - csum[a] <= budget
        bounds.append(min(hi, lo + max(b, a + 1)))
    return bounds


def default_budget(dev):
    """Half of the device memory that is free or held unused by torch's caching allocator."""
    free, _ = torch.cuda.mem_get_info(dev)
    return (free + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)) // 2


def item_info(item, rating, n_items, device="cuda"):
    """(average, norm2, count) per item over its records (recommenderSim.py:29-62): [n_items, 3] float64."""
    L = N.lib()
    dev = torch.device(device)
    item = torch.as_tensor(item, dtype=torch.int64).to(dev)
    rating = torch.as_tensor(rating, dtype=torch.float64).to(dev)
    oi = torch.argsort(item, stable=True)
    item_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
    item_ptr[1:] = torch.cumsum(torch.bincount(item, minlength=n_items), 0)
    info = torch.zeros((n_items, 3), dtype=torch.float64, device=dev)
    N.check(L.xmap_recsim_item_info(N.ptr(item_ptr), N.ptr(rating[oi].contiguous()), n_items, N.ptr(info),
                                    N.stream()), "xmap_recsim_item_info")
    return info


class _Profile(object):
    """The profile records grouped by user (list order kept: it fixes the arrival order of a pair's entries), the item
    info and the co-rating entries of every item row."""

    def __init__(self, user, item, rating, n_items, device):
        dev = torch.device(device)
        user = torch.as_tensor(user, dtype=torch.int64).to(dev)
        item = torch.as_tensor(item, dtype=torch.int32).to(dev).contiguous()
        rating = torch.as_tensor(rating, dtype=torch.float64).to(dev).contiguous()
        self.dev, self.n_items, self.n_rec = dev, n_items, int(user.numel())
        self.info = item_info(item, rating, n_items, dev)
        ou = torch.argsort(user, stable=True)
        self.item, self.rating = item[ou].contiguous(), rating[ou].contiguous()
        _, d = torch.unique_consecutive(user[ou], return_counts=True)
        self.n_users = int(d.numel())
        self.user_ptr = torch.zeros(self.n_users + 1, dtype=torch.int64, device=dev)
        self.user_ptr[1:] = torch.cumsum(d, 0)
        self.rec_end = torch.repeat_interleave(self.user_ptr[1:], d)       # end of each record's user
        self.row_ent = row_entries(user, item, n_items)

    def pairs(self, i0, i1, num_atleast):
        """Fill, sort and reduce the co-rating entries of the item rows [i0, i1): (i, j, n, sim, ls) of every pair
        (i, j) with i in the rows, sorted by (i, j), and the entry count."""
        L, dev = N.lib(), self.dev
        i64 = dict(dtype=torch.int64, device=dev)
        pos = torch.arange(self.n_rec, **i64)
        inr = ((self.item >= i0) & (self.item < i1)).long()
        in_before = torch.zeros(self.n_rec + 1, **i64)
        in_before[1:] = torch.cumsum(inr, 0)
        ent_before = torch.zeros(self.n_rec + 1, **i64)
        ent_before[1:] = torch.cumsum(inr * (self.rec_end - pos - 1) + in_before[self.rec_end] - in_before[1:], 0)
        del pos, inr
        total = int(ent_before[-1].item()) if self.n_rec else 0
        key = torch.empty(total, **i64)
        src = torch.empty(total, **i64)
        N.check(L.xmap_recsim_fill_rows(N.ptr(self.user_ptr), self.n_users, N.ptr(in_before), N.ptr(ent_before), self.n_rec,
                                        N.ptr(self.item), self.n_items, int(i0), int(i1), total, N.ptr(key), N.ptr(src),
                                        N.stream()), "xmap_recsim_fill_rows")
        del in_before, ent_before
        key_s, perm = torch.sort(key, stable=True)          # CUB radix sort (library plumbing); stable: arrival order kept
        del key
        src_s = src[perm].contiguous()
        del src, perm
        seg_key, cnt = torch.unique_consecutive(key_s, return_counts=True)
        del key_s
        n_pairs = int(seg_key.numel())
        seg_ptr = torch.zeros(n_pairs + 1, **i64)
        seg_ptr[1:] = torch.cumsum(cnt, 0)
        out_i = torch.empty(n_pairs, dtype=torch.int32, device=dev)
        out_j = torch.empty(n_pairs, dtype=torch.int32, device=dev)
        out_n = torch.empty(n_pairs, **i64)
        out_sim = torch.empty(n_pairs, dtype=torch.float64, device=dev)
        out_ls = torch.empty(n_pairs, dtype=torch.float64, device=dev)
        N.check(L.xmap_recsim_pairs(N.ptr(seg_ptr), N.ptr(seg_key.contiguous()), N.ptr(src_s), N.ptr(self.rating),
                                    N.ptr(self.info), self.n_items, n_pairs, int(num_atleast), N.ptr(out_i), N.ptr(out_j),
                                    N.ptr(out_n), N.ptr(out_sim), N.ptr(out_ls), N.stream()), "xmap_recsim_pairs")
        return RecSim(out_i, out_j, out_n, out_sim, out_ls, self.info, total)

    def plan(self, budget, lo=0, hi=None):
        return pass_plan(self.row_ent, default_budget(self.dev) if budget is None else budget, lo, hi)


def pair_passes(user, item, rating, n_items, num_atleast=50, budget=None, device="cuda"):
    """cosine_item pass by pass: yields one RecSim per block of item rows (the pairs (i, j) with i in the block),
    blocks in row order, each filled, sorted and reduced within `budget` bytes (default: half the free memory)."""
    prof = _Profile(user, item, rating, n_items, device)
    bounds = prof.plan(budget)
    for i0, i1 in zip(bounds[:-1], bounds[1:]):
        yield prof.pairs(i0, i1, num_atleast)


def cosine_item(user, item, rating, n_items, num_atleast=50, device="cuda", budget=None):
    """user / item / rating: the flat profile records in the order the reference receives them
    (only the order of a user's records matters: it fixes the arrival order of a pair's entries).
    The pairs are computed in blocks of item rows of at most `budget` bytes each (pair_passes) and concatenated;
    the result does not depend on the budget."""
    parts = list(pair_passes(user, item, rating, n_items, num_atleast, budget, device))
    return RecSim(*(torch.cat([getattr(p, f) for p in parts]) for f in ("i", "j", "n", "sim", "ls")), parts[0].info,
                  sum(p.n_entries for p in parts))


@dataclass
class Neighbors:
    idx: torch.Tensor        # int32 [n_items, k]
    sim: torch.Tensor        # f64   [n_items, k]
    len: torch.Tensor        # int32 [n_items]


def _row_ptr(i, lo, n_rows):
    """[n_rows + 1] extents of the rows lo .. lo + n_rows - 1 in an i-sorted pair list whose rows lie in that range."""
    ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=i.device)
    ptr[1:] = torch.cumsum(torch.bincount(i.long() - lo, minlength=n_rows), 0)
    return ptr


def _neighbors_into(rs, i0, i1, nb):
    """Non-private selection for the rows [i0, i1) of nb (rs: the pairs of exactly those rows)."""
    N.check(N.lib().xmap_recsim_neighbors(N.ptr(_row_ptr(rs.i, i0, i1 - i0)), N.ptr(rs.j.contiguous()),
                                          N.ptr(rs.sim.contiguous()), i1 - i0, int(nb.idx.shape[1]),
                                          N.ptr(nb.idx[i0:i1]), N.ptr(nb.sim[i0:i1]), N.ptr(nb.len[i0:i1]),
                                          N.stream()), "xmap_recsim_neighbors")


def empty_tables(n_rows, k, dev):
    """Neighbour tables with no neighbour in any row: idx -1, sim 0, len 0."""
    return Neighbors(torch.full((n_rows, k), -1, dtype=torch.int32, device=dev),
                     torch.zeros((n_rows, k), dtype=torch.float64, device=dev),
                     torch.zeros(n_rows, dtype=torch.int32, device=dev))


def neighbors(rs, n_items, k=10):
    """RecommenderPrivacy.nonprivate_neighbor_selection + nonnoise_perturbation (recommenderPrivacy.py:141-189):
    {item: [(neighbour, sim)] first k by |sim|} as fixed-width tables."""
    nb = empty_tables(n_items, k, rs.i.device)
    if n_items > 0:
        _neighbors_into(rs, 0, n_items, nb)
    return nb


def per_item_uniforms(u, have, n_items, dev):
    """One injected uniform per item that has neighbours (have: those items, ascending) -> [n_items], or None."""
    if u is None:
        return None
    u = torch.as_tensor(u, dtype=torch.float64).to(dev)
    if u.numel() != have.numel():
        raise ValueError("need one uniform per item that has neighbours (%d), got %d" % (have.numel(), u.numel()))
    full = torch.zeros(n_items, dtype=torch.float64, device=dev)
    full[have] = u
    return full


def private_options(private, have, n_rows, dev):
    """private (a dict of private_neighbors' keywords) over their defaults, with u_pick / u_noise spread to one uniform
    per row (have: the rows that have a pair, ascending).  An unknown keyword raises TypeError."""
    opts = dict(privacy_epsilon=0.6, rpo=0.1, u_pick=None, u_noise=None, seed=0)
    unknown = set(private) - set(opts)
    if unknown:
        raise TypeError("unknown private selection options: %s" % sorted(unknown))
    opts.update(private)
    for u in ("u_pick", "u_noise"):
        opts[u] = per_item_uniforms(opts[u], have, n_rows, dev)
    return opts


def private_draw(row, nbr, sim, ls, rows, nb, mapping_range, opts):
    """Private selection into the rows `rows` (an index tensor or a slice) of nb from their pairs (row, nbr, sim, ls),
    each row's pairs in neighbour order.  opts: private_options.  The kernel runs over every row of nb, so the Philox
    counter and the uniforms stay indexed by the global row; rows without pairs here come out empty."""
    dev = sim.device
    n_rows = int(nb.idx.shape[0])
    row_ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
    row_ptr[1:] = torch.cumsum(torch.bincount(row, minlength=n_rows), 0)
    # |sim| descending, stable (ties keep the neighbour order), inside every row (recommenderPrivacy.py:123)
    o1 = torch.sort(sim.abs(), descending=True, stable=True).indices
    o = o1[torch.sort(row[o1], stable=True).indices]
    nbr, sim, ls = nbr[o].contiguous(), sim[o].contiguous(), ls[o].contiguous()
    scratch = torch.empty(max(int(sim.numel()), 1), dtype=torch.float64, device=dev)
    out = empty_tables(n_rows, 1, dev)
    N.check(N.lib().xmap_recsim_private_neighbor(N.ptr(row_ptr), N.ptr(nbr), N.ptr(sim), N.ptr(ls), n_rows,
                                                 int(mapping_range), float(opts["privacy_epsilon"]) / 2.0,
                                                 float(opts["rpo"]), N.ptr(opts["u_pick"]), N.ptr(opts["u_noise"]),
                                                 int(opts["seed"]) & (2 ** 64 - 1), N.ptr(scratch), N.ptr(out.idx),
                                                 N.ptr(out.sim), N.ptr(out.len), N.stream()),
            "xmap_recsim_private_neighbor")
    for a, b in zip((nb.idx, nb.sim, nb.len), (out.idx, out.sim, out.len)):
        a[rows] = b[rows]


def private_neighbors(rs, n_items, mapping_range=10, privacy_epsilon=0.6, rpo=0.1, u_pick=None, u_noise=None, seed=0):
    """RecommenderPrivacy.private_neighbor_selection + noise_perturbation (recommenderPrivacy.py:35-139, 152-171) as the
    reference behaves under Python 3: ONE neighbour per item, drawn by the exponential mechanism over all its neighbours,
    its similarity plus Laplace noise.  u_pick / u_noise: one injected uniform per item THAT HAS NEIGHBOURS, in item
    order (the reference's np.random draws replayed), or None -> Philox4x32-10(seed, item).  Returns Neighbors with k = 1."""
    dev = rs.i.device
    have = torch.nonzero(torch.bincount(rs.i.long(), minlength=n_items) > 0).flatten()
    opts = private_options(dict(privacy_epsilon=privacy_epsilon, rpo=rpo, u_pick=u_pick, u_noise=u_noise, seed=seed),
                           have, n_items, dev)
    nb = empty_tables(n_items, 1, dev)
    if n_items > 0:
        private_draw(rs.i.long(), rs.j, rs.sim, rs.ls, slice(0, n_items), nb, mapping_range, opts)
    return nb


@dataclass
class ItemKnn:
    """item_knn's result: the neighbour tables, the item info that predict reads, and what the passes did."""
    nb: Neighbors
    info: torch.Tensor       # f64 [n_items, 3] = (average, norm2, count)
    n_entries: int           # co-rating entries of the rows this process computed
    passes: int              # blocks of item rows this process filled, sorted and reduced
    max_row_entries: int     # entries of the largest item row (of the whole profile)


def item_knn(user, item, rating, n_items, num_atleast=50, k=10, private=None, budget=None, shard=False, group=None,
             device="cuda"):
    """RecommenderSim cosine_item followed by neighbour selection, pass by pass: each block of item rows (at most
    `budget` bytes of co-rating entries, default half the free memory) is filled, sorted and reduced, and only its
    rows of the neighbour tables are kept, so the pairs of the whole profile never exist at once.  The tables equal
    neighbors / private_neighbors on cosine_item's result, whatever the budget.

    private: None for the non-private selection of the first k neighbours, or a dict of private_neighbors' keywords
    (privacy_epsilon, rpo, u_pick, u_noise, seed) for the private one with mapping_range k.
    shard: split the item rows over the ranks of `group` (torch.distributed; every rank passes the whole profile) in
    contiguous blocks of equal entry counts; one all-gather then gives every rank the whole tables."""
    prof = _Profile(user, item, rating, n_items, device)
    dev = prof.dev
    if budget is None:
        budget = default_budget(dev)
    sh = M.RowShard(prof.row_ent, M.dist.get_rank(group), M.dist.get_world_size(group)) if shard else None
    lo, hi = (sh.lo, sh.hi) if sh is not None else (0, n_items)
    bounds = prof.plan(budget, lo, hi)                           # checks every row, so all ranks fail alike
    if private is not None:
        # an item has a pair iff it owns an entry
        opts = private_options(private, torch.nonzero(prof.row_ent > 0).flatten(), n_items, dev)
    nb = empty_tables(n_items, 1 if private is not None else k, dev)
    n_entries = passes = 0
    for i0, i1 in zip(bounds[:-1], bounds[1:]):
        if i1 == i0:
            continue
        rs = prof.pairs(i0, i1, num_atleast)
        n_entries += rs.n_entries
        passes += 1
        if private is None:
            _neighbors_into(rs, i0, i1, nb)
        else:
            private_draw(rs.i.long(), rs.j, rs.sim, rs.ls, slice(i0, i1), nb, k, opts)
        del rs
    if sh is not None:
        M.gather_selected([nb.idx, nb.sim, nb.len], sh, group=group)
    return ItemKnn(nb, prof.info, n_entries, passes,
                   int(prof.row_ent.max().item()) if n_items else 0)


def predict(user, item, rating, ts, n_users, rs, nb, test_user, test_item, test_rating=None, alpha=0.03):
    """RecommenderPrediction.item_based_recommendation + calculate_mae (recommenderPrediction.py:26-139) on the
    profile records (list order).  rs: a RecSim or an ItemKnn (only its item info is read).  Returns (pred_nodecay, pred_decay, mae_nodecay, mae_decay); predictions are -1
    where the test item has no neighbour list, the MAEs are None without test ratings."""
    L = N.lib()
    dev = rs.info.device
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
                                  float(alpha), N.ptr(p0), N.ptr(p1), N.ptr(err), N.stream()), "xmap_recsim_predict")
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


def index_set(t, n_max, dev, name="users"):
    """t as int64 on dev, checked to be a 1-D integer tensor of indices in [0, n_max)."""
    t = torch.as_tensor(t)
    if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
        raise ValueError("%s must be a 1-D integer tensor" % name)
    t = t.to(device=dev, dtype=torch.int64)
    if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n_max):
        raise ValueError("%s outside [0, %d)" % (name, n_max))
    return t


def query_users(users, n_users, dev):
    """The rows a call computes: every user for None, else `users` checked as an index set of distinct users."""
    if users is None:
        return torch.arange(max(n_users, 0), dtype=torch.int64, device=dev)
    sel = index_set(users, n_users, dev)
    if int(torch.unique(sel).numel()) != int(sel.numel()):
        raise ValueError("users must be distinct")
    return sel


def list_length(n, hi=N.TOPN_MAX):
    """n checked as the length of a top-N list: an integer in [1, hi]."""
    if isinstance(n, bool) or int(n) != n or not 1 <= int(n) <= hi:
        raise ValueError("n must be an integer in [1, %d], got %r" % (hi, n))
    return int(n)


def empty_lists(n_rows, n, dev):
    """(idx, score, len) of n_rows top-N lists of width n before any is filled: idx -1, score NaN, len 0."""
    return (torch.full((n_rows, n), -1, dtype=torch.int32, device=dev),
            torch.full((n_rows, n), float("nan"), dtype=torch.float64, device=dev),
            torch.zeros(n_rows, dtype=torch.int32, device=dev))


@dataclass
class TopN:
    """top_n's result: every user's list, and what the kernels did for the users this process ran."""
    idx: torch.Tensor        # int32 [n_users, n], -1 padded
    score: torch.Tensor      # f64   [n_users, n], NaN padded: the prediction before bound_rating
    len: torch.Tensor        # int32 [n_users]
    visits: int              # reverse-index entries visited
    candidates: int          # distinct overlap candidates scored or found NaN
    warp_users: int          # users of the one-warp shape
    cta_users: int           # users of the one-CTA shape


def reverse_index(nb):
    """For every item j the items i that list j as a neighbour, ascending: (rev_ptr int64 [n_items + 1], rev_item int32).
    One sort of the (neighbour, item) keys."""
    n_items, k = int(nb.idx.shape[0]), int(nb.idx.shape[1])
    dev = nb.idx.device
    valid = torch.arange(k, device=dev).unsqueeze(0) < nb.len.long().unsqueeze(1)
    j = nb.idx.long()[valid]
    i = torch.arange(n_items, device=dev).unsqueeze(1).expand(n_items, k)[valid]
    key = torch.sort(j * n_items + i).values
    rev_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
    rev_ptr[1:] = torch.cumsum(torch.bincount(j, minlength=n_items), 0)
    return rev_ptr, (key % max(n_items, 1)).to(torch.int32).contiguous()


def top_n(user, item, rating, ts, n_users, knn, nb, n, decay=False, alpha=0.03, shard=False, group=None, users=None):
    """Every user's first n items (1 <= n <= 64) by the item-based prediction BEFORE bound_rating
    (recommenderPrediction.py:26-103, the value predict rounds), without or with temporal decay.  The reference has
    no such function.  Candidates are the items with a neighbour list the user has no record on (real and synthetic
    records alike); order: score descending, then the smaller item index (-0.0 equals 0.0); a NaN score is never
    recommended.  An item none of whose neighbours the user rated scores its average, so a user without records gets
    the top of the average order, and a user with fewer than n candidates a shorter list.

    user / item / rating / ts: the profile records in list order; knn: an ItemKnn or a RecSim (its item info is read);
    nb: the neighbour tables (any k).  shard: split the users over the ranks of `group` (torch.distributed; every rank
    passes the whole profile and tables) in contiguous blocks of equal work; one all-gather then gives every rank
    every list.  The result does not depend on the launch shape, the tiling of the item axis or the world size.
    users: None for every user, or a 1-D integer tensor of distinct users in [0, n_users): only their rows are filled
    (the others keep the padding), and the counts refer to them; shard then splits these users.
    Raises NativeError (error 4) when a candidate gathers more than 128 matching profile records, as predict does."""
    n = list_length(n)
    L = N.lib()
    dev = knn.info.device
    n_items = int(nb.idx.shape[0])
    # checked in int64 before the narrowing copies: the kernels index the profile by user and the tables by item
    user = torch.as_tensor(user, dtype=torch.int64).to(dev).flatten()
    item = torch.as_tensor(item, dtype=torch.int64).to(dev).flatten()
    n_rec = int(user.numel())
    if int(item.numel()) != n_rec:
        raise ValueError("user and item differ in length (%d, %d)" % (n_rec, int(item.numel())))
    if n_users < 0 or (n_rec and (int(user.min()) < 0 or int(user.max()) >= n_users)):
        raise ValueError("user outside [0, %d)" % n_users)
    if n_rec and (int(item.min()) < 0 or int(item.max()) >= n_items):
        raise ValueError("item outside [0, %d)" % n_items)
    sel = query_users(users, n_users, dev)
    # the records grouped by user, stably by item inside each user: a candidate's entries are runs in list order
    o = torch.argsort(user * n_items + item, stable=True)
    prof_ptr = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
    prof_ptr[1:] = torch.cumsum(torch.bincount(user, minlength=n_users), 0)
    p_item = item[o].to(torch.int32).contiguous()
    p_rating = torch.as_tensor(rating, dtype=torch.float64).to(dev).flatten()[o].contiguous()
    p_ts = torch.as_tensor(ts, dtype=torch.int64).to(dev).flatten()[o].contiguous()
    rev_ptr, rev_item = reverse_index(nb)
    # per user: sum over its records j of |rev(j)|, the bound on the overlap candidates it visits (one scatter-add)
    bound = torch.zeros(n_users, dtype=torch.int64, device=dev).index_add_(0, user, (rev_ptr[1:] - rev_ptr[:-1])[item])
    sh, mine = M.shard_selected(sel, bound[sel], group) if shard else (None, sel)
    light = bound[mine] <= N.TOPN_WARP_BOUND
    warp_users = mine[light].to(torch.int32).contiguous()
    heavy = mine[~light]
    cta_users = heavy[torch.argsort(bound[heavy], descending=True, stable=True)].to(torch.int32).contiguous()
    # the items that score their average when unreached, by (average desc, index asc); + 0.0 makes -0.0 sort as 0.0
    avg = knn.info[:, 0]
    fb = torch.nonzero((nb.len > 0) & (avg == avg)).flatten()
    fb = fb[torch.sort(avg[fb] + 0.0, descending=True, stable=True).indices].to(torch.int32).contiguous()
    out_idx, out_score, out_len = empty_lists(n_users, n, dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    N.check(L.xmap_recsim_top_n(N.ptr(prof_ptr), N.ptr(p_item), N.ptr(p_rating), N.ptr(p_ts), N.ptr(knn.info.contiguous()),
                                N.ptr(nb.idx.contiguous()), N.ptr(nb.sim.contiguous()), N.ptr(nb.len.contiguous()),
                                int(nb.idx.shape[1]), n_items, N.ptr(rev_ptr), N.ptr(rev_item), N.ptr(fb), int(fb.numel()),
                                N.ptr(warp_users), int(warp_users.numel()), N.ptr(cta_users), int(cta_users.numel()), n,
                                float(alpha), 1 if decay else 0, N.ptr(out_idx), N.ptr(out_score), N.ptr(out_len),
                                N.ptr(stats), N.ptr(err), N.stream()), "xmap_recsim_top_n")
    if int(err.item()):
        raise N.NativeError("top-N kernel error %d (4: more than 128 matching profile records)" % int(err.item()))
    if sh is not None:
        M.gather_selected([out_idx, out_score, out_len], sh, None if users is None else sel, group)
    visits, cands = stats.tolist()
    return TopN(out_idx, out_score, out_len, visits, cands, int(warp_users.numel()), int(cta_users.numel()))


# 1 / log2(p + 2) for the list slots, computed on the host so that no device log2 enters a metric
DISCOUNT = 1.0 / np.log2(np.arange(N.TOPN_MAX, dtype=np.float64) + 2.0)


@dataclass
class RankMetrics:
    """rank_metrics' result: per evaluated user (in the order given) and the means over them."""
    hits: torch.Tensor       # int32 [n_eval]   hits among the first n slots
    precision: torch.Tensor  # f64   hits / n
    recall: torch.Tensor     # f64   hits / |R|
    ndcg: torch.Tensor       # f64   DCG / ideal DCG of min(n, |R|) hits
    ap: torch.Tensor         # f64   average precision, over min(n, |R|)
    mean: dict               # precision, recall, ndcg, map: exact sum (math.fsum) / n_eval; None without users
    coverage: float          # distinct recommended items / catalogue (None without a catalogue size)


def rank_metrics(top, users, rel_ptr, rel_item, n, catalogue=None):
    """Precision, recall, NDCG and average precision at n of the top-N lists of `users` (a TopN, or anything with
    idx [n_users, width] and len) against each user's relevant items: user users[q] has rel_item[rel_ptr[q]:
    rel_ptr[q + 1]], sorted ascending and unique, at least one (an item no list can hold still counts in |R|).
    The first min(len, n) slots of a list count (1 <= n <= width).  The reference has no ranking metrics; the
    definitions are in DESIGN.md section 3.6.  catalogue: the number of items that can be recommended (those with a
    neighbour list); coverage = distinct items in the counted slots / catalogue.  Raises ValueError before the launch."""
    import math
    idx, ln = top.idx, top.len
    dev = idx.device
    if idx.dim() != 2 or ln.dim() != 1 or int(ln.numel()) != int(idx.shape[0]):
        raise ValueError("top lists: idx must be [n_users, width] and len [n_users]")
    width = int(idx.shape[1])
    n = list_length(n, min(width, N.TOPN_MAX))
    u = index_set(users, int(idx.shape[0]), dev)           # repeats allowed
    m = int(u.numel())
    ptr = torch.as_tensor(rel_ptr).to(device=dev, dtype=torch.int64).flatten()
    it = torch.as_tensor(rel_item).to(device=dev, dtype=torch.int64).flatten()
    if int(ptr.numel()) != m + 1 or int(ptr[0]) != 0 or int(ptr[-1]) != int(it.numel()):
        raise ValueError("rel_ptr must have len(users) + 1 entries, from 0 to len(rel_item)")
    if m and int((ptr[1:] - ptr[:-1]).min()) < 1:
        raise ValueError("every evaluated user needs at least one relevant item")
    if it.numel() and (int(it.min()) < 0 or int(it.max()) > INT32_MAX):
        raise ValueError("rel_item outside [0, 2^31)")
    if it.numel() > 1:
        start = torch.zeros(int(it.numel()), dtype=torch.bool, device=dev)
        start[ptr[:-1]] = True
        if bool(((it[1:] <= it[:-1]) & ~start[1:]).any()):
            raise ValueError("each user's relevant items must be sorted ascending and unique")
    out = [torch.zeros(m, dtype=torch.int32, device=dev)] + [torch.zeros(m, dtype=torch.float64, device=dev)
                                                             for _ in range(4)]
    # the narrowed copies stay referenced until the launch: a freed temporary's block could back the next one
    disc = torch.from_numpy(DISCOUNT).to(dev)
    idx_c, ln32 = idx.contiguous(), ln.to(torch.int32).contiguous()
    u32, it32 = u.to(torch.int32).contiguous(), it.to(torch.int32).contiguous()
    N.check(N.lib().xmap_recsim_rank_metrics(N.ptr(idx_c), N.ptr(ln32), width, N.ptr(u32), m, N.ptr(ptr), N.ptr(it32),
                                             N.ptr(disc), n, *(N.ptr(t) for t in out), N.stream()),
            "xmap_recsim_rank_metrics")
    mean = None
    if m:
        mean = {k: math.fsum(t.cpu().tolist()) / m for k, t in zip(("precision", "recall", "ndcg", "map"), out[1:])}
    coverage = None
    if catalogue:
        slots = torch.arange(n, device=dev).unsqueeze(0) < ln[u].long().unsqueeze(1)
        coverage = int(torch.unique(idx[u][:, :n][slots]).numel()) / int(catalogue)
    return RankMetrics(*out, mean, coverage)
