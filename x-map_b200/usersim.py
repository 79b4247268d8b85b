"""User-based kNN on the AlterEgo profile (C ABI section 9, DESIGN.md section 3.9).

The project's definition: user-based = the item-based stage (recsim.py) with the roles of user and item exchanged,
stage by stage.  cosine_user similarity and its neighbour selection run in csrc/usersim.cu, one similarity row per
query user accumulated on chip (the pairs of the whole profile are never materialised); the prediction is
xmap_recsim_predict on the transposed profile (predict); the top-N has its own kernel (top_n).
"""
from dataclasses import dataclass

import torch

from . import _native as N
from . import multi as M
from . import recsim as RS


def scale_base(max_dup):
    """qbase = 62 - ceil(log2 m) of the fixed-point inner product, m the largest record count of one (user, item)."""
    return 62 - max(0, (int(max_dup) - 1).bit_length())


def norm_exponents(norm):
    """E per user with 2^(E-1) <= norm < 2^E (0 for a zero norm), as frexp gives it."""
    _, e = torch.frexp(norm)
    return torch.where(norm > 0, e, torch.zeros_like(e)).to(torch.int32).contiguous()


class UserProfile(object):
    """The profile twice: grouped by item, sorted by (item, user, list position), and each user's records as positions
    in that order; the user info (average, norm2, count) over each user's records in list order."""

    def __init__(self, user, item, rating, n_users, n_items, device="cuda", ts=None):
        dev = torch.device(device)
        user = torch.as_tensor(user, dtype=torch.int64).to(dev).flatten()
        item = torch.as_tensor(item, dtype=torch.int64).to(dev).flatten()
        rating = torch.as_tensor(rating, dtype=torch.float64).to(dev).flatten()
        n_rec = int(user.numel())
        if int(item.numel()) != n_rec or int(rating.numel()) != n_rec:
            raise ValueError("user, item and rating differ in length")
        if n_rec and (int(user.min()) < 0 or int(user.max()) >= n_users):
            raise ValueError("user outside [0, %d)" % n_users)
        if n_rec and (int(item.min()) < 0 or int(item.max()) >= n_items):
            raise ValueError("item outside [0, %d)" % n_items)
        if n_rec and not bool(torch.isfinite(rating).all()):
            raise ValueError("ratings must be finite")
        self.dev, self.n_users, self.n_items, self.n_rec = dev, n_users, n_items, n_rec
        self.info = RS.item_info(user, rating, n_users, dev)         # the item info of the transposed profile
        o = torch.argsort(item * max(n_users, 1) + user, stable=True)          # (item, user, list position)
        self.t_user = user[o].to(torch.int32).contiguous()
        self.t_item = item[o].to(torch.int32).contiguous()
        self.t_rating = rating[o].contiguous()
        self.t_ts = None if ts is None else torch.as_tensor(ts, dtype=torch.int64).to(dev).flatten()[o].contiguous()
        c = torch.bincount(item, minlength=n_items)
        self.item_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
        self.item_ptr[1:] = torch.cumsum(c, 0)
        self.u_rec = torch.argsort(self.t_user.long(), stable=True).contiguous()   # ascending positions per user
        self.u_ptr = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
        self.u_ptr[1:] = torch.cumsum(torch.bincount(user, minlength=n_users), 0)
        self.uexp = norm_exponents(self.info[:, 1])
        dup = torch.unique(user * max(n_items, 1) + item, return_counts=True)[1]
        self.qbase = scale_base(int(dup.max()) if n_rec else 1)
        # per user: co-rating products (sum over its records of c_i - 1), the bound on its distinct neighbours
        self.row_products = torch.zeros(n_users, dtype=torch.int64, device=dev).index_add_(0, user, c[item] - 1)


@dataclass
class UserKnn:
    """user_knn's result: the neighbour tables over users, the user info that predict reads, and what the kernels did
    for the rows this process computed."""
    nb: RS.Neighbors
    info: torch.Tensor       # f64 [n_users, 3] = (average, norm2, count)
    products: int            # co-rating products accumulated
    pairs: int               # distinct (row, neighbour) pairs
    passes: int              # tiles of the neighbour axis walked, over all rows
    warp_rows: int
    cta_rows: int
    blocks: int              # emit blocks (private mode), else 0


def _launch(prof, rows, cta, tile, num_atleast, k, nb, emit, stats, err):
    e_ptr, e_v, e_n, e_sim, e_ls, e_len = emit if emit is not None else (None,) * 6
    if int(rows.numel()) == 0:
        return
    N.check(N.lib().xmap_usersim_rows(N.ptr(prof.item_ptr), N.ptr(prof.t_user), N.ptr(prof.t_item), N.ptr(prof.t_rating),
                                      N.ptr(prof.u_ptr), N.ptr(prof.u_rec), N.ptr(prof.info), N.ptr(prof.uexp),
                                      prof.n_users, prof.qbase, int(num_atleast), int(k), N.ptr(rows), int(rows.numel()),
                                      1 if cta else 0, int(tile), N.ptr(nb.idx) if nb else None,
                                      N.ptr(nb.sim) if nb else None, N.ptr(nb.len) if nb else None, N.ptr(e_ptr),
                                      N.ptr(e_v), N.ptr(e_n), N.ptr(e_sim), N.ptr(e_ls), N.ptr(e_len), N.ptr(stats),
                                      N.ptr(err), N.stream()), "xmap_usersim_rows")


def user_knn(user, item, rating, n_users, n_items, num_atleast=50, k=10, private=None, users=None, budget=None,
             shard=False, group=None, device="cuda", shape=None, tile=None, emit_cap=None):
    """RecommenderSim cosine_user followed by neighbour selection: the item-based stage with the roles of user and item
    exchanged (DESIGN.md 3.9).  Returns UserKnn; its tables have a row per user, filled for the query users.

    private: None for the non-private first k neighbours (select mode: the running top-k stays on chip), or a dict of
    recsim.private_neighbors' keywords (privacy_epsilon, rpo, u_pick, u_noise, seed) for the private one with
    mapping_range k: the rows' pairs are emitted in blocks of query users of at most `budget` bytes (default half the
    free memory), sorted stably by |sim| and drawn by xmap_recsim_private_neighbor.  u_pick / u_noise hold one uniform
    per user that has a pair, in user order, as recsim's do per item.
    users: None for every user, or a 1-D integer tensor of distinct users: only their rows are computed (the others
    keep length 0).  shard: split the query users over the ranks of `group` in blocks of equal products, then one
    all-gather.  The result does not depend on shard, users (for the rows computed), budget, shape or tile.
    shape: None (warp rows up to XMAP_USERSIM_WARP_BOUND products, CTA rows above), "warp" or "cta" for every row;
    tile: cells per pass (None: the shape's default); emit_cap: per-row extent override, for tests of the overflow."""
    prof = UserProfile(user, item, rating, n_users, n_items, device)
    dev = prof.dev
    sel = RS.query_users(users, n_users, dev)
    sh, mine = M.shard_selected(sel, prof.row_products[sel], group) if shard else (None, sel)
    heavy = _launch_shape(prof.row_products[mine] > N.USERSIM_WARP_BOUND, shape)
    groups = [(mine[~heavy], False), (mine[heavy], True)]
    stats = torch.zeros(3, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    blocks = 0
    if private is None:
        nb = RS.empty_tables(n_users, k, dev)
        for rows, cta in groups:
            t = tile or (N.USERSIM_CTA_TILE if cta else N.USERSIM_WARP_TILE)
            _launch(prof, rows.to(torch.int32).contiguous(), cta, t, num_atleast, k, nb, None, stats, err)
    else:
        # a user has a pair iff it owns a product
        opts = RS.private_options(private, torch.nonzero(prof.row_products > 0).flatten(), n_users, dev)
        nb = RS.empty_tables(n_users, 1, dev)
        for rows, row, v, _n, sim, ls in _emit_blocks(prof, groups, num_atleast, budget, tile, emit_cap, stats, err):
            blocks += 1
            RS.private_draw(row, v, sim, ls, rows, nb, k, opts)
    if int(err.item()):
        raise N.NativeError("user similarity kernel error %d" % int(err.item()))
    if sh is not None:
        M.gather_selected([nb.idx, nb.sim, nb.len], sh, None if users is None else sel, group)
    products, pairs, passes = stats.tolist()
    return UserKnn(nb, prof.info, products, pairs, passes, int((~heavy).sum()), int(heavy.sum()), blocks)


def _launch_shape(heavy, shape):
    """heavy (the rows their work sends to the one-CTA shape), or every row in the shape `shape` names."""
    if shape == "warp":
        return torch.zeros_like(heavy)
    if shape == "cta":
        return torch.ones_like(heavy)
    if shape is not None:
        raise ValueError("shape must be None, 'warp' or 'cta'")
    return heavy


def _emit_blocks(prof, groups, num_atleast, budget, tile, emit_cap, stats, err):
    """Emit mode over the query rows of each (rows, cta) group, in blocks of at most `budget` bytes: yields (rows of
    the block, then of every pair emitted for them its row, v, n, sim and ls), each row's pairs in user order."""
    dev = prof.dev
    if budget is None:
        budget = RS.default_budget(dev)
    for rows, cta in groups:
        bound = torch.clamp(prof.row_products[rows], max=prof.n_users)
        # recsim.ENTRY_BYTES per pair: (v, n, sim, ls) and the private draw's two stable sorts fit in it
        bounds = RS.pass_plan(bound, budget)
        t = tile or (N.USERSIM_EMIT_CTA_TILE if cta else N.USERSIM_WARP_TILE)
        for b0, b1 in zip(bounds[:-1], bounds[1:]):
            if b1 == b0:
                continue
            r = rows[b0:b1]
            cap = bound[b0:b1] if emit_cap is None else torch.full_like(bound[b0:b1], int(emit_cap))
            e_ptr = torch.zeros(b1 - b0 + 1, dtype=torch.int64, device=dev)
            e_ptr[1:] = torch.cumsum(cap, 0)
            tot = int(e_ptr[-1])
            pairs = [torch.empty(max(tot, 1), dtype=dt, device=dev)                     # v, n, sim, ls
                     for dt in (torch.int32, torch.int64, torch.float64, torch.float64)]
            e_len = torch.zeros(b1 - b0, dtype=torch.int64, device=dev)
            _launch(prof, r.to(torch.int32).contiguous(), cta, t, num_atleast, 1, None, (e_ptr, *pairs, e_len), stats,
                    err)
            if int(err.item()):
                raise N.NativeError("user similarity kernel error %d (2: a row has more pairs than its extent)"
                                    % int(err.item()))
            row_of = torch.repeat_interleave(torch.arange(b1 - b0, device=dev), cap)
            keep = torch.arange(tot, device=dev) - e_ptr[:-1][row_of] < e_len[row_of]    # the written part of each extent
            yield (r, r[row_of[keep]]) + tuple(p[:tot][keep] for p in pairs)


def pair_blocks(user, item, rating, n_users, n_items, num_atleast=50, budget=None, device="cuda"):
    """cosine_user block by block: yields (u, v, n, sim, ls) of every pair (u, v) of a block of users (ascending),
    sorted by (u, v), each block emitted within `budget` bytes (default: half the free memory)."""
    prof = UserProfile(user, item, rating, n_users, n_items, device)
    rows = torch.arange(n_users, dtype=torch.int64, device=prof.dev)
    stats = torch.zeros(3, dtype=torch.int64, device=prof.dev)
    err = torch.zeros(1, dtype=torch.int32, device=prof.dev)
    for _, u, v, n, sim, ls in _emit_blocks(prof, [(rows, False)], num_atleast, budget, None, None, stats, err):
        yield u.to(torch.int32), v, n, sim, ls


def predict(user, item, rating, ts, n_items, knn, nb, test_user, test_item, test_rating=None, alpha=0.03):
    """The user-based prediction: recsim.predict on the transposed profile (p0(u, i) = avg_u + sum over the
    neighbours v of u and v's records on i of sim (r - avg_v) / sum |sim|; -1 where u has no neighbour list).
    knn: a UserKnn (its user info is read); nb: its tables.  Returns (pred_nodecay, pred_decay, mae_nodecay, mae_decay)."""
    return RS.predict(item, user, rating, ts, n_items, knn, nb, test_item, test_user, test_rating, alpha)


def top_n(user, item, rating, ts, n_users, n_items, knn, nb, n, decay=False, alpha=0.03, users=None, shape=None,
          tile=None):
    """Every (or each listed) user's first n (1 <= n <= 64) items by the user-based prediction before bound_rating,
    without or with decay, over the profile items the user has no record on; order: score descending, then the smaller
    item; NaN never listed.  An item none of the user's neighbours rated scores avg_u.  A user with no neighbour list
    gets an empty list.  Returns recsim.TopN (rows of users not listed keep the padding).  shape: None (one warp per user
    whose neighbours hold at most XMAP_TOPN_WARP_BOUND records, one CTA above), "warp" or "cta"."""
    n = RS.list_length(n)
    if ts is None:
        raise ValueError("ts is required: the decay order and the kernels read a time per record")
    if tile is not None and (isinstance(tile, bool) or int(tile) < 32):
        raise ValueError("tile must be an integer >= 32, got %r" % (tile,))
    dev = knn.info.device
    prof = UserProfile(user, item, rating, n_users, n_items, dev, ts=ts)
    sel = RS.query_users(users, n_users, dev)
    user = torch.as_tensor(user, dtype=torch.int64).to(dev).flatten()
    item = torch.as_tensor(item, dtype=torch.int64).to(dev).flatten()
    o = torch.argsort(user * max(n_items, 1) + item, stable=True)
    up_item = item[o].to(torch.int32).contiguous()
    d = prof.u_ptr[1:] - prof.u_ptr[:-1]
    k = int(nb.idx.shape[1])
    valid = torch.arange(k, device=dev).unsqueeze(0) < nb.len.long().unsqueeze(1)
    bound = (d[nb.idx.long().clamp(min=0)] * valid).sum(1)
    heavy = _launch_shape(bound[sel] > N.TOPN_WARP_BOUND, shape)
    out_idx, out_score, out_len = RS.empty_lists(n_users, n, dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    info, nbi, nbs, nbl = knn.info.contiguous(), nb.idx.contiguous(), nb.sim.contiguous(), nb.len.contiguous()
    for cta in (False, True):
        rows = sel[heavy if cta else ~heavy].to(torch.int32).contiguous()
        if int(rows.numel()) == 0:
            continue
        N.check(N.lib().xmap_usersim_top_n(N.ptr(prof.u_ptr), N.ptr(up_item), N.ptr(prof.item_ptr), N.ptr(prof.t_user),
                                           N.ptr(prof.t_rating), N.ptr(prof.t_ts), N.ptr(info), N.ptr(nbi), N.ptr(nbs),
                                           N.ptr(nbl), k, n_items, N.ptr(rows), int(rows.numel()), 1 if cta else 0,
                                           int(tile or 0), n,
                                           float(alpha), 1 if decay else 0, N.ptr(out_idx), N.ptr(out_score),
                                           N.ptr(out_len), N.ptr(stats), N.ptr(err), N.stream()), "xmap_usersim_top_n")
    if int(err.item()):
        raise N.NativeError("top-N kernel error %d (4: more than 128 matching profile records)" % int(err.item()))
    visits, cands = stats.tolist()
    return RS.TopN(out_idx, out_score, out_len, visits, cands, int((~heavy).sum()), int(heavy.sum()))
