"""Explicit-feedback ALS on the device (C ABI section 8): the form of MLlib's explicit ALS (ALS-WR), defined in
DESIGN.md section 3.8 so that every bit of the factors follows from the inputs (tests/als_exact.py restates it).

    model = als.train(user, item, rating, n_users, n_items, rank=10, iterations=5, lam=0.01)
    score = als.predict(model, u, i)                       # f64, NaN where a side has no factors
    top = als.top_n(model, 10, user, item)                 # every user's 10 best unrated items, recsim.TopN layout

The MLlib-shaped facade over these calls is core/als.py."""
import math
from dataclasses import dataclass

import torch

from . import _native as N
from . import multi as M
from . import recsim as RS

SEGMENT = N.ALS_SEGMENT
# Bytes of segment partials (fp64 normal equations) one normal / solve launch pair may hold: the rows of a half-step
# are cut into launches under it.  The factors do not depend on it; tests shrink it to run many launches.
SCRATCH_BYTES = 1 << 31


@dataclass
class AlsModel:
    """train's result.  A row without records has no factors: its row is zero and its count 0."""
    user_factors: torch.Tensor   # f32 [n_users, rank]
    item_factors: torch.Tensor   # f32 [n_items, rank]
    user_count: torch.Tensor     # int64 [n_users] records per user
    item_count: torch.Tensor     # int64 [n_items] records per item
    rank: int
    lam: float
    iterations: int
    half_ms: list                # per half-step {"side", "normal_ms", "solve_ms"} when events were passed, else None


def _int(v, name, lo, hi=None):
    if isinstance(v, bool) or int(v) != v or int(v) < lo or (hi is not None and int(v) > hi):
        raise ValueError("%s must be an integer in [%d, %s], got %r" % (name, lo, "inf" if hi is None else hi, v))
    return int(v)


def _records(user, item, n_users, n_items, dev, rating=None):
    """The records as int64 device tensors (and the ratings as f64), checked before any launch."""
    u = torch.as_tensor(user).to(dev).flatten()
    i = torch.as_tensor(item).to(dev).flatten()
    for t, name in ((u, "user"), (i, "item")):
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError("%s must be integer" % name)
    u, i = u.long(), i.long()
    n = int(u.numel())
    if int(i.numel()) != n:
        raise ValueError("user and item differ in length (%d, %d)" % (n, int(i.numel())))
    if n and (int(u.min()) < 0 or int(u.max()) >= n_users):
        raise ValueError("user outside [0, %d)" % n_users)
    if n and (int(i.min()) < 0 or int(i.max()) >= n_items):
        raise ValueError("item outside [0, %d)" % n_items)
    if rating is None:
        return u, i
    r = torch.as_tensor(rating, dtype=torch.float64).to(dev).flatten()
    if int(r.numel()) != n:
        raise ValueError("rating differs in length from user (%d, %d)" % (int(r.numel()), n))
    if n and not bool(torch.isfinite(r).all()):
        raise ValueError("ratings must be finite")
    return u, i, r


class _Side(object):
    """The rows of one side (items or users) with the other side's index and the rating of each record, stably sorted
    by row, cut into segments of SEGMENT records and into launches under SCRATCH_BYTES."""

    def __init__(self, row, col, rating, n_rows, rank, lo, hi):
        dev = row.device
        o = torch.argsort(row, stable=True)
        self.col = col[o].to(torch.int32).contiguous()
        self.rating = rating[o].contiguous()
        self.count = torch.bincount(row, minlength=n_rows)
        ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
        ptr[1:] = torch.cumsum(self.count, 0)
        self.n_rows, self.lo, self.hi = n_rows, lo, hi
        rows = torch.nonzero(self.count[lo:hi] > 0).flatten() + lo
        n = self.count[rows]
        nseg = (n + SEGMENT - 1) // SEGMENT
        P = rank * (rank + 1) // 2 + rank
        per = max(1, SCRATCH_BYTES // (P * 8))              # segments one launch may hold
        cs = torch.cumsum(nseg, 0).cpu()
        bounds, a = [0], 0
        while a < int(rows.numel()):
            b = max(int(torch.searchsorted(cs, (int(cs[a - 1]) if a else 0) + per, right=True)), a + 1)
            bounds.append(b)
            a = b
        self.launches = []
        for a, b in zip(bounds[:-1], bounds[1:]):
            ns = nseg[a:b]
            seg_ptr = torch.zeros(b - a + 1, dtype=torch.int64, device=dev)
            seg_ptr[1:] = torch.cumsum(ns, 0)
            total = int(seg_ptr[-1])
            owner = torch.repeat_interleave(torch.arange(b - a, device=dev), ns)
            k = torch.arange(total, device=dev) - seg_ptr[owner]
            seg_lo = ptr[rows[a:b]][owner] + k * SEGMENT
            seg_n = torch.minimum(n[a:b][owner] - k * SEGMENT, torch.tensor(SEGMENT, device=dev)).to(torch.int32)
            self.launches.append((rows[a:b].to(torch.int32).contiguous(), seg_ptr, n[a:b].contiguous(),
                                  seg_lo.contiguous(), seg_n.contiguous(), total))
        self.max_seg = max([L[5] for L in self.launches], default=0)

    def solve(self, other, rank, lam, name, timer=None):
        """New factors of the rows [lo, hi) from the other side's factors (the other rows stay zero), and a status
        byte per row (1: a pivot was not > 0)."""
        L = N.lib()
        dev = other.device
        out = torch.zeros((self.n_rows, rank), dtype=torch.float32, device=dev)
        status = torch.zeros(self.n_rows, dtype=torch.int8, device=dev)
        P = rank * (rank + 1) // 2 + rank
        partial = torch.empty(max(self.max_seg * P, 1), dtype=torch.float64, device=dev)
        for rows, seg_ptr, n, seg_lo, seg_n, total in self.launches:
            with _phase(timer, "normal"):
                N.check(L.xmap_als_normal(N.ptr(self.col), N.ptr(self.rating), N.ptr(seg_lo), N.ptr(seg_n), total,
                                          N.ptr(other), rank, N.ptr(partial), N.stream()), "xmap_als_normal")
            with _phase(timer, "solve"):
                N.check(L.xmap_als_solve(N.ptr(rows), N.ptr(seg_ptr), N.ptr(n), int(rows.numel()), N.ptr(partial),
                                         rank, float(lam), N.ptr(out), N.ptr(status), N.stream()), "xmap_als_solve")
        return out, status


class _phase(object):
    """CUDA events around one kernel: appended to timer[name] (a dict of lists) when timer is not None."""

    def __init__(self, timer, name):
        self.timer, self.name = timer, name

    def __enter__(self):
        if self.timer is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.timer is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            self.timer.setdefault(self.name, []).append((self.a, b))


def _check_status(status, name, lam):
    bad = torch.nonzero(status).flatten()
    if int(bad.numel()):
        raise N.NativeError("ALS: the Cholesky factor of %s row %d has a pivot that is not > 0 (lambda = %r); "
                            "only lambda = 0 allows it" % (name, int(bad[0]), lam))


def init_factors(n_rows, rank, seed=None, device="cuda"):
    """The initial user factors of train: row u = Philox4x32-10(seed, u) -> rank standard normals (Box-Muller) divided
    by their L2 norm, fp32 [n_rows, rank].  seed None means 0."""
    n_rows = _int(n_rows, "n_rows", 0, 2 ** 31 - 1)
    rank = _int(rank, "rank", 1, N.ALS_RANK_MAX)
    seed = 0 if seed is None else _int(seed, "seed", 0, 2 ** 64 - 1)
    X = torch.empty((n_rows, rank), dtype=torch.float32, device=device)
    N.check(N.lib().xmap_als_init(n_rows, rank, seed, N.ptr(X), N.stream()), "xmap_als_init")
    return X


def train(user, item, rating, n_users, n_items, rank, iterations, lam, seed=None, init=None, shard=False, group=None,
          events=None, device="cuda"):
    """Explicit ALS on the records (user[k], item[k], rating[k]), taken as given (duplicates count).  Each iteration
    solves every item from the user factors, then every user from the new item factors (DESIGN.md 3.8).
    init: fp32 [n_users, rank] initial user factors, or None -> Philox4x32-10(seed, user) normals of unit norm
    (seed None means 0).  shard: each rank of `group` (torch.distributed; every rank passes every record) solves a
    contiguous block of rows of equal record count, and one all-gather per half-step shares them; the factors do not
    depend on the world size.  events: a dict that receives the per-half-step kernel times in model.half_ms.
    Raises ValueError before any launch, NativeError when a pivot fails (possible only with lam = 0)."""
    n_users = _int(n_users, "n_users", 0, 2 ** 31 - 1)
    n_items = _int(n_items, "n_items", 0, 2 ** 31 - 1)
    rank = _int(rank, "rank", 1, N.ALS_RANK_MAX)
    iterations = _int(iterations, "iterations", 1)
    if isinstance(lam, bool) or not isinstance(lam, (int, float)) or not math.isfinite(lam) or lam < 0:
        raise ValueError("lam must be a finite number >= 0, got %r" % (lam,))
    lam = float(lam)
    seed = 0 if seed is None else _int(seed, "seed", 0, 2 ** 64 - 1)
    dev = torch.device(device)
    u, i, r = _records(user, item, n_users, n_items, dev, rating)
    if init is not None:
        init = torch.as_tensor(init)
        if init.dtype != torch.float32 or tuple(init.shape) != (n_users, rank):
            raise ValueError("init must be float32 [%d, %d], got %s %s" % (n_users, rank, init.dtype, tuple(init.shape)))
    N.lib()
    sh_u = sh_i = None
    if shard:
        rk, world = M.dist.get_rank(group), M.dist.get_world_size(group)
        sh_i = M.RowShard(torch.bincount(i, minlength=n_items), rk, world)
        sh_u = M.RowShard(torch.bincount(u, minlength=n_users), rk, world)
    items = _Side(i, u, r, n_items, rank, *((sh_i.lo, sh_i.hi) if sh_i else (0, n_items)))
    users = _Side(u, i, r, n_users, rank, *((sh_u.lo, sh_u.hi) if sh_u else (0, n_users)))
    X = init.to(dev).contiguous().clone() if init is not None else init_factors(n_users, rank, seed, dev)
    Y = None
    half = [] if events is not None else None
    for _ in range(iterations):
        for side, sh, name in ((items, sh_i, "item"), (users, sh_u, "user")):
            timer = {} if events is not None else None
            out, status = side.solve(X if name == "item" else Y, rank, lam, name, timer)
            if sh is not None:
                M.allgather_rows([out, status], sh, group)
            _check_status(status, name, lam)
            if name == "item":
                Y = out
            else:
                X = out
            if timer is not None:
                events.setdefault("%s_normal" % name, []).extend(timer.get("normal", []))
                events.setdefault("%s_solve" % name, []).extend(timer.get("solve", []))
                half.append((name, timer))
    if half is not None:
        torch.cuda.synchronize(dev)
        half = [{"side": name, **{"%s_ms" % k: sum(a.elapsed_time(b) for a, b in t.get(k, [])) for k in ("normal", "solve")}}
                for name, t in half]
    return AlsModel(X, Y, users.count, items.count, rank, lam, iterations, half)


def predict(model, u, i):
    """score(u, i) = sum_k x_u[k] y_i[k] in fp64 (DESIGN.md 3.8), NaN where the user or the item has no factors."""
    dev = model.user_factors.device
    n_users, n_items = int(model.user_factors.shape[0]), int(model.item_factors.shape[0])
    pu, pi = _records(u, i, n_users, n_items, dev)
    out = torch.empty(int(pu.numel()), dtype=torch.float64, device=dev)
    pu32, pi32 = pu.to(torch.int32).contiguous(), pi.to(torch.int32).contiguous()
    N.check(N.lib().xmap_als_predict(N.ptr(model.user_factors), N.ptr(model.item_factors), N.ptr(model.user_count),
                                     N.ptr(model.item_count), model.rank, N.ptr(pu32), N.ptr(pi32), int(pu.numel()),
                                     N.ptr(out), N.stream()), "xmap_als_predict")
    return out


@dataclass
class AlsTopN:
    """top_n's result, in the layout of recsim.TopN (recsim.rank_metrics reads idx and len)."""
    idx: torch.Tensor        # int32 [n_users, n], -1 padded
    score: torch.Tensor      # f64   [n_users, n], NaN padded
    len: torch.Tensor        # int32 [n_users]
    candidates: int          # candidate items with factors


def top_n(model, n, user=None, item=None, candidates=None, users=None, exclude_rated=True, shard=False, group=None):
    """Each user's first n (1 <= n <= 64) candidate items by score descending, then the smaller item index (-0.0
    equals 0.0; a NaN score is never listed).  candidates: ascending distinct items (None: every item); items without
    factors are dropped.  exclude_rated: drop the items of the user's records among user / item (the training records).
    users: None for every user, or distinct users whose rows alone are filled (the others keep the padding).  A user
    without factors gets an empty list.  shard: split the users over the ranks of `group` and all-gather the lists.
    The result does not depend on the launch shape, the tiling or the world size."""
    n = RS.list_length(n)
    dev = model.user_factors.device
    n_users, n_items = int(model.user_factors.shape[0]), int(model.item_factors.shape[0])
    rated_ptr = rated_item = None
    if exclude_rated:
        if user is None or item is None:
            raise ValueError("exclude_rated needs the training records user / item")
        ru, ri = _records(user, item, n_users, n_items, dev)
        key = torch.unique(ru * max(n_items, 1) + ri)
        rated_ptr = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
        rated_ptr[1:] = torch.cumsum(torch.bincount(key // max(n_items, 1), minlength=n_users), 0)
        rated_item = (key % max(n_items, 1)).to(torch.int32).contiguous()
    if candidates is None:
        cand = torch.arange(n_items, device=dev)
    else:
        cand = RS.index_set(candidates, n_items, dev, "candidates")
        if cand.numel() > 1 and bool((cand[1:] <= cand[:-1]).any()):
            raise ValueError("candidates must be ascending and distinct")
    cand = cand[model.item_count[cand] > 0].to(torch.int32).contiguous()
    sel = RS.query_users(users, n_users, dev)
    sh, mine = M.shard_selected(sel, torch.zeros(int(sel.numel()), device=dev), group) if shard else (None, sel)
    run = mine[model.user_count[mine] > 0].to(torch.int32).contiguous()
    out_idx, out_score, out_len = RS.empty_lists(n_users, n, dev)
    N.check(N.lib().xmap_als_top_n(N.ptr(model.user_factors), N.ptr(model.item_factors), model.rank, N.ptr(run),
                                   int(run.numel()), N.ptr(cand), int(cand.numel()), N.ptr(rated_ptr),
                                   N.ptr(rated_item), n, N.ptr(out_idx), N.ptr(out_score), N.ptr(out_len), N.stream()),
            "xmap_als_top_n")
    if sh is not None:
        M.gather_selected([out_idx, out_score, out_len], sh, None if users is None else sel, group)
    return AlsTopN(out_idx, out_score, out_len, int(cand.numel()))
