"""Clean stage on encoded records (C ABI section 6; SURVEY.md 8(f) #4).

Reference: BaselinerClean.parse_data's period test, filter_data and clean_data (baselinerClean.py:47-52, 62-92,
94-97).  Splitting the text lines and building the id dictionaries stay on the host (core/baselinerClean.py)."""
from datetime import datetime

import torch

from . import _native as N


def period_bounds(date_from, date_to):
    """The two instants the LOCAL-time years [date_from, date_to] span: the reference tests
    datetime.fromtimestamp(ts).year in range(date_from, date_to + 1) (baselinerClean.py:36, 50)."""
    return datetime(int(date_from), 1, 1).timestamp(), datetime(int(date_to) + 1, 1, 1).timestamp()


def clean_encoded(user, item, ts, n_users, t_lo, t_hi, num_atleast, device="cuda"):
    """user / item: int32 indices of the records in arrival order, ts: float64 seconds.
    Returns (keep uint8 [n], distinct in-period items per user int32 [n_users])."""
    dev = torch.device(device)
    user = torch.as_tensor(user, dtype=torch.int32).to(dev).contiguous()
    item = torch.as_tensor(item, dtype=torch.int32).to(dev).contiguous()
    ts = torch.as_tensor(ts, dtype=torch.float64).to(dev).contiguous()
    order = clean_order(user, item, ts, t_lo, t_hi)
    return clean_sorted(user, item, ts, order, n_users, t_lo, t_hi, num_atleast)


def clean_order(user, item, ts, t_lo, t_hi):
    """Record indices sorted, stable, by (out-of-period last, user, item): a (user, item) group is a run in arrival
    order.  user < 2^30."""
    inp = (ts >= t_lo) & (ts < t_hi)
    key = ((~inp).long() << 62) | (user.long() << 32) | item.long()
    return torch.argsort(key, stable=True).contiguous()                # CUB radix sort through torch: library plumbing


def clean_sorted(user, item, ts, order, n_users, t_lo, t_hi, num_atleast):
    """clean_encoded on device tensors with their clean_order already computed."""
    L = N.lib()
    dev = user.device
    n = int(user.numel())
    keep = torch.empty(n, dtype=torch.uint8, device=dev)
    user_items = torch.empty(max(int(n_users), 1), dtype=torch.int32, device=dev)
    N.check(L.xmap_clean_records(N.ptr(user), N.ptr(item), N.ptr(ts), N.ptr(order), n, int(n_users),
                                 float(t_lo), float(t_hi), int(num_atleast), N.ptr(keep), N.ptr(user_items),
                                 torch.cuda.current_stream().cuda_stream), "xmap_clean_records")
    return keep, user_items[: int(n_users)]
