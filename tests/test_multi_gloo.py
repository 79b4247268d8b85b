"""CPU, gloo: work-balanced row sharding, the neighbour-record exchange, the table all-gather and the gather of
selected rows."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from xmap_b200.multi import RowShard, allgather_rows
    g = torch.Generator().manual_seed(3)
    work = (torch.rand(1001, generator=g) ** 4 * 1e5).long()
    sh = RowShard(work, rank, world)
    assert sh.bounds[0] == 0 and sh.bounds[-1] == 1001 and sh.bounds == sorted(sh.bounds)
    full = torch.arange(1001 * 6, dtype=torch.float64).reshape(1001, 2, 3)
    mine = torch.zeros_like(full)
    mine[sh.lo:sh.hi] = full[sh.lo:sh.hi]
    allgather_rows(mine, sh)
    flags = torch.zeros(1001, dtype=torch.uint8)
    flags[sh.lo:sh.hi] = (torch.arange(sh.lo, sh.hi) % 3 == 0).to(torch.uint8)
    allgather_rows(flags, sh)
    ok = bool(torch.equal(mine, full)) and bool(torch.equal(flags, (torch.arange(1001) % 3 == 0).to(torch.uint8)))
    # several tensors of different dtypes / row widths packed into ONE all-gather
    fulls = [torch.arange(1001, dtype=torch.int64) * 7, torch.arange(1001 * 4, dtype=torch.int32).reshape(1001, 2, 2),
             torch.arange(1001 * 2, dtype=torch.float64).reshape(1001, 2) / 3.0, (torch.arange(1001) % 5).to(torch.uint8)]
    parts = []
    for f in fulls:
        m = torch.zeros_like(f); m[sh.lo:sh.hi] = f[sh.lo:sh.hi]; parts.append(m)
    allgather_rows(parts, sh)
    ok = ok and all(bool(torch.equal(a, b)) for a, b in zip(parts, fulls))
    loads = [float(work[sh.bounds[r]:sh.bounds[r + 1]].sum()) for r in range(world)]
    q.put((rank, ok, loads))
    dist.destroy_process_group()


def test_row_shard_and_allgather_world2():
    import sys
    from tests import parity  # noqa: F401  (puts the repo root on sys.path for the children)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert all(ok for _, ok, _ in res)
    loads = res[0][2]
    assert max(loads) / (sum(loads) / 2) < 1.25        # blocks balanced by work, not by row count


def _selected_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from xmap_b200.multi import gather_selected, shard_selected
    n_rows, width = 500, 3
    g = torch.Generator().manual_seed(7)
    work = (torch.rand(n_rows, generator=g) ** 4 * 1e4).long()
    subset = torch.randperm(n_rows, generator=g)[:317]          # a permuted subset of the rows

    def lists(rows):                   # top-N-shaped tables with the rows `rows` filled by a function of the row
        t = [torch.full((n_rows, width), -1, dtype=torch.int32), torch.full((n_rows, width), -1.0, dtype=torch.float64),
             torch.zeros(n_rows, dtype=torch.int32)]
        t[0][rows] = (rows.unsqueeze(1) * 10 + torch.arange(width)).int()
        t[1][rows] = rows.unsqueeze(1).double() / 7.0 + torch.arange(width)
        t[2][rows] = (rows % (width + 1)).int()
        return t
    ok = True
    for sel in (subset, None):
        rows = torch.arange(n_rows) if sel is None else sel
        sh, mine = shard_selected(rows, work[rows])
        got = lists(mine)
        gather_selected(got, sh, sel)
        ok = ok and all(bool(torch.equal(a, b)) for a, b in zip(got, lists(rows)))
    q.put((rank, ok))
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gather_selected_rows_equals_unsharded(world):
    """The shard-then-gather of the sharded top-N and user-kNN calls, on a permuted subset of the rows and on every
    row in order: every rank ends with the tables one process computing every selected row would hold."""
    from tests import parity  # noqa: F401
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_selected_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res)


def _exchange_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from xmap_b200.multi import RowShard, exchange_records
    I = 257
    g = torch.Generator().manual_seed(5)
    cap = torch.randint(0, 9, (I,), generator=g) * world
    ptr = torch.zeros(I + 1, dtype=torch.int64); ptr[1:] = torch.cumsum(cap, 0)
    sh = RowShard(cap + 1, rank, world)
    # rank r produced, for row i, (i * 7 + r) % (cap/world + 1) records tagged (i, r, position)
    def produced(r):
        return torch.minimum((torch.arange(I) * 7 + r) % 5, cap // world)
    cnt = produced(rank).to(torch.int32)
    rec = torch.full((int(ptr[-1]) + 1, 2), -1, dtype=torch.int64)
    rec_n = torch.full((int(ptr[-1]) + 1,), -1, dtype=torch.int32)     # the counts travel with their records
    for i in range(I):
        for p in range(int(cnt[i])):
            rec[int(ptr[i]) + p, 0] = i * 1000 + rank * 100 + p
            rec[int(ptr[i]) + p, 1] = rank
            rec_n[int(ptr[i]) + p] = (i * 1000 + rank * 100 + p) % 977
    exchange_records(rec, ptr, cnt, sh, rec_n=rec_n)
    ok = True
    for i in range(I):
        want = sorted(i * 1000 + r * 100 + p for r in range(world) for p in range(int(produced(r)[i]))) \
            if sh.lo <= i < sh.hi else []
        a, b = int(ptr[i]), int(ptr[i]) + int(cnt[i])
        got = sorted(rec[a:b, 0].tolist())
        ok = ok and got == want and (rec[a:b, 0] % 977).tolist() == rec_n[a:b].tolist()
    q.put((rank, ok))
    dist.destroy_process_group()


def test_record_exchange_world2():
    from tests import parity  # noqa: F401
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_exchange_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res)


def _xsim_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from xmap_b200.multi import sum_unit_results
    n, m = 37, 4
    g = torch.Generator().manual_seed(9)
    full = (torch.randint(1, 50, (n,), generator=g, dtype=torch.int32), torch.randint(1, 500, (n,), generator=g),
            torch.randint(0, 90, (n, m), generator=g, dtype=torch.int32),
            torch.randn(n, m, generator=g, dtype=torch.float64), torch.randint(0, m + 1, (n,), generator=g, dtype=torch.int32))
    order = torch.randperm(n, generator=g)                   # the descending-work order of the units
    mine = torch.zeros(n, dtype=torch.bool); mine[order[rank::world]] = True
    part = tuple(torch.where(mine.view((n,) + (1,) * (t.dim() - 1)), t, torch.zeros_like(t)) for t in full)
    out = sum_unit_results(part)
    ok = all(torch.equal(a, b) for a, b in zip(out, full))
    q.put((rank, ok))
    dist.destroy_process_group()


def test_xsim_allreduce_world2():
    from tests import parity  # noqa: F401
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_xsim_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res)


def test_user_shard_balances_ratings():
    from xmap_b200.multi import UserShard
    g = torch.Generator().manual_seed(4)
    deg = (torch.rand(5000, generator=g) ** 3 * 200).int()
    ptr = torch.zeros(5001, dtype=torch.int32); ptr[1:] = torch.cumsum(deg, 0)
    for world in (1, 2, 4, 8):
        sh = [UserShard(ptr, r, world) for r in range(world)]
        assert sh[0].lo == 0 and sh[-1].hi == 5000 and all(a.hi == b.lo for a, b in zip(sh, sh[1:]))
        loads = [int(ptr[s.hi] - ptr[s.lo]) for s in sh]
        assert max(loads) <= sum(loads) / world + 200
    e = UserShard(torch.zeros(1, dtype=torch.int32), 0, 2)
    assert (e.lo, e.hi) == (0, 0)


def test_row_shard_single_rank_and_edge_cases():
    from xmap_b200.multi import RowShard
    sh = RowShard(torch.tensor([5, 0, 7]), 0, 1)
    assert (sh.lo, sh.hi) == (0, 3)
    for world in (2, 4, 8):
        w = torch.zeros(3, dtype=torch.long)
        b = [RowShard(w, r, world) for r in range(world)]
        assert b[0].lo == 0 and b[-1].hi == 3 and all(x.hi == y.lo for x, y in zip(b, b[1:]))
