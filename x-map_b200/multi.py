"""Multi-GPU sharding of the similarity + selection stage (one process per GPU).

Item rows are cut into contiguous blocks of equal *work* (sum of rater degrees,
not row count); every rank keeps the whole ratings layout (replicated; the
reference broadcasts its side tables the same way, assist.py:69,73).  A rank
evaluates the triangular similarity rows of its block, which produces neighbour
records for BOTH ends of every pair -- the end it owns and the (more popular)
end another rank may own.  So the path has one real exchange step, followed by
the gathers the reference performs as collect + broadcast:

  1. all-to-all of the neighbour records addressed to rows of other ranks
     (replaces the reduceByKey shuffle of baselinerSim.py:210-211, 232-233);
  2. max-all-reduce of the BB flags (the SQL DISTINCT + collect + broadcast of
     assist.py:82-87) -- n_items bytes;
  3. all-gather of the neighbour tables after selection (the collectAsMap +
     broadcast of assist.py:121-132) -- n_items * 2k * 20 bytes.

X-SIM extension shards by work unit (a start, or one range of the hashed end axis
of a heavy start: units are independent; every rank builds the same plan from the
gathered tables and runs every world-th unit of the descending-work order); the
per-unit results are summed across ranks (each is non-zero on exactly one rank)
and every rank merges them per start.  Generation shards by user: the item map is
tiny and replicated, every rank rewrites the ratings of a contiguous block of
users holding an equal share of the ratings, and the AlterEgo records stay
sharded (the reference's result is an RDD) unless the caller gathers them.

Because the accumulators are order-free integers and selection uses a total
order, the result is bit-identical for any world size.  The exchange helpers are
device-agnostic so they can be exercised with the gloo backend on CPU tensors.
"""
import torch
import torch.distributed as dist


class RowShard(object):
    """Contiguous, work-balanced block of item rows owned by `rank`."""

    def __init__(self, row_work, rank=0, world=1):
        self.rank, self.world = rank, world
        n = int(row_work.numel())
        self.n_items = n
        if world == 1:
            self.bounds = [0, n]
        else:
            cw = torch.cumsum(row_work.double() + 1.0, 0)          # +1: empty rows still cost a visit
            total = float(cw[-1]) if n else 0.0
            targets = torch.tensor([total * r / world for r in range(1, world)], dtype=torch.float64,
                                   device=cw.device)
            cuts = torch.searchsorted(cw, targets).tolist() if n else [0] * (world - 1)
            self.bounds = [0] + [int(c) for c in cuts] + [n]
            for i in range(1, len(self.bounds)):
                self.bounds[i] = max(self.bounds[i], self.bounds[i - 1])
        self.lo, self.hi = self.bounds[rank], self.bounds[rank + 1]
        self.max_rows = max(self.bounds[r + 1] - self.bounds[r] for r in range(world))

    def rows(self, device):
        return torch.arange(self.lo, self.hi, dtype=torch.int32, device=device)


def allgather_rows(t, shard, group=None):
    """t: tensor (or list of tensors) whose dim 0 is the item axis, valid on [shard.lo, shard.hi).
    After the call every rank holds every row.  The rows of all the tensors are packed side by side into
    one byte matrix, padded to the largest block, so that ONE equal-size all-gather moves everything."""
    ts = list(t) if isinstance(t, (list, tuple)) else [t]
    if shard.world == 1 or not ts:
        return t
    dev = ts[0].device
    own = shard.hi - shard.lo
    flat = [x[shard.lo:shard.hi].contiguous().view(own, -1).view(torch.uint8) if own else
            x.new_zeros((0, 1)).view(torch.uint8).view(0, -1) for x in ts]
    width = [int(x[:1].numel()) * x.element_size() for x in ts]       # bytes per row of every tensor
    W = sum(width)
    send = torch.zeros((shard.max_rows, W), dtype=torch.uint8, device=dev)
    if own:
        col = 0
        for f, w in zip(flat, width):
            send[:own, col:col + w] = f.view(own, w)
            col += w
    recv = torch.empty((shard.world * shard.max_rows, W), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(recv, send, group=group)
    recv = recv.view(shard.world, shard.max_rows, W)
    for r in range(shard.world):
        lo, hi = shard.bounds[r], shard.bounds[r + 1]
        if r == shard.rank or hi <= lo:
            continue
        col = 0
        for x, w in zip(ts, width):
            blk = recv[r, : hi - lo, col:col + w].contiguous().view(x.dtype)
            x[lo:hi] = blk.view((hi - lo,) + tuple(x.shape[1:]))
            col += w
    return t


def shard_selected(sel, weight, group=None):
    """Split the selected rows sel over the ranks of `group` in contiguous blocks of sel of equal total weight
    (weight[q]: the work of row sel[q]).  Returns (the shard of positions in sel, the rows this rank computes)."""
    sh = RowShard(weight, dist.get_rank(group), dist.get_world_size(group))
    return sh, sel[sh.lo:sh.hi]


def gather_selected(ts, shard, sel=None, group=None):
    """ts: tensors whose dim 0 is the row axis, each rank having filled the rows sel[shard.lo:shard.hi].  After the
    call every rank holds every selected row; sel None means every row in order."""
    if sel is None:
        allgather_rows(ts, shard, group)
        return
    rows = [t[sel] for t in ts]                 # the selected rows side by side, in the order of sel
    allgather_rows(rows, shard, group)
    for t, r in zip(ts, rows):
        t[sel] = r


def _all_to_all(recv, send, group=None):
    """dist.all_to_all where the backend has it (NCCL); point-to-point otherwise (gloo)."""
    if dist.get_backend(group) == "nccl":
        dist.all_to_all(recv, send, group=group)
        return
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    recv[rank].copy_(send[rank])
    ops = []
    for s in range(world):
        if s == rank:
            continue
        if send[s].numel():
            ops.append(dist.P2POp(dist.isend, send[s], s, group))
        if recv[s].numel():
            ops.append(dist.P2POp(dist.irecv, recv[s], s, group))
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()


def _list_slots(base, seg):
    """Flat indices base[r] + 0 .. seg[r]-1 for every row r, rows concatenated."""
    tot = int(seg.sum())
    if tot == 0:
        return torch.zeros(0, dtype=torch.int64, device=seg.device), 0
    first = torch.cumsum(seg, 0) - seg
    r = torch.repeat_interleave(torch.arange(seg.numel(), device=seg.device), seg)
    return base[r] + (torch.arange(tot, device=seg.device) - first[r]), tot


def _segmented_copy(src, src_pos, dst, dst_pos, seg_len, total=None):
    """dst[dst_pos[g] + k] = src[src_pos[g] + k] for k < seg_len[g] (16-byte records or their int32 counts, CUDA)."""
    from . import _native as N
    seg_off = (torch.cumsum(seg_len, 0) - seg_len).contiguous()
    if total is None:
        total = int(seg_len.sum())
    fn = N.lib().xmap_segmented_copy4 if src.dtype == torch.int32 else N.lib().xmap_segmented_copy16
    N.check(fn(N.ptr(src), N.ptr(src_pos.contiguous()), N.ptr(dst), N.ptr(dst_pos.contiguous()), N.ptr(seg_off),
               int(seg_len.numel()), total, torch.cuda.current_stream().cuda_stream), "xmap_segmented_copy")


def exchange_records_cuda(rec, rec_ptr, rec_cnt, shard, group=None, rec_n=None):
    """exchange_records on the GPU: one packing kernel, one all-to-all of the lengths, one all-to-all
    of the records (NCCL), one appending kernel; two small device -> host reads for the split sizes."""
    world, rank, dev = shard.world, shard.rank, rec.device
    I = shard.n_items
    lo, hi = shard.lo, shard.hi
    own = hi - lo
    bounds = torch.tensor(shard.bounds, dtype=torch.int64, device=dev)
    cnt = rec_cnt.long()
    out_cnt = cnt.clone()
    out_cnt[lo:hi] = 0                                       # rows are rank-major, so is the packed buffer
    csum = torch.zeros(I + 1, dtype=torch.int64, device=dev)
    csum[1:] = torch.cumsum(out_cnt, 0)
    in_split = (csum[bounds[1:]] - csum[bounds[:-1]])         # records for each destination
    # lengths first (device all-to-all of int64 vectors of unequal size)
    send_cnt = [out_cnt[shard.bounds[s]:shard.bounds[s + 1]].contiguous() for s in range(world)]
    recv_cnt = [torch.empty(own, dtype=torch.int64, device=dev) for _ in range(world)]
    _all_to_all(recv_cnt, send_cnt, group)
    RC = torch.stack(recv_cnt)                               # [world, own]; row `rank` is zero
    sizes = torch.cat([in_split, RC.sum(1)]).tolist()         # the one host read
    in_sizes, out_sizes = sizes[:world], sizes[world:]
    n_in, n_out = sum(in_sizes), sum(out_sizes)
    # append: source-major segments (s, row) land after the row's own records and the earlier sources'
    before = torch.cumsum(RC, 0) - RC + cnt[lo:hi].unsqueeze(0)
    seg_len = RC.reshape(-1)
    src_pos = torch.cumsum(seg_len, 0) - seg_len
    dst_pos = (rec_ptr[lo:hi].unsqueeze(0) + before).reshape(-1)
    for arr in (rec,) if rec_n is None else (rec, rec_n):          # the int32 counts travel like the records
        tail = tuple(arr.shape[1:])
        send = torch.empty((max(n_in, 1),) + tail, dtype=arr.dtype, device=dev)
        _segmented_copy(arr, rec_ptr[:-1], send, csum[:-1], out_cnt, total=n_in)
        recv = torch.empty((max(n_out, 1),) + tail, dtype=arr.dtype, device=dev)
        dist.all_to_all_single(recv[:n_out], send[:n_in], out_sizes, in_sizes, group=group)
        _segmented_copy(recv, src_pos, arr, dst_pos, seg_len, total=n_out)
    new_cnt = cnt[lo:hi] + RC.sum(0)
    rec_cnt.zero_()
    rec_cnt[lo:hi] = new_cnt.to(rec_cnt.dtype)


def exchange_records(rec, rec_ptr, rec_cnt, shard, group=None, rec_n=None):
    """rec [total, 2] int64 records (rec_n [total] int32: their co-rating counts, moved alongside),
    rec_ptr [I + 1] list extents, rec_cnt [I] list lengths.
    On entry the lists hold the records THIS rank produced, for every row; on exit the lists of the
    rows this rank owns hold the records of every rank and the other lists are empty."""
    if shard.world == 1:
        return
    if rec.is_cuda:
        return exchange_records_cuda(rec, rec_ptr, rec_cnt, shard, group, rec_n)
    world, rank = shard.world, shard.rank
    cnt = rec_cnt.long()
    blocks = [(shard.bounds[s], shard.bounds[s + 1]) for s in range(world)]
    send_cnt = [cnt[lo:hi].contiguous() for lo, hi in blocks]
    own = shard.hi - shard.lo
    recv_cnt = [torch.empty(own, dtype=torch.int64, device=rec.device) for _ in range(world)]
    _all_to_all(recv_cnt, send_cnt, group)
    for arr in (rec,) if rec_n is None else (rec, rec_n):
        tail = tuple(arr.shape[1:])
        send_buf = []
        for s, (lo, hi) in enumerate(blocks):
            if s == rank:
                send_buf.append(arr.new_empty((0,) + tail))
                continue
            src, _ = _list_slots(rec_ptr[lo:hi], send_cnt[s])
            send_buf.append(arr[src])
        recv_buf = [arr.new_empty((0 if s == rank else int(recv_cnt[s].sum()),) + tail) for s in range(world)]
        _all_to_all(recv_buf, send_buf, group)
        cur = cnt[shard.lo:shard.hi].clone()
        for s in range(world):
            if s == rank:
                continue
            dst, tot = _list_slots(rec_ptr[shard.lo:shard.hi] + cur, recv_cnt[s])
            if tot:
                arr[dst] = recv_buf[s]
            cur += recv_cnt[s]
    rec_cnt.zero_()
    rec_cnt[shard.lo:shard.hi] = cur.to(rec_cnt.dtype)


def similarity_shard(engine, rank=0, world=1):
    """Row blocks balanced by the cost of both phases: the products a row evaluates (accumulate,
    ~30 ps each) and the records it will have to select from (~1/6 of its list capacity at ~18 ps)."""
    return RowShard(engine.tri_work + engine.rec_cap_bound // 6, rank, world)


def similarity_step(engine, shard, group=None):
    """Triangular rows of the owned block -> record exchange -> BB flags -> selection -> gather."""
    rows = None if shard.world == 1 else shard.rows(engine.device)
    if shard.world > 1 and not getattr(engine, "_sizing_agreed", False):
        # whether the exact-sizing branch (which holds an all-reduce) runs must be the same decision on
        # every rank: each rank judged its own free memory, so any rank that needs it forces it everywhere
        need = torch.tensor([1 if engine.rec is None else 0], dtype=torch.int32, device=engine.device)
        dist.all_reduce(need, op=dist.ReduceOp.MAX, group=group)
        if int(need.item()) and engine.rec is not None:
            engine.release_lists()
        engine._sizing_agreed = True
    if engine.rec is None and shard.world > 1:
        # exact list sizing: a rank's lists hold its own records for every row, plus, for the rows it
        # owns, the records the other ranks will send
        own = engine._size_lists(rows)
        tot = own.clone()
        dist.all_reduce(tot, op=dist.ReduceOp.SUM, group=group)
        own[shard.lo:shard.hi] = tot[shard.lo:shard.hi]
        engine._alloc_lists(own)
    engine.reset()
    stats = engine.accumulate(rows)
    if shard.world > 1:
        engine._timed("exchange", lambda: exchange_records(engine.rec, engine.rec_ptr, engine.rec_cnt, shard, group,
                                                                   rec_n=engine.rec_n))
        dist.all_reduce(engine.bb, op=dist.ReduceOp.MAX, group=group)
    engine.select(rows)
    nkept = None
    if shard.world > 1:
        nkept = engine.rec_cnt.clone()          # the lists stay sharded: only the lengths are gathered
        allgather_rows([engine.row_npairs, nkept, engine.tab_len, engine.tab_idx, engine.tab_sim,
                        engine.tab_mutu, engine.tab_n], shard, group)
    return engine.tables(dict(accumulate=stats, rows=(shard.lo, shard.hi)), row_nkept=nkept)


def sum_unit_results(tensors, group=None):
    """X-SIM work units are dealt to the ranks (every world-th unit of the descending-work order); a unit's
    result (distinct ends, paths, top-m list) is non-zero on exactly one rank, so a sum assembles the full
    unit tables on every rank.  Device-agnostic (NCCL on the GPUs, gloo in the CPU tests)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return tensors
    for t in tensors:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return tensors


class UserShard(object):
    """Contiguous block of users holding ~1/world of the ratings (csr_ptr: int32 [n_users + 1])."""

    def __init__(self, csr_ptr, rank=0, world=1):
        n = int(csr_ptr.numel()) - 1
        nnz = int(csr_ptr[-1]) if n >= 0 and csr_ptr.numel() else 0
        if world == 1 or n <= 0:
            bounds = [0] + [max(n, 0)] * world
        else:
            targets = torch.tensor([nnz * r // world for r in range(1, world)], dtype=csr_ptr.dtype,
                                   device=csr_ptr.device)
            cuts = torch.searchsorted(csr_ptr[:-1].contiguous(), targets).tolist()
            bounds = [0] + [int(c) for c in cuts] + [n]
            for i in range(1, len(bounds)):
                bounds[i] = max(bounds[i], bounds[i - 1])
        self.rank, self.world, self.bounds = rank, world, bounds
        self.lo, self.hi = bounds[rank], bounds[rank + 1]


def build_alterego_sharded(layout, ts, mapping, shard, gather=False, group=None):
    """AlterEgo records of the users this rank owns (generator.py:113-157); gather=True
    concatenates every rank's records, in user order, on every rank."""
    from . import generate as G
    import copy
    lo, hi = shard.lo, shard.hi
    e_lo, e_hi = int(layout.csr_ptr[lo]), int(layout.csr_ptr[hi])
    sub = copy.copy(layout)
    sub.n_users, sub.nnz = hi - lo, e_hi - e_lo
    sub.csr_ptr = (layout.csr_ptr[lo:hi + 1] - e_lo).contiguous()
    sub.csr_ent = layout.csr_ent[e_lo:e_hi]
    sub.csr_src = layout.csr_src[e_lo:e_hi]
    ou, oi, orr, ot = G.build_alterego(sub, ts, mapping)
    ou = ou + lo
    if not gather or shard.world == 1:
        return ou, oi, orr, ot
    n = torch.tensor([ou.numel()], dtype=torch.int64, device=ou.device)
    sizes = [torch.zeros_like(n) for _ in range(shard.world)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(x) for x in sizes]
    cap = max(max(sizes), 1)
    out = []
    for t in (ou, oi, orr, ot):
        send = torch.zeros(cap, dtype=t.dtype, device=t.device)
        send[: t.numel()] = t
        recv = [torch.empty_like(send) for _ in range(shard.world)]
        dist.all_gather(recv, send, group=group)
        out.append(torch.cat([r[:m] for r, m in zip(recv, sizes)]))
    return tuple(out)
