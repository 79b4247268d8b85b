"""Rating text files -> device-resident training set (C ABI section 7, csrc/ingest.cu; SURVEY.md 8(f) #4).

    train, test = ingest.clean_split_pipeline(None, clean_source, clean_target, split_tool,
                                              path_source, path_target, is_debug)

gives the records of baseliner_clean_data_pipeline (once per domain) followed by baseliner_split_data_pipeline
(assist.py:9-39), without a Python object per record: the files go to the GPU as bytes, the lines are found, split
and parsed there (one warp per 32 lines), the ids are ranked by sorting their packed bytes, the record rules of the
clean stage run in xmap_clean_records, and the split places every record with one sort of per-record keys.  Only the
per-user draws of the split (randomSplit's uniforms, random.sample from the global generator BaselinerSplit seeded)
run on the host, over arrays of users.  `train` carries the Session (layout, item codes) the next pipeline stage
uses, so session_of never encodes records; records are built only if somebody collects an RDD.

`ingest_arrays` returns the same result as arrays (IngestArrays) for callers that do not want RDDs.

What this reader accepts is a subset of what the host path accepts: see DESIGN.md section 6."""
import os
import random
import re
from collections.abc import Sequence
from dataclasses import dataclass, field
from datetime import datetime

import numpy as np
import torch

from . import _native as N
from . import clean as CL
from . import encode as ENC
from . import engine as E
from .rdd import LazyRDD, split_cells

ID_MAX = N.INGEST_ID_MAX
TS_MIN = -62135596800.0 + 2 * 86400        # 0001-01-03 UTC: datetime.fromtimestamp works in any time zone
TS_MAX = 253402300799.0 - 2 * 86400        # 9999-12-29 UTC
MAX_ITEMS = 1 << 24                        # the 24-bit item field of the layout entries
MAX_LINES = (1 << 31) - 1
INT32_MAX = (1 << 31) - 1

OK, BLANK, FEW_FIELDS, NON_ASCII, NUL, BAD_TIME, TIME_RANGE, BAD_RATING, UID_LONG, IID_LONG = range(10)
_REFUSAL = {
    FEW_FIELDS: (IndexError, "expected 'uid iid rating timestamp'", None),
    NON_ASCII: (ValueError, "non-ASCII byte", "byte"),
    NUL: (ValueError, "NUL byte", "byte"),
    BAD_TIME: (ValueError, "timestamp is not a decimal number of at most 15 significant digits and exponent "
                           "within +-22", 3),
    TIME_RANGE: (ValueError, "timestamp outside the years 1-9999", 3),
    BAD_RATING: (ValueError, "rating is not a decimal number of at most 15 significant digits and exponent "
                             "within +-22", 2),
    UID_LONG: (ValueError, "user id longer than %d bytes" % ID_MAX, 0),
    IID_LONG: (ValueError, "item id + domain label longer than %d bytes" % ID_MAX, 1),
}
_TOKEN = re.compile(rb"[^\t-\r\x1c-\x20]+")


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _Timer(object):
    """Optional CUDA-event timing of the phases (tools/ingest_time.py): {name: [(start, end) events]}."""

    def __init__(self, events):
        self.events = events

    def __call__(self, name):
        return _Phase(self.events, name)


class _Phase(object):
    def __init__(self, events, name):
        self.events, self.name = events, name

    def __enter__(self):
        if self.events is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.events is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            self.events.setdefault(self.name, []).append((self.a, b))


class _Times(Sequence):
    """enc.times of an ingested training set: datetime.fromtimestamp of the float64 seconds, made on access."""

    def __init__(self, ts):
        self._ts = ts

    def __len__(self):
        return len(self._ts)

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [datetime.fromtimestamp(t) for t in self._ts[k].tolist()]
        return datetime.fromtimestamp(float(self._ts[k]))


@dataclass
class IngestArrays:
    """The training and test sets of clean_split_pipeline as arrays.
    Train records (in the host path's record order): user / item index `uids` / `iids` (sorted unique ids of the
    training set, as encode.encode_records numbers them), rating and ts (float64 seconds) on the device; `meta` holds
    the item codes of `iids`.  Test records index `all_uids` / `all_iids` (every id of the two files, sorted).
    train_users / train_ptr: the train RDD's records in order, record k = user all_uids[train_users[k]] with the
    train arrays [train_ptr[k], train_ptr[k+1]) (a test user may have none); test_users / test_ptr the same for
    the test records."""
    user: torch.Tensor
    item: torch.Tensor
    rating: torch.Tensor
    ts: torch.Tensor
    test_user: torch.Tensor
    test_item: torch.Tensor
    test_rating: torch.Tensor
    test_ts: torch.Tensor
    uids: np.ndarray
    iids: np.ndarray
    all_uids: np.ndarray
    all_iids: np.ndarray
    meta: E.ItemMeta
    train_users: np.ndarray
    train_ptr: np.ndarray
    test_users: np.ndarray
    test_ptr: np.ndarray
    codes: dict = field(default_factory=dict)      # the item codes on the host (encode.item_codes names)


# ---- reading and parsing -------------------------------------------------------------------------------------------
class _File(object):
    def __init__(self, path, dev, timer):
        self.path = path
        with open(path, "rb") as f:
            size = os.fstat(f.fileno()).st_size
            self.host = torch.empty(size + 32, dtype=torch.uint8, pin_memory=True)
            view = self.host.numpy()
            got = 0
            while got < size:
                k = f.readinto(memoryview(view[got:size]))
                if not k:
                    break
                got += k
        size = got
        if size and view[size - 1] not in (10, 13):       # a last line without terminator
            view[size] = 10
            size += 1
        pad = (size + 15) // 16 * 16
        view[size:pad] = 0
        self.size = size
        with timer("h2d"):
            self.buf = self.host[:max(pad, 16)].to(dev, non_blocking=True)
        L = N.lib()
        nch = (size + 15) // 16
        nblk = (nch + 255) // 256
        masks = torch.empty(nch, dtype=torch.int16, device=dev)
        cnt = torch.empty(nblk, dtype=torch.int32, device=dev)
        with timer("line_masks"):
            N.check(L.xmap_ingest_line_masks(N.ptr(self.buf), size, N.ptr(masks), N.ptr(cnt), _stream()),
                    "xmap_ingest_line_masks")
        csum = torch.cumsum(cnt, 0, dtype=torch.int64)
        n = int(csum[-1]) if nblk else 0
        self.offs = torch.empty(n, dtype=torch.int64, device=dev)
        with timer("line_offsets"):
            N.check(L.xmap_ingest_line_offsets(N.ptr(masks), size, N.ptr(csum - cnt), N.ptr(self.offs), _stream()),
                    "xmap_ingest_line_offsets")
        self.n = n

    def line(self, k):
        """Bytes of line k (0-based), without its terminator."""
        o = self.offs[max(k - 1, 0): k + 1].cpu().tolist()
        lo = 0 if k == 0 else o[0] + 1
        return bytes(self.host.numpy()[lo:o[-1]]).rstrip(b"\r")


def _refuse(f, k, code):
    exc, what, which = _REFUSAL[code]
    line = f.line(k)
    toks = [(m.start(), m.group()) for m in _TOKEN.finditer(line)]
    if which is None:
        tok = line
    elif which == "byte":
        pos = next(i for i, c in enumerate(line) if c == 0 or c >= 0x80)
        tok = next((t for s, t in toks if s <= pos < s + len(t)), line)
    else:
        tok = toks[which][1]
    raise exc("%s, line %d: %s: %r" % (f.path, k + 1, what, tok.decode("latin-1")))


class _Lines(object):
    """Per line of both files (source lines first): status, rating, ts, and the packed id words."""

    def __init__(self, files, labels, dev, timer):
        L = N.lib()
        self.n = n = sum(f.n for f in files)
        if n > MAX_LINES:
            raise ValueError("%d lines: at most 2^31 - 1 are supported" % n)
        self.status = torch.empty(n, dtype=torch.uint8, device=dev)
        self.rating = torch.empty(n, dtype=torch.float64, device=dev)
        self.ts = torch.empty(n, dtype=torch.float64, device=dev)
        self.uw = torch.zeros(ID_MAX // 8, max(n, 1), dtype=torch.int64, device=dev)
        self.iw = torch.zeros(ID_MAX // 8, max(n, 1), dtype=torch.int64, device=dev)
        self.ulen = torch.empty(n, dtype=torch.uint8, device=dev)
        self.ilen = torch.empty(n, dtype=torch.uint8, device=dev)
        self.lo = []
        lo = 0
        for f, lab in zip(files, labels):
            self.lo.append(lo)
            if f.n:
                with timer("parse"):
                    N.check(L.xmap_ingest_parse(
                        N.ptr(f.buf), N.ptr(f.offs), f.n, lab, len(lab), TS_MIN, TS_MAX, max(n, 1),
                        N.ptr(self.status[lo:]), N.ptr(self.rating[lo:]), N.ptr(self.ts[lo:]), N.ptr(self.uw[:, lo:]),
                        N.ptr(self.ulen[lo:]), N.ptr(self.iw[:, lo:]), N.ptr(self.ilen[lo:]), _stream()),
                        "xmap_ingest_parse")
            lo += f.n
        self.lo.append(lo)
        if n:
            bad = (self.status >= FEW_FIELDS).view(torch.uint8)
            k = int(torch.argmax(bad))
            if int(bad[k]):
                d = 0 if k < self.lo[1] else 1
                _refuse(files[d], k - self.lo[d], int(self.status[k]))

    def domain_of(self, k):
        return 0 if k < self.lo[1] else 1


def _rank(words, lens, n, dev, timer):
    """Dense ranks of the ids (np.unique order) by an LSD sequence of stable sorts of their words; rep[r] = a line
    holding rank r.  Returns (rank int32 [n], rep int64 [n_distinct], words per id)."""
    L = N.lib()
    nw = max(1, (int(lens.max()) + 7) // 8) if n else 1
    with timer("rank_sort"):
        perm = torch.argsort(words[nw - 1, :n], stable=True)
        for w in range(nw - 2, -1, -1):
            perm = perm.index_select(0, torch.argsort(words[w, :n].index_select(0, perm), stable=True))
    flag = torch.empty(n, dtype=torch.int32, device=dev)
    with timer("rank_flags"):
        N.check(L.xmap_ingest_rank_flags(N.ptr(words), words.shape[1], nw, N.ptr(perm), n, N.ptr(flag), _stream()),
                "xmap_ingest_rank_flags")
    csum = torch.cumsum(flag, 0, dtype=torch.int64)
    nd = int(csum[-1]) if n else 0
    rank = torch.empty(n, dtype=torch.int32, device=dev)
    rep = torch.empty(nd, dtype=torch.int64, device=dev)
    with timer("rank_scatter"):
        N.check(L.xmap_ingest_rank_scatter(N.ptr(perm), N.ptr(flag), N.ptr(csum), n, N.ptr(rank), N.ptr(rep),
                                           _stream()), "xmap_ingest_rank_scatter")
    return rank, rep, nw


def _strings(words, rep, nw):
    """The id strings of the ranks (host numpy str array, ascending)."""
    if rep.numel() == 0:
        return np.zeros(0, dtype="<U1")
    a = words[:nw].index_select(1, rep).t().contiguous().cpu().numpy()
    return np.ascontiguousarray(a.astype(">i8")).view("S%d" % (8 * nw)).ravel().astype(str)


def _item_codes(P, rep, dev, timer, with_labels=True):
    """encode.item_codes of the items rep (ascending id order) on the device."""
    L = N.lib()
    n = int(rep.numel())
    labels = torch.zeros(0, dtype=torch.int32, device=dev)
    if with_labels and n:
        present = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
        with timer("item_codes"):
            N.check(L.xmap_ingest_item_suffix(N.ptr(P.iw), P.iw.shape[1], N.ptr(P.ilen), N.ptr(rep), n, N.ptr(present),
                                              _stream()), "xmap_ingest_item_suffix")
        labels = torch.nonzero(present).flatten().to(torch.int32)
        if labels.numel() > 8:
            raise ValueError("more than 8 distinct 2-character id suffixes; at most 8 domain labels are supported")
    prefix_new = torch.empty(n, dtype=torch.int32, device=dev)
    dom = torch.empty(n, dtype=torch.uint8, device=dev)
    contains = torch.empty(n, dtype=torch.uint8, device=dev)
    has_S = torch.empty(n, dtype=torch.bool, device=dev)
    has_T = torch.empty(n, dtype=torch.bool, device=dev)
    with timer("item_codes"):
        N.check(L.xmap_ingest_item_codes(N.ptr(P.iw), P.iw.shape[1], N.ptr(P.ilen), N.ptr(rep), n, N.ptr(labels),
                                         int(labels.numel()), N.ptr(prefix_new), N.ptr(dom), N.ptr(contains),
                                         N.ptr(has_S), N.ptr(has_T), _stream()), "xmap_ingest_item_codes")
    prefix = (torch.cumsum(prefix_new, 0, dtype=torch.int32) - 1) if n else prefix_new
    return E.ItemMeta(prefix, dom, contains, has_S, has_T)


# ---- clean and split -----------------------------------------------------------------------------------------------
def _clean(P, d, urank, irank, n_users, tool, is_debug, dev, timer):
    """The lines of domain d kept by baseliner_clean_data_pipeline, in its record order (users in first-appearance
    order, a user's items in first-appearance order): global line indices."""
    L = N.lib()
    lo, hi = P.lo[d], P.lo[d + 1]
    n = hi - lo
    if n == 0 or len(tool.period) == 0:
        return torch.zeros(0, dtype=torch.int64, device=dev)
    user, item, ts = urank[lo:hi], irank[lo:hi], P.ts[lo:hi]
    t_lo, t_hi = CL.period_bounds(tool.period[0], tool.period[-1])
    with timer("clean"):
        order = CL.clean_order(user, item, ts, t_lo, t_hi)
        keep, user_items = CL.clean_sorted(user, item, ts, order, n_users, t_lo, t_hi, tool.num_atleast_rating)
        first_user = torch.full((max(n_users, 1),), INT32_MAX, dtype=torch.int32, device=dev)
        pair_first = torch.empty(n, dtype=torch.int32, device=dev)
        N.check(L.xmap_ingest_first(N.ptr(user), N.ptr(item), N.ptr(ts), N.ptr(order), N.ptr(keep), n, t_lo, t_hi,
                                    N.ptr(first_user), N.ptr(pair_first), _stream()), "xmap_ingest_first")
        kept = torch.nonzero(keep).flatten()
        if is_debug:                                     # take_partial_data: the first size_subset users
            ok = (user_items >= tool.num_atleast_rating) & (first_user[:n_users] < INT32_MAX)
            users = torch.nonzero(ok).flatten()
            users = users[torch.argsort(first_user[users])][: tool.size_subset]
            sel = torch.zeros(n_users, dtype=torch.bool, device=dev)
            sel[users] = True
            kept = kept[sel[user[kept].long()]]
        key = (first_user[user[kept].long()].long() << 32) | pair_first[kept].long()
        kept = kept[torch.argsort(key)]
    return kept + lo


def ingest_arrays(clean_source, clean_target, split_tool, path_source, path_target, is_debug, device="cuda",
                  events=None):
    """clean (both domains) + split of two rating files on the device; see the module docstring.  events: optional
    dict that receives CUDA-event pairs per phase."""
    dev = torch.device(device)
    timer = _Timer(events)
    labels = []
    for tool in (clean_source, clean_target):
        lab = str(tool.label).encode("ascii")
        if len(lab) > 16:
            raise ValueError("domain label %r: at most 16 bytes are supported" % tool.label)
        labels.append(lab)
    files = [_File(path_source, dev, timer), _File(path_target, dev, timer)]
    P = _Lines(files, labels, dev, timer)
    n = P.n
    urank, urep, unw = _rank(P.uw, P.ulen, n, dev, timer)
    irank, irep, inw = _rank(P.iw, P.ilen, n, dev, timer)
    n_users, n_items = int(urep.numel()), int(irep.numel())
    if n_users >= 1 << 30:
        raise ValueError("%d distinct users: at most 2^30 are supported" % n_users)
    all_uids, all_iids = _strings(P.uw, urep, unw), _strings(P.iw, irep, inw)

    src = _clean(P, 0, urank, irank, n_users, clean_source, is_debug, dev, timer)
    tgt = _clean(P, 1, urank, irank, n_users, clean_target, is_debug, dev, timer)

    # ---- split: per-user draws on the host (users in the clean stage's order) --------------------------------------
    with timer("split"):
        rec = torch.cat([src, tgt])                        # lines in the order of source list + target list
        ru, ri = urank[rec], irank[rec]
        su = torch.unique_consecutive(urank[src]).cpu().numpy()
        tu = torch.unique_consecutive(urank[tgt]).cpu().numpy()
    in_s = np.zeros(n_users, dtype=bool)
    in_t = np.zeros(n_users, dtype=bool)
    in_s[su] = True
    in_t[tu] = True
    ov = su[in_t[su]]                                    # overlap users in source order = reduceByKey order
    cells = split_cells([split_tool.ratio_split, split_tool.ratio_both,
                         1 - split_tool.ratio_split - split_tool.ratio_both], split_tool.seed, len(ov))
    ns, nt = su[~in_t[su]], tu[~in_s[tu]]
    grp = np.full(n_users, -1, dtype=np.int8)
    upos = np.zeros(n_users, dtype=np.int32)
    grp[ns], upos[ns] = 0, np.arange(len(ns))
    grp[nt], upos[nt] = 1, np.arange(len(nt))
    grp[ov], upos[ov] = np.array([4, 2, 3], dtype=np.int8)[cells], np.arange(len(ov))
    test_users = ov[cells == 0]
    with timer("split"):
        meta_all = _item_codes(P, irep, dev, timer, with_labels=False)
        grp_d, upos_d = torch.from_numpy(grp).to(dev), torch.from_numpy(upos).to(dev)
        ru_l = ru.long()
        tidx = torch.nonzero((grp_d[ru_l] == 4) & ~meta_all.has_S[ri.long()]).flatten()
        tpos = upos_d[ru_l[tidx]].long()
        o = torch.argsort(tpos, stable=True)
        tidx, tpos = tidx[o], tpos[o]
        cnt = torch.bincount(tpos, minlength=len(ov)).cpu().numpy() if len(ov) else np.zeros(0, np.int64)
    start = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    srank_flat = np.full(int(start[-1]), -1, dtype=np.int32)
    for u in test_users:                                 # split_data's loop: one random.sample per test user
        k = upos[u]
        drawn = random.sample(range(int(cnt[k])), split_tool.num_left)
        srank_flat[start[k] + np.asarray(drawn, dtype=np.int64)] = np.arange(len(drawn), dtype=np.int32)
    if len(srank_flat) and srank_flat.max() + 1 >= 1 << 26:
        raise ValueError("num_left %d: at most 2^26 - 2 are supported" % split_tool.num_left)
    L = N.lib()
    with timer("split"):
        srank_flat_d = torch.from_numpy(srank_flat).to(dev)
        srank = torch.full((rec.numel(),), -1, dtype=torch.int32, device=dev)
        srank[tidx] = srank_flat_d
        key = torch.empty(rec.numel(), dtype=torch.int64, device=dev)
        N.check(L.xmap_ingest_train_keys(N.ptr(ru), N.ptr(ri), N.ptr(grp_d), N.ptr(upos_d), N.ptr(meta_all.has_S),
                                         N.ptr(srank), rec.numel(), N.ptr(key), _stream()), "xmap_ingest_train_keys")
        tr = torch.nonzero(key >= 0).flatten()
        tr = tr[torch.argsort(key[tr], stable=True)]
        train_line, test_line = rec[tr], rec[tidx[srank_flat_d < 0]]

    # ---- train-only numbering: a flag scan over the ranks, no second sort --------------------------------------------
    with timer("encode"):
        tu_all, ti_all = urank[train_line].long(), irank[train_line].long()
        used_u = torch.zeros(n_users, dtype=torch.int32, device=dev)
        used_i = torch.zeros(n_items, dtype=torch.int32, device=dev)
        used_u[tu_all] = 1
        used_i[ti_all] = 1
        user = (torch.cumsum(used_u, 0, dtype=torch.int32) - 1)[tu_all] if n_users else tu_all.int()
        item = (torch.cumsum(used_i, 0, dtype=torch.int32) - 1)[ti_all] if n_items else ti_all.int()
        used_u_h, used_i_h = used_u.bool().cpu().numpy(), used_i.bool().cpu().numpy()
    n_train_items = int(used_i_h.sum())
    if n_train_items > MAX_ITEMS:
        raise ValueError("%d training items: at most 2^24 are supported" % n_train_items)
    meta = _item_codes(P, irep[torch.from_numpy(used_i_h).to(dev)], dev, timer)
    rating = P.rating[train_line]
    bad = (rating.float().double() != rating).view(torch.uint8)
    if rating.numel() and int(bad.max()):
        k = int(train_line[int(torch.argmax(bad))])
        d = P.domain_of(k)
        tok = [t for t in _TOKEN.findall(files[d].line(k - P.lo[d]))][2]
        raise ValueError("%s, line %d: %r: ratings must be exactly representable in binary32 (integer / half-star "
                         "scales are); got values that are not" % (files[d].path, k - P.lo[d] + 1, tok.decode()))

    train_users = np.concatenate([ns, nt, ov[cells == 1], ov[cells == 2], test_users]).astype(np.int64)
    tcount = np.bincount(tu_all.cpu().numpy(), minlength=n_users) if n_users else np.zeros(0, np.int64)
    test_u = urank[test_line].long()
    ecount = np.bincount(test_u.cpu().numpy(), minlength=n_users) if n_users else np.zeros(0, np.int64)
    ptr = lambda users, c: np.concatenate([[0], np.cumsum(c[users])]).astype(np.int64)
    codes = dict(zip(("prefix_code", "dom_code", "contains", "has_S", "has_T"),
                     (meta.prefix_code.cpu().numpy(), meta.dom_code.cpu().numpy(), meta.contains.cpu().numpy(),
                      meta.has_S.cpu().numpy(), meta.has_T.cpu().numpy())))
    return IngestArrays(user=user.int(), item=item.int(), rating=rating, ts=P.ts[train_line],
                        test_user=test_u.int(), test_item=irank[test_line], test_rating=P.rating[test_line],
                        test_ts=P.ts[test_line], uids=all_uids[used_u_h], iids=all_iids[used_i_h],
                        all_uids=all_uids, all_iids=all_iids, meta=meta,
                        train_users=train_users, train_ptr=ptr(train_users, tcount),
                        test_users=test_users.astype(np.int64), test_ptr=ptr(test_users, ecount), codes=codes)


# ---- RDD facade ----------------------------------------------------------------------------------------------------
def _records(users, ptr, uids, iids, item, rating, ts):
    """(uid, [(iid, rating, datetime)]) records; item indexes iids."""
    it = iids[item].tolist() if len(item) else []
    r, t = rating.tolist(), ts.tolist()
    out = []
    for k, u in enumerate(users.tolist()):
        a, b = int(ptr[k]), int(ptr[k + 1])
        out.append((str(uids[u]), [(it[q], r[q], datetime.fromtimestamp(t[q])) for q in range(a, b)]))
    return out


def encoded(A):
    """encode.Encoded of the training set (what encode_records(train.collect()) holds), times made on access."""
    c = A.codes
    uids = A.uids if len(A.uids) else np.zeros(0, dtype="<U1")
    iids = A.iids if len(A.iids) else np.zeros(0, dtype="<U1")
    return ENC.Encoded(uids, iids, A.user.cpu().numpy(), A.item.cpu().numpy(), A.rating.cpu().numpy(),
                       _Times(A.ts.cpu().numpy()), c["prefix_code"], c["dom_code"], c["contains"], c["has_S"],
                       c["has_T"])


def clean_split_pipeline(sc, clean_source, clean_target, split_tool, path_source, path_target, is_debug,
                         device="cuda"):
    """baseliner_clean_data_pipeline(sc, clean_source, path_source, is_debug, ...), the same for the target, then
    baseliner_split_data_pipeline: returns (train, test) LazyRDDs with the same records in the same order.  `train`
    carries the Session the similarity stage uses.  sc must be None (no Spark)."""
    if sc is not None:
        raise ValueError("clean_split_pipeline runs without Spark: sc must be None")
    from .session import Session
    A = ingest_arrays(clean_source, clean_target, split_tool, path_source, path_target, is_debug, device)
    enc = encoded(A)
    train_host = (A.train_users, A.train_ptr, A.all_uids, A.iids, enc.item, enc.rating, A.ts.cpu().numpy())
    train = LazyRDD(lambda: _records(*train_host), handle=A)
    test_host = (A.test_users, A.test_ptr, A.all_uids, A.all_iids, A.test_item.cpu().numpy(),
                 A.test_rating.cpu().numpy(), A.test_ts.cpu().numpy())
    test = LazyRDD(lambda: _records(*test_host), handle=A)
    if len(enc.user):
        train._xmap_session = Session(enc, device, user=A.user, item=A.item, rating=A.rating, meta=A.meta)
    return train, test
