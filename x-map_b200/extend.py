"""X-SIM extension driver (C ABI section 3).

Turns the fixed-width neighbour tables of the similarity stage into the three
index structures the kernel walks, exactly following the reference's wiring:

  attach(b)    NB items n that list bridge item b in NB_BB(n), with NB_NN(n)
               (extender.py:48-59, reduceByKey :171-173)
  src pairs    (t, s): s a bridge item with "S:" in its id and a non-empty attach
               list, t any key of knn_BB[s] with "T:" in its id   (extender.py:61-70)
  tgt pairs    (t, s): t a bridge item with "T:" and attach, s a key of knn_BB[t]
               with "S:"                                           (extender.py:72-81)
  joint        src pairs that are also tgt pairs (the inner join, extender.py:178)
  right(s)     s ; (s,n) ; (s,n,x) for x in NB_NN(n)               (extender.py:134-138)
  left(t)      (n,t) ; (x,n,t)                                     (extender.py:160-167)

Edge values are symmetric in this implementation (sim(a,b) == sim(b,a)
bitwise), so the reference's 4-way lookup precedence (extender.py:100-112)
cannot change a value and every edge is read from the row that lists it.

All index building is torch (sort / cumsum / repeat_interleave) on whatever
device the tables live on; the path evaluation itself is the CUDA kernel.
"""
import os
from dataclasses import dataclass

import torch

from . import _native as N



def _excl_cumsum(x):
    return torch.cumsum(x, 0) - x


def _segment_ids(lengths):
    return torch.repeat_interleave(torch.arange(lengths.numel(), device=lengths.device), lengths)


@dataclass
class XsimPlan:
    n_items: int
    start_item: torch.Tensor
    leg_ptr: torch.Tensor
    leg_t: torch.Tensor
    leg_joint_only: torch.Tensor
    leg_vals: tuple              # e1, m1, f1, e2, m2, f2
    par_ptr: torch.Tensor
    par_s: torch.Tensor
    par_joint: torch.Tensor
    par_vals: tuple              # e, m, f
    rs_ptr: torch.Tensor
    rs_end: torch.Tensor
    rs_vals: tuple               # e1, m1, f1, e2, m2, f2
    ub: torch.Tensor             # per start: combos (= reference paths) it will evaluate
    ub_leg: torch.Tensor         # per leg
    n_src: int
    n_joint: int
    t_items: torch.Tensor        # bridge targets, indexed by leg_t / par_ptr
    s_items: torch.Tensor        # bridge sources, indexed by par_s / rs_ptr


def build_plan(tabs, item_count, has_S, has_T):
    """tabs: engine.SimTables (global, i.e. holding every item's lists)."""
    dev = tabs.tab_idx.device
    I, k = tabs.n_items, tabs.k
    i64 = torch.int64
    bb = (tabs.row_flags & 1).bool()
    tlen = tabs.tab_len.long()
    valid_nb = (~bb) & (tlen[:, 0] > 0)
    r = torch.arange(k, device=dev)

    def flat(slot, rowmask):
        """All (row, nbr, e, m, f) entries of `slot` for rows in rowmask, row-major."""
        m = rowmask[:, None] & (r[None, :] < tlen[:, slot, None])
        rows, pos = torch.nonzero(m, as_tuple=True)
        nbr = tabs.tab_idx[rows, slot, pos].long()
        sim = tabs.tab_sim[rows, slot, pos]
        mutu = tabs.tab_mutu[rows, slot, pos].double()
        n = tabs.tab_n[rows, slot, pos].double()
        frac = 1.0 * mutu / (item_count[rows] + item_count[nbr] - n)     # baselinerSim.py:171-173
        return rows, nbr, sim * mutu, mutu, frac

    # ---- attach edges (b <- n), ordered by (b, n) -------------------------
    n_row, b_nbr, a_e, a_m, a_f = flat(0, valid_nb)
    o = torch.argsort(b_nbr * I + n_row)
    att_b, att_n = b_nbr[o], n_row[o]
    att_e, att_m, att_f = a_e[o], a_m[o], a_f[o]
    a_cnt = torch.bincount(att_b, minlength=I)
    nn_len = torch.where(valid_nb, tlen[:, 1], torch.zeros_like(tlen[:, 1]))
    # NB_NN entries, row-major; nn_ptr[n] indexes them
    nn_row, nn_x, nn_e, nn_m, nn_f = flat(1, valid_nb)
    nn_ptr = torch.zeros(I + 1, dtype=i64, device=dev)
    nn_ptr[1:] = torch.cumsum(nn_len, 0)

    # ---- bridge pairs -----------------------------------------------------
    kb_row0, kb_nbr0, kb_e0, kb_m0, kb_f0 = flat(0, bb)
    kb_row1, kb_nbr1, kb_e1, kb_m1, kb_f1 = flat(1, bb)
    kb_row = torch.cat([kb_row0, kb_row1]); kb_nbr = torch.cat([kb_nbr0, kb_nbr1])
    kb_e = torch.cat([kb_e0, kb_e1]); kb_m = torch.cat([kb_m0, kb_m1]); kb_f = torch.cat([kb_f0, kb_f1])
    has_att = a_cnt > 0
    src_m = has_S[kb_row] & has_att[kb_row] & has_T[kb_nbr]
    src_t, src_s = kb_nbr[src_m], kb_row[src_m]
    src_e, src_m_, src_f = kb_e[src_m], kb_m[src_m], kb_f[src_m]
    tgt_m = has_T[kb_row] & has_att[kb_row] & has_S[kb_nbr]
    tgt_key = torch.unique(kb_row[tgt_m] * I + kb_nbr[tgt_m])
    src_key = src_t * I + src_s
    o = torch.argsort(src_key)
    src_key, src_t, src_s = src_key[o], src_t[o], src_s[o]
    src_e, src_m_, src_f = src_e[o], src_m_[o], src_f[o]
    if tgt_key.numel() and src_key.numel():
        p = torch.searchsorted(tgt_key, src_key).clamp(max=tgt_key.numel() - 1)
        joint = tgt_key[p] == src_key
    else:
        joint = torch.zeros_like(src_key, dtype=torch.bool)

    # ---- right segments per bridge source s -------------------------------
    s_items = torch.unique(src_s)
    s_index = torch.full((I,), -1, dtype=i64, device=dev)
    s_index[s_items] = torch.arange(s_items.numel(), device=dev)
    am = s_index[att_b] >= 0
    ra_s, ra_n = s_index[att_b[am]], att_n[am]
    ra_e, ra_m, ra_f = att_e[am], att_m[am], att_f[am]
    blk = 1 + nn_len[ra_n]
    R = torch.ones(s_items.numel(), dtype=i64, device=dev)
    R.index_add_(0, ra_s, blk)
    rs_ptr = torch.zeros(s_items.numel() + 1, dtype=i64, device=dev)
    rs_ptr[1:] = torch.cumsum(R, 0)
    total_rs = int(rs_ptr[-1].item()) if s_items.numel() else 0
    rs_end = torch.empty(total_rs, dtype=torch.int32, device=dev)
    f64 = dict(dtype=torch.float64, device=dev)
    rs_e1 = torch.zeros(total_rs, **f64); rs_m1 = torch.zeros(total_rs, **f64); rs_f1 = torch.ones(total_rs, **f64)
    rs_e2 = torch.zeros(total_rs, **f64); rs_m2 = torch.zeros(total_rs, **f64); rs_f2 = torch.ones(total_rs, **f64)
    if total_rs:
        rs_end[rs_ptr[:-1]] = s_items.to(torch.int32)                    # the bare (t, s) path ends at s
        # block start of attach edge a inside its s: 1 + blocks before it in the same s
        cs = _excl_cumsum(blk)
        first_of_s = torch.zeros(s_items.numel(), dtype=i64, device=dev)
        cnt_s = torch.bincount(ra_s, minlength=s_items.numel())
        first_edge = _excl_cumsum(cnt_s)
        nz = cnt_s > 0
        first_of_s[nz] = cs[first_edge[nz]]
        blk_start = rs_ptr[ra_s] + 1 + (cs - first_of_s[ra_s])
        a_of = _segment_ids(blk)
        q = torch.arange(a_of.numel(), device=dev) - _excl_cumsum(blk)[a_of]
        pos = blk_start[a_of] + q
        is_n = q == 0
        nnp = (nn_ptr[ra_n[a_of]] + q - 1).clamp(min=0)
        rs_end[pos] = torch.where(is_n, ra_n[a_of], nn_x[nnp] if nn_x.numel() else ra_n[a_of]).to(torch.int32)
        rs_e1[pos] = ra_e[a_of]; rs_m1[pos] = ra_m[a_of]; rs_f1[pos] = ra_f[a_of]
        if nn_x.numel():
            one = torch.ones_like(nn_f[nnp]); zero = torch.zeros_like(nn_e[nnp])
            rs_e2[pos] = torch.where(is_n, zero, nn_e[nnp])
            rs_m2[pos] = torch.where(is_n, zero, nn_m[nnp])
            rs_f2[pos] = torch.where(is_n, one, nn_f[nnp])

    # ---- partners per bridge target t -------------------------------------
    t_items = torch.unique(src_t)
    t_index = torch.full((I,), -1, dtype=i64, device=dev)
    t_index[t_items] = torch.arange(t_items.numel(), device=dev)
    par_cnt = torch.bincount(t_index[src_t], minlength=t_items.numel()) if src_t.numel() else \
        torch.zeros(0, dtype=i64, device=dev)
    par_ptr = torch.zeros(t_items.numel() + 1, dtype=i64, device=dev)
    par_ptr[1:] = torch.cumsum(par_cnt, 0)
    par_s = s_index[src_s].to(torch.int32)               # src pairs are already sorted by (t, s)
    Rs = R[s_index[src_s]] if src_s.numel() else torch.zeros(0, dtype=i64, device=dev)
    rt_all = torch.zeros(t_items.numel(), dtype=i64, device=dev)
    rt_joint = torch.zeros(t_items.numel(), dtype=i64, device=dev)
    if src_t.numel():
        rt_all.index_add_(0, t_index[src_t], Rs)
        rt_joint.index_add_(0, t_index[src_t], Rs * joint.long())

    # ---- legs per start ---------------------------------------------------
    zt = torch.zeros(t_items.numel(), **f64); ot = torch.ones(t_items.numel(), **f64)
    # type 0: the bridge target itself starts the non-joint paths (extender.py:180)
    L_start = [t_items]; L_t = [torch.arange(t_items.numel(), device=dev)]
    L_jo = [torch.zeros(t_items.numel(), dtype=torch.uint8, device=dev)]
    L_type = [torch.zeros(t_items.numel(), dtype=i64, device=dev)]
    L_vals = [[zt], [zt], [ot], [zt], [zt], [ot]]
    # types 1, 2: attach edges of targets that have at least one joint partner
    tj = torch.zeros(I, dtype=torch.bool, device=dev)
    if src_t.numel():
        tj[src_t[joint]] = True
    lm = tj[att_b]
    la_t, la_n = att_b[lm], att_n[lm]
    la_e, la_m, la_f = att_e[lm], att_m[lm], att_f[lm]
    na = la_t.numel()
    if na:
        L_start.append(la_n); L_t.append(t_index[la_t])
        L_jo.append(torch.ones(na, dtype=torch.uint8, device=dev))
        L_type.append(torch.ones(na, dtype=i64, device=dev))
        for lst, v in zip(L_vals, (la_e, la_m, la_f, torch.zeros(na, **f64), torch.zeros(na, **f64),
                                   torch.ones(na, **f64))):
            lst.append(v)
        ln = nn_len[la_n]
        a_of = _segment_ids(ln)
        if a_of.numel():
            q = torch.arange(a_of.numel(), device=dev) - _excl_cumsum(ln)[a_of]
            nnp = nn_ptr[la_n[a_of]] + q
            L_start.append(nn_x[nnp]); L_t.append(t_index[la_t[a_of]])
            L_jo.append(torch.ones(a_of.numel(), dtype=torch.uint8, device=dev))
            L_type.append(torch.full((a_of.numel(),), 2, dtype=i64, device=dev))
            # path (x, n, t): edge (x, n) first, then (n, t)
            for lst, v in zip(L_vals, (nn_e[nnp], nn_m[nnp], nn_f[nnp], la_e[a_of], la_m[a_of], la_f[a_of])):
                lst.append(v)
    lg_start = torch.cat(L_start); lg_t = torch.cat(L_t); lg_jo = torch.cat(L_jo); lg_type = torch.cat(L_type)
    lg_vals = [torch.cat(v) for v in L_vals]
    # stable sort by (start, type): construction order inside a type is already (t, n, q)
    o = torch.argsort(lg_start * 4 + lg_type, stable=True)
    lg_start, lg_t, lg_jo = lg_start[o], lg_t[o], lg_jo[o]
    lg_vals = [v[o] for v in lg_vals]
    start_item, leg_cnt = torch.unique_consecutive(lg_start, return_counts=True)
    leg_ptr = torch.zeros(start_item.numel() + 1, dtype=i64, device=dev)
    leg_ptr[1:] = torch.cumsum(leg_cnt, 0)
    ub_leg = torch.where(lg_jo.bool(), rt_joint[lg_t], rt_all[lg_t]) if lg_t.numel() else \
        torch.zeros(0, dtype=i64, device=dev)
    ub = torch.zeros(start_item.numel(), dtype=i64, device=dev)
    if lg_t.numel():
        ub.index_add_(0, _segment_ids(leg_cnt), ub_leg)
    return XsimPlan(
        n_items=I, start_item=start_item.to(torch.int32), leg_ptr=leg_ptr, leg_t=lg_t.to(torch.int32),
        leg_joint_only=lg_jo.contiguous(), leg_vals=tuple(v.contiguous() for v in lg_vals),
        par_ptr=par_ptr, par_s=par_s.contiguous(), par_joint=joint.to(torch.uint8).contiguous(),
        par_vals=(src_e.contiguous(), src_m_.contiguous(), src_f.contiguous()),
        rs_ptr=rs_ptr, rs_end=rs_end, rs_vals=(rs_e1, rs_m1, rs_f1, rs_e2, rs_m2, rs_f2),
        ub=ub, ub_leg=ub_leg, n_src=int(src_t.numel()), n_joint=int(joint.sum().item()) if joint.numel() else 0,
        t_items=t_items, s_items=s_items)


PI_MULT = 0x9E3779B1            # pi(y) = (y * PI_MULT) mod 2^32 orders every right-segment list (csrc/xsim.cu)
XSIM_CELLS_LG = int(os.environ.get("XMAP_XSIM_CELLS_LG", "9"))    # 512-cell shared-memory table per warp ...
XSIM_WARPS = int(os.environ.get("XMAP_XSIM_WARPS", "20"))         # ... 20 warps per CTA (limited by registers: 94 x 640)
XSIM_LOAD = float(os.environ.get("XMAP_XSIM_LOAD", "0.62"))       # target fill of a table
XSIM_RHO = float(os.environ.get("XMAP_XSIM_RHO", "1.25"))         # assumed paths per distinct end when a start's pass count is chosen
                                # (measured at cfg2: 10 % quantile 1.30, median 1.62; a pass that turns out
                                # too full is split on the device)
XSIM_UNIT_WORK = 1 << int(os.environ.get("XMAP_XSIM_UNIT_LG", "17"))   # paths per unit (= per warp): heavier starts are
                                # cut into more units (disjoint end ranges)
XSIM_MAX_PASSES = int(os.environ.get("XMAP_XSIM_MAX_PASSES", "1000000000"))   # cap on the passes a start is cut into for
                                # table capacity; a unit whose ends then exceed the shared-memory table keeps its table in
                                # global memory (L2).  Measured at cfg2: 32 passes + L2 tables 968 ms, shared memory only
                                # (no cap) 732 ms -- dependent read-modify-writes at L2 latency lose to narrow passes
XSIM_GCELLS_LG = 16             # largest global-memory table of a unit (cells)
XSIM_MODE = os.environ.get("XMAP_XSIM_MODE", "hybrid")                # "warp": one warp per unit (xsim_warp_kernel); "cta": one CTA
                                                                   # per unit with one 8x larger table (xsim_cta_kernel)
XSIM_FUSE = os.environ.get("XMAP_XSIM_FUSE", "1") != "0"          # fused bridge lists B(t) for the joint-only legs
XSIM_FUSE_MAX = 1 << 31         # entries (28 B each + sort scratch) above which the lists are not fused: a fixed number, not a
                                # function of free memory, so that every rank takes the same decision
XSIM_BALANCE = os.environ.get("XMAP_XSIM_BALANCE", "heat")     # how a heavy start's tiles are cut into units: equal "heat"
                                # (expected paths) or "uniform" (equal numbers of tiles)
XSIM_HOT_PATHS = float(os.environ.get("XMAP_XSIM_HOT_PATHS", str(1 << 19)))   # hybrid mode: a unit expected to hold more paths
                                # than this is run by the CTA kernel (8 warps on one unit) instead of one warp
XSIM_CTA_CELLS_LG = int(os.environ.get("XMAP_XSIM_CTA_CELLS_LG", "12"))
XSIM_CTA_UNIT_LG = int(os.environ.get("XMAP_XSIM_CTA_UNIT_LG", "17"))     # 2^17 paths per unit: short critical path when units are dealt to 8 GPUs


@dataclass
class XsimResult:
    start_item: torch.Tensor     # int32 [n_starts]
    count: torch.Tensor          # int32 distinct ends per start
    combos: torch.Tensor         # int64 paths evaluated per start
    top_end: torch.Tensor        # int32 [n_starts, top_m], |xsim| desc, ties to smaller end
    top_xsim: torch.Tensor
    top_len: torch.Tensor
    launches: int
    unit_count: torch.Tensor = None   # int32 [n_units] distinct ends per work unit (sizes the emit pass)


class XsimEngine:
    """Runs the extension kernels over an XsimPlan (C ABI section 3).

    The accumulator of a start lives in shared memory.  The end axis is hashed (pi) and cut into 2^gb
    tiles; a start evaluates its paths in passes over tile ranges small enough for a warp's table, a warp
    runs one unit = one or more passes of one start, heavy starts are spread over several units.  The
    summation order of a (start, end) cell depends on the path structure and this plan only, so results
    are bit-identical from run to run and for any number of GPUs."""

    def __init__(self, plan, top_m=10, cells_lg=None, rho=XSIM_RHO, unit_work=None,
                 load=XSIM_LOAD, warps=XSIM_WARPS, max_passes=XSIM_MAX_PASSES, mode=XSIM_MODE, fuse=None,
                 fuse_max_entries=XSIM_FUSE_MAX, hot_paths=None, balance=XSIM_BALANCE):
        if mode not in ("hybrid", "warp", "cta"):
            raise ValueError("mode must be 'hybrid', 'warp' or 'cta'")
        self.mode = mode
        self.hot_paths = float(XSIM_HOT_PATHS if hot_paths is None else hot_paths)
        if fuse is None:
            fuse = XSIM_FUSE
        if cells_lg is None:
            cells_lg = XSIM_CTA_CELLS_LG if mode == "cta" else XSIM_CELLS_LG
        if unit_work is None:
            unit_work = (1 << XSIM_CTA_UNIT_LG) if mode == "cta" else XSIM_UNIT_WORK
        if mode == "cta":
            max_passes = 10 ** 9                 # shared memory only
            if cells_lg < 9:
                raise ValueError("cta mode needs cells_lg >= 9")
        if not (1 <= top_m <= N.KMAX):
            raise ValueError("top_m must be in [1, %d]" % N.KMAX)
        if not (6 <= cells_lg <= N.XSIM_MAX_CELLS_LG):
            raise ValueError("cells_lg must be in [6, %d]" % N.XSIM_MAX_CELLS_LG)
        warps = int(warps)
        while mode != "cta" and warps > 1 and N.lib().xmap_xsim_smem_bytes(int(cells_lg), warps) > 227 * 1024:
            warps -= 1
        self.plan, self.top_m, self.cells_lg, self.warps = plan, int(top_m), int(cells_lg), warps
        self.unit_counter = torch.zeros(1, dtype=torch.int32, device=plan.start_item.device)
        p = plan
        dev = self.device = p.start_item.device
        self.launches = 0
        i64, i32 = torch.int64, torch.int32
        n = int(p.start_item.numel())
        self.error_flag = torch.zeros(1, dtype=i32, device=dev)
        # ---- legs: left segment folded in path order (edge (x,n) first, then (n,t)) ---------------------
        e1, m1, f1, e2, m2, f2 = p.leg_vals
        self.leg_n, self.leg_d, self.leg_c = (e1 + e2).contiguous(), (m1 + m2).contiguous(), (f1 * f2).contiguous()
        # ---- partners: the joint ones first within every bridge target, so that a joint-only leg (the
        # reference's inner join, extender.py:178) uses a prefix of the list ----------------------------
        par_cnt = p.par_ptr[1:] - p.par_ptr[:-1]
        t_of_par = _segment_ids(par_cnt)
        joint = p.par_joint.long()
        perm_par = torch.argsort(t_of_par * 2 + (1 - joint), stable=True) if joint.numel() else joint
        self.par_s = p.par_s[perm_par].contiguous()
        self.par_e, self.par_m, self.par_f = (v[perm_par].contiguous() for v in p.par_vals)
        jcnt = torch.zeros_like(par_cnt)
        if joint.numel():
            jcnt.index_add_(0, t_of_par, joint)
        lt = p.leg_t.long()
        leg_npar = torch.where(p.leg_joint_only.bool(), jcnt[lt], par_cnt[lt]) if lt.numel() else \
            torch.zeros(0, dtype=i64, device=dev)
        leg_par_base = p.par_ptr[lt] if lt.numel() else torch.zeros(0, dtype=i64, device=dev)
        # ---- right segments: the two edges folded into one (N, D, C) triple (the sums are reassociated
        # by at most one rounding; D is an exact integer either way), every list ordered by pi(end) ------
        r1, rm1, rf1, r2, rm2, rf2 = p.rs_vals
        rl = p.rs_ptr[1:] - p.rs_ptr[:-1]
        n_s = int(rl.numel())
        seg = _segment_ids(rl)
        pi = (p.rs_end.long() * PI_MULT) & 0xFFFFFFFF
        perm = torch.argsort(seg * (1 << 32) + pi, stable=True) if seg.numel() else seg
        rs_end = p.rs_end[perm].contiguous()
        rs_ndc = [(r1 + r2)[perm].contiguous(), (rm1 + rm2)[perm].contiguous(), (rf1 * rf2)[perm].contiguous()]
        pi = pi[perm] if seg.numel() else pi
        rs_ptr = p.rs_ptr
        self.end_cap = int(torch.unique(p.rs_end).numel()) if p.rs_end.numel() else 1
        # ---- fused bridge lists: what follows a joint-only leg (x .. t) does not depend on the start, so
        # for every bridge target t the (bridge edge, right segment) combinations of its joint partners are
        # materialised once as ONE list B(t) = {(end, e + N_r, m + D_r, f * C_r)}, ordered by pi(end) like any
        # right-segment list.  A joint-only leg then has a single (virtual) partner whose list is B(t): a pass
        # resolves one sub-range per LEG instead of one per (leg, partner) pair, and the sub-ranges are as many
        # times longer.  (N_l + (e + N_r) instead of (N_l + e) + N_r: one more reassociation, DESIGN 6.5.)
        # The legs of type 0 (the bridge target itself, all partners) keep the pair lists.
        self.fused_entries = 0
        n_t = int(par_cnt.numel())
        jl = p.leg_joint_only.bool() if lt.numel() else torch.zeros(0, dtype=torch.bool, device=dev)
        if fuse and n_t and joint.numel() and bool(jl.any()):
            used = torch.zeros(n_t, dtype=torch.bool, device=dev)
            used[lt[jl]] = True
            jp = torch.nonzero((joint[perm_par] == 1) & used[t_of_par]).flatten()      # joint partners, (t, joint-first) order
            ln = rl[self.par_s[jp].long()]
            F = int(ln.sum().item())
            if 0 < F <= fuse_max_entries:
                a_of = _segment_ids(ln)
                q = torch.arange(F, device=dev) - _excl_cumsum(ln)[a_of]
                r = rs_ptr[self.par_s[jp].long()][a_of] + q
                pa = jp[a_of]
                tt = t_of_par[pa]
                o = torch.argsort(tt * (1 << 32) + pi[r], stable=True)
                del q, a_of
                r, pa, tt = r[o], pa[o], tt[o]
                del o
                f_end = rs_end[r]
                f_n = self.par_e[pa] + rs_ndc[0][r]
                f_d = self.par_m[pa] + rs_ndc[1][r]
                f_c = self.par_f[pa] * rs_ndc[2][r]
                f_pi = pi[r]
                del r, pa
                fl = torch.bincount(tt, minlength=n_t)
                total_rs = int(rs_ptr[-1].item())
                rs_ptr = torch.cat([rs_ptr[:-1], total_rs + _excl_cumsum(fl), rs_ptr.new_tensor([total_rs + F])])
                seg = torch.cat([seg, n_s + tt]); del tt
                pi = torch.cat([pi, f_pi]); del f_pi
                rs_end = torch.cat([rs_end, f_end]); del f_end
                rs_ndc = [torch.cat([rs_ndc[0], f_n]), torch.cat([rs_ndc[1], f_d]), torch.cat([rs_ndc[2], f_c])]
                del f_n, f_d, f_c
                rl = torch.cat([rl, fl])
                n_par = int(self.par_s.numel())
                self.par_s = torch.cat([self.par_s, (n_s + torch.arange(n_t, device=dev)).to(i32)])
                zt = torch.zeros(n_t, dtype=torch.float64, device=dev)
                self.par_e = torch.cat([self.par_e, zt]); self.par_m = torch.cat([self.par_m, zt])
                self.par_f = torch.cat([self.par_f, torch.ones_like(zt)])
                leg_par_base = torch.where(jl, n_par + lt, leg_par_base)
                leg_npar = torch.where(jl, torch.ones_like(leg_npar), leg_npar)
                n_s += n_t
                self.fused_entries = F
        if n_s and int(rl.max()) >= (1 << (26 if mode == "warp" else 23)):
            raise N.NativeError("a right-segment list is too long for the 32-bit product counter of a macro-batch "
                                "(2^26 entries, warp mode; 2^23, cta mode)")
        self.rs_ptr, self.rs_end, self.rs_ndc = rs_ptr.contiguous(), rs_end.contiguous(), tuple(v.contiguous() for v in rs_ndc)
        self.leg_npar = leg_npar.to(i32).contiguous()
        self.leg_par_base = leg_par_base.contiguous()
        self.lp_ptr = torch.zeros(lt.numel() + 1, dtype=i64, device=dev)
        self.lp_ptr[1:] = torch.cumsum(self.leg_npar.long(), 0)
        # ---- pair descriptors: one record per (leg, partner) pair in walking order, so that the kernels resolve a
        # pair with one coalesced load instead of a leg search and a chain of dependent gathers ------------------
        lop = _segment_ids(self.leg_npar.long())
        pp = self.leg_par_base[lop] + (torch.arange(lop.numel(), device=dev) - self.lp_ptr[:-1][lop])
        self.pd_s = self.par_s[pp].contiguous()
        self.pd_n = (self.leg_n[lop] + self.par_e[pp]).contiguous()           # sums in path order (extender.py:85-88)
        self.pd_d = (self.leg_d[lop] + self.par_m[pp]).contiguous()
        self.pd_c = (self.leg_c[lop] * self.par_f[pp]).contiguous()
        del lop, pp
        # ---- passes per start: enough for the estimated distinct ends, and enough units for its paths ---
        cap = max(16.0, load * (1 << self.cells_lg))
        ub = p.ub.double()
        e_est = torch.clamp(ub / float(rho), max=float(self.end_cap))
        T_fit = torch.clamp(torch.ceil(e_est / cap), min=1).long()             # passes whose ends fit shared memory
        n_units_x = torch.clamp(torch.ceil(ub / float(unit_work)), min=1).long()
        n_units_x = torch.minimum(n_units_x, T_fit)                             # at most one unit per such pass
        # few, wide passes keep the sub-range of a (leg, partner) pair long (full sectors, few duplicates per
        # 32-path step, few pair look-ups); a pass whose ends exceed the shared-memory table runs with a larger
        # table in global memory.  Heavy starts still get one pass per unit (parallelism).
        T = torch.maximum(torch.clamp(T_fit, max=max(1, int(max_passes))), n_units_x)
        t_max = int(T.max().item()) if n else 1
        # 2^gb tiles: at least the largest pass count (its passes are sized by the true bound end_cap and never
        # overflow); lighter starts have many tiles per pass, so an overflowing pass can be halved on the device
        self.gb = min(14, max(4, (t_max - 1).bit_length()))
        G = 1 << self.gb
        T = torch.clamp(T, max=G)
        n_units_x = torch.clamp(n_units_x, max=G)
        ppu = (T + n_units_x - 1) // n_units_x                                 # passes per unit
        tile = (pi >> (32 - self.gb)) if self.gb else torch.zeros_like(pi)
        # tile_ptr[s][g] = entries of list s in tiles < g.  Built a block of lists at a time (32-bit counts scattered
        # into the pointer rows, then a row-wise scan), so the scratch stays ~1 GB whatever the number of lists.
        self.tile_ptr = torch.zeros((n_s, G + 1), dtype=i32, device=dev)
        if seg.numel():
            blk = max(1, (1 << 27) // (G + 1))
            cuts = list(range(0, n_s, blk)) + [n_s]
            ent = self.rs_ptr[torch.tensor(cuts, device=dev)].tolist()
            for a0, a1, e0, e1 in zip(cuts[:-1], cuts[1:], ent[:-1], ent[1:]):
                if e1 == e0:
                    continue
                rows = self.tile_ptr[a0:a1]
                rows.view(-1).scatter_add_(0, (seg[e0:e1] - a0) * (G + 1) + tile[e0:e1] + 1,
                                           torch.ones(e1 - e0, dtype=i32, device=dev))
                rows.copy_(torch.cumsum(rows, 1, dtype=i32))
        # tile heat: the paths a start's walk is expected to spend in every tile = entries per tile weighted by the number
        # of (leg, partner) pairs that walk the list.  Popular ends are popular for every start, so this global profile
        # tells which tile range of a heavy start is hot (cfg2: one 2-tile unit of the heaviest start holds 7.8 M paths
        # where a uniform split expects 0.36 M).
        heat = torch.zeros(G, dtype=torch.float64, device=dev)
        if seg.numel() and self.pd_s.numel():
            usage = torch.bincount(self.pd_s.long(), minlength=n_s).double()
            heat.index_add_(0, tile, usage[seg])
        cum_heat = torch.zeros(G + 1, dtype=torch.float64, device=dev)
        cum_heat[1:] = torch.cumsum(heat, 0)
        del tile, seg, pi
        # ---- units -------------------------------------------------------------------------------------
        self.start_unit_ptr = torch.zeros(n + 1, dtype=i32, device=dev)
        self.start_unit_ptr[1:] = torch.cumsum(n_units_x, 0).to(i32)
        self.n_units = int(self.start_unit_ptr[-1].item()) if n else 0
        us = _segment_ids(n_units_x)
        kq = torch.arange(self.n_units, device=dev) - self.start_unit_ptr[:-1].long()[us]
        nu = n_units_x[us]
        self.unit_start = us
        tot_heat = float(cum_heat[-1].item()) if G else 0.0
        if balance == "heat" and tot_heat > 0 and self.n_units:
            # the units of a start take equal shares of the tile HEAT, not equal numbers of tiles (every unit keeps at
            # least one tile): cut k of nu sits where the cumulative heat reaches k / nu of the total
            cut = torch.searchsorted(cum_heat, kq.double() / nu.double() * tot_heat, right=False)
            cut = torch.where(kq == 0, torch.zeros_like(cut), cut)
            big = 2 * (G + 1)
            v = torch.cummax(cut - kq + us * big, 0).values - us * big + kq       # strictly increasing inside a start
            g0 = torch.minimum(v, G - (nu - kq))                                      # room for the units that follow
            nxt = torch.cat([g0[1:], g0.new_tensor([G])])
            g1 = torch.where(kq + 1 == nu, torch.full_like(g0, G), nxt)
            self.unit_g0, self.unit_g1 = g0.to(i32).contiguous(), g1.to(i32).contiguous()
            width = (g1 - g0)
            need = torch.clamp((T[us] * width + G - 1) // G, min=1)                   # ends are spread evenly over the tiles
            self.unit_npass = torch.minimum(need, width).to(i32).contiguous()
        else:
            self.unit_g0 = (kq * G // nu).to(i32).contiguous()
            self.unit_g1 = ((kq + 1) * G // nu).to(i32).contiguous()
            self.unit_npass = torch.minimum(ppu[us], (self.unit_g1 - self.unit_g0).long()).to(i32).contiguous()
        self.unit_leg_lo = p.leg_ptr[:-1][us].contiguous()
        self.unit_leg_hi = p.leg_ptr[1:][us].contiguous()
        # table a unit wants: its share of the start's estimated ends at the target load
        e_unit = e_est[us] / T[us].double()
        want = torch.ceil(torch.log2(torch.clamp(e_unit / float(load), min=2.0))).long()
        self.gcells_lg = int(min(XSIM_GCELLS_LG, max(int(want.max().item()) if self.n_units else 0, self.cells_lg)))
        self.unit_clg = torch.clamp(want, min=self.cells_lg, max=self.gcells_lg).to(i32).contiguous()
        self.gws = None
        if self.gcells_lg > self.cells_lg:
            sms = torch.cuda.get_device_properties(dev).multi_processor_count if dev.type == "cuda" else 1
            self.gws = torch.empty(sms * self.warps * (20 << self.gcells_lg), dtype=torch.uint8, device=dev)
        # expected paths of a unit: the start's paths times the heat share of the unit's tile range
        share = (cum_heat[self.unit_g1.long()] - cum_heat[self.unit_g0.long()]) / max(tot_heat, 1e-300) if tot_heat > 0 else \
            (self.unit_g1 - self.unit_g0).double() / float(G)
        unit_work_est = ub[us] * share
        self.unit_est_paths = unit_work_est
        self.unit_order = torch.argsort(unit_work_est, descending=True, stable=True).to(i32).contiguous()
        self.T, self.n_units_x = T, n_units_x
        # ---- hybrid: the units one warp would take too long over (a straggler bounds the multi-GPU time) are run by the
        # CTA kernel, 8 warps on one unit with one 8x larger table, the rest by the warp kernel.  The class of a unit is a
        # function of the plan only, so results do not depend on the number of GPUs.
        self.cta_cells_lg = XSIM_CTA_CELLS_LG
        if mode == "hybrid":
            hot = unit_work_est > self.hot_paths
            # fewer passes on the larger table (never more than the unit has tiles)
            grow = 1 << max(0, self.cta_cells_lg - self.cells_lg)
            np_hot = torch.clamp((self.unit_npass.long() + grow - 1) // grow, min=1)
            self.unit_npass = torch.where(hot, np_hot, self.unit_npass.long()).to(i32).contiguous()
            uo = self.unit_order.long()
            self.hot_order = self.unit_order[hot[uo]].contiguous()
            self.cold_order = self.unit_order[~hot[uo]].contiguous()
        elif mode == "cta":
            self.hot_order, self.cold_order = self.unit_order, self.unit_order[:0]
        else:
            self.hot_order, self.cold_order = self.unit_order[:0], self.unit_order

    # ------------------------------------------------------------------
    def _args(self, keep):
        p = self.plan
        a = N.XsimArgs()

        def P(t):
            t = t.contiguous()
            keep.append(t)
            return N.ptr(t)
        a.n_starts = int(p.start_item.numel())
        a.unit_leg_lo, a.unit_leg_hi = P(self.unit_leg_lo), P(self.unit_leg_hi)
        a.unit_g0, a.unit_g1, a.unit_npass = P(self.unit_g0), P(self.unit_g1), P(self.unit_npass)
        a.start_unit_ptr = P(self.start_unit_ptr)
        a.lp_ptr = P(self.lp_ptr)
        a.pd_s, a.pd_n, a.pd_d, a.pd_c = P(self.pd_s), P(self.pd_n), P(self.pd_d), P(self.pd_c)
        a.rs_ptr, a.rs_end = P(self.rs_ptr), P(self.rs_end)
        a.rs_n, a.rs_d, a.rs_c = [P(v) for v in self.rs_ndc]
        a.tile_ptr, a.gb = P(self.tile_ptr), self.gb
        a.cells_lg, a.top_m, a.warps = self.cells_lg, self.top_m, self.warps
        a.unit_counter = N.ptr(self.unit_counter)
        a.unit_clg, a.gws, a.gcells_lg = P(self.unit_clg), N.ptr(self.gws), self.gcells_lg
        a.error_flag = N.ptr(self.error_flag)
        return a

    def _launch_units(self, a, rank, world, st):
        """This rank's units: the hot ones first (CTA kernel: they are the long poles), then the rest (warp kernel).
        Every world-th unit of either descending-work order."""
        L = N.lib()
        hot = self.hot_order if world == 1 else self.hot_order[rank::world].contiguous()
        cold = self.cold_order if world == 1 else self.cold_order[rank::world].contiguous()
        self._orders = (hot, cold)                         # keep the device arrays alive until the kernels ran
        side = None
        if hot.numel() and cold.numel() and self.device.type == "cuda":
            # the two kernels run side by side: the hot CTAs are dispatched first, the persistent CTAs of the warp
            # kernel take the SMs over as the hot ones drain
            if getattr(self, "_side", None) is None:
                self._side = torch.cuda.Stream(device=self.device)
            side = self._side
            side.wait_stream(torch.cuda.current_stream(self.device))
        if hot.numel():
            clg = a.cells_lg
            a.cells_lg = self.cta_cells_lg if self.mode == "hybrid" else self.cells_lg
            a.unit_order, a.n_units = N.ptr(hot), int(hot.numel())
            N.check(L.xmap_xsim_extend_cta(a, side.cuda_stream if side is not None else st), "xmap_xsim_extend_cta")
            a.cells_lg = clg
            self.launches += 1
        if cold.numel():
            a.unit_order, a.n_units = N.ptr(cold), int(cold.numel())
            N.check(L.xmap_xsim_extend(a, st), "xmap_xsim_extend")
            self.launches += 1
        if side is not None:
            torch.cuda.current_stream(self.device).wait_stream(side)

    def _check(self):
        e = int(self.error_flag.item())
        if e:
            self.error_flag.zero_()
            raise N.NativeError("X-SIM kernel error %d (2: a pass overflows its table even at one hash tile)" % e)

    def run(self, rank=0, world=1, group=None):
        """count + top-m for every start of the plan.  world > 1: this rank runs every world-th unit of the
        descending-work order, the unit results are summed across ranks (each is non-zero on one rank) and
        every rank merges them, so all ranks return the full, identical result."""
        L = N.lib()
        p, dev, n, nu, m = self.plan, self.device, int(self.plan.start_item.numel()), self.n_units, self.top_m
        keep = []
        a = self._args(keep)
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        ucount, ucombos = z(nu, torch.int32), z(nu, torch.int64)
        ute, utx, utl = z((nu, m), torch.int32), z((nu, m), torch.float64), z(nu, torch.int32)
        cnt, comb = z(n, torch.int32), z(n, torch.int64)
        te = torch.full((n, m), -1, dtype=torch.int32, device=dev)
        tx, tl = z((n, m), torch.float64), z(n, torch.int32)
        a.unit_count, a.unit_combos = N.ptr(ucount), N.ptr(ucombos)
        a.unit_top_end, a.unit_top_xsim, a.unit_top_len = N.ptr(ute), N.ptr(utx), N.ptr(utl)
        a.out_count, a.out_combos = N.ptr(cnt), N.ptr(comb)
        a.top_end, a.top_xsim, a.top_len = N.ptr(te), N.ptr(tx), N.ptr(tl)
        st = torch.cuda.current_stream().cuda_stream
        if n and nu:
            self._launch_units(a, rank, world, st)
            if world > 1:
                from .multi import sum_unit_results
                sum_unit_results((ucount, ucombos, ute, utx, utl), group)
            N.check(L.xmap_xsim_merge(a, st), "xmap_xsim_merge")
            self.launches += 1
        self._check()
        return XsimResult(p.start_item, cnt, comb, te, tx, tl, self.launches, ucount)

    def emit(self, res):
        """Every (start, end, xsim), sorted by (start, end): the materialised return
        value of extender_pipeline (assist.py:80-102)."""
        L = N.lib()
        p, dev, nu = self.plan, self.device, self.n_units
        ptr = torch.zeros(nu + 1, dtype=torch.int64, device=dev)
        ptr[1:] = torch.cumsum(res.unit_count.long(), 0)
        total = int(ptr[-1].item()) if nu else 0
        e_end = torch.empty(total, dtype=torch.int32, device=dev)
        e_x = torch.empty(total, dtype=torch.float64, device=dev)
        if total:
            keep = []
            a = self._args(keep)
            m = self.top_m
            z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
            scratch = [z(nu, torch.int32), z(nu, torch.int64), z((nu, m), torch.int32), z((nu, m), torch.float64),
                       z(nu, torch.int32)]
            a.unit_count, a.unit_combos, a.unit_top_end, a.unit_top_xsim, a.unit_top_len = [N.ptr(t) for t in scratch]
            a.emit_ptr, a.emit_end, a.emit_xsim = N.ptr(ptr), N.ptr(e_end), N.ptr(e_x)
            self._launch_units(a, 0, 1, torch.cuda.current_stream().cuda_stream)
            self._check()
            if not torch.equal(scratch[0], res.unit_count):
                raise N.NativeError("X-SIM emit pass disagrees with the counting pass")
        start = torch.repeat_interleave(p.start_item.long()[self.unit_start], res.unit_count.long())
        o = torch.argsort(start * p.n_items + e_end.long())
        return start[o], e_end[o].long(), e_x[o]
