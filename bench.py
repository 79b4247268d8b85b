#!/usr/bin/env python
"""Benchmark of the AlterEgo-construction hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|...] [--dump-outputs DIR]

--dump-outputs DIR (--impl ours only: the reference arm times a CPU port on samples and returns no tables) writes
what the last timed step returned, the neighbour tables of engine.SimTables, as DIR/<name>.npy.

A "step" is one pass of the similarity stage (all item rows: co-rating SpGEMM +
epilogue + top-k selection, passes 1 and 2) over the synthetic two-domain
workload; `value` = directed co-rated item pairs evaluated per second with the
ratings layout already resident in HBM.  `e2e` is the same metric through the
host-facing call: pinned host triples -> H2D -> layout build -> similarity ->
D2H of the neighbour tables, all inside the timed region.  The line also
carries the pipeline wall-time (similarity + X-SIM extension + generation), the
roofline of the dominant kernel and a CPU baseline (the oracle port, timed on a
bounded sample on this box's host cores).

Under torchrun (N > 1) every rank holds the replicated layout, owns a
work-balanced block of item rows, and the ranks exchange BB flags and neighbour
tables with NCCL all-gathers; timing is max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (users, items/domain, draws, domains, overlap, k)
    "cfg2": (1_000_000, 200_000, 20_000_000, 2, 0.05, 10),         # BASELINE.json configs[1]
    "cfg4": (2_000_000, 250_000, 80_000_000, 4, 0.05, 10),         # configs[3]: one source->target pipeline per source domain
    "cfg4_small": (200_000, 25_000, 8_000_000, 4, 0.05, 10),
    "cfg2_small": (100_000, 20_000, 2_000_000, 2, 0.05, 10),
    "tiny": (20_000, 3_000, 400_000, 2, 0.05, 10),
}
METRIC = "item_pair_sims_per_sec"
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
# (profiles/), keyed by kernel group; None until captured.
NCU_TRAFFIC = {"tri_cta_kernel": 7.229e9 / 14,   # dram__bytes_read + dram__bytes_write summed over the 14 launches of one stage,
               "xsim_warp_kernel": 3.688e11}     # ... and of the one X-SIM launch: profiles/r2_ncu_full_cfg2.csv; per launch like
                                                 # `achieved` (cfg2, one GPU)


def _compact(name, sr, keep, k, tag):
    """One two-domain problem cut from the rating set: users / items renumbered in sorted-id order."""
    from xmap_b200 import synth
    from xmap_b200.encode import item_codes
    user, item, rating, ts = (sr.user, sr.item, sr.rating, sr.ts) if keep is None else \
        (sr.user[keep], sr.item[keep], sr.rating[keep], sr.ts[keep])
    present = np.unique(item)
    iids = np.array([synth.item_id(int(g), sr.n_items_per_domain, sr.labels) for g in present])
    order = np.argsort(iids)
    present, iids = present[order], iids[order]
    imap = np.full(int(item.max()) + 1, -1, dtype=np.int64)
    imap[present] = np.arange(len(present))
    uu = np.unique(user)
    umap = np.full(int(user.max()) + 1, -1, dtype=np.int64)
    umap[uu] = np.arange(len(uu))
    pc, dc, ct, hs, ht = item_codes(iids)
    du = np.bincount(umap[user]).astype(np.int64)
    return dict(name=name + tag, user=umap[user].astype(np.int32), item=imap[item].astype(np.int32),
                rating=rating.astype(np.float32), ts=ts, n_users=len(uu), n_items=len(iids), k=k,
                meta=dict(prefix_code=pc, dom_code=dc, contains=ct, has_S=hs, has_T=ht),
                nnz=int(len(user)), W=int((du * (du - 1)).sum()))


def _generate_pipelines(name):
    from xmap_b200 import synth
    nu, ni, nd, ndom, ov, k = WORKLOADS[name]
    sr = synth.make_ratings(nu, ni, nd, n_domains=ndom, overlap=ov)
    if ndom == 2:
        return [_compact(name, sr, None, k, "")]
    tgt = ndom - 1
    return [_compact(name, sr, (sr.domain == d) | (sr.domain == tgt), k, "[%s->T:]" % sr.labels[d]) for d in range(tgt)]


def make_pipelines(name):
    """The two-domain problems of a workload: one for a two-domain shape; for a multi-domain shape one
    source -> target problem per source domain, cut from ONE rating set, exactly as multidomain_demo.py:101-128
    runs them (independent pipelines whose AlterEgo records are unioned).
    Under torchrun the ranks of a node share one generation: local rank 0 writes the arrays to /dev/shm, the others
    read them (the generator is deterministic; this only avoids N processes competing for the host cores)."""
    world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world <= 1 or not os.path.isdir("/dev/shm"):
        return _generate_pipelines(name)
    import pickle
    tag = "%s_%s_%s" % (name, "_".join(str(x) for x in WORKLOADS[name]), os.environ.get("MASTER_PORT", "0"))
    path = "/dev/shm/xmap_b200_%s.pkl" % tag
    if local == 0:
        pipes = _generate_pipelines(name)
        with open(path + ".tmp", "wb") as f:
            pickle.dump(pipes, f, protocol=4)
        os.replace(path + ".tmp", path)
        return pipes
    t0 = time.time()
    while not os.path.exists(path):
        if time.time() - t0 > 1800:
            raise RuntimeError("timed out waiting for %s" % path)
        time.sleep(0.5)
    with open(path, "rb") as f:
        return pickle.load(f)


def make_workload(name):
    """First (for a two-domain shape: the only) pipeline of a workload."""
    return make_pipelines(name)[0]


DUMP_BUDGET = 48 << 20       # bytes --dump-outputs may write (the tables of a large workload: a fixed sample of rows)
DUMP_FIELDS = (("row_flags", np.float32), ("row_npairs", np.float64), ("row_nkept", np.float64), ("tab_len", np.float32),
               ("tab_idx", np.float32), ("tab_sim", np.float64), ("tab_mutu", np.float32), ("tab_n", np.float32))


def dump_rows(pipes, k):
    """Item rows whose tables --dump-outputs writes, per pipeline: all of them if they fit DUMP_BUDGET, else a fixed,
    seeded sample (the same rows in every run with the same arguments), sorted."""
    n_rows = DUMP_BUDGET // (len(pipes) * (36 + 40 * k))        # bytes per row of the files DUMP_FIELDS make
    return [np.arange(wl["n_items"]) if wl["n_items"] <= n_rows else
            np.sort(np.random.default_rng(0).choice(wl["n_items"], n_rows, replace=False)) for wl in pipes]


def snapshot_tables(tabs_all, rows_all):
    """Host copy of what a caller of the similarity step receives (engine.SimTables), on the dumped rows: ids and
    counts of items and users as float32 (exact below 2^24), pair counts and similarities as float64."""
    import torch
    out = {}
    for q, (tabs, rows) in enumerate(zip(tabs_all, rows_all)):
        pre = "" if len(tabs_all) == 1 else "pipeline%d_" % q
        r = torch.as_tensor(rows, device=tabs.tab_sim.device)
        out[pre + "rows"] = rows.astype(np.float64)
        out[pre + "n_pairs_total"] = np.array([tabs.n_pairs_total], dtype=np.float64)
        for name, dt in DUMP_FIELDS:
            a = getattr(tabs, name).index_select(0, r).cpu().numpy()
            assert dt != np.float32 or a.size == 0 or np.abs(a).max() < 1 << 24, name
            out[pre + name] = a.astype(dt)
    return out


def workload_label(wl, method):
    return "%s: %d users, %d items, %d ratings (Zipf), W=%d products, top-k=%d, %s" % (
        wl["name"], wl["n_users"], wl["n_items"], wl["nnz"], wl["W"], wl["k"], method)


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML; nvidia-smi as a fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.sm_max, self.stop_flag = index, [], set(), None, False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _nvml_sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
                          ("sw_power_cap", 0x4)):
            if r & bit:
                self.reasons.add(name)

    def _smi_sample(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        self.sm.append(float(f[0])); self.sm_max = float(f[1])
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            try:
                self._nvml_sample() if self.nvml else self._smi_sample()
            except Exception:
                pass
            time.sleep(0.005 if self.nvml else 0.1)

    def summary(self):
        self.stop_flag = True
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self.nvml else "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------
# CPU baseline: the oracle port on a bounded sample of the same workload
# --------------------------------------------------------------------------
def _cpu_block(args):
    from oracle import restate as RS
    user, item, rating, nU, nI, pc, method, na = args
    t0 = time.perf_counter()
    P = RS.sim_pairs(user, item, rating, nU, nI, pc, method, na)
    return P["n_pairs_total"], len(P["i"]), time.perf_counter() - t0


def _sample(wl, phase, stride):
    """Every `stride`-th user starting at `phase` (a uniform sample of light and heavy users),
    with users and items renumbered densely."""
    m = (wl["user"] % stride) == phase
    user, item = wl["user"][m].astype(np.int64) // stride, wl["item"][m].astype(np.int64)
    n_u = int(user.max()) + 1 if len(user) else 1
    present = np.unique(item)
    imap = np.full(wl["n_items"], -1, dtype=np.int64); imap[present] = np.arange(len(present))
    return (user, imap[item], wl["rating"][m].astype(np.float64), n_u, len(present),
            wl["meta"]["prefix_code"][present]), int(m.sum())


def cpu_baseline(wl, method="adjust_cosine", num_atleast=50, target_ratings=250_000, cores=1):
    """oracle/restate.py (numpy/scipy restatement of baselinerSim.py:17-216) on a bounded sample of
    the workload: `cores` disjoint strided user samples of ~target_ratings ratings each, one process
    per sample (the reference's per-task arithmetic is single-threaded)."""
    stride = max(cores, int(round(wl["nnz"] / max(1, target_ratings))))
    jobs, nr = [], 0
    for c in range(cores):
        args, r = _sample(wl, c, stride)
        jobs.append(args + (method, num_atleast)); nr += r
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_block(jobs[0])]
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_cpu_block, jobs)
    dt = time.perf_counter() - t0
    n_pairs = sum(r[0] for r in res)
    out = {"value": n_pairs / dt, "unit": "item pairs/s", "cores": cores, "kind": "port",
           "sample": "%d sample(s), every %d-th user of %s (%d ratings, %d co-rated pairs, %.1f s wall): "
                     "oracle/restate.py, the numpy/scipy restatement of the reference arithmetic "
                     "(no Spark/JVM/shuffle serialisation)" % (cores, stride, wl["name"], nr, n_pairs, dt)}
    # the reference's OWN Python on the same kind of sample cannot be timed here (/root/reference does not travel to
    # the GPU box): quote the measurement taken in the build container (tools/ref_shim_time.py), labelled as such
    p = os.path.join(ROOT, "profiles", "r2_reference_own_python_sample.json")
    if os.path.isfile(p):
        try:
            r = json.load(open(p))
            out["reference_own_python"] = {"value": r["pairs_per_s"], "unit": "item pairs/s", "cores": r["cores"],
                                           "sample": r["sample"], "seconds": r["seconds"], "what": r["what"],
                                           "measured": "build container, not this box"}
        except Exception:
            pass
    return out


def run_reference_arm(args, emit):
    """--impl reference: the reference's CPU arithmetic for the path on this box's host cores.
    /root/reference (pure Python on Spark) does not travel to the GPU box and Spark is absent,
    so the oracle port (oracle/restate.py) is what is timed, on a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = make_workload(args.workload)
    vals, secs = [], []
    cores = min(os.cpu_count() or 1, 16)           # fixed ceiling: the denominator must not move with the box size
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        cb = cpu_baseline(wl, method=args.method, target_ratings=150_000, cores=cores)
        if s >= args.warmup:
            vals.append(cb["value"]); secs.append(time.perf_counter() - t0)
    v = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "item pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_label(wl, args.method), "note": "each step = one bounded sample (see cpu_baseline.sample); "
                       "Spark is not installed on this image, /root/reference (pure Python on Spark RDDs) does "
                       "not travel to the GPU box, so the timed code is the oracle port of its arithmetic"},
            "cpu_baseline": dict(cb, value=v),
            "e2e": {"value": v, "unit": "item pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--method", default="adjust_cosine")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the extension/generation timing")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the neighbour tables of the last timed step to DIR/<name>.npy (float32 / float64; "
                         "a fixed sample of item rows when they exceed %d MB)" % (DUMP_BUDGET >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the tables of the GPU path (--impl ours)")
    # exactly one JSON line may reach stdout: libraries (NCCL's version banner) write there too, so
    # stdout is pointed at stderr for the duration of the run and restored for the final print
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference_arm(args, emit)

    import torch
    import torch.distributed as dist
    from xmap_b200 import engine as E
    from xmap_b200 import extend as X
    from xmap_b200 import generate as G
    from xmap_b200 import multi as MG
    from xmap_b200.engine import to_device_meta

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    pipes = make_pipelines(args.workload)
    k = pipes[0]["k"]
    pin = lambda a: torch.from_numpy(a).pin_memory()
    for wl in pipes:
        wl["dmeta"] = to_device_meta(wl["meta"], dev)
        wl["h"] = (pin(wl["user"]), pin(wl["item"]), pin(wl["rating"]))
    h2d_bytes = sum(wl["h"][0].numel() * 4 * 3 for wl in pipes)
    W_total, nnz_total, I_total = (sum(wl[q] for wl in pipes) for q in ("W", "nnz", "n_items"))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # resident layouts + engines for the device-timed metric (one per source -> target pipeline); the record lists of
    # several engines must fit together, so each gets an equal share of the free memory (else: exact sizing pass)
    free_b, _ = torch.cuda.mem_get_info(dev)
    budget = None if len(pipes) == 1 else int(free_b * 0.6 / len(pipes))
    for wl in pipes:
        wl["lay"] = E.build_layout(*wl["h"], wl["n_users"], wl["n_items"], device=dev)
        wl["ts_dev"] = torch.as_tensor(wl["ts"], dtype=torch.int64).to(dev)       # rating times, resident like the layout
        wl["eng"] = E.SimEngine(wl["lay"], wl["dmeta"], args.method, 50, k, rec_budget=budget)
        wl["shard"] = MG.similarity_shard(wl["eng"], rank, world)

    def sim_step():
        return [MG.similarity_step(wl["eng"], wl["shard"]) for wl in pipes]

    for _ in range(args.warmup):
        sim_step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    l0 = sum(wl["eng"].launches for wl in pipes)
    barrier()
    for s in range(args.steps):
        ev[s][0].record()
        tabs_all = sim_step()
        ev[s][1].record()
    barrier()
    clocks = sampler.summary()
    for wl in pipes:
        wl["eng"]._check_error()
    launches = sum(wl["eng"].launches for wl in pipes) - l0
    # the tables live in engine buffers that the next steps overwrite: copy what the last timed step computed now
    dumped = snapshot_tables(tabs_all, dump_rows(pipes, k)) if args.dump_outputs and rank == 0 else None
    # per-kernel CUDA-event times: a second set of steps with every launch serialised on one stream
    for wl in pipes:
        wl["eng"].enable_profile()
    for s in range(args.steps):
        sim_step()
    prof = {}
    for wl in pipes:
        for kk, (n, ms_k) in wl["eng"].profile_ms().items():
            prof[kk] = (prof.get(kk, (0, 0.0))[0] + n, prof.get(kk, (0, 0.0))[1] + ms_k)
        wl["eng"].profile = None
    barrier()
    ms = torch.tensor([a.elapsed_time(b) for a, b in ev], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms.mean())
    P_total = sum(t.n_pairs_total for t in tabs_all)
    P_kept = sum(int(t.row_nkept.sum().item()) for t in tabs_all)
    value = P_total / (ms_step * 1e-3)

    # multi-GPU parity, carried in the line: rank 0 runs the single-GPU stage (untimed) on the first pipeline and
    # compares every table, later the X-SIM top-m and the item map, bit for bit
    multi_parity, ref_tabs = None, None
    if world > 1:
        ok = True
        if rank == 0:
            wl = pipes[0]
            ref_eng = E.SimEngine(wl["lay"], wl["dmeta"], args.method, 50, k, rec_budget=budget)
            ref_tabs = ref_eng.run()
            ok = all(torch.equal(getattr(ref_tabs, f), getattr(tabs_all[0], f)) for f in
                     ("row_flags", "row_npairs", "row_nkept", "tab_len", "tab_idx", "tab_sim", "tab_mutu", "tab_n"))
            ref_eng._give_back()
            del ref_eng
        multi_parity = {"similarity_tables": bool(ok)}
        barrier()

    # e2e: host triples -> layout -> similarity -> neighbour tables back on the host
    def e2e_step():
        nb = 0
        for wl in pipes:
            lay2 = E.build_layout(*wl["h"], wl["n_users"], wl["n_items"], device=dev)
            eng2 = E.SimEngine(lay2, wl["dmeta"], args.method, 50, k, rec_budget=budget)
            t = MG.similarity_step(eng2, MG.similarity_shard(eng2, rank, world))
            out = eng2.tables_to_host(t, reuse=True)     # pinned host buffers, synchronises
            nb += sum(o.numel() * o.element_size() for o in out.values())
            eng2._give_back()
        return nb
    e2e_step()
    n_e2e = max(3, min(args.steps, 7))
    e2e_times = []
    for _ in range(n_e2e):
        barrier()
        t0 = time.perf_counter()
        d2h_bytes = e2e_step()
        barrier()
        e2e_times.append(time.perf_counter() - t0)
    # median of the per-step wall-clock times (the host is shared: a single descheduling would skew a mean)
    e2e_s = torch.tensor([float(np.median(e2e_times))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_val = P_total / float(e2e_s)

    # pipeline wall-time: similarity + X-SIM extension (sharded by work unit) + generation (sharded by user), per
    # source -> target pipeline, summed
    pipe = None
    for timed in ((False, True, True) if not args.no_pipeline else ()):  # one untimed pass, then the faster of two
        acc = dict(plan=0.0, xsim=0.0, xsim_kernel=0.0, gen=0.0, combos=0, starts=0, pairs=0, recs=0, src=0, joint=0, units=0, hot=0)
        for q, wl in enumerate(pipes):
            lay, meta, tabs = wl["lay"], wl["dmeta"], tabs_all[q]
            barrier()
            t0 = time.perf_counter()
            plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
            torch.cuda.synchronize(); t1 = time.perf_counter()
            xe = X.XsimEngine(plan, 10)
            torch.cuda.synchronize(); t1b = time.perf_counter()
            res = xe.run(rank, world)
            barrier(); t2 = time.perf_counter()
            ch = G.choose_mapping(res, "argmax", sim_method=args.method)
            mp = G.invert_mapping(res.start_item, ch, wl["n_items"])
            ou, oi, orr, ot = MG.build_alterego_sharded(lay, wl["ts_dev"], mp, MG.UserShard(lay.csr_ptr, rank, world))
            n_rec = torch.tensor([ou.numel()], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(n_rec)
            barrier(); t3 = time.perf_counter()
            acc["plan"] += t1 - t0; acc["xsim"] += t2 - t1; acc["xsim_kernel"] += t2 - t1b; acc["gen"] += t3 - t2
            acc["combos"] += int(res.combos.sum().item()); acc["starts"] += int(res.start_item.numel())
            acc["pairs"] += int(res.count.sum().item()); acc["recs"] += int(n_rec.item())
            acc["src"] += plan.n_src; acc["joint"] += plan.n_joint; acc["units"] += xe.n_units; acc["hot"] += int(xe.hot_order.numel())
            if world > 1 and q == 0 and multi_parity is not None and "xsim_top_m" not in multi_parity:
                ok = True
                if rank == 0:
                    plan1 = X.build_plan(ref_tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
                    res1 = X.XsimEngine(plan1, 10).run()
                    ok = all(torch.equal(getattr(res1, f), getattr(res, f)) for f in
                             ("count", "combos", "top_end", "top_xsim", "top_len"))
                    mp1 = G.invert_mapping(res1.start_item, G.choose_mapping(res1, "argmax", sim_method=args.method), wl["n_items"])
                    multi_parity["item_map"] = bool(torch.equal(mp1, mp))
                    del plan1, res1
                multi_parity["xsim_top_m"] = bool(ok)
                barrier()
            del plan, xe, res
        total_ms = ms_step + (acc["plan"] + acc["xsim"] + acc["gen"]) * 1e3
        if not timed or (pipe is not None and pipe["alterego_pipeline_ms"] <= total_ms):
            continue
        pipe = {"similarity_ms": ms_step, "extend_plan_ms": acc["plan"] * 1e3, "extend_kernel_ms": acc["xsim"] * 1e3,
                "extend_engine_build_ms": (acc["xsim"] - acc["xsim_kernel"]) * 1e3, "xsim_kernels_ms": acc["xsim_kernel"] * 1e3,
                "generate_ms": acc["gen"] * 1e3, "alterego_pipeline_ms": total_ms,
                "xsim_paths": acc["combos"], "xsim_paths_per_s": acc["combos"] / max(acc["xsim_kernel"], 1e-9),
                "xsim_starts": acc["starts"], "xsim_pairs": acc["pairs"], "xsim_units": acc["units"],
                "xsim_hot_units": acc["hot"],
                "alterego_synthetic_records": acc["recs"], "bridge_pairs": acc["src"], "joint_pairs": acc["joint"],
                "pipelines": len(pipes),
                "sharding": "X-SIM by work unit x%d, generation by user x%d (host wall-clock of rank 0 between barriers, "
                            "faster of two passes after one untimed pass)" % (world, world)}
    if multi_parity is not None:
        flag = torch.tensor([1 if all(multi_parity.values()) else 0], device=dev)
        dist.broadcast(flag, 0)
        multi_parity["all"] = bool(flag.item())

    if rank == 0:
        peaks, peak_src = measured_peaks()
        # the stage evaluates every unordered pair once: W/2 products of 8 B, one pass over the CSC
        # (24 B per rating: entry + suffix extent + rater mean), 2 x 20 B records written and read back per kept pair,
        # and the tables out
        alg_bytes = 8.0 * (W_total / 2) + 24.0 * nnz_total + 40.0 * P_kept + 80.0 * k * I_total
        stage_gbs = alg_bytes / (ms_step * 1e-3) / 1e9
        # kernels: the accumulate launches are one kernel function per group width
        fam_ms, fam_n, fam_bytes = {}, {}, {}
        for kk, (n, ms_k) in prof.items():
            if kk.startswith("accumulate_c") or kk.startswith("accumulate_g"):
                fam = "tri_warp_kernel" if kk.endswith("_t32") else ("tri_gmem_kernel" if "_g" in kk else "tri_cta_kernel")
            elif kk == "accumulate_split":
                fam = "tri_split_kernel"
            elif kk == "select_warp":
                fam = "select_warp_kernel"
            elif kk == "select_cta":
                fam = "select_cta_kernel"
            else:
                fam = kk
            fam_ms[fam] = fam_ms.get(fam, 0.0) + ms_k
            fam_n[fam] = fam_n.get(fam, 0) + n
        for q, wl in enumerate(pipes):
            eng, tabs = wl["eng"], tabs_all[q]
            launches_plan, _, split_plan = eng.plan(None if world == 1 else wl["shard"].rows(dev))
            for r, cells_cap, threads, in_gmem, _hdr in launches_plan:
                fam = "tri_gmem_kernel" if in_gmem else ("tri_warp_kernel" if threads == 32 else "tri_cta_kernel")
                fam_bytes[fam] = fam_bytes.get(fam, 0.0) + 8.0 * float(eng.tri_work[r.long()].sum().item())
            if split_plan is not None:
                fam_bytes["tri_split_kernel"] = fam_bytes.get("tri_split_kernel", 0.0) + \
                    8.0 * float(eng.tri_work[split_plan["rows"].long()].sum().item())
            long_rows = tabs.row_nkept > 8192
            fam_bytes["select_cta_kernel"] = fam_bytes.get("select_cta_kernel", 0.0) + 16.0 * float(tabs.row_nkept[long_rows].sum().item())
            fam_bytes["select_warp_kernel"] = fam_bytes.get("select_warp_kernel", 0.0) + 16.0 * float(tabs.row_nkept[~long_rows].sum().item())
        kinds = {kk: (fam_n[kk], fam_ms[kk]) for kk in fam_ms}
        dom = max((kk for kk in kinds if kk in fam_bytes), key=lambda kk: kinds[kk][1])
        dom_bytes_step = fam_bytes.get(dom, 0.0)
        dom_ms_step = kinds[dom][1] / args.steps
        achieved = dom_bytes_step / (dom_ms_step * 1e-3) / 1e9 if dom_ms_step > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": "item pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64 epilogue over i64 fixed-point accumulators", "data": "synthetic",
            "config": {"workload": " + ".join(workload_label(wl, args.method) for wl in pipes),
                       "pairs_evaluated": P_total, "pairs_kept": P_kept,
                       "l2_policy": "inputs (CSR+CSC+tables) larger than L2; no explicit flush",
                       "parallelism": "item row-blocks x%d, ratings replicated, neighbour records exchanged" % world},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "item pairs/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": float(e2e_s) * 1e3,
                    "steps": n_e2e, "statistic": "median of per-step host wall-clock, max over ranks"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC.get(dom),
                         "peak_source": peak_src, "algorithmic_bytes_per_step": dom_bytes_step,
                         "kernel_ms_per_step": dom_ms_step, "launches_per_step": kinds[dom][0] / args.steps,
                         "kernel_share_of_step": dom_ms_step / max(sum(v[1] for v in kinds.values()) / args.steps, 1e-9),
                         "per_kernel_ms_per_step": {kk: v[1] / args.steps for kk, v in kinds.items()},
                         "stage_algorithmic_gbs": stage_gbs, "stage_frac": stage_gbs / peaks["hbm_gbs"],
                         "per_launch_ms_per_step": {kk: v[1] / args.steps for kk, v in prof.items()},
                         "timing": "per-kernel times come from %d extra steps with every launch serialised on one stream "
                                   "(CUDA events around each launch); the timed steps overlap the small launches on a "
                                   "side stream" % args.steps,
                         "note": "achieved = algorithmic bytes of the kernel (8 B per co-rating product for the "
                                 "accumulate kernels, 16 B per neighbour record for the selection kernels) / its "
                                 "CUDA-event time; stage figure = (8*W/2 + 24*nnz + 40*P_kept + 80*k*I) / step time"},
            "pipeline": pipe,
        }
        if pipe is not None:
            # the X-SIM kernel is the other half of BASELINE.json's metric (pipeline wall-time): SURVEY.md 8(d) counts
            # 16 B of accumulator read-modify-write per path; here the accumulators never leave shared memory, so the
            # figure is an equivalent-traffic rate, next to the 28 B right-segment read each path really makes
            xk = pipe["xsim_kernels_ms"] * 1e-3
            gb16, gb28 = 16.0 * pipe["xsim_paths"] / xk / 1e9, 28.0 * pipe["xsim_paths"] / xk / 1e9
            xname = {"hybrid": "xsim_warp_kernel (+ xsim_cta_kernel for the hot units)", "warp": "xsim_warp_kernel",
                     "cta": "xsim_cta_kernel"}[X.XSIM_MODE]
            line["pipeline_roofline"] = {"kernel": xname, "bound": "hbm", "achieved": gb16, "peak": peaks["hbm_gbs"],
                                         "unit": "GB/s", "frac": gb16 / peaks["hbm_gbs"], "traffic": NCU_TRAFFIC.get(xname.split()[0]),
                                         "algorithmic_bytes_per_path": 16, "paths": pipe["xsim_paths"],
                                         "kernel_ms": pipe["xsim_kernels_ms"], "right_segment_read_gbs": gb28,
                                         "note": "host wall-clock around the kernel launches + merge (max over ranks via the barrier)"}
        if multi_parity is not None:
            line["multi_parity"] = multi_parity
        if not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(pipes[0], args.method)
        if dumped is not None:
            assert sum(a.nbytes for a in dumped.values()) <= 64 * 10 ** 6
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
