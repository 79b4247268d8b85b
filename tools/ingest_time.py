"""Rating text files -> training set on the device (ingest.clean_split_pipeline), timed, against the host path.

  python tools/ingest_time.py [out_dir]       (the JSON line goes to stdout, and to out_dir/ingest_time.json if given)

Writes cfg2_small- and cfg2-shaped rating files (bench.py WORKLOADS, synth.make_ratings; 33-byte lines
`u%08d <tab> xx%07d <tab> r <tab> ts`) into a temporary directory and reports, per shape, in one JSON line:
  host_read_h2d_ms   reading both files into pinned memory + the copy to the device (synchronised)
  ingest_ms          ingest_arrays wall time (file read included), median of 3 after a warm-up
  phase_ms           CUDA-event time of every phase of one ingest (summed over the two files where there are two)
  byte_pass_GBps     (file bytes read + masks written and read + offsets written) / (line_masks + line_offsets)
  byte_pass_hbm      that rate over 7.7 TB/s (HGX B200 data sheet)
  e2e_ms             text -> AlterEgo arrays: ingest + similarity + X-SIM + mapping + generation, synchronised
and, at cfg2_small, the host path: baseliner_clean_data_pipeline x2 + baseliner_split_data_pipeline + encode_records.
The GPU name and power limit are read in the same run.
"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12
SHAPES = {"cfg2_small": (100_000, 20_000, 2_000_000, 0.05), "cfg2": (1_000_000, 200_000, 20_000_000, 0.05)}


def write_files(sr, tmp, tag):
    """Fixed-width lines built with numpy (what synth.to_text_lines writes, at 18 M lines)."""
    import numpy as np
    from xmap_b200 import synth
    paths = []
    for d in range(2):
        m = sr.domain == d
        u, i, r, t = sr.user[m], sr.item[m] % sr.n_items_per_domain, sr.rating[m], sr.ts[m]
        n = len(u)
        a = np.empty((n, 33), dtype=np.uint8)

        def digits(col, v, w):
            v = v.astype(np.int64).copy()
            for k in range(w - 1, -1, -1):
                a[:, col + k] = 48 + v % 10
                v //= 10
        a[:, 0] = ord("u")
        digits(1, u, 8)
        a[:, 9] = 9
        a[:, 10:12] = np.frombuffer(synth.PREFIXES[d].encode(), dtype=np.uint8)
        digits(12, i, 7)
        a[:, 19] = 9
        digits(20, r, 1)
        a[:, 21] = 9
        digits(22, t, 10)
        a[:, 32] = 10
        p = os.path.join(tmp, "%s_%d.txt" % (tag, d))
        a.tofile(p)
        paths.append(p)
    return paths


def tools():
    from xmap_b200.core import BaselinerClean, BaselinerSplit
    return (BaselinerClean(10, 10 ** 9, 2012, 2013, "S:"), BaselinerClean(10, 10 ** 9, 2012, 2013, "T:"),
            BaselinerSplit(0, 0.2, 0.8, 666666))


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def measure(paths):
    import numpy as np
    import torch
    from xmap_b200 import ingest, generate as G
    from xmap_b200.core import (BaselinerSim, ExtendSim, Generator, baseliner_calculate_sim_pipeline,
                                extender_pipeline)
    from xmap_b200.session import session_of
    dev = torch.device("cuda")
    res = {"bytes": int(sum(os.path.getsize(p) for p in paths))}

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for p in paths:
        h = torch.empty(os.path.getsize(p), dtype=torch.uint8, pin_memory=True)
        with open(p, "rb") as f:
            f.readinto(memoryview(h.numpy()))
        d = h.to(dev, non_blocking=True)
    torch.cuda.synchronize()
    res["host_read_h2d_ms"] = (time.perf_counter() - t0) * 1e3
    del h, d

    walls = []
    for rep in range(4):
        cs, ct, sp = tools()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        A = ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False)
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
        del A
    res["ingest_ms"] = float(np.median(walls[1:]))
    res["ingest_ms_runs"] = [round(w, 2) for w in walls]

    ev = {}
    cs, ct, sp = tools()
    A = ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False, events=ev)
    torch.cuda.synchronize()
    res["phase_ms"] = {k: round(sum(a.elapsed_time(b) for a, b in v), 3) for k, v in ev.items()}
    res["train_records"], res["test_records"] = int(A.user.numel()), int(A.test_user.numel())
    res["train_users"], res["train_items"] = len(A.uids), len(A.iids)
    lines = res["bytes"] // 33
    moved = res["bytes"] + 2 * res["bytes"] / 8 + 8 * lines
    t_pass = (res["phase_ms"].get("line_masks", 0) + res["phase_ms"].get("line_offsets", 0)) / 1e3
    res["byte_pass_GBps"] = round(moved / t_pass / 1e9, 1) if t_pass else None
    res["byte_pass_hbm"] = round(moved / t_pass / HBM_BPS, 3) if t_pass else None
    del A

    def e2e():
        cs, ct, sp = tools()
        tr, _ = ingest.clean_split_pipeline(None, cs, ct, sp, paths[0], paths[1], False)
        sim_tool = BaselinerSim("adjust_cosine", 50)
        simRDD = baseliner_calculate_sim_pipeline(None, sim_tool, tr)
        xs = extender_pipeline(None, None, sim_tool, ExtendSim(10), simRDD)
        sess = session_of(tr)
        gen = Generator(1, 0.6, "adjust_cosine", 0.1)
        xres, chosen = gen._map(xs, sess, gen.private_mode)
        mapping = G.invert_mapping(xres.start_item, chosen, sess.enc.n_items)
        out = G.build_alterego(sess.layout, np.arange(sess.layout.nnz, dtype=np.int64), mapping)
        torch.cuda.synchronize()
        return int(out[0].numel())
    e2e()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res["alterego_records"] = e2e()
    res["e2e_ms"] = (time.perf_counter() - t0) * 1e3
    return res


def host_path(paths):
    from xmap_b200.core import baseliner_clean_data_pipeline, baseliner_split_data_pipeline
    from xmap_b200.encode import encode_records
    cs, ct, sp = tools()
    T = {}
    t0 = time.perf_counter()
    s = baseliner_clean_data_pipeline(None, cs, paths[0], False, 30)
    T["clean_source_ms"] = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    t = baseliner_clean_data_pipeline(None, ct, paths[1], False, 30)
    T["clean_target_ms"] = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    tr, _ = baseliner_split_data_pipeline(None, sp, s, t)
    T["split_ms"] = (time.perf_counter() - t0) * 1e3
    recs = tr.collect()
    t0 = time.perf_counter()
    encode_records(recs)
    T["encode_records_ms"] = (time.perf_counter() - t0) * 1e3
    T["total_ms"] = sum(T.values())
    return T


def main():
    from xmap_b200 import synth
    out_dir = sys.argv[1] if len(sys.argv) > 1 else None
    os.environ["TZ"] = "UTC"
    time.tzset()
    line = dict(tool="ingest_time", **gpu_info())
    with tempfile.TemporaryDirectory() as tmp:
        for name in ("cfg2_small", "cfg2"):
            nu, ni, nd, ov = SHAPES[name]
            paths = write_files(synth.make_ratings(nu, ni, nd, overlap=ov), tmp, name)
            line[name] = measure(paths)
            if name == "cfg2_small":
                line[name]["host_path_ms"] = host_path(paths)
            for p in paths:
                os.remove(p)
    s = json.dumps(line)
    print(s)
    if out_dir is not None:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "ingest_time.json"), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
