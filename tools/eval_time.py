"""Held-out evaluation (evaluate.evaluate) of the two-domain experiment at cfg2 scale, device-timed per stage.

  python tools/eval_time.py [workload=cfg2] [out_dir]

Writes the cfg2-shaped pair of rating files (ingest_time.SHAPES, ingest_time.write_files) into a temporary directory,
runs ingest_arrays once, then evaluate twice on the same arrays:
  NX-MAP  non-private generation (Generator.cross_nonprivate_mapping) and non-private neighbour selection;
  X-MAP   exponential-mechanism generation at eps = 0.6 and the private neighbour selection, both seeded.
One JSON line: per-stage device times (CUDA events) and the wall time of each run, the held-out pairs predicted and
skipped by kind, the evaluated users, MAE without and with decay, P/R/NDCG/MAP@10, catalogue coverage, and the GPU name
and power limit read in the same run.  With out_dir the line is also written to out_dir/eval_time_<workload>.json.

The synthetic ratings carry no signal (synth.make_ratings draws them independently of user and item), so the numbers
only show that the evaluation runs end to end at this scale; its parity with the facade chain is pinned by
tests/test_gpu_evaluate.py.
"""
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

N = 10
SEEDS = dict(generator=20261018, privacy=20261022)


def runs():
    """(label, tool factory, private_gen, private_rec): fresh, identically seeded tools per run."""
    from xmap_b200.core import BaselinerSim, ExtendSim, Generator, RecommenderSim, RecommenderPrivacy

    def make():
        return (BaselinerSim("adjust_cosine", 50), ExtendSim(10),
                Generator(1, 0.6, "adjust_cosine", 0.1, private_mode="exp_mech", seed=SEEDS["generator"]),
                RecommenderSim("cosine_item", 50), RecommenderPrivacy(10, 0.6, 0.1, seed=SEEDS["privacy"]))
    return [("nx_map", make, False, False), ("x_map", make, True, True)]


def summary(ev, wall_ms):
    m = ev.metrics
    r = lambda x: None if x is None else round(x, 6)
    return {"stage_ms": {k: round(v, 3) for k, v in ev.stage_ms.items()}, "wall_ms": round(wall_ms, 1),
            **ev.counts, "top_n_visits": ev.top.visits, "top_n_candidates": ev.top.candidates,
            "top_n_warp_users": ev.top.warp_users, "top_n_cta_users": ev.top.cta_users,
            "mae_nodecay": r(ev.mae_nodecay), "mae_decay": r(ev.mae_decay),
            **{"%s@%d" % (k, ev.n): r(v) for k, v in (m.mean or {}).items()}, "coverage@%d" % ev.n: r(m.coverage)}


def main():
    import torch
    from ingest_time import SHAPES, gpu_info, tools, write_files
    from xmap_b200 import evaluate, ingest, synth
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    out_dir = sys.argv[2] if len(sys.argv) > 2 else None
    os.environ["TZ"] = "UTC"
    time.tzset()
    nu, ni, nd, ov = SHAPES[name]
    with tempfile.TemporaryDirectory() as tmp:
        paths = write_files(synth.make_ratings(nu, ni, nd, overlap=ov), tmp, name)
        if not torch.cuda.is_available():
            raise SystemExit("eval_time: wrote %s (%d bytes); no CUDA device, and the evaluation runs on the GPU only"
                             % (paths, sum(os.path.getsize(p) for p in paths)))
        line = {"tool": "eval_time", "workload": "%s: %d users, %d items per domain, %d draws, overlap %g"
                % (name, nu, ni, nd, ov), **gpu_info(), "n": N, "seeds": SEEDS}
        ev = {}
        cs, ct, sp = tools()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        A = ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False, events=ev)
        torch.cuda.synchronize()
        line["ingest_wall_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        line["ingest_phase_ms"] = {k: round(sum(a.elapsed_time(b) for a, b in v), 3) for k, v in ev.items()}
    line.update(train_records=int(A.user.numel()), test_records=int(A.test_user.numel()),
                test_users=len(A.test_users), train_users=len(A.uids), train_items=len(A.iids))
    for label, make, private_gen, private_rec in runs():
        sim, ext, gen, rsim, priv = make()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = evaluate.evaluate(A, sim, ext, gen, private_gen, rsim, priv, private_rec, n=N, events={})
        torch.cuda.synchronize()
        line[label] = summary(res, (time.perf_counter() - t0) * 1e3)
        del res
    line["note"] = ("the synthetic ratings have no signal (drawn independently of user and item): the MAE and the "
                    "top-N accuracy only show that the evaluation runs end to end at this scale; parity with the "
                    "facade chain is pinned by tests/test_gpu_evaluate.py")
    s = json.dumps(line)
    print(s)
    if out_dir is not None:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "eval_time_%s.json" % name), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
