"""Explicit ALS (als.py) at cfg2 scale: device time per half-step, split into normal equations and solve, the top-N
time, the fp64 operation counts and rates, and the held-out accuracy (evaluate.evaluate_als).

  python tools/als_time.py [workload=cfg2] [out_dir]

Writes the cfg2-shaped pair of rating files (ingest_time.SHAPES, ingest_time.write_files) into a temporary directory,
runs ingest_arrays once, then evaluate_als four times: trained on every training record of both domains (the
MLlib-ALS baseline) and on the NX-MAP AlterEgo profile (non-private generation), each at rank 10 (MLlib's default) and
rank 64, 5 iterations, lambda 0.01.  Per run, one more als.top_n covers every user.  One JSON line, with the GPU name
and power limit read in the same run; with out_dir the line is also written to out_dir/als_time_<workload>.json.

Operation counts are computed from the shapes: a half-step forms records x (T + rank) fp64 multiply-adds of normal
equations (T = rank (rank + 1) / 2 packed entries), and each row with records takes (rank^3 - rank) / 6 multiply-adds
of Cholesky and rank (rank - 1) of substitutions.  The synthetic ratings carry no signal (synth.make_ratings draws them
independently of user and item), so the accuracy numbers only show that the evaluation runs end to end."""
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

N = 10
ITERATIONS = 5
LAMBDA = 0.01
SEED = 20261022


def counts(model, n_records):
    r = model.rank
    T = r * (r + 1) // 2
    rows = {"item": int((model.item_count > 0).sum()), "user": int((model.user_count > 0).sum())}
    return {side: {"normal_madd": n_records * (T + r), "solve_madd": rows[side] * ((r ** 3 - r) // 6 + r * (r - 1)),
                   "rows": rows[side]} for side in rows}


def summary(ev, wall_ms, all_ms, n_records):
    m, model = ev.metrics, ev.model
    rnd = lambda x: None if x is None else round(x, 6)
    ops = counts(model, n_records)
    halves = []
    for h in model.half_ms:
        c = ops[h["side"]]
        halves.append({"side": h["side"], "normal_ms": round(h["normal_ms"], 3), "solve_ms": round(h["solve_ms"], 3),
                       "normal_gflops": round(2 * c["normal_madd"] / h["normal_ms"] / 1e6, 1),
                       "solve_gflops": round(2 * c["solve_madd"] / h["solve_ms"] / 1e6, 1)})
    return {"rank": model.rank, "train_records": n_records, "stage_ms": {k: round(v, 3) for k, v in ev.stage_ms.items()},
            "wall_ms": round(wall_ms, 1), "half_steps": halves, "op_counts": ops,
            "train_ms": round(ev.stage_ms["als_train"], 3), "top_n_test_users_ms": round(ev.stage_ms["top_n"], 3),
            "top_n_all_users_ms": round(all_ms, 3), **ev.counts, "mae": rnd(ev.mae), "mae_bounded": rnd(ev.mae_bounded),
            **{"%s@%d" % (k, ev.n): rnd(v) for k, v in (m.mean or {}).items()}, "coverage@%d" % ev.n: rnd(m.coverage)}


def main():
    import torch
    from ingest_time import SHAPES, gpu_info, tools, write_files
    from xmap_b200 import als, evaluate, ingest, synth
    from xmap_b200.core import BaselinerSim, ExtendSim, Generator
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    out_dir = sys.argv[2] if len(sys.argv) > 2 else None
    os.environ["TZ"] = "UTC"
    time.tzset()
    nu, ni, nd, ov = SHAPES[name]
    with tempfile.TemporaryDirectory() as tmp:
        paths = write_files(synth.make_ratings(nu, ni, nd, overlap=ov), tmp, name)
        if not torch.cuda.is_available():
            raise SystemExit("als_time: wrote %s (%d bytes); no CUDA device, and ALS runs on the GPU only"
                             % (paths, sum(os.path.getsize(p) for p in paths)))
        line = {"tool": "als_time", "workload": "%s: %d users, %d items per domain, %d draws, overlap %g"
                % (name, nu, ni, nd, ov), **gpu_info(), "n": N, "iterations": ITERATIONS, "lambda": LAMBDA,
                "seed": SEED}
        cs, ct, sp = tools()
        A = ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False)
    line.update(train_records=int(A.user.numel()), test_records=int(A.test_user.numel()),
                test_users=len(A.test_users), train_users=len(A.uids), train_items=len(A.iids))
    arms = [("baseline", None),
            ("nx_map", lambda: (BaselinerSim("adjust_cosine", 50), ExtendSim(10),
                                Generator(1, 0.6, "adjust_cosine", 0.1, private_mode="exp_mech", seed=SEED), False))]
    # warm-up: module load and the first launches of every kernel shape, outside the timed runs
    evaluate.evaluate_als(A, rank=10, iterations=1, lambda_=LAMBDA, seed=SEED)
    evaluate.evaluate_als(A, rank=64, iterations=1, lambda_=LAMBDA, seed=SEED)
    for label, make in arms:
        for rank in (10, 64):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev = evaluate.evaluate_als(A, rank=rank, iterations=ITERATIONS, lambda_=LAMBDA, seed=SEED,
                                       alterego=None if make is None else make(), n=N, events={})
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            allt = als.top_n(ev.model, N, ev.train_user, ev.train_item,
                             candidates=torch.nonzero(A.meta.has_T[ev.profile_items] &
                                                      (ev.model.item_count > 0)).flatten())
            b.record()
            torch.cuda.synchronize()
            s = summary(ev, wall, a.elapsed_time(b), int(ev.train_user.numel()))
            s["top_n_all_users"] = int((allt.len > 0).sum())
            line["%s_rank%d" % (label, rank)] = s
            del ev, allt
    line["multi_gpu"] = "not measured"
    line["note"] = ("the synthetic ratings have no signal (drawn independently of user and item): the MAE and the "
                    "top-N accuracy only show that the evaluation runs end to end at this scale; the factors equal "
                    "the numpy restatement bit for bit (tests/test_gpu_als.py)")
    s = json.dumps(line)
    print(s)
    if out_dir is not None:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "als_time_%s.json" % name), "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
