"""Freeze the records of the clean / split stages on a small synthetic input into tests/golden/cleansplit.npz.

TEST INFRASTRUCTURE ONLY:   python -m oracle.make_golden_cleansplit [--snapshot]

With the original X-MAP source available (oracle/harness.py, XMAP_REFERENCE_CODE) the stored records are the
reference's own, and the host classes (xmap_b200.core.BaselinerClean / BaselinerSplit driven through
baseliner_clean_data_pipeline / baseliner_split_data_pipeline) must produce the same records, or nothing is written.
Without the source nothing is written unless --snapshot asks for a regression snapshot of the host classes' records.
The file's `source` field says which of the two it holds.

The committed tests/golden/cleansplit.npz is such a snapshot: the original source was not available when it was
recorded, so it pins the host classes to their own earlier output, not to the reference.
tests/test_host_cleansplit.py::test_clean_and_split_match_reference compares with the reference where it is available.

Everything runs under TZ=UTC: the clean stage reads the rating times in local time (baselinerClean.py:36) and keeps
the ratings of a range of years, so which records survive depends on the time zone.  Times are stored as POSIX
seconds.
"""
import contextlib
import hashlib
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden", "cleansplit.npz")
STAGES = ("source", "target", "train", "test")
MODES = (("debug", True), ("full", False))


@contextlib.contextmanager
def utc():
    old = os.environ.get("TZ")
    os.environ["TZ"] = "UTC"
    time.tzset()
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("TZ", None)
        else:
            os.environ["TZ"] = old
        time.tzset()


def write_inputs(tmp):
    """Two rating files (user \\t item \\t rating \\t time), one per domain; returns their paths."""
    from xmap_b200 import synth
    sr = synth.make_ratings(400, 60, 9000, overlap=0.3, seed=4)
    paths = []
    for d, nm in ((0, "book"), (1, "movie")):
        lines = synth.to_text_lines(sr, d)
        # duplicates with other timestamps / out-of-period years exercise the filters
        extra = [l.rsplit("\t", 1)[0] + "\t" + str(int(l.rsplit("\t", 1)[1]) + k * 40000000)
                 for k, l in enumerate(lines[:200])]
        p = os.path.join(tmp, nm + ".txt")
        with open(p, "w") as f:
            f.write("\n".join(lines + extra) + "\n")
        paths.append(p)
    return paths


def inputs_digest(paths):
    h = hashlib.sha256()
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def run(mods, sc, paths):
    """{mode: [source, target, train, test]}, each a sorted list of (user, sorted [(item, rating, POSIX time)])."""
    out = {}
    for mode, dbg in MODES:
        cs = mods["BaselinerClean"](5, 150, 2012, 2013, "S:")
        ct = mods["BaselinerClean"](5, 150, 2012, 2013, "T:")
        sp = mods["BaselinerSplit"](0, 0.2, 0.8, 666666)
        s = mods["clean"](sc, cs, paths[0], dbg, 30)
        t = mods["clean"](sc, ct, paths[1], dbg, 30)
        tr, te = mods["split"](sc, sp, s, t)
        norm = lambda rdd: sorted((u, sorted((i, float(r), int(x.timestamp())) for i, r, x in l)) for u, l in rdd.collect())
        out[mode] = [norm(s), norm(t), norm(tr), norm(te)]
    return out


def run_host(paths):
    from xmap_b200.core import (BaselinerClean, BaselinerSplit, baseliner_clean_data_pipeline,
                                baseliner_split_data_pipeline)
    return run(dict(BaselinerClean=BaselinerClean, BaselinerSplit=BaselinerSplit,
                    clean=baseliner_clean_data_pipeline, split=baseliner_split_data_pipeline), None, paths)


def run_reference(paths):
    from oracle import harness as H
    R = H.load_reference()
    return run(dict(BaselinerClean=R["BaselinerClean"], BaselinerSplit=R["BaselinerSplit"],
                    clean=R["assist"].baseliner_clean_data_pipeline,
                    split=R["assist"].baseliner_split_data_pipeline), R["sc"], paths)


def encode(out):
    arrs = {}
    for mode, _ in MODES:
        for stage, recs in zip(STAGES, out[mode]):
            p = "%s_%s_" % (mode, stage)
            arrs[p + "user"] = np.array([u for u, _ in recs], dtype=str)
            arrs[p + "count"] = np.array([len(l) for _, l in recs], dtype=np.int32)
            arrs[p + "item"] = np.array([i for _, l in recs for i, _, _ in l], dtype=str)
            arrs[p + "rating"] = np.array([r for _, l in recs for _, r, _ in l], dtype=np.float64)
            arrs[p + "time"] = np.array([t for _, l in recs for _, _, t in l], dtype=np.int64)
    return arrs


SOURCES = ("reference", "host classes (regression snapshot)")


def load():
    """(records in the form run() returns, sha256 of the input files they were made from, their source: one of
    SOURCES)."""
    g = np.load(GOLDEN)
    out = {}
    for mode, _ in MODES:
        out[mode] = []
        for stage in STAGES:
            p = "%s_%s_" % (mode, stage)
            ptr = np.concatenate([[0], np.cumsum(g[p + "count"])])
            recs = list(zip(g[p + "item"].tolist(), g[p + "rating"].tolist(), g[p + "time"].tolist()))
            out[mode].append([(u, recs[a:b]) for u, a, b in zip(g[p + "user"].tolist(), ptr[:-1], ptr[1:])])
    return out, str(g["inputs_sha256"]), str(g["source"])


def main():
    from oracle import harness as H
    with_ref = H.reference_available()
    if not with_ref and "--snapshot" not in sys.argv[1:]:
        sys.exit("the original X-MAP source is not available (XMAP_REFERENCE_CODE): nothing written; pass --snapshot "
                 "to record the host classes' records as a regression snapshot instead")
    with utc(), tempfile.TemporaryDirectory() as tmp:
        paths = write_inputs(tmp)
        recs = run_host(paths)
        if with_ref:
            ref = run_reference(paths)
            assert ref == recs, "the host classes and the reference disagree: nothing written"
            recs = ref
        np.savez_compressed(GOLDEN, inputs_sha256=np.array(inputs_digest(paths)),
                            source=np.array(SOURCES[0] if with_ref else SOURCES[1]), **encode(recs))
    print("%s (%d KB), records of the %s" % (GOLDEN, os.path.getsize(GOLDEN) // 1024,
                                             SOURCES[0] if with_ref else SOURCES[1]))


if __name__ == "__main__":
    main()
