"""CPU: the host-side clean / split stages against the unmodified reference run through the oracle shim (needs the
original X-MAP source, XMAP_REFERENCE_CODE; skipped without it), and against the records stored in
tests/golden/cleansplit.npz (oracle/make_golden_cleansplit.py), which run everywhere."""
import subprocess
import sys

import pytest

from oracle import harness as H
from oracle import make_golden_cleansplit as CS
from tests import parity as PT

_REFERENCE_RUN = """
import sys
sys.path.insert(0, %(root)r)
from oracle import make_golden_cleansplit as CS
paths = CS.write_inputs(%(tmp)r)
mine, ref = CS.run_host(paths), CS.run_reference(paths)
for mode in mine:
    for stage, a, b in zip(CS.STAGES, mine[mode], ref[mode]):
        assert a == b, (mode, stage, len(a), len(b))
    assert len(mine[mode][2]) > 0 and len(mine[mode][3]) > 0
print("ok")
"""


@pytest.mark.skipif(not H.reference_available(), reason="needs the original X-MAP source (XMAP_REFERENCE_CODE)")
def test_clean_and_split_match_reference(tmp_path):
    """Both modes (debug sample and full data), in the local time zone: the four record sets of the clean and split
    stages equal those of the unmodified reference on the same input."""
    code = _REFERENCE_RUN % dict(root=PT.ROOT, tmp=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=PT.ROOT)
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


def test_clean_and_split_match_stored_records(tmp_path):
    """Both modes, under TZ=UTC: the four record sets equal those stored in tests/golden/cleansplit.npz.  The file says
    where its records come from; the committed one is a regression snapshot of the host classes (the original source
    was not available when it was recorded), so this pins the stages to their earlier output, not to the reference:
    test_clean_and_split_match_reference does that where the source is available."""
    want, digest, source = CS.load()
    assert source in CS.SOURCES, source
    with CS.utc():
        paths = CS.write_inputs(str(tmp_path))
        assert CS.inputs_digest(paths) == digest, "the synthetic input is not the one the stored records were made from"
        mine = CS.run_host(paths)
    for mode in want:
        for stage, a, b in zip(CS.STAGES, mine[mode], want[mode]):
            assert a == b, (mode, stage, source, len(a), len(b))
        assert len(mine[mode][2]) > 0 and len(mine[mode][3]) > 0


def test_local_rdd_surface():
    from xmap_b200.rdd import LocalRDD, LazyRDD
    r = LocalRDD([("a", 1), ("b", 2), ("a", 3)])
    assert r.reduceByKey(lambda x, y: x + y).collectAsMap() == {"a": 4, "b": 2}
    assert r.map(lambda kv: kv[1]).filter(lambda v: v > 1).collect() == [2, 3]
    assert r.join(LocalRDD([("a", "x")])).collect() == [("a", (1, "x")), ("a", (3, "x"))]
    assert r.keys().distinct().collect() == ["a", "b"]
    calls = []
    lz = LazyRDD(lambda: calls.append(1) or [1, 2, 3])
    assert not calls and lz.count() == 3 and lz.collect() == [1, 2, 3] and len(calls) == 1
    parts = LocalRDD(range(1000)).randomSplit([0.2, 0.8], seed=7)
    assert sum(p.count() for p in parts) == 1000 and 120 < parts[0].count() < 280


def test_encoder_replicates_reference_string_tests():
    from xmap_b200.encode import encode_records, item_codes
    from datetime import datetime
    t = datetime(2012, 5, 1)
    recs = [("u2", [("mv01T:", 4.0, t), ("bkS:9S:", 2.5, t)]), ("u1", [("bk07S:", 5.0, t)])]
    e = encode_records(recs)
    assert list(e.uids) == ["u1", "u2"] and list(e.iids) == ["bk07S:", "bkS:9S:", "mv01T:"]
    assert list(e.prefix_code) == [0, 0, 1] and list(e.dom_code) == [0, 0, 1]
    assert list(e.has_S) == [True, True, False] and list(e.has_T) == [False, False, True]
    assert list(e.contains) == [1, 1, 2]
    with pytest.raises(ValueError):
        encode_records([("u", [("bkS:", 3.7000001, t)])])
    pc, dc, ct, hs, ht = item_codes(["xxT:S:"])       # a label inside the raw id still counts (substring test)
    assert ct[0] == 3 or ct[0] == 1


def test_clean_restatement_matches_host_class(monkeypatch):
    """The array-level restatement of the clean stage's record rules (tests/parity.clean_encoded_numpy -- what the device
    kernel is checked against) drives BaselinerClean.device_pipeline to exactly the records of the host class, which
    test_clean_and_split_match_reference pins to the unmodified reference."""
    import numpy as np
    import torch
    from xmap_b200 import synth, clean as CL
    from xmap_b200.core import BaselinerClean
    from xmap_b200.rdd import LocalRDD
    monkeypatch.setattr(CL, "clean_encoded", lambda u, i, t, nu, lo, hi, k, device="cpu":
                        tuple(torch.as_tensor(x) for x in PT.clean_encoded_numpy(u, i, t, nu, lo, hi, k)))
    sr = synth.make_ratings(300, 50, 6000, overlap=0.3, seed=5)
    lines = synth.to_text_lines(sr, 1)
    bump = lambda l, dt: l.rsplit("\t", 1)[0] + "\t" + str(int(l.rsplit("\t", 1)[1]) + dt)
    lines = lines + [bump(l, k * 40000000) for k, l in enumerate(lines[:150])] + [bump(l, -3600) for l in lines[150:250]] + \
        ["\t".join(l.split("\t")[:2] + ["1", l.split("\t")[3]]) for l in lines[250:350]]
    rng = np.random.default_rng(1)
    lines = [lines[k] for k in rng.permutation(len(lines))]
    assert CL.period_bounds(2012, 2013)[0] < 1.34e9 < CL.period_bounds(2012, 2013)[1]
    for atleast in (1, 4, 9):
        tool = BaselinerClean(atleast, 10 ** 9, 2012, 2013, "T:")
        want = tool.clean_data(tool.filter_data(tool.parse_data(LocalRDD(lines)))).collect()
        got = tool.device_pipeline(LocalRDD(lines)).collect()
        assert len(want) > 0 and got == want, atleast
