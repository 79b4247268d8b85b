"""GPU: ingest.clean_split_pipeline (rating files -> device-resident training set, csrc/ingest.cu) against the host
path it replaces, baseliner_clean_data_pipeline x2 + baseliner_split_data_pipeline, record for record and in order;
its Encoded against encode_records; the refusals of its stricter reader; and the downstream stages on both."""
import contextlib
import os
import time

import numpy as np
import pytest
import torch

from oracle import make_golden_cleansplit as CS

pytestmark = pytest.mark.gpu

DST_TZ = "EST+5EDT,M3.2.0/2,M11.1.0/2"


@contextlib.contextmanager
def tz(name):
    old = os.environ.get("TZ")
    os.environ["TZ"] = name
    time.tzset()
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("TZ", None)
        else:
            os.environ["TZ"] = old
        time.tzset()


def _tools(cfg):
    from xmap_b200.core import BaselinerClean, BaselinerSplit
    cs = BaselinerClean(cfg["atleast"], cfg["subset"], cfg["date_from"], cfg["date_to"], cfg["labels"][0])
    ct = BaselinerClean(cfg["atleast"], cfg["subset"], cfg["date_from"], cfg["date_to"], cfg["labels"][1])
    sp = BaselinerSplit(cfg["num_left"], cfg["ratio_split"], cfg["ratio_both"], cfg["seed"])   # seeds `random`
    return cs, ct, sp


def run_host(paths, cfg, dbg):
    from xmap_b200.core import baseliner_clean_data_pipeline, baseliner_split_data_pipeline
    cs, ct, sp = _tools(cfg)
    s = baseliner_clean_data_pipeline(None, cs, paths[0], dbg, 30)
    t = baseliner_clean_data_pipeline(None, ct, paths[1], dbg, 30)
    tr, te = baseliner_split_data_pipeline(None, sp, s, t)
    return tr, te


def run_device(paths, cfg, dbg):
    from xmap_b200 import ingest
    cs, ct, sp = _tools(cfg)
    return ingest.clean_split_pipeline(None, cs, ct, sp, paths[0], paths[1], dbg)


def _cfg(**kw):
    c = dict(atleast=5, subset=150, date_from=2012, date_to=2013, labels=("S:", "T:"), num_left=0, ratio_split=0.2,
             ratio_both=0.8, seed=666666)
    c.update(kw)
    return c


def check_encoded(train, host_train):
    from xmap_b200.encode import encode_records
    got = train._xmap_session.enc
    want = encode_records(host_train)
    assert np.array_equal(got.uids, want.uids) and np.array_equal(got.iids, want.iids)
    assert got.user.dtype == want.user.dtype and np.array_equal(got.user, want.user)
    assert got.item.dtype == want.item.dtype and np.array_equal(got.item, want.item)
    assert np.array_equal(got.rating.view(np.int64), want.rating.view(np.int64))
    for k in ("prefix_code", "dom_code", "contains", "has_S", "has_T"):
        a, b = getattr(got, k), getattr(want, k)
        assert a.dtype == b.dtype and np.array_equal(a, b), k
    assert len(got.times) == len(want.times) and list(got.times) == list(want.times)


def check_parity(paths, cfg, dbg, encoded=True):
    htr, hte = run_host(paths, cfg, dbg)
    htr, hte = htr.collect(), hte.collect()
    dtr, dte = run_device(paths, cfg, dbg)
    got_tr = dtr.collect()
    assert got_tr == htr
    assert dte.collect() == hte
    if encoded and htr:
        check_encoded(dtr, htr)
    return htr, hte


# ---- 1. the golden input -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,dbg", CS.MODES)
def test_golden_input_matches_host(tmp_path, mode, dbg):
    want, _, _ = CS.load()
    with CS.utc():
        paths = CS.write_inputs(str(tmp_path))
        htr, hte = check_parity(paths, _cfg(), dbg)
    norm = lambda recs: sorted((u, sorted((i, float(r), int(x.timestamp())) for i, r, x in l)) for u, l in recs)
    assert norm(htr) == want[mode][2] and norm(hte) == want[mode][3]
    assert len(htr) > 0 and len(hte) > 0


# ---- 2. randomised inputs ------------------------------------------------------------------------------------------
def _synth_files(tmp, seed, n_users=20000):
    from xmap_b200 import synth
    import calendar
    sr = synth.make_ratings(n_users, 3000, 240000, overlap=0.3, seed=seed)
    rng = np.random.default_rng(seed)
    paths = []
    for d, nm in ((0, "src"), (1, "tgt")):
        lines = synth.to_text_lines(sr, d)
        n = len(lines)
        pick = lambda k: [lines[q] for q in rng.integers(0, n, k)]
        parts = lambda l: l.split("\t")
        extra = []
        for l in pick(n // 10):                          # re-ratings, later or earlier
            u, i, r, t = parts(l)
            extra.append("\t".join([u, i, str(rng.integers(1, 6)), str(int(t) + int(rng.integers(-10 ** 7, 10 ** 7)))]))
        for l in pick(n // 20):                          # equal-time duplicates: the first one wins
            u, i, r, t = parts(l)
            extra.append("\t".join([u, i, str(rng.integers(1, 6)), t]))
        for l in pick(n // 20):                          # out of the period
            u, i, r, t = parts(l)
            extra.append("\t".join([u, i, r, str(int(t) + int(rng.choice([-1, 1])) * 3 * 10 ** 8)]))
        edges = [calendar.timegm((y, 1, 1, 0, 0, 0)) for y in (2012, 2014)]
        for l in pick(n // 20):                          # within an hour of a year boundary, in UTC and in local time
            u, i, r, t = parts(l)
            e = int(rng.choice(edges)) + int(rng.choice([0, 5 * 3600]))
            extra.append("\t".join([u, i, r, str(e + int(rng.integers(-3600, 3600)))]))
        allx = lines + extra
        allx = [allx[q] for q in rng.permutation(len(allx))]
        p = os.path.join(tmp, nm + ".txt")
        with open(p, "w") as f:
            f.write("\n".join(allx) + "\n")
        paths.append(p)
    return paths


@pytest.mark.parametrize("num_left,subset,dbg", [(0, 10 ** 9, False), (2, 10 ** 9, False), (0, 700, True),
                                                 (2, 10 ** 9, True), (2, 3000, True)])
def test_random_inputs_match_host(tmp_path, num_left, subset, dbg):
    with tz(DST_TZ):
        paths = _synth_files(str(tmp_path), 11 + num_left)
        htr, hte = check_parity(paths, _cfg(atleast=3, subset=subset, num_left=num_left, ratio_split=0.3,
                                            ratio_both=0.4, seed=2 ** 40 + 17), dbg)
    assert len(htr) > 100 and len(hte) > 0


# ---- 3. grammar ----------------------------------------------------------------------------------------------------
def _grammar_files(tmp, seed, final_newline):
    rng = np.random.default_rng(seed)
    ratings = ["4", "4.", ".5", "+4.0", "-0", "4e0", "45E-1", "0.5e1", "3.50", "-2.5", "00012", "1E+0"]
    stamps = ["1356998400", "1356998400.25", "1.3569984e9", "+1356998400", "1356998400.", "13569984000E-1",
              "1388534399", "1325376000"]
    seps = [" ", "\t", "   ", "\x0b", "\x1f", "\x0c", " \t ", "\x1c"]
    terms = ["\n", "\r\n", "\r"]
    pre8, pre16 = "abcdefgh", "abcdefghijklmnop"
    uids = ["u", "u1", pre8, pre8 + "1", pre8 + "12", pre16, pre16 + "x", pre16 + "xy", "u" * 40, "zS:", "zT:"]
    raw = ["i", "i1", pre8, pre8 + "a", pre16, pre16 + "b", pre16 + "bc", "k" * 40, "xS:y", "yT:", "S:", "T:S:",
           "mvS:1", "a" * 23]
    paths = []
    for d in range(2):
        out = []
        for k in range(1500):
            if rng.random() < 0.04:
                out.append(str(rng.choice(["", "  ", "\t", "\x1c\x1d", " \x0b "])))
                continue
            f = [str(rng.choice(uids)), str(rng.choice(raw)), str(rng.choice(ratings)), str(rng.choice(stamps))]
            if rng.random() < 0.2:
                f += ["extra", "fields"][: rng.integers(1, 3)]
            line = "".join(a + str(rng.choice(seps)) for a in f[:-1]) + f[-1]
            if rng.random() < 0.2:
                line = str(rng.choice(seps)) + line
            if rng.random() < 0.2:
                line = line + str(rng.choice(seps))
            out.append(line)
        text = ""
        for k, line in enumerate(out):
            t = str(rng.choice(terms))
            if t == "\r" and k + 1 < len(out) and out[k + 1] == "":
                t = "\n"                                   # "\r" + "" + "\n" would read as one "\r\n"
            text += line + t
        if not final_newline:
            text = text.rstrip("\r\n")
        p = os.path.join(tmp, "g%d.txt" % d)
        with open(p, "w", newline="") as fh:
            fh.write(text)
        paths.append(p)
    return paths


@pytest.mark.parametrize("final_newline", [True, False])
@pytest.mark.parametrize("num_left", [0, 1])
def test_grammar_matches_host(tmp_path, final_newline, num_left):
    with CS.utc():
        paths = _grammar_files(str(tmp_path), 3 + num_left, final_newline)
        htr, hte = check_parity(paths, _cfg(atleast=1, num_left=num_left, ratio_split=0.5, ratio_both=0.3), False)
    assert len(htr) > 10


def test_number_parser_is_bit_equal_to_float(tmp_path):
    """20 000 random decimal spellings within the grammar, read as ratings of test records (which the binary32 check
    does not cover): the parsed values equal float() bit for bit."""
    from xmap_b200 import ingest
    rng = np.random.default_rng(5)
    toks = []
    for _ in range(20000):
        digits = "".join(str(x) for x in rng.integers(0, 10, rng.integers(1, 16)))
        dot = int(rng.integers(0, len(digits) + 1))
        s = digits[:dot] + "." + digits[dot:] if rng.random() < 0.7 else digits
        if rng.random() < 0.5:
            s += "e%+d" % rng.integers(-7, 9)
        toks.append(str(rng.choice(["", "+", "-"])) + s)
    src = os.path.join(str(tmp_path), "s.txt")
    tgt = os.path.join(str(tmp_path), "t.txt")
    with open(src, "w") as f:
        f.write("".join("u%05d i 1 1356998400\n" % k for k in range(len(toks))))
    with open(tgt, "w") as f:
        f.write("".join("u%05d j %s 1356998400\n" % (k, t) for k, t in enumerate(toks)))
    cs, ct, sp = _tools(_cfg(atleast=1, num_left=0, ratio_split=1.0, ratio_both=0.0))
    with CS.utc():
        A = ingest.ingest_arrays(cs, ct, sp, src, tgt, False)
    got = A.test_rating.cpu().numpy()
    want = np.array([float(t) for t in toks])
    assert len(got) == len(toks) and np.array_equal(got.view(np.int64), want.view(np.int64))


# ---- 4. refusals ---------------------------------------------------------------------------------------------------
_GOOD = ["u1\ti1\t4\t1356998400", "u2\ti1\t5\t1356998500"]


@pytest.mark.parametrize("bad,exc,token", [
    (b"u3\ti1\t4", IndexError, None),
    (b"u3\ti\xc3\xa91\t4\t1356998400", ValueError, "i\xc3\xa91"),
    (b"u3\ti1\t4\t13569\x0084", ValueError, None),
    (b"u3\ti1\tnan\t1356998400", ValueError, "nan"),
    (b"u3\ti1\t1_0\t1356998400", ValueError, "1_0"),
    (b"u3\ti1\t12345678901234567\t1356998400", ValueError, "12345678901234567"),
    (b"u3\ti1\t4\t1e20", ValueError, "1e20"),
    (b"u3\ti1\t3.7000001\t1356998400", ValueError, "3.7000001"),
    (b"u3\t" + b"i" * 47 + b"\t4\t1356998400", ValueError, "i" * 47),
    (b"u" * 49 + b"\ti1\t4\t1356998400", ValueError, "u" * 49),
])
def test_refusals_name_the_line(tmp_path, bad, exc, token):
    from xmap_b200 import ingest
    src = os.path.join(str(tmp_path), "s.txt")
    tgt = os.path.join(str(tmp_path), "t.txt")
    with open(src, "wb") as f:
        f.write(("\n".join(_GOOD) + "\n").encode() + bad + b"\n")
    with open(tgt, "w") as f:
        f.write("u1\tj1\t4\t1356998400\n")
    cs, ct, sp = _tools(_cfg(atleast=1))
    with CS.utc(), pytest.raises(exc) as e:
        ingest.clean_split_pipeline(None, cs, ct, sp, src, tgt, False)
    msg = str(e.value)
    assert "s.txt, line 3" in msg, msg
    if token is not None:
        assert repr(token) in msg, msg


def test_refuses_more_than_eight_suffixes(tmp_path):
    from xmap_b200 import ingest
    from xmap_b200.encode import encode_records
    src = os.path.join(str(tmp_path), "s.txt")
    tgt = os.path.join(str(tmp_path), "t.txt")
    with open(src, "w") as f:
        f.write("".join("u1\ti%d\t4\t1356998400\n" % k for k in range(9)))
    with open(tgt, "w") as f:
        f.write("u9\tj1\t4\t1356998400\n")
    cfg = _cfg(atleast=1, labels=("S", "T"))
    with CS.utc():
        htr, _ = run_host((src, tgt), cfg, False)
        with pytest.raises(ValueError, match="more than 8"):
            encode_records(htr.collect())
        cs, ct, sp = _tools(cfg)
        with pytest.raises(ValueError, match="more than 8"):
            ingest.clean_split_pipeline(None, cs, ct, sp, src, tgt, False)


def test_empty_files_and_sc(tmp_path):
    from xmap_b200 import ingest
    src = os.path.join(str(tmp_path), "s.txt")
    tgt = os.path.join(str(tmp_path), "t.txt")
    open(src, "w").close()
    with open(tgt, "w") as f:
        f.write("\n  \n")
    cs, ct, sp = _tools(_cfg())
    tr, te = ingest.clean_split_pipeline(None, cs, ct, sp, src, tgt, False)
    assert tr.collect() == [] and te.collect() == []
    with pytest.raises(ValueError):
        ingest.clean_split_pipeline(object(), cs, ct, sp, src, tgt, False)


# ---- 5. downstream -------------------------------------------------------------------------------------------------
def test_downstream_stages_equal(tmp_path):
    from xmap_b200.core import (BaselinerSim, ExtendSim, Generator, baseliner_calculate_sim_pipeline,
                                extender_pipeline, generator_pipeline)
    from xmap_b200.session import session_of
    with CS.utc():
        paths = _synth_files(str(tmp_path), 11)
        cfg = _cfg(atleast=3, num_left=2, ratio_split=0.3, ratio_both=0.4)
        out = []
        for run in (run_host, run_device):
            tr, _ = run(paths, cfg, False)
            sim_tool = BaselinerSim("adjust_cosine", 5)
            simRDD = baseliner_calculate_sim_pipeline(None, sim_tool, tr)
            xs = extender_pipeline(None, None, sim_tool, ExtendSim(10), simRDD)
            alter = generator_pipeline(Generator(1, 0.6, "adjust_cosine", 0.1), tr, xs, True).collect()
            out.append((session_of(tr).tables, xs.collect(), alter))
    (ta, xa, aa), (tb, xb, ab) = out
    for k in ("row_flags", "row_nkept", "tab_idx", "tab_sim", "tab_mutu", "tab_n", "tab_len"):
        if hasattr(ta, k):
            assert torch.equal(getattr(ta, k), getattr(tb, k)), k
    assert xa == xb and len(xa) > 0
    assert aa == ab and len(aa) > 0
