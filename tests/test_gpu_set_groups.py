"""RegexSets in pattern groups on the GPU (DESIGN.md §2): sets of more than 256 patterns and sets whose product
automaton is over the table budget.  Every answer is compared with the oracle's set_matches, and with the
product-automaton object of the same patterns wherever one exists."""
import ctypes
import os
import re as pyre
import sys
import threading

import numpy as np
import pytest

import regex_b200 as R
from helpers import sherlock_text, tiled_corpus, vectors
from oracle import oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import corpus as C  # noqa: E402

pytestmark = pytest.mark.gpu

SET_PATTERNS = [r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+", "Holmes", "Watson", "Sherlock", r"Holmes|Watson", r"^The", r"\.$",
                r"(?m)^$", r"[0-9]{4}", r"(?i)holmes", "zqj", r"[a-z]+ing", r"(?-u:\b)never(?-u:\b)"]
SMALL = 16 << 10
_SETS = {}


def words():
    return [w.decode() for w in sorted(set(pyre.findall(rb"[A-Za-z]{4,}", sherlock_text())))]


def edge_patterns():
    """Empty, anchored and boundary members spread over several groups of 3."""
    w = words()
    return [w[10], "", w[20], w[30], r"^The", w[40], w[50], r"\.$", w[60], r"(?m)^$", w[70], w[80], r"(?-u:\b)", "zqjx", w[90]]


def make(name):
    """(set, patterns, product-automaton set or None) -- cached: the over-budget set takes seconds to compile."""
    if name in _SETS:
        return _SETS[name]
    w = words()
    product = None
    if name == "w257":
        pats = w[:257]
        s = R.BytesRegexSet(pats)
    elif name == "w1024":
        pats = w[:1024]
        s = R.BytesRegexSet(pats)
    elif name == "w1024i":
        pats = ["(?i)" + x for x in w[2000:3024]]
        s = R.BytesRegexSet(pats)
    elif name == "c4_small":
        pats = C.c4_patterns()
        s = R.BytesRegexSet(pats, dfa_size_limit=SMALL)
        product = R.BytesRegexSet(pats)
    elif name == "set_small":
        pats = SET_PATTERNS
        s = R.BytesRegexSet(pats, dfa_size_limit=SMALL)
        product = R.BytesRegexSet(pats)
    elif name == "over_budget":
        pats = [r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+"] + [rf"(?i){x}\s+\w+" for x in w[200:260]]
        s = R.BytesRegexSet(pats)
    elif name == "c4_k5":
        pats = C.c4_patterns()
        s = R.BytesRegexSet(pats)
        s.set_option("set_group_patterns", 5)
        product = R.BytesRegexSet(pats)
    elif name == "c4_k65":
        pats = C.c4_patterns() + SET_PATTERNS + ["zqjx" + str(i) for i in range(60)]
        s = R.BytesRegexSet(pats)
        s.set_option("set_group_patterns", 65)
        product = None
    elif name == "edge":
        pats = edge_patterns()
        s = R.BytesRegexSet(pats)
        s.set_option("set_group_patterns", 3)
        product = R.BytesRegexSet(pats)
    else:
        raise KeyError(name)
    assert len(s.groups()) > 1, name
    _SETS[name] = (s, pats, product)
    return _SETS[name]


GROUPED = ["w257", "w1024", "w1024i", "c4_small", "set_small", "over_budget", "c4_k5", "c4_k65", "edge"]


def _starts(text):
    mid = text.index(b"\n", len(text) // 2) - 7  # inside a line
    return [0, 1, 17, mid, len(text)]


@pytest.mark.parametrize("name", GROUPED)
def test_whole_haystack_calls_on_sherlock(name):
    import torch
    s, pats, product = make(name)
    text = sherlock_text()
    o = O.OracleRegex(pats)
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for start in _starts(text):
        exp = o.set_matches(text, start)
        assert s.matches(text, start) == exp, (name, start)
        mask = s.matches_mask(text, start)
        assert [i for i in range(len(pats)) if (mask[i // 64] >> (i % 64)) & 1] == exp
        assert s.is_match(text, start) == bool(exp)
        assert s.matches_device(d, start) == exp, (name, start)
        if product is not None:
            assert product.matches(text, start) == exp
    assert s.last_stats()["groups"] == len(s.groups())


@pytest.mark.parametrize("name", ["c4_small", "w1024", "over_budget"])
def test_tiled_32mib_corpus(name):
    """The oracle checks C4 over the whole corpus (it runs at about 1 MB/s); the larger sets are compared with
    another group plan of the same patterns and with the oracle on the first 2 MiB."""
    import torch
    s, pats, product = make(name)
    text = tiled_corpus(32 << 20)
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    o = O.OracleRegex(pats)
    other = R.BytesRegexSet(pats, dfa_size_limit=SMALL if name == "c4_small" else 2 << 20)
    other.set_option("set_group_patterns", 16)
    assert other.groups() != s.groups()
    for start in (0, (20 << 20) + 5):
        got = s.matches_device(d, start)
        assert s.matches(text, start) == got, start
        assert other.matches_device(d, start) == got, start
        if product is not None:
            assert product.matches_device(d, start) == got
        if name == "c4_small" and start == 0:
            assert got == o.set_matches(text, start)
    head = text[:2 << 20]
    assert s.matches(head, 5) == o.set_matches(head, 5)


def test_rure_set_matches_through_ctypes_past_256_patterns():
    s, pats, _ = make("w1024")
    text = sherlock_text()
    lib = R.lib()
    for start in (0, 1000):
        out = (ctypes.c_bool * len(pats))()
        p, n, keep = R._buf(text)
        any_ = lib.rure_set_matches(s._h, p, n, start, out)
        exp = O.OracleRegex(pats).set_matches(text, start)
        assert [i for i in range(len(pats)) if out[i]] == exp
        assert bool(any_) == bool(exp)
        assert lib.rure_set_is_match(s._h, p, n, start) == bool(exp)


@pytest.mark.parametrize("k", [1, 5])
def test_golden_set_vectors_in_forced_groups(k):
    n, bad = 0, []
    for x in vectors():
        if x["kind"] not in ("matset", "nomatset"):
            continue
        text = bytes.fromhex(x["text_hex"])
        for mode in x["modes"]:
            utf8 = mode == "str"
            try:
                s = (R.RegexSet if utf8 else R.BytesRegexSet)(x["res"])
            except R.Error as e:
                assert "word boundar" in str(e)
                continue
            s.set_option("set_group_patterns", k)
            got = s.matches(text)
            if got != x["expected"] or s.is_match(text) != bool(got):
                bad.append((x["name"], mode, got, x["expected"]))
            off = np.array([0, len(text)], dtype=np.uint64)
            row = s.matches_batch(text, off)[0]
            if [i for i in range(len(x["res"])) if (int(row[i // 64]) >> (i % 64)) & 1] != x["expected"]:
                bad.append(("batch", x["name"], mode))
            n += 1
    assert n > 10
    assert not bad, bad[:10]


def test_narrowing_across_groups():
    """56 MiB at wave0 = 1 MiB: waves [0, 1 MiB), [1, 17 MiB) and the rest, so narrowing on and off both take three
    or more; the late matches lie in the last wave."""
    import torch
    base = tiled_corpus(56 << 20)
    late = b" zyxwvut 987654 "
    text = base[:40 << 20] + late + base[40 << 20:]
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    pats = [r"\w+", r"\d+", r"Holmes", r"zyxwvut", r"9876\d+", r"qqqqqq", r"(?i)WATSON\s", r"^The", r"\.$", r"xyzzy|plugh",
            r"[A-Z][a-z]+ing"] + C.c4_patterns()
    product = R.BytesRegexSet(pats)
    exp = product.matches_device(d)
    assert 3 in exp and 4 in exp  # the late matches
    head = O.OracleRegex(pats).set_matches(text[:1 << 20])
    answers = []
    for narrow in (1, 0):
        s = R.BytesRegexSet(pats, dfa_size_limit=SMALL)
        assert len(s.groups()) > 1
        s.set_option("wave0", 1 << 20)
        s.set_option("narrow_sets", narrow)
        answers.append(s.matches_device(d))
        assert s.last_stats()["waves"] >= 3
        assert s.matches_device(d) == answers[-1]  # steady state: the narrowed subset is cached
        assert s.matches(text[:1 << 20]) == head
    assert answers[0] == answers[1] == exp


def test_only_the_last_group_matches_near_the_start():
    import torch
    s, pats, _ = make("w1024")
    text = bytearray(b"." * (32 << 20))
    text[10:10 + len(pats[-1])] = pats[-1].encode()
    d = torch.frombuffer(text, dtype=torch.uint8).cuda()
    s.set_option("wave0", 1 << 20)
    assert s.is_match(bytes(text))
    st = s.last_stats()
    assert st["waves"] == 1 and st["groups"] == len(s.groups())
    exp = O.OracleRegex(pats).set_matches(bytes(text[:4096]))
    assert len(pats) - 1 in exp
    assert s.matches_device(d) == exp
    s.set_option("wave0", 64 << 20)


def _batch_expect(pats, text, offs):
    o = O.OracleRegex(pats)
    return [o.set_matches(text[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]


def _rows(m, n_pat):
    m = np.asarray(m).astype(np.uint64)
    return [[i for i in range(n_pat) if (int(row[i // 64]) >> (i % 64)) & 1] for row in m]


@pytest.mark.parametrize("name", GROUPED)
def test_batched_sherlock_lines(name):
    import torch
    s, pats, product = make(name)
    lines = sherlock_text().split(b"\n")[:800]
    lines[3] = b""
    lines[7] = b""
    text = b"\n".join(lines)
    offs, pos = [0], 0
    for l in lines:
        pos += len(l) + 1
        offs.append(min(pos, len(text)))
    offs = np.array(offs, dtype=np.uint64)
    exp = _batch_expect(pats, text, offs.tolist())
    got = _rows(s.matches_batch(text, offs), len(pats))
    assert got == exp
    mw = (len(pats) + 63) // 64
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    d_off = torch.from_numpy(offs.astype(np.int64)).cuda()
    d_masks = torch.full((len(offs) - 1, mw), -1, dtype=torch.int64, device="cuda")
    s.matches_batch_device(d_text, d_off, d_masks)
    assert _rows(d_masks.cpu().numpy().view(np.uint64), len(pats)) == exp
    if product is not None:
        assert _rows(product.matches_batch(text, offs), len(pats)) == exp
    # zero records
    assert s.matches_batch(text, np.array([0], dtype=np.uint64)).shape[0] == 0


def test_batched_record_that_only_the_last_group_matches():
    for name in ("w1024", "c4_k5", "c4_k65"):
        s, pats, _ = make(name)
        lo, hi = s.groups()[-1]
        rec = [b"", b"......", pats[-1].encode() if name != "c4_k5" else b"Mrs. ", b"zz"]
        text = b"".join(rec)
        offs = np.cumsum([0] + [len(r) for r in rec]).astype(np.uint64)
        got = _rows(s.matches_batch(text, offs), len(pats))
        assert got == _batch_expect(pats, text, offs.tolist()), name
        assert any(i >= lo for i in got[2])


def test_batched_million_c3_lines():
    import torch
    dev = torch.device("cuda", 0)
    text, offsets = C.log_lines(1_000_000, dev)
    for name in ("c4_small", "c4_k5", "w1024"):
        s, pats, product = make(name)
        mw = (len(pats) + 63) // 64
        out = torch.empty((1_000_000, mw), dtype=torch.int64, device=dev)
        s.matches_batch_device(text, offsets, out)
        got = out.cpu().numpy().view(np.uint64)
        if product is not None:
            ref = torch.empty_like(out)
            product.matches_batch_device(text, offsets, ref)
            assert (ref.cpu().numpy().view(np.uint64) == got).all(), name
        k = 5000
        host, offs = text[:int(offsets[k])].cpu().numpy().tobytes(), offsets[:k + 1].tolist()
        assert _rows(got[:k], len(pats)) == _batch_expect(pats, host, offs), name


def test_four_threads_share_one_grouped_handle():
    s, pats, _ = make("over_budget")
    text = sherlock_text()
    exp = {start: O.OracleRegex(pats).set_matches(text, start) for start in (0, 1000, 200000)}
    lib = R.lib()
    p, n, keep = R._buf(text)
    errors = []

    def work(t):
        for start in (0, 1000, 200000):
            out = (ctypes.c_bool * len(pats))()
            lib.rure_set_matches(s._h, p, n, start, out)
            if [i for i in range(len(pats)) if out[i]] != exp[start]:
                errors.append((t, start))

    threads = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors


def test_explicit_errors_of_grouped_sets():
    import torch
    s, pats, _ = make("c4_small")
    with pytest.raises(R.Error, match="pattern groups"):
        s.dfa(R.DFA_FWD_UNANCHORED_ALL)
    text = sherlock_text()
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    io = {"own_lo": 0, "own_hi": len(text), "is_first": True, "is_last": True, "entry_state": 0xFFFFFFFF}
    with pytest.raises(R.Error, match="pattern groups"):
        s.forward_shard_device(d, io)
