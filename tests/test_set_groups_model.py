"""CPU checks of RegexSets in pattern groups (DESIGN.md §2), by compiling only.

A set whose product automaton is over the table budget, or that has more than 256 patterns, is searched as
contiguous pattern ranges with one automaton each.  These tests check the plan (coverage, size, budget, split
points), the errors that stay, and a model of the search: each planned range compiled as its own set, its
forward all-match tables walked with dfa_sim.Sim.forward_scan, and the shifted OR of the masks compared with
the oracle's set_matches."""
import re as pyre
import sys
import os

import pytest

import regex_b200 as R
from dfa_sim import Sim
from helpers import sherlock_text, vectors
from oracle import oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import corpus as C  # noqa: E402

SET_PATTERNS = [r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+", "Holmes", "Watson", "Sherlock", r"Holmes|Watson", r"^The", r"\.$",
                r"(?m)^$", r"[0-9]{4}", r"(?i)holmes", "zqj", r"[a-z]+ing", r"(?-u:\b)never(?-u:\b)"]
SMALL = 16 << 10


def words():
    return [w.decode() for w in sorted(set(pyre.findall(rb"[A-Za-z]{4,}", sherlock_text())))]


def check_plan(s, pats, dfa_size_limit=2 << 20, max_group=256):
    g = s.groups()
    assert g[0][0] == 0 and g[-1][1] == len(pats)
    for (lo, hi), (lo2, _) in zip(g, g[1:]):
        assert hi == lo2
    for lo, hi in g:
        assert 0 < hi - lo <= min(256, max_group)
        R.BytesRegexSet(pats[lo:hi], dfa_size_limit=dfa_size_limit)  # each group compiles alone
    return g


def split_points_ok(g, n, chunk):
    """Every split that is not a chunk boundary came from halving a range; ranges over 64 patterns split on
    multiples of 64, so every group of more than 64 patterns starts and ends on one (or at n)."""
    for lo, hi in g:
        if hi - lo > 64:
            assert lo % 64 == 0 or lo % chunk == 0, (lo, hi)
            assert hi % 64 == 0 or hi == n or hi % chunk == 0, (lo, hi)


def test_257_and_1024_words_compile_in_groups_of_256():
    w = words()
    s = R.BytesRegexSet(w[:257])
    assert check_plan(s, w[:257]) == [(0, 256), (256, 257)]
    s = R.BytesRegexSet(w[:1024])
    assert check_plan(s, w[:1024]) == [(0, 256), (256, 512), (512, 768), (768, 1024)]
    assert len(s.groups()) >= 4
    assert R.BytesRegexSet(w[:256]).groups() == [(0, 256)]  # the product automaton, as before


@pytest.mark.parametrize("name", ["c4", "set_patterns"])
def test_budget_split_sets(name):
    pats = C.c4_patterns() if name == "c4" else SET_PATTERNS
    assert R.BytesRegexSet(pats).groups() == [(0, len(pats))]
    s = R.BytesRegexSet(pats, dfa_size_limit=SMALL)
    g = check_plan(s, pats, SMALL)
    assert len(g) > 1
    split_points_ok(g, len(pats), 256)
    with pytest.raises(R.Error, match="pattern groups"):
        s.dfa(R.DFA_FWD_UNANCHORED_ALL)


def test_over_budget_set_of_64_patterns():
    w = words()
    pats = [r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+"] + [rf"(?i){x}\s+\w+" for x in w[200:260]]
    s = R.BytesRegexSet(pats)
    g = check_plan(s, pats)
    assert len(g) >= 2
    split_points_ok(g, len(pats), 256)


@pytest.mark.parametrize("k", [1, 5, 63, 64, 65])
def test_forced_group_sizes(k):
    for pats in (C.c4_patterns(), SET_PATTERNS):
        s = R.BytesRegexSet(pats)
        s.set_option("set_group_patterns", k)
        g = check_plan(s, pats, max_group=max(k, 1))
        if k < len(pats):
            assert len(g) == (len(pats) + k - 1) // k
            assert all(lo % k == 0 for lo, _ in g)
        else:
            assert g == [(0, len(pats))]
        s.set_option("set_group_patterns", 0)
        assert s.groups() == [(0, len(pats))]


def test_forced_groups_split_further_by_budget():
    pats = C.c4_patterns()
    s = R.BytesRegexSet(pats, dfa_size_limit=SMALL)
    s.set_option("set_group_patterns", 64)
    g = check_plan(s, pats, SMALL)
    assert len(g) > 1
    s.set_option("set_group_patterns", 5)
    assert all(hi - lo <= 5 for lo, hi in check_plan(s, pats, SMALL))


def test_errors_that_stay():
    with pytest.raises(R.Error, match="exceeds size limit"):
        R.BytesRegexSet([r"error.{0,100}timeout", r"x"])  # an over-budget singleton
    with pytest.raises(R.Error, match="exceeds size limit"):
        R.BytesRegexSet([r"x", r"error.{0,100}timeout"], dfa_size_limit=SMALL)
    w = words()
    with pytest.raises(R.Error, match="exceeds size limit of 10485760 bytes"):
        R.BytesRegexSet([rf"{x}=\w+" for x in w[:96]])  # the program-size limit
    with pytest.raises(R.Error, match="exceeds size limit of 0 bytes"):
        R.BytesRegexSet([r"\w{100}"], size_limit=0)
    with pytest.raises(R.Error, match="word boundar"):
        R.RegexSet(w[:300] + [r"\bfoo\b"])


def model_matches(pats, groups, text, start, utf8, dfa_size_limit):
    cls = R.RegexSet if utf8 else R.BytesRegexSet
    acc = 0
    for lo, hi in groups:
        _, m = Sim(cls(pats[lo:hi], dfa_size_limit=dfa_size_limit)).forward_scan(text, start)
        acc |= m << lo
    return [i for i in range(len(pats)) if (acc >> i) & 1]


def test_model_on_golden_set_vectors():
    n = 0
    for x in vectors():
        if x["kind"] not in ("matset", "nomatset"):
            continue
        text = bytes.fromhex(x["text_hex"])
        for mode in x["modes"]:
            utf8 = mode == "str"
            pats = x["res"]
            try:
                s = (R.RegexSet if utf8 else R.BytesRegexSet)(pats)
            except R.Error as e:
                assert "word boundar" in str(e)
                continue
            for k in (1, 2):
                if k >= len(pats):
                    continue
                s.set_option("set_group_patterns", k)
                g = s.groups()
                assert len(g) == (len(pats) + k - 1) // k
                exp = O.OracleRegex(pats, only_utf8=utf8).set_matches(text)
                assert model_matches(pats, g, text, 0, utf8, 2 << 20) == exp, (x["name"], k)
                assert exp == x["expected"] or x["kind"] == "nomatset"
                n += 1
    assert n > 10


@pytest.mark.parametrize("utf8", [False, True])
def test_model_on_sherlock_slices(utf8):
    text = sherlock_text()
    cases = [(SET_PATTERNS, SMALL), (C.c4_patterns(), SMALL)]
    for pats, lim in cases:
        s = (R.RegexSet if utf8 else R.BytesRegexSet)(pats, dfa_size_limit=lim)
        g = s.groups()
        assert len(g) > 1
        o = O.OracleRegex(pats, only_utf8=utf8)
        for lo in (0, 20000, 300000):
            sl = text[lo:lo + 3000]
            for start in (0, 1, 17, 1500, len(sl)):
                assert model_matches(pats, g, sl, start, utf8, lim) == o.set_matches(sl, start), (lo, start)


@pytest.mark.parametrize("k", [0, 1, 5])
def test_forced_groups_on_empty_and_one_pattern_sets(k):
    """The golden set vectors include an empty set and one-pattern sets: the option applies to every set."""
    for cls in (R.BytesRegexSet, R.RegexSet):
        s = cls([])
        s.set_option("set_group_patterns", k)
        assert s.groups() == []
        s = cls(["a+"])
        s.set_option("set_group_patterns", k)
        assert s.groups() == [(0, 1)]
        s.dfa(R.DFA_FWD_UNANCHORED_ALL)  # one group is the product automaton
