"""CPU model of the per-record find_iter of the batch_iter kernels, walked on the product's exported tables.

Each record is its own haystack: from p, the end of the leftmost-first match (forward unanchored
leftmost-first automaton, start state by the flags at p), its start by the reverse longest automaton over
the slice [p..] (so p is judged as beginning of text), then the empty-match rule of the reference
iterator (re_trait.rs:197-220).  The model states those steps once more, on the tables the kernels read,
and is compared record by record with the oracle's find_iter.  It also checks the count-pass shortcut of
the kernels: a pattern that cannot match empty and has no look-around is counted by the forward automaton
alone (p = e after every match)."""
import numpy as np

import regex_b200 as R
from dfa_sim import Sim, flags_forward
from helpers import vectors, xorshift_bytes
from oracle import oracle as O
from test_fuzz_tables_vs_oracle import _pattern


def _forward_end(sim, t, p):
    d = sim.d(R.DFA_FWD_UNANCHORED_LF)
    n = len(t)
    st = int(d["start"][flags_forward(t, p)])
    e, q = None, p
    while st != 0:
        st = sim.step(d, st, t[q]) if q < n else sim.eof(d, st)
        if st >= d["match_lo"]:
            e = q
        if q >= n:
            break
        q += 1
    return e


def iter_record(sim, t):
    out, p, lm, n = [], 0, None, len(t)
    while p <= n:
        e = _forward_end(sim, t, p)
        if e is None:
            break
        s = p if e == p else sim.slice_start(t, p, e)
        if s is None:
            break
        if s == e:
            p = sim.next_after_empty(t, e)
            if e == lm:
                continue
        else:
            p = e
        lm = e
        out.append((s, e))
    return out


def count_forward_only(sim, t):
    k, p, n = 0, 0, len(t)
    while p <= n:
        e = _forward_end(sim, t, p)
        if e is None:
            break
        k += 1
        p = e
    return k


def _check(r, o, records, utf8):
    sim = Sim(r)
    info = r.pattern_info()
    shortcut = not info["can_match_empty"] and not info["has_looks"]
    for t in records:
        if utf8:
            try:
                t.decode()
            except UnicodeDecodeError:
                continue
        got = iter_record(sim, t)
        assert got == o.find_iter(t), (r.pattern, utf8, t)
        if shortcut:
            assert count_forward_only(sim, t) == len(got), (r.pattern, utf8, t)
    return shortcut


def test_model_on_matiter_vectors():
    n = 0
    for x in vectors():
        if x["kind"] != "matiter":
            continue
        text = bytes.fromhex(x["text_hex"])
        for mode in x["modes"]:
            utf8 = mode == "str"
            try:
                r = (R.Regex if utf8 else R.BytesRegex)(x["re"])
            except R.Error as e:
                assert "word boundar" in str(e), (x["name"], str(e))
                continue
            assert iter_record(Sim(r), text) == [tuple(s) for s in x["expected"]], (x["name"], mode)
            # the same text cut into records: every record is its own haystack
            _check(r, O.OracleRegex(x["re"], only_utf8=utf8), [text[:i] for i in range(len(text) + 1)][-3:] + text.split(b"\n"), utf8)
            n += 1
    assert n > 70, n


RECORDS = [b"", b"a", b"\n", b"ab c\n", b"abc abc ab\n", b"  a b  \n", "aé αβ b\n".encode(), "x αβγ1".encode(), b"ab\xff\xc3a\xa9 b",
           xorshift_bytes(3, 40, b"abc \n"), xorshift_bytes(4, 33, b"ab1 _\n"), b"a" * 17, b"b" * 16 + b"a", "aδ☃𝄞b".encode()]


def test_model_on_random_patterns():
    rng = np.random.Generator(np.random.PCG64(0xBA7C4))
    cases = shortcuts = 0
    for _ in range(240):
        p = _pattern(rng)
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            try:
                r = cls(p)
            except R.Error:
                continue
            shortcuts += _check(r, O.OracleRegex(p, only_utf8=utf8), RECORDS, utf8)
            cases += 1
    assert cases > 300 and shortcuts > 30, (cases, shortcuts)


def test_model_on_log_line_patterns():
    lines = [b"2014-01-02 host-0001 svc[12]: reading the file\n", "٢٠١٤-٠١-٠٢ arabic\n".encode(), b"", b"\xff\xfe 2001-02-03 \xc3\n",
             b"x" * 15 + b"2020-10-10", b"no newline 2030-01-01"]
    for pat in [r"(\d{4})-(\d{2})-(\d{2})", r"[a-z]+ing", r"\w+", r"", r"a*", r"\s*", r"(?m)^\w+", r"\w+$", r"(?-u:\b)\d{2}(?-u:\b)",
                r"^[ab]{2,}\w*?|(?m:$)"]:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            _check(cls(pat), O.OracleRegex(pat, only_utf8=utf8), lines, utf8)
