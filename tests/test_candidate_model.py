"""CPU model of candidate-start mode (DESIGN.md §2), walked on the product's exported tables.

Patterns whose unanchored automata exceed the table budget compile to the anchored automata only (kinds 0 and 3).
Every search then runs from candidate starts: positions whose first min(min_len, 4) bytes lie in the byte sets of
the anchored automaton.  find_at(p) = (s*, A(s*)), s* = the first candidate >= p at which the anchored automaton A
finds a match (with look-arounds the start comes from the reverse-on-slice rule); shortest_match = the least first
match end over the candidates >= start.  The model states those rules once more and is compared with the oracle."""
import numpy as np
import pytest

import regex_b200 as R
from dfa_sim import Sim, flags_forward
from helpers import xorshift_bytes
from oracle import oracle as O

OVER_BUDGET = [r"error.{0,100}timeout", r"(?i)warn.{0,64}disk", r"user=\w+.{0,50}failed", r"Holmes.{0,40}Watson",
               r"[a-z]+.{0,30}ing", r"a.{20}b", r"[A-Z][a-z]+ [A-Z][a-z]+.{0,80}said", r"[a-q][^u-z]{13}x",
               r"(?-u:\b)error(?-u:\b).{0,60}timeout", r"(a.{20}b)?"]
_CACHE = {}


def _re(pat, utf8):
    if (pat, utf8) not in _CACHE:
        _CACHE[(pat, utf8)] = (R.Regex if utf8 else R.BytesRegex)(pat)
    return _CACHE[(pat, utf8)]


@pytest.mark.parametrize("utf8", [False, True])
def test_over_budget_patterns_compile_to_the_anchored_automata(utf8):
    for pat in OVER_BUDGET:
        r = _re(pat, utf8)
        r.dfa(R.DFA_FWD_ANCHORED_LF)
        r.dfa(R.DFA_REV_ANCHORED_LONGEST)
        for kind in (R.DFA_REV_UNANCHORED_ALL, R.DFA_FWD_UNANCHORED_ALL, R.DFA_FWD_UNANCHORED_LF):
            with pytest.raises(R.Error, match="candidate starts"):
                r.dfa(kind)


def test_budget_errors_that_stay():
    with pytest.raises(R.Error, match="exceeds size limit"):
        R.BytesRegex(r"[ab]*a[ab]{14}", dfa_size_limit=1024)  # kind 0 is over the budget too
    with pytest.raises(R.Error, match="exceeds size limit"):
        R.BytesRegexSet([r"error.{0,100}timeout", r"x"])  # set semantics need the all-match product automaton
    r = R.BytesRegex(r"(?m)^.{0,20}x$")  # fits: every kind is there
    for kind in range(5):
        r.dfa(kind)


class CandModel:
    def __init__(self, regex):
        self.sim = Sim(regex)
        self.d0 = self.sim.d(R.DFA_FWD_ANCHORED_LF)
        info = regex.pattern_info()
        self.looks, self.empty = info["has_looks"], info["can_match_empty"]
        self.depth = min(info["min_len"], 4)
        self.utf8 = self.sim.utf8
        d = self.d0
        trans, classes = d["trans"], d["classes"]
        starts = {int(d["start"][32])} if d["uniform_start"] else {int(s) for s in d["start"]}
        reach = np.zeros(trans.shape[0], dtype=bool)
        reach[list(starts)] = True
        reach[0] = False
        self.sets = []
        for _ in range(self.depth):  # bytes with which some start state survives d + 1 steps
            live = trans[reach][:, classes] != 0  # [reached states][256 bytes]
            self.sets.append(live.any(axis=0))
            nxt = np.zeros_like(reach)
            nxt[np.unique(trans[reach][:, classes][live])] = True
            nxt[0] = False
            reach = nxt

    def cand(self, t, s):
        n = len(t)
        if any(s + d >= n or not self.sets[d][t[s + d]] for d in range(self.depth)):
            return False
        return not (self.utf8 and self.empty and s < n and (t[s] & 0xC0) == 0x80)

    def first_end(self, t, s):
        d, n = self.d0, len(t)
        st = int(d["start"][flags_forward(t, s)])
        q = s
        while st != 0:
            st = self.sim.step(d, st, t[q]) if q < n else self.sim.eof(d, st)
            if st >= d["match_lo"]:
                return q
            if q >= n:
                break
            q += 1
        return None

    def find_at(self, t, p):
        for s in range(p, len(t) + 1):
            if self.cand(t, s):
                e = self.sim.anchored_end(t, s)
                if e is not None:
                    return s, e
        return None

    def find_iter(self, t):
        out, p, lm = [], 0, None
        while p <= len(t):
            m = self.find_at(t, p)
            if m is None:
                break
            s, e = m
            if self.looks and e != p:
                s = self.sim.slice_start(t, p, e)
                if s is None:
                    break
            if s == e:
                p = self.sim.next_after_empty(t, e)
                if e == lm:
                    continue
            else:
                p = e
            lm = e
            out.append((s, e))
        return out

    def shortest_match_at(self, t, start):
        best = None
        for s in range(start, len(t) + 1):
            if best is not None and s >= best:
                break
            if any(s + d >= len(t) or not self.sets[d][t[s + d]] for d in range(self.depth)):
                continue
            e = self.first_end(t, s)
            if e is not None and (best is None or e < best):
                best = e
        return best


def _haystacks(seed):
    alpha = b"errortimeoutWARNdiskuser=failedHolmesWatsonSaidingabxX \n"
    out = [b"", b"a" + b"z" * 20 + b"b", xorshift_bytes(seed, 3000, alpha)]
    planted = bytearray(xorshift_bytes(seed + 1, 2500, alpha))
    for at, m in ((0, b"error then timeout"), (700, b"Holmes met Watson"), (1300, b"user=bob x failed"), (1900, b"warn: DISK")):
        planted[at:at + len(m)] = m
    out.append(bytes(planted) + b"a" + b"q" * 20 + b"b")
    if seed % 2:
        out.append("naïve café — warn ☃ disk ing".encode() * 20)
    return out


@pytest.mark.parametrize("utf8", [False, True])
def test_model_equals_oracle(utf8):
    for i, pat in enumerate(OVER_BUDGET + [r"(?m)^.{0,20}x$", r"x{0,3}(?-u:\b)", r"(?-u:\B)[a-z]{2}.{0,5}"]):
        r = _re(pat, utf8) if pat in OVER_BUDGET else (R.Regex if utf8 else R.BytesRegex)(pat)
        m, o = CandModel(r), O.OracleRegex(pat, only_utf8=utf8)
        for t in _haystacks(i):
            if utf8:
                try:
                    t.decode()
                except UnicodeDecodeError:
                    continue
            assert m.find_iter(t) == o.find_iter(t), (pat, utf8, t[:30])
            for start in sorted({0, min(1, len(t)), len(t) // 3, len(t)}):
                assert m.shortest_match_at(t, start) == o.shortest_match_at(t, start), (pat, utf8, start)
                assert (m.shortest_match_at(t, start) is not None) == o.is_match_at(t, start), (pat, utf8, start)
