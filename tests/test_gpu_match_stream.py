"""Match streams (include/rure_b200.h, Regex.match_stream / RegexSet.match_stream): is_match, shortest_match and
RegexSet matches over text written in pieces through a bounded device window must give exactly the resident answer on
the concatenation -- for single patterns, pattern groups, candidate-start patterns, matches across piece edges and str
mode with scalars split across writes -- and the forward host calls through the window (option "host_window") must
equal the resident calls."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import regex_b200 as R
from helpers import sherlock_text, tiled_corpus
from oracle import oracle as O
from test_gpu_candidate import PATTERNS as CAND_PATTERNS, _adversarial
from test_gpu_set_groups import SET_PATTERNS, make as make_set

pytestmark = pytest.mark.gpu

N = 12 << 20
PIECES = (1 << 20, 3 << 20)
WRITE_SIZES = [0, 1, 255, 257, 1 << 20, 3 << 20, 5 << 20]
SINGLE = [r"Holmes", r"[a-zA-Z]+ing", r"(?-u:\b)the(?-u:\b)", r"(?m)^\w+$", r"a*", r"", r"zqxwv"]


@pytest.fixture(scope="module")
def corpus():
    return tiled_corpus(N)


def _writes(data, rng, sizes=WRITE_SIZES):
    pos = 0
    while pos < len(data):
        k = int(rng.choice(sizes))
        yield data[pos:pos + k]
        pos += k


def _feed(s, data, seed, sizes=WRITE_SIZES):
    """Ragged writes (bytes and arrays), then finish; returns whether the stream was decided before finish."""
    rng = np.random.Generator(np.random.PCG64(seed))
    for i, w in enumerate(_writes(data, rng, sizes)):
        s.write(w if i % 3 else np.frombuffer(w, dtype=np.uint8))
    early = s.decided
    s.finish()
    assert s.decided
    return early


def _shortest(r, data, piece, seed, hold=0, sizes=WRITE_SIZES):
    with r.match_stream(piece=piece, hold=hold) as s:
        _feed(s, data, seed, sizes)
        assert s.found == (s.end is not None)
        return s.end


@pytest.mark.parametrize("utf8", [False, True])
def test_single_patterns(corpus, utf8):
    for pat in SINGLE:
        r = (R.Regex if utf8 else R.BytesRegex)(pat)
        exp = r.shortest_match(corpus)
        assert r.is_match(corpus) == (exp is not None)
        for j, piece in enumerate(PIECES):
            assert _shortest(r, corpus, piece, seed=31 * j + len(pat)) == exp, (pat, piece)


def test_against_oracle(corpus):
    prefix = corpus[:1 << 20]
    for pat in SINGLE:
        got = _shortest(R.BytesRegex(pat), prefix, 1 << 16, seed=5, sizes=[0, 1, 255, 257, 70000])
        assert got == O.OracleRegex(pat).shortest_match_at(prefix, 0), pat


def test_dead_state_decides_early(corpus):
    r = R.BytesRegex(r"^foo")
    with r.match_stream(piece=1 << 20) as s:
        s.write(corpus[:3 << 20])
        assert s.decided and not s.found
        searched = s.searched
        assert searched == 1 << 20  # the first piece took the automaton to the dead state
        s.write(corpus[3 << 20:])  # later writes succeed and search nothing
        assert s.searched == searched
        s.finish()
        assert not s.found and s.searched == searched


def test_end_of_text_step(corpus):
    data = corpus[:(3 << 20) - 3] + b"foo"
    r = R.BytesRegex(r"foo$")
    assert r.shortest_match(data) == len(data)
    with r.match_stream(piece=1 << 20) as s:
        s.write(data)
        assert not s.found and not s.decided
        s.finish()
        assert s.found and s.end == len(data)


def test_matches_across_piece_edges(corpus):
    piece = 1 << 20
    base = corpus[:5 << 20]
    for pat, m in ((r"zqxwvut", b"zqxwvut"), (r"(?-u:\b)zqxwvut(?-u:\b)", b" zqxwvut "), (r"(?m)zqxwvut$", b"zqxwvut\n")):
        r = R.BytesRegex(pat)
        for edge in (piece, 2 * piece, 3 * piece):
            for d in (-len(m) // 2, -1, 0, 1, -len(m), -len(m) + 1):
                buf = bytearray(base)
                buf[edge + d:edge + d + len(m)] = m
                data = bytes(buf)
                exp = r.shortest_match(data)
                assert exp is not None
                assert _shortest(r, data, piece, seed=edge + d) == exp, (pat, edge, d)


def test_str_mode_split_scalars():
    words = "Шерлок Холмс и доктор Ватсон — ёж, щука, яблоко. ".encode("utf-8")
    text = (words * ((6 << 20) // len(words) + 1))[: 6 << 20]
    text = text[: len(text) - len(text.split(b" ")[-1])] + "яблокож".encode("utf-8")
    for pat in (r"яблокож", r"\w+ж$", r"[а-я]+ож", r"Холмс"):
        r = R.Regex(pat)
        exp = r.shortest_match(text)
        assert exp is not None
        assert _shortest(r, text, 1 << 20, seed=7) == exp, pat  # odd write sizes split two-byte scalars


def _set_stream(s, data, piece, seed, masks):
    with s.match_stream(piece=piece, masks=masks) as st:
        early = _feed(st, data, seed)
        return (st.mask if masks else None), st.found, early


@pytest.mark.parametrize("name", ["product", "edge", "w257", "c4_small"])
def test_sets(corpus, name):
    if name == "product":
        s = R.BytesRegexSet(SET_PATTERNS)
        assert len(s.groups()) == 1
    else:
        s = make_set(name)[0]
    data = corpus[:6 << 20]
    exp_mask, exp_any = s.matches_mask(data), s.is_match(data)
    for j, piece in enumerate(PIECES):
        mask, found, _ = _set_stream(s, data, piece, seed=j, masks=True)
        assert mask == exp_mask, (name, piece)
        assert found == any(exp_mask)
        _, found, _ = _set_stream(s, data, piece, seed=j + 7, masks=False)
        assert found == exp_any, (name, piece)
    with s.match_stream(piece=1 << 20) as st:
        _feed(st, data, 3)
        assert st.matches == s.matches(data)


def test_set_decided_once_every_pattern_matched(corpus):
    s = R.BytesRegexSet(["Holmes", r"\w+", "Watson"])
    with s.match_stream(piece=1 << 20) as st:
        st.write(corpus[:3 << 20])
        assert st.decided and st.matches == [0, 1, 2]
        searched = st.searched
        assert searched < 3 << 20
        st.write(corpus[3 << 20:])
        assert st.searched == searched
        st.finish()
        assert st.matches == [0, 1, 2]
    with s.match_stream(piece=1 << 20, masks=False) as st:  # is_match: decided at the first match
        st.write(corpus[:3 << 20])
        assert st.decided and st.found


def _cand(pat, utf8=False, **opts):
    r = (R.Regex if utf8 else R.BytesRegex)(pat)
    r.set_option("prefilter", 0)
    r.set_option("candidate_starts", 1)
    for k, v in opts.items():
        r.set_option(k, v)
    return r


def test_candidate_patterns(corpus):
    small = [0, 1, 255, 257, 5000]
    for pat in CAND_PATTERNS:
        r = _cand(pat)
        adversarial = _adversarial(pat)[len(CAND_PATTERNS[pat]) + 1:]  # without the match at 0: the first ones lie at piece edges
        for name, text in (("sherlock", sherlock_text()), ("adversarial", adversarial), ("corpus", corpus)):
            exp = r.shortest_match(text)
            pieces = PIECES if name == "corpus" else (4096, 1 << 16)
            for j, piece in enumerate(pieces):
                got = _shortest(r, text, piece, seed=j, sizes=WRITE_SIZES if name == "corpus" else small)
                assert got == exp, (pat, name, piece)
            if name == "adversarial":
                o = O.OracleRegex(pat)
                for d in (4096, 8192, 12288):  # prefixes ending at the planted edges
                    assert _shortest(r, text[:d + 5], 4096, seed=d, sizes=small) == o.shortest_match_at(text[:d + 5], 0), (pat, d)


def test_candidate_bound_past_piece_end():
    """The candidate at 4000 ends at 4201, past the first piece; the one at 4100 ends earlier, in the next piece."""
    text = b"0" * 4000 + b"a" + b"x" * 99 + b"c" + b"x" * 100 + b"z" + b"0" * 5000
    r = _cand(r"a[a-z]*z|c")
    assert r.shortest_match(text) == 4101
    assert _shortest(r, text, 4096, seed=1, sizes=[0, 1, 255, 257, 5000]) == 4101


def test_candidate_lookahead_regrowth_and_hold():
    # one candidate (the x; every letter of the run would be one for `[a-z]+...`, each running to the same end)
    text = b"0" * 4000 + b"x" + b"a" * 200_000 + b"ing" + b"0" * 600_000
    r = _cand(r"x[a-z]+.{0,30}ing")
    exp = r.shortest_match(text)
    assert exp == 4001 + 200_000 + 3
    # look-ahead 64 KiB, then 512 KiB: the run from the first piece reaches the window's end undecided once, and the
    # end found past the piece is the bound the later pieces keep
    with r.match_stream(piece=4096, hold=1 << 20) as s:
        for k in range(0, len(text), 70_000):
            s.write(text[k:k + 70_000])
        assert s.decided and s.end == exp
        s.finish()
        assert s.end == exp
    with r.match_stream(piece=4096, hold=1 << 16) as s:
        with pytest.raises(R.Error, match=r"a match is longer than the stream window \(65536 bytes\)"):
            s.write(text)
        with pytest.raises(R.Error):
            s.write(b"more")  # a failed stream stays failed


def _starts(text):
    mid = text.index(b"\n", len(text) // 2) - 7  # inside a line
    return [0, 1, 17, mid, len(text)]


def test_host_window_equals_resident(corpus):
    data = corpus[:(10 << 20) + 123]
    lib = R.lib()
    for pat in (r"Holmes", r"[a-zA-Z]+ing", r"(?m)^\w+$", r"zqxwv", r"^foo", r"Holmes.{0,40}Watson"):
        r = R.BytesRegex(pat)
        if pat == r"Holmes.{0,40}Watson":
            r.set_option("candidate_starts", 1)
        exp = [(r.is_match_at(data, s), r.shortest_match_at(data, s)) for s in _starts(data)]
        exp_c = lib.rure_is_match(r._h, data, len(data), 0)
        r.set_option("host_window", 4 << 20)  # pieces and hold of 512 KiB
        assert [(r.is_match_at(data, s), r.shortest_match_at(data, s)) for s in _starts(data)] == exp, pat
        assert r.is_match(data) == exp[0][0] and r.shortest_match(data) == exp[0][1]
        assert lib.rure_is_match(r._h, data, len(data), 0) == exp_c
        assert r.last_stats()["waves"] >= 1
    for s, name in ((R.BytesRegexSet(SET_PATTERNS), "product"), (make_set("edge")[0], "edge")):
        n_pat = len(s)
        exp = [(s.is_match(data, st), s.matches(data, st)) for st in _starts(data)]
        s.set_option("host_window", 4 << 20)
        try:
            assert [(s.is_match(data, st), s.matches(data, st)) for st in _starts(data)] == exp, name
            out = (ctypes.c_bool * n_pat)()
            assert lib.rure_set_matches(s._h, data, len(data), 0, out) == bool(exp[0][1])
            assert [i for i in range(n_pat) if out[i]] == exp[0][1]
        finally:
            s.set_option("host_window", 0)


def test_early_exit_stops_feeding(corpus):
    """A match near the front: the host call through the window searches one piece, not the whole text."""
    data = b"Holmes" + corpus[:8 << 20]
    r = R.BytesRegex(r"Holmes")
    r.set_option("host_window", 1 << 20)
    assert r.shortest_match(data) == 6
    assert r.last_stats()["waves"] == 1


def test_errors():
    r = R.BytesRegex(r"a+")
    with r.match_stream() as s:
        s.write(b"")  # zero-length write
        s.write(b"xx aa")
        s.finish()
        assert s.found and s.end == 4 and s.decided
        with pytest.raises(R.Error, match="write after finish"):
            s.write(b"a")
    for pat, exp in ((r"zqj", None), (r"", 0), (r"a*", 0)):
        with R.BytesRegex(pat).match_stream() as s:  # empty text
            s.finish()
            assert s.decided and s.end == exp
    with R.BytesRegexSet([r"a", r"b"]).match_stream() as s:
        s.finish()
        assert s.matches == [] and not s.found
    with R.BytesRegexSet([]).match_stream() as s:
        assert s.decided
        s.write(b"abc")
        s.finish()
        assert s.matches == []


def test_set_stream_c_example(corpus, tmp_path):
    """tests/capi/set_stream.c: fread in 1 MiB blocks into a set match stream, strict ANSI C."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_dir = os.path.join(root, "regex_b200")
    exe = str(tmp_path / "set_stream_example")
    subprocess.check_call(["gcc", "-ansi", "-Wall", "-Werror", os.path.join(root, "tests", "capi", "set_stream.c"), "-I" + os.path.join(root, "include"),
                           "-L" + lib_dir, "-lrure_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    path = tmp_path / "hay.txt"
    data = corpus[:5 << 20]
    path.write_bytes(data)
    for pats in (SET_PATTERNS, ["Holmes", r"\w+", "Watson"]):
        out = subprocess.run([exe, str(path), *pats], capture_output=True, text=True, timeout=300, check=True).stdout.split()
        assert [int(x) for x in out] == R.BytesRegexSet(pats).matches(data), pats
