"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU
oracle and the committed golden vectors.  Bit-exact: spans, counts, masks are integers."""
import os

import numpy as np
import pytest

import regex_b200 as R
from helpers import GOLDEN, sherlock_counts, sherlock_text, tiled_corpus, vectors, xorshift_bytes
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _spans(a):
    return [tuple(int(v) for v in r) for r in np.asarray(a).reshape(-1, 2).tolist()]


# ------------------------------------------------------------ golden vectors --
def test_reference_vectors_through_c_abi():
    """tests/*.rs vectors via rure_find / find_iter / rure_is_match / rure_shortest_match /
    rure_set_matches on the GPU.  Unicode-\\b patterns must raise the explicit error."""
    bad, n, unsupported = [], 0, 0
    for x in vectors():
        text = bytes.fromhex(x["text_hex"])
        for mode in x["modes"]:
            utf8 = mode == "str"
            try:
                if x["kind"] in ("matset", "nomatset"):
                    s = (R.RegexSet if utf8 else R.BytesRegexSet)(x["res"])
                    got = s.matches(text)
                    assert s.is_match(text) == bool(got)
                else:
                    r = (R.Regex if utf8 else R.BytesRegex)(x["re"])
                    if x["kind"] == "mat":
                        got = r.find(text)
                        got = list(got) if got else None
                        assert r.is_match(text) == (got is not None)
                        assert (r.shortest_match(text) is not None) == (got is not None)
                        found, spans = r.find_batch(text, [0, len(text)])
                        assert (list(map(int, spans[0])) if found[0] else None) == got, ("batch", x["name"])
                    elif x["kind"] == "matiter":
                        got = [list(t) for t in r.find_iter(text)]
                    elif x["kind"] == "ismatch":
                        got = r.is_match(text)
                    elif x["kind"] == "shortmat":
                        got = r.shortest_match(text)
            except R.Error as e:
                assert "word boundar" in str(e), (x["name"], str(e))
                unsupported += 1
                continue
            n += 1
            if got != x["expected"]:
                bad.append((x["file"], x["name"], mode, x["expected"], got))
    assert n > 1000
    assert not bad, bad[:10]


def test_misc_is_match_known_answers():
    """bench/src/misc.rs is_match expectations through the C ABI (str Regex); a pattern whose
    DFA exceeds the budget must say so instead of answering."""
    from helpers import misc_is_match
    answered = 0
    for name, pat, expected, hay in misc_is_match():
        try:
            r = R.Regex(pat)
        except R.Error as e:
            assert "exceeds size limit" in str(e), (name, e)
            continue
        assert r.is_match(hay) == expected, name
        assert (r.shortest_match(hay) is not None) == expected, name
        assert (r.find(hay) is not None) == expected, name
        answered += 1
    assert answered >= 30


def test_sherlock_counts_and_spans():
    """bench/src/sherlock.rs counts + full span parity with the oracle."""
    text = sherlock_text()
    for x in sherlock_counts():
        try:
            r = R.Regex(x["re"])
        except R.Error as e:
            # the two explicit errors of this backend (north star): Unicode \b, and the
            # one bench pattern whose DFA blows up ([a-q][^u-z]{13}x: 73k states > u16 ids)
            assert "word boundar" in str(e) or (x["name"] == "repeated_class_negation" and "exceeds size limit" in str(e))
            continue
        got = r.find_all(text)
        assert len(got) == x["count"], x
        exp = O.OracleRegex(x["re"], only_utf8=True).find_iter(text)
        assert _spans(got) == exp, x["name"]


def test_regexdna_shootout():
    seq = open(os.path.join(GOLDEN, "regexdna-input.txt"), "rb").read()
    expect = open(os.path.join(GOLDEN, "regexdna-output.txt")).read().split("\n")
    spans = _spans(R.Regex(r">[^\n]*\n|\n").find_all(seq))
    out, last = [], 0
    for s, e in spans:
        out.append(seq[last:s])
        last = e
    out.append(seq[last:])
    clean = b"".join(out)
    assert len(clean) == int(expect[11])
    for i in range(9):
        name, count = expect[i].rsplit(" ", 1)
        assert R.Regex(name).count_all(clean) == int(count), name


# ---------------------------------------------------------- chunk boundaries --
PATTERNS_STRESS = [
    r"[a-zA-Z]+ing", r"Holmes|Watson", r"\w+", r"the\s+\w+", r"(?i)sherlock|holmes|watson", r"a", r"aa", r"aaa",
    r"[a-z]*", r"\s*", r"", r"(?m)^\w+", r"(?m)\w+$", r"(?m)^$", r"(?-u:\b)\w+(?-u:\b)", r"(?-u:\B)[a-z]",
    r"[a-z ]{0,12}Holmes", r"[^\n]*", r".*", r"e[a-z ]{2,6}?a", r"\p{Lu}\p{Ll}+",
]


@pytest.mark.parametrize("generic", [False, True], ids=["fast", "generic"])
@pytest.mark.parametrize("seg,chunk,warm", [(64, 64, 16), (128, 64, 0), (64, 256, 64), (0, 4096, 0)])
def test_small_segments_force_boundary_logic(seg, chunk, warm, generic):
    """Tiny segments/chunks put a boundary inside almost every match: exercises the
    warm-up verification, redo rounds and chain stitching."""
    text = sherlock_text()[:20000] + b"aaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaa" * 20
    for pat in PATTERNS_STRESS:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            r = cls(pat)
            r.set_tuning(seg=seg, chunk=chunk, warm=warm)
            r.force_generic(generic)
            got = _spans(r.find_all(text))
            exp = O.OracleRegex(pat, only_utf8=utf8).find_iter(text)
            assert got == exp, (pat, utf8, seg, chunk, got[:5], exp[:5])
            for cut in (63, 64, 65, 1000):  # ragged ends / tiny haystacks through the same kernels
                assert _spans(r.find_all(text[:cut])) == O.OracleRegex(pat, only_utf8=utf8).find_iter(text[:cut]), (pat, cut)


@pytest.mark.parametrize("seg", [0, 64, 256])
def test_unicode_classes_hot_table_and_cold_fallback(seg):
    """Unicode-aware classes compile to hundreds of DFA states of which ASCII text visits a
    handful: the fast kernels keep those hot rows in shared memory and a lane that meets
    a byte outside the hot set (multi-byte UTF-8, invalid bytes) redoes the group on the
    full table.  Mixed text makes lanes leave and re-enter the hot set all the time."""
    ascii_part = sherlock_text()[:6000]
    mixed = ("naïve café über straße Ωμέγα привет мир 日本語のテキスト ２０１４ ٣٤ x²+y² ".encode("utf-8")) * 8
    junk = bytes([0xFF, 0xC3, 0x28, 0xE2, 0x82, 0x41, 0xF0, 0x9F, 0x98, 0x80, 0x80, 0xBF]) * 5
    rng = np.random.Generator(np.random.PCG64(0x4807))
    parts = []
    for _ in range(60):
        o = int(rng.integers(0, len(ascii_part) - 400))
        parts.append(ascii_part[o:o + int(rng.integers(1, 400))])
        parts.append(mixed[int(rng.integers(0, 40)):][:int(rng.integers(1, 120))] if rng.random() < 0.7 else junk[:int(rng.integers(1, 30))])
    text_bytes = b"".join(parts)
    text_str = (ascii_part[:3000].decode("latin-1") + mixed.decode("utf-8") * 2 + ascii_part[3000:5000].decode("latin-1")).encode("utf-8")
    pats = [r"\w+", r"the\s+\w+", r"\d+", r"(\d{4})-(\d{2})-(\d{2})", r"\pL+ing", r"[^\s]+\s", r"(?i)sher\w*", r"\w+\s*[,.]"]
    for pat in pats:
        for cls, utf8, text in ((R.BytesRegex, False, text_bytes), (R.Regex, True, text_str)):
            r = cls(pat)
            if seg:
                r.set_tuning(seg=seg, chunk=max(seg, 256), warm=0)
            exp = O.OracleRegex(pat, only_utf8=utf8).find_iter(text)
            got = _spans(r.find_all(text))
            assert got == exp, (pat, utf8, seg, got[:5], exp[:5])
            r.force_generic(True)
            assert _spans(r.find_all(text)) == exp, (pat, utf8, "generic")


@pytest.mark.parametrize("k", [25, 40, 60])
def test_word_alternations_mid_size_tables(k):
    """Alternations of k frequent words: 86 / 126 / 188 reverse-DFA states.  These sit on the
    shared-memory hot path with one-byte state ids above 127 (k = 60) and, from k = 40 on,
    with tables too large to share the CTA with a fused walk (separate walk kernel)."""
    from collections import Counter
    text = sherlock_text()[:300000]
    words = [w.decode() for w in sherlock_text().split() if w.isalpha() and len(w) >= 4]
    top = [w for w, _ in Counter(words).most_common(400)]
    pat = "|".join(top[10:10 + k])
    exp = O.OracleRegex(pat).find_iter(text)
    r = R.BytesRegex(pat)
    assert _spans(r.find_all(text)) == exp
    lines = text.split(b"\n")[:2000]
    off = np.concatenate([[0], np.cumsum([len(l) for l in lines])]).astype(np.uint64)
    found, spans = r.find_batch(b"".join(lines), off)
    o = O.OracleRegex(pat)
    for i, l in enumerate(lines):
        m = o.find_at(l)
        assert bool(found[i]) == (m is not None), i
        if m:
            assert tuple(int(v) for v in spans[i]) == m, i
    r.force_generic(True)
    assert _spans(r.find_all(text)) == exp


def test_forward_scan_fast_path_shortest_match():
    """Whole-haystack is_match / shortest_match: scan_fwd_fast (hot table + TMA ring) for the
    full segments, scan_fwd_reduce for the edges and the EOF step; match placed early, late,
    across segment boundaries, only at EOF, and after non-ASCII bytes (cold fallback)."""
    base = sherlock_text()[:400000].replace(b"Watson", b"W4tson").replace(b"ing", b"1ng")
    cases = []
    for pos in (0, 63, 4095, 4096, 4097, 131072 - 3, 250000, len(base) - 6):
        t = bytearray(base)
        t[pos:pos + 6] = b"Watson"
        cases.append(bytes(t))
    cases.append(base)                                   # no match at all
    cases.append(base + b"Watson")                       # match ends exactly at EOF
    cases.append(base[:200000] + "ünï 日本 ".encode() * 50 + base[200000:300000] + b"xx Watson yy")
    pats = ["Watson", r"Wat\w+", r"[a-zA-Z]+ing", r"Watson$", r"(?m)^Watson", r"\w+son\s", r"W.{2,5}n"]
    for text in cases:
        for pat in pats:
            o = O.OracleRegex(pat)
            for cls in (R.BytesRegex,):
                r = cls(pat)
                for start in (0, 64, 4096, 199936):
                    exp = o.shortest_match_at(text, start)
                    assert r.shortest_match_at(text, start) == exp, (pat, start, exp)
                    assert r.is_match_at(text, start) == (exp is not None), (pat, start)
                r.force_generic(True)
                assert r.shortest_match(text) == o.shortest_match_at(text, 0), (pat, "generic")


def test_random_patterns_vs_oracle():
    """Seeded fuzz over a small regex grammar on a 4-letter alphabet (dense matches)."""
    rng = np.random.Generator(np.random.PCG64(0xB200))
    atoms = ["a", "b", "c", "d", "[ab]", "[^a]", ".", "(?:ab|c)", "a*", "b+", "c?", "(?:a|bc)*", "d{2,3}", "[a-c]{1,2}?"]
    text = xorshift_bytes(7, 5000, b"abcd\n")
    for it in range(120):
        k = int(rng.integers(1, 5))
        pat = "".join(atoms[int(i)] for i in rng.integers(0, len(atoms), size=k))
        if rng.random() < 0.3:
            pat = pat + "|" + "".join(atoms[int(i)] for i in rng.integers(0, len(atoms), size=2))
        if rng.random() < 0.15:
            pat = "(?m)^" + pat
        if rng.random() < 0.15:
            pat = pat + "$"
        r = R.BytesRegex(pat)
        r.set_tuning(seg=64, chunk=128, warm=0)
        exp = O.OracleRegex(pat, only_utf8=False).find_iter(text)
        assert _spans(r.find_all(text)) == exp, pat
        assert r.shortest_match(text) == O.OracleRegex(pat).shortest_match_at(text), pat


def test_find_at_and_iter_offsets():
    text = b"xx 2014-01-02 yy 2015-12-31 zz"
    r = R.BytesRegex(r"(\d{4})-(\d{2})-(\d{2})")
    o = O.OracleRegex(r"(\d{4})-(\d{2})-(\d{2})")
    for start in range(len(text) + 2):
        assert r.find_at(text, start) == o.find_at(text, start), start
        assert r.is_match_at(text, start) == o.is_match_at(text, start) if start <= len(text) else True
        assert r.shortest_match_at(text, start) == o.shortest_match_at(text, start) if start <= len(text) else True


def test_empty_and_tiny_haystacks():
    for pat in [r"", r"a", r"a*", r"^", r"$", r"^$", r"(?m)^", r"\s*"]:
        for text in [b"", b"a", b"\n", b"ab"]:
            for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
                r, o = cls(pat), O.OracleRegex(pat, only_utf8=utf8)
                assert _spans(r.find_all(text)) == o.find_iter(text), (pat, text)
                assert r.is_match(text) == o.is_match_at(text), (pat, text)
                assert r.shortest_match(text) == o.shortest_match_at(text), (pat, text)


def test_utf8_empty_matches_step_by_scalar():
    text = "aδ☃𝄞b".encode()
    for pat in [r"", r"x*", r"(?-u:\B)"]:
        assert _spans(R.Regex(pat).find_all(text)) == O.OracleRegex(pat, only_utf8=True).find_iter(text), pat
        assert _spans(R.BytesRegex(pat).find_all(text)) == O.OracleRegex(pat, only_utf8=False).find_iter(text), pat


# -------------------------------------------------------------------- batch ----
def _log_lines(n, seed=0x5EED0003):
    rng = np.random.Generator(np.random.PCG64(seed))
    words = [w for w in set(sherlock_text()[:200000].split()) if w.isalpha()][:500]
    lines = []
    for i in range(n):
        if rng.random() < 0.7:
            ts = f"{rng.integers(1990, 2030):04d}-{rng.integers(1, 13):02d}-{rng.integers(1, 29):02d}T{rng.integers(0, 24):02d}:00:00Z"
        else:
            ts = str(int(rng.integers(10**9, 2 * 10**9)))
        msg = b" ".join(words[int(j)] for j in rng.integers(0, len(words), size=int(rng.integers(3, 13))))
        lines.append(f"{ts} host-{rng.integers(0, 10000):04d} svc[{rng.integers(1, 65536)}]: ".encode() + msg + b"\n")
    return lines


def test_batched_lines_match_scalar_api():
    lines = _log_lines(3000)
    lines[17] = b""  # empty record
    # records that leave the hot (ASCII-reachable) part of Unicode-class tables, short
    # records, and records shorter / longer than the 16-byte window of batch_fast
    lines[0] = b"2014-01-02"
    lines[1] = "٢٠١٤-٠١-٠٢ arabic-indic digits are \\d too\n".encode()
    lines[2] = "naïve 1999-12-31 café\n".encode()
    lines[3] = b"\xff\xfe 2001-02-03 \xc3\n"
    lines[4] = b"7"
    lines[5] = b"x" * 15 + b"2020-10-10"
    lines[6] = b"x" * 16 + b"2020-10-10" + b"y" * 33
    lines[-1] = b"no newline at the very end 2030-01-01"
    text = b"".join(lines)
    off = np.concatenate([[0], np.cumsum([len(l) for l in lines])]).astype(np.uint64)
    for pat in [r"(\d{4})-(\d{2})-(\d{2})", r"(?-u)(\d{4})-(\d{2})-(\d{2})", r"^\d+ host", r"svc\[\d+\]:$", r"(?i)holmes", r"\n$",
                r"\w+\s\w+$", r"(?-u:\b)\d{2}(?-u:\b)", r"^$", r"[a-z]+ing"]:
        o = O.OracleRegex(pat)
        # batch_fast (one record per lane per round), batch_refill for is_match (1 the default, 2 whatever the batch size), generic
        for generic, refill in ((False, 1), (False, 0), (False, 2), (True, 1)):
            r = R.BytesRegex(pat)
            r.force_generic(generic)
            r.set_option("batch_refill", refill)
            m = r.is_match_batch(text, off)
            found, spans = r.find_batch(text, off)
            for i, l in enumerate(lines):
                exp = o.find_at(l)
                assert bool(m[i]) == (exp is not None), (pat, i, generic, refill)
                assert bool(found[i]) == (exp is not None), (pat, i, generic, refill)
                if exp:
                    assert tuple(int(v) for v in spans[i]) == exp, (pat, i, generic, refill)


SET_PATTERNS = [r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+", "Holmes", "Watson", "Sherlock", r"Holmes|Watson", r"^The", r"\.$",
                r"(?m)^$", r"[0-9]{4}", r"(?i)holmes", "zqj", r"[a-z]+ing", r"\bnever\b".replace(r"\b", r"(?-u:\b)")]


def test_regex_set_whole_and_batched():
    text = sherlock_text()[:50000]
    s = R.BytesRegexSet(SET_PATTERNS)
    s.set_tuning(seg=128, warm=0)
    o = O.OracleRegex(SET_PATTERNS)
    assert s.matches(text) == o.set_matches(text)
    assert s.is_match(text)
    lines = [l + b"\n" for l in text.split(b"\n")][:800]
    body = b"".join(lines)
    off = np.concatenate([[0], np.cumsum([len(l) for l in lines])]).astype(np.uint64)
    masks = s.matches_batch(body, off)
    for i, l in enumerate(lines):
        exp = sum(1 << j for j in o.set_matches(l))
        assert int(masks[i, 0]) == exp, (i, l)


def test_regex_set_more_than_64_patterns():
    pats = [f"w{i}x" for i in range(70)] + [r"\d+"]
    s = R.BytesRegexSet(pats)
    text = b"w3x w69x 12 w70x"
    assert s.matches(text) == [3, 69, 70]


# ------------------------------------------------------- size-independent props --
def test_large_haystack_properties():
    """256 MiB tiled corpus on device: count equals the sum over an independent split at
    line boundaries (matches cannot span '\\n' for these patterns), spans are sorted,
    non-overlapping and every span re-matches when checked by the oracle on a sample."""
    import torch
    base = tiled_corpus(1 << 24)
    reps = 16
    d = torch.frombuffer(bytearray(base), dtype=torch.uint8).cuda().repeat(reps)
    n = d.numel()
    for pat in [r"[a-zA-Z]+ing", r"Holmes|Watson", r"the\s+\w+"]:
        r = R.BytesRegex(pat)
        base_spans = O.OracleRegex(pat).find_iter(base)
        # base ends at an arbitrary byte; compare on the device against the oracle of the first copy
        out = torch.empty((len(base_spans) * reps + 1024, 2), dtype=torch.int64, device="cuda")
        total = r.find_all_device(d, out)
        got = out[:total].cpu().numpy()
        assert (got[:, 0] < got[:, 1]).all() and (got[1:, 0] >= got[:-1, 1]).all()
        first = got[got[:, 1] <= len(base) - 64]
        exp = np.array([s for s in base_spans if s[1] <= len(base) - 64], dtype=np.int64).reshape(-1, 2)
        assert first.shape == exp.shape and (first == exp).all(), pat
        # count-only mode must agree with emit mode
        assert r.find_all_device(d) == total
        assert n == len(base) * reps


# ------------------------------------------------------------------- shards ----
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_search_matches_whole_haystack(world):
    """Several byte-range shards driven through one GPU (one thread per shard, in-process
    collectives): results must equal find_iter over the whole haystack."""
    import threading
    import torch
    from regex_b200 import sharded
    text = tiled_corpus(3 << 20) + b"a" * 70000 + b"\n" + tiled_corpus(1 << 20, seed=5)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for pat in [r"[a-zA-Z]+ing", r"Holmes|Watson", r"aaa", r"(?m)^\w+", r"a*", r"[^\n]{5,}"]:
        exp = O.OracleRegex(pat).find_iter(text)
        comm = sharded.ThreadComm(world)
        out = [None] * world
        errs = []

        def work(rank):
            try:
                re_ = R.BytesRegex(pat)
                info = re_.pattern_info()
                geom = sharded.plan(len(text), world, rank, halo=1 << 17)
                buf = d_text[geom.buf_lo:geom.buf_hi].clone()
                eng = sharded.GpuShardEngine(re_, buf, cap=len(exp) + 16)
                n_local, offset, total, rounds = sharded.find_all_sharded(eng, geom, comm.view(rank), info["can_match_empty"], info["has_looks"])
                spans = (eng.spans[:n_local] + geom.buf_lo).cpu().numpy()
                out[rank] = (offset, spans, total)
            except Exception as e:  # surface failures instead of dead-locking the barrier
                errs.append(e)
                comm._barrier.abort()

        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errs, errs
        merged = []
        for off, sp, total in out:
            assert off == len(merged) and total == len(exp)
            merged += [tuple(int(v) for v in r) for r in sp.tolist()]
        assert merged == exp, (pat, world)


# -------------------------------------------------- the reference's own C test ----
CTEST_CASES = {"test_is_match", "test_shortest_match", "test_find", "test_captures", "test_iter", "test_iter_capture_names", "test_flags",
               "test_compile_error", "test_compile_error_size_limit", "test_regex_set_match", "test_regex_set_options",
               "test_regex_set_match_start"}


def _build_c_program(src, exe, flags):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_dir = os.path.join(root, "regex_b200")
    subprocess.check_call(["gcc", *flags, src, "-I" + os.path.join(root, "include"), "-L" + lib_dir, "-lrure_b200",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    return exe


def test_reference_ctest_binary(tmp_path):
    """The reference's C API test and iterator example (regex-capi/ctest/test.c and
    examples/iter.c, restated in tests/capi/), compiled against include/rure.h as strict ANSI C
    with warnings as errors and linked to librure_b200.so.  All twelve tests must pass,
    the three that read capture groups included; the example must find what the oracle finds.
    With REGEX_CAPI_DIR naming a checkout of the reference's regex-capi directory, its own two
    files are compiled unchanged and run as well."""
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    strict = ["-ansi", "-Wall", "-Werror"]
    sources = [("restated", os.path.join(here, "capi", "ctest.c"), os.path.join(here, "capi", "iter.c"), ["-DDEBUG", *strict], strict)]
    upstream = os.environ.get("REGEX_CAPI_DIR")
    if upstream:
        sources.append(("upstream", os.path.join(upstream, "ctest", "test.c"), os.path.join(upstream, "examples", "iter.c"), ["-DDEBUG"], []))
    for kind, test_c, iter_c, test_flags, iter_flags in sources:
        exe = _build_c_program(test_c, str(tmp_path / f"ctest_{kind}"), test_flags)
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        lines = [l for l in r.stderr.splitlines() if l.startswith(("PASSED", "FAILED"))]
        failed = {l.split(": ")[1] for l in lines if l.startswith("FAILED")}
        passed = {l.split(": ")[1] for l in lines if l.startswith("PASSED")}
        assert not failed, (kind, failed, r.stderr[-2000:])
        assert passed >= CTEST_CASES, (kind, passed, r.stderr[-2000:])
        # the iterator example (captures iterator) must run to completion over sherlock.txt
        exe = _build_c_program(iter_c, str(tmp_path / f"iter_{kind}"), iter_flags)
        it = subprocess.run([exe], capture_output=True, text=True, timeout=120, cwd=GOLDEN)
        assert it.returncode == 0, (kind, it.stderr[-500:])
        if kind == "restated":
            exp = O.OracleRegex(r"(?i)(\w+)\s+Holmes").find_iter(sherlock_text())
            got = [tuple(int(v) for v in l.split(":")[0].split()[-1].split("..")) for l in it.stdout.splitlines() if l.startswith("match at")]
            assert got == exp and it.stdout.splitlines()[-1] == f"{len(exp)} matches"


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_search_short_haystacks(world):
    """Haystacks so short that an early rank's halo reaches the end of the text (its buffer
    then ends where the haystack does: end-of-text semantics, no halo overflow) and trailing
    ranks own nothing."""
    import threading
    import torch
    from regex_b200 import sharded
    base = sherlock_text()[5000:9000]
    for pat in (r"[a-zA-Z]+ing", r"\w+", r"a*", r"(?m)^\w+$", r"[a-z]+\s*$"):
        re_ = R.BytesRegex(pat)
        info = re_.pattern_info()
        exp_all = O.OracleRegex(pat)
        for n in (0, 1, 255, 256, 257, 600, 1100, 4000):
            t = base[:n]
            comm = sharded.ThreadComm(world)
            out = [None] * world

            def work(rank):
                geom = sharded.plan(len(t), world, rank, halo=512)
                buf = torch.frombuffer(bytearray(t[geom.buf_lo:geom.buf_hi] or b"\0"), dtype=torch.uint8).cuda()[:geom.n_buf]
                # one compiled regex per rank: reuse_scan keeps the start bitmap inside the object
                eng = sharded.GpuShardEngine(R.BytesRegex(pat), buf, cap=len(t) + 8)
                n_local, offset, total, _ = sharded.find_all_sharded(eng, geom, comm.view(rank), info["can_match_empty"], info["has_looks"])
                spans = eng.spans[:n_local].cpu().numpy().astype(np.int64) + geom.buf_lo if n_local else np.zeros((0, 2), dtype=np.int64)
                out[rank] = (offset, [tuple(int(v) for v in r) for r in spans], total)

            threads = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
            for th in threads:
                th.start()
            for th in threads:
                th.join(timeout=60)
                assert not th.is_alive(), (pat, n, world, "a rank failed or hung")
            merged = []
            for off, sp, _ in sorted(out):
                assert off == len(merged), (pat, n, world)
                merged += sp
            assert merged == exp_all.find_iter(t), (pat, n, world)


@pytest.mark.gpu
def test_pipelined_host_find_all(monkeypatch):
    """rure_b200_find_all on host memory uploads in pieces and searches each piece as a shard
    while later pieces are still in flight; spans must equal the upload-then-search path --
    with ragged last pieces, empty matches, look-arounds, and a match longer than the halo
    (which makes the pipeline give up and redo the haystack in one piece)."""
    n = 12 << 20
    corpus = tiled_corpus(n)
    special = bytearray(corpus)
    special[5_000_000:5_300_000] = b"a" * 300_000
    for data in (corpus, bytes(special)):
        for pat in [r"[a-zA-Z]+ing", r"\w+", r"a+", r"(?m)^\w+", r"a*", r"(?-u:\b)the(?-u:\b)"]:
            r = R.BytesRegex(pat)
            monkeypatch.setenv("RB200_PIPELINE_PIECE", "0")
            plain = r.find_all(data, cap=4_000_000)
            for piece in (1 << 20, 3 << 20):
                monkeypatch.setenv("RB200_PIPELINE_PIECE", str(piece))
                got = r.find_all(data, cap=4_000_000)
                assert got.shape == plain.shape and np.array_equal(got, plain), (pat, piece)
    exp = O.OracleRegex(r"[a-zA-Z]+ing").find_iter(corpus[:3 << 20])
    monkeypatch.setenv("RB200_PIPELINE_PIECE", str(1 << 20))
    got = _spans(R.BytesRegex(r"[a-zA-Z]+ing").find_all(corpus))
    assert got[:len(exp) - 1] == exp[:len(exp) - 1]


# ------------------------------------------- look-arounds at every kind of boundary ----
def _run_gpu_shards(pat, text, d_text, world, exp_len, halo=256, tuning=None, options=None, stats=None):
    """Byte-range shards of `text` through one GPU (one thread per shard, in-process collectives).
    `stats`: a dict that receives each rank's last_stats() once the boundary protocol is through."""
    import threading
    from regex_b200 import sharded
    comm = sharded.ThreadComm(world)
    out, errs = [None] * world, []

    def work(rank):
        try:
            re_ = R.BytesRegex(pat)
            if tuning:
                re_.set_tuning(**tuning)
            for k, v in (options or {}).items():
                re_.set_option(k, v)
            info = re_.pattern_info()
            geom = sharded.plan(len(text), world, rank, halo=halo)
            buf = d_text[geom.buf_lo:geom.buf_hi].clone()
            eng = sharded.GpuShardEngine(re_, buf, cap=exp_len + 16)
            n_local, offset, total, _ = sharded.find_all_sharded(eng, geom, comm.view(rank), info["can_match_empty"], info["has_looks"])
            out[rank] = (offset, (eng.spans[:n_local] + geom.buf_lo).cpu().numpy(), total)
            if stats is not None:
                stats[rank] = re_.last_stats()
        except Exception as e:  # noqa: BLE001 -- surface instead of dead-locking the barrier
            errs.append(e)
            comm._barrier.abort()

    threads = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=120)
        assert not t.is_alive()
    if errs:
        real = [e for e in errs if "BrokenBarrier" not in type(e).__name__]
        raise real[0] if real else errs[0]
    merged = []
    for off, sp, total in out:
        assert off == len(merged) and total == exp_len
        merged += [tuple(int(v) for v in r) for r in sp.tolist()]
    return merged


def test_look_around_patterns_at_chunk_and_shard_boundaries():
    """>= 2000 random patterns WITH look-arounds (the grammar of test_fuzz_tables_vs_oracle: ^ $ (?m:^)
    (?m:$) \\b \\B next to classes, lazy/greedy repeats, alternations) on 64-byte segments and
    64-bit chunks, whole haystack and 2-4 shards, against the oracle: the reference's
    reverse-on-slice rule (src/exec.rs:651-657) at speculative chunk / shard entries, chunks
    without candidates, empty matches at boundaries."""
    import torch
    from test_fuzz_tables_vs_oracle import _pattern
    rng = np.random.Generator(np.random.PCG64(0x100C5))
    cases = shard_cases = explicit = 0
    tries = 0
    while cases < 2000 and tries < 20000:
        tries += 1
        p = _pattern(rng)
        if all(x not in p for x in ("α", "é", "3b1", "pL")):
            p = "(?-u)" + p
        try:
            r = R.BytesRegex(p)
        except R.Error:
            continue
        if not r.pattern_info()["has_looks"]:
            continue
        o = O.OracleRegex(p)
        text = xorshift_bytes(int(rng.integers(0, 1 << 30)), int(rng.integers(600, 2600)), b"abc \n" if rng.random() < 0.7 else b"ab1 _\n")
        exp = o.find_iter(text)
        r.set_tuning(seg=64, chunk=64, warm=int(rng.integers(0, 2)) * 16)
        r.force_generic(bool(rng.integers(0, 2)))
        got = _spans(r.find_all(text))
        assert got == exp, (p, text, got[:5], exp[:5])
        cases += 1
        if cases % 4 == 0:
            d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
            try:
                got = _run_gpu_shards(p, text, d_text, int(rng.integers(2, 5)), len(exp), tuning=dict(seg=64, chunk=64, warm=0))
            except R.Error as e:
                assert "enlarge" in str(e), (p, str(e))  # halo / left context too short: explicit, not wrong
                explicit += 1
                continue
            assert got == exp, ("sharded", p, text)
            shard_cases += 1
    assert cases >= 2000 and shard_cases >= 300, (cases, shard_cases, explicit)


def test_round1_slice_rule_case_on_the_gpu():
    pat = r"^[ab]{2,}\w*?|(?m:$)"
    import torch
    for seed in range(8):
        text = xorshift_bytes(seed, 948, b"abc \n")
        exp = O.OracleRegex(pat).find_iter(text)
        for seg, chunk in ((64, 64), (64, 256), (0, 4096)):
            r = R.BytesRegex(pat)
            r.set_tuning(seg=seg, chunk=chunk, warm=0)
            assert _spans(r.find_all(text)) == exp, (seed, seg, chunk)
        d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
        assert _run_gpu_shards(pat, text, d_text, 3, len(exp)) == exp, seed
