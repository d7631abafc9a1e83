"""Per-record find_iter (find_iter_batch / count_batch) and per-record captures (captures_batch) on the GPU,
every record against the oracle run on that record alone."""
import numpy as np
import pytest

import regex_b200 as R
from helpers import vectors
from oracle import oracle as O
from test_gpu_parity import _log_lines

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFFFFFFFFFF


def _offsets(records):
    return np.concatenate([[0], np.cumsum([len(l) for l in records])]).astype(np.uint64)


def _edge_lines():
    lines = _log_lines(3000)
    lines[17] = b""
    lines[0] = b"2014-01-02"
    lines[1] = "٢٠١٤-٠١-٠٢ arabic-indic digits are \\d too\n".encode()
    lines[2] = "naïve 1999-12-31 café\n".encode()
    lines[3] = b"\xff\xfe 2001-02-03 \xc3\n"
    lines[4] = b"7"
    lines[5] = b"x" * 15
    lines[6] = b"x" * 6 + b"2020-10-10"
    lines[7] = b"ab" * 8 + b"a"
    lines[8] = "aδ☃𝄞b".encode()
    lines[9] = b"x" * 16 + b"2020-10-10" + b"y" * 33
    lines[-1] = b"no newline at the very end 2030-01-01"
    return lines


PATTERNS = [r"(\d{4})-(\d{2})-(\d{2})", r"\w+", r"", r"a*", r"\s*", r"(?m)^\w+", r"\w+$", r"(?-u:\b)\d{2}(?-u:\b)",
            r"^[ab]{2,}\w*?|(?m:$)", r"[a-z]+ing"]


def _check_iter(r, o, lines, text, off, tag):
    moff, spans = r.find_iter_batch(text, off)
    counts = r.count_batch(text, off)
    assert moff.shape == (len(lines) + 1,) and int(moff[0]) == 0 and int(moff[-1]) == spans.shape[0], tag
    assert (np.diff(moff) == counts).all(), tag
    found, first = r.find_batch(text, off)
    for i, l in enumerate(lines):
        exp = o.find_iter(l)
        got = [tuple(int(v) for v in s) for s in spans[int(moff[i]):int(moff[i + 1])]]
        assert got == exp, (tag, i, l)
        assert bool(found[i]) == bool(exp), (tag, i)
        if exp:
            assert tuple(int(v) for v in first[i]) == exp[0], (tag, i)  # the iterator's first span is find's
    return moff, spans


@pytest.mark.parametrize("generic", [False, True])
def test_find_iter_batch_log_lines(generic):
    lines = _edge_lines()
    text, off = b"".join(lines), _offsets(lines)
    for pat in PATTERNS:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            recs = lines if not utf8 else [l for l in lines if _valid(l)]
            t, o_ = (text, off) if not utf8 else (b"".join(recs), _offsets(recs))
            r = cls(pat)
            r.force_generic(generic)
            _check_iter(r, O.OracleRegex(pat, only_utf8=utf8), recs, t, o_, (pat, utf8, generic))


def _valid(b):
    try:
        b.decode()
        return True
    except UnicodeDecodeError:
        return False


def test_utf8_empty_matches_per_record():
    lines = ["aδ☃𝄞b".encode(), "δ".encode(), b"", "☃☃".encode()]
    text, off = b"".join(lines), _offsets(lines)
    for pat in [r"", r"x*", r"(?-u:\B)"]:
        for cls, utf8 in ((R.Regex, True), (R.BytesRegex, False)):
            _check_iter(cls(pat), O.OracleRegex(pat, only_utf8=utf8), lines, text, off, (pat, utf8))


def test_unaligned_haystack_cap_count_only_and_empty_batch():
    import torch
    lines = _edge_lines()[:600]
    text, off = b"".join(lines), _offsets(lines)
    pat = r"\w+"
    o = O.OracleRegex(pat)
    exp = [o.find_iter(l) for l in lines]
    exp_moff = np.concatenate([[0], np.cumsum([len(e) for e in exp])]).astype(np.uint64)
    flat = [s for e in exp for s in e]
    r = R.BytesRegex(pat)
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    buf = torch.frombuffer(bytearray(b"#" + text), dtype=torch.uint8).cuda()
    d_text = buf[1:]  # starts at byte 1: not 16-byte aligned, the generic kernel runs
    assert d_text.data_ptr() % 16 != 0
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    d_moff = torch.full((len(lines) + 1,), -1, dtype=torch.int64, device="cuda")
    # count only
    assert r.find_iter_batch_device(d_text, d_off, d_moff) == len(flat)
    assert (d_moff.cpu().numpy().astype(np.uint64) == exp_moff).all()
    # cap below the total: offsets and total complete, the first cap spans stored
    cap = len(flat) // 3
    d_out = torch.full((cap, 2), -1, dtype=torch.int64, device="cuda")
    d_moff.fill_(-1)
    assert r.find_iter_batch_device(d_text, d_off, d_moff, d_out) == len(flat)
    assert (d_moff.cpu().numpy().astype(np.uint64) == exp_moff).all()
    assert [tuple(s) for s in d_out.cpu().tolist()] == flat[:cap]
    # aligned, everything stored
    d_al = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    d_out = torch.empty((len(flat), 2), dtype=torch.int64, device="cuda")
    assert r.find_iter_batch_device(d_al, d_off, d_moff, d_out) == len(flat)
    assert [tuple(s) for s in d_out.cpu().tolist()] == flat
    # host call with a small cap: complete offsets and count
    moff, spans = r.find_iter_batch(text, off, cap=5)
    assert (moff == exp_moff).all() and [tuple(int(v) for v in s) for s in spans] == flat
    # no records
    d_moff = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    assert r.find_iter_batch_device(d_al, d_off[:1], d_moff) == 0 and int(d_moff[0]) == 0
    moff, spans = r.find_iter_batch(b"", np.zeros(1, dtype=np.uint64))
    assert moff.tolist() == [0] and spans.shape == (0, 2)
    assert r.count_batch(b"", [0]).shape == (0,)


def test_sets_are_rejected():
    import ctypes
    s = R.BytesRegexSet([r"a", r"b"])
    moff, off, total = np.zeros(2, dtype=np.uint64), np.array([0, 2], dtype=np.uint64), ctypes.c_size_t()
    assert not R.lib().rure_b200_find_iter_batch(s._h, b"ab", off.ctypes.data, 1, moff.ctypes.data, None, 0, ctypes.byref(total))
    assert "exactly one pattern" in R._last_error()


def _check_captures(r, o, lines, tag):
    text, off = b"".join(lines), _offsets(lines)
    found, slots = r.captures_batch(text, off)
    g = r.captures_len()
    assert slots.shape == (len(lines), g, 2), tag
    for i, l in enumerate(lines):
        exp = o.captures_at(l)
        assert bool(found[i]) == (exp is not None), (tag, i, l)
        if exp is None:
            assert (slots[i] == NONE).all(), (tag, i)
            continue
        got = [None if int(a) == NONE else (int(a), int(b)) for a, b in slots[i]]
        assert got == exp[:g] + [None] * (g - len(exp)), (tag, i, l)


def test_captures_batch_golden_vectors():
    n = 0
    for x in vectors():
        if x["kind"] != "mat" or len(x["groups"]) < 2:
            continue
        text = bytes.fromhex(x["text_hex"])
        for mode in x["modes"]:
            utf8 = mode == "str"
            try:
                r = (R.Regex if utf8 else R.BytesRegex)(x["re"])
            except R.Error as e:
                assert "word boundar" in str(e), (x["name"], str(e))
                continue
            o = O.OracleRegex(x["re"], only_utf8=utf8)
            _check_captures(r, o, [text], (x["name"], mode))  # one record: the reference's captures
            found, slots = r.captures_batch(text, [0, len(text)])
            exp = x["groups"]
            got = [None if int(a) == NONE else [int(a), int(b)] for a, b in slots[0]][:len(exp)] if found[0] else [None]
            assert got == exp[:len(got)], (x["name"], got, exp)
            # several records: the text, its halves, an empty record
            h = len(text) // 2
            recs = [text, text[:h], b"", text[h:], text]
            _check_captures(r, o, [t for t in recs if not utf8 or _valid(t)], (x["name"], mode, "multi"))
            n += 1
    assert n > 100, n


def test_captures_batch_log_lines_and_absent_groups():
    lines = _edge_lines()
    for pat in [r"(\d{4})-(\d{2})-(\d{2})", r"(?P<host>host-\d+) svc\[(\d+)\]", r"(a)|(b)", r"(\w+)$", r"^(\d+)?(x*)"]:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            recs = lines if not utf8 else [l for l in lines if _valid(l)]
            _check_captures(cls(pat), O.OracleRegex(pat, only_utf8=utf8), recs, (pat, utf8))
    r = R.BytesRegex(r"(a)|(b)")
    found, slots = r.captures_batch(b"xbxaz", [0, 2, 4, 5])
    assert found.tolist() == [True, True, False]
    assert slots[0].tolist() == [[1, 2], [NONE, NONE], [1, 2]]
    assert slots[1].tolist() == [[1, 2], [1, 2], [NONE, NONE]]
    assert (slots[2] == NONE).all()


def test_captures_batch_device():
    import torch
    lines = _edge_lines()[:500]
    text, off = b"".join(lines), _offsets(lines)
    pat = r"(\d{4})-(\d{2})-(\d{2})"
    r = R.BytesRegex(pat)
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    o = O.OracleRegex(pat)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    g = r.captures_len()
    d_slots = torch.empty(len(lines) * g * 2, dtype=torch.int64, device="cuda")
    d_bits = torch.zeros((len(lines) + 31) // 32, dtype=torch.int32, device="cuda")
    r.captures_batch_device(d_text, d_off, d_slots, d_bits)
    slots = d_slots.cpu().numpy().view(np.uint64).reshape(len(lines), g, 2)
    bits = np.unpackbits(d_bits.cpu().numpy().view(np.uint8), bitorder="little")
    for i, l in enumerate(lines):
        exp = o.captures_at(l)
        assert bool(bits[i]) == (exp is not None), i
        if exp:
            assert [None if int(a) == NONE else (int(a), int(b)) for a, b in slots[i]] == exp, i


@pytest.mark.parametrize("pat", [r"(\d{4})-(\d{2})-(\d{2})", r"[a-z]+ing"])
def test_c3_full_size(pat):
    """C3 log lines at 1 M lines: every line against the oracle."""
    import os
    import sys
    import torch
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import corpus as C
    n_lines = 1_000_000
    d_text, d_off = C.log_lines(n_lines, torch.device("cuda", 0))
    r = R.BytesRegex(pat)
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    d_moff = torch.empty(n_lines + 1, dtype=torch.int64, device="cuda")
    total = r.find_iter_batch_device(d_text, d_off, d_moff)
    d_out = torch.empty((total, 2), dtype=torch.int64, device="cuda")
    assert r.find_iter_batch_device(d_text, d_off, d_moff, d_out) == total
    host = d_text.cpu().numpy().tobytes()
    offs = d_off.cpu().tolist()
    moff = d_moff.cpu().tolist()
    spans = d_out.cpu().numpy()
    o = O.OracleRegex(pat)
    bad = 0
    for i in range(n_lines):
        exp = o.find_iter(host[offs[i]:offs[i + 1]])
        got = spans[moff[i]:moff[i + 1]]
        if len(exp) != got.shape[0] or (len(exp) and not (got == np.array(exp, dtype=np.int64)).all()):
            bad += 1
    assert bad == 0 and total > 0, (pat, bad, total)
    if pat.startswith("("):
        found, slots = r.captures_batch(host, np.array(offs, dtype=np.uint64))
        for i in range(0, n_lines, 50):
            exp = o.captures_at(host[offs[i]:offs[i + 1]])
            assert bool(found[i]) == (exp is not None), i
            if exp:
                assert [(int(a), int(b)) for a, b in slots[i]] == exp, i
