"""Per-record replacen / splitn / captures_iter (replacen_batch, split_batch, splitn_batch, captures_iter_batch and
their device variants) on the GPU: every record against the reference loops run on that record alone over the
oracle's spans, and a sample of records against the single-haystack calls."""
import os
import sys

import numpy as np
import pytest

import regex_b200 as R
from oracle import oracle as O
from test_batch_bulk_model import _rep_fn, split_batch
from test_gpu_batch_iter import PATTERNS, _edge_lines, _offsets, _valid

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFFFFFFFFFF
DATE = r"(\d{4})-(\d{2})-(\d{2})"
LOOKS = [r"^[ab]{2,}\w*?|(?m:$)", r"(?-u:\b)\d{2}(?-u:\b)", r"(?m)^\w+"]
# captures_iter and find_iter disagree on this record: group 0 of the second match is (3, 3), its find_iter
# span (1, 3) (the reverse-on-slice rule of the DFA path); found by a seeded search over the oracle
DIVERGING = (r"^[ab]{2,}\w*?|(?m:$)", b"\nab")


def _records(utf8):
    lines = _edge_lines()
    return [l for l in lines if _valid(l)] if utf8 else lines


def _replace_rec(rec, spans, limit, rep_fn):
    out, last = [], 0
    for i, (s, e) in enumerate(spans):
        if limit and i >= limit:
            break
        out += [rec[last:s], rep_fn(rec[s:e])]
        last = e
    return b"".join(out) + rec[last:]


def _split_recs(recs, per, has_limit, limit):
    """Pieces per record from the oracle's spans (the model of tests/test_batch_bulk_model.py)."""
    moff = np.concatenate([[0], np.cumsum([len(p) for p in per])]).astype(np.int64)
    spans = np.array([s for p in per for s in p], dtype=np.int64).reshape(-1, 2)
    poff, pieces = split_batch(recs, moff, spans, has_limit, limit)
    return [[tuple(int(v) for v in x) for x in pieces[poff[r]:poff[r + 1]]] for r in range(len(recs))]


def _rows(slots, g):
    return [[None if int(a) == NONE else (int(a), int(b)) for a, b in row[:g]] for row in slots]


def _pad(caps, g):
    return [c[:g] + [None] * (g - len(c)) for c in caps]


@pytest.mark.parametrize("generic", [False, True])
def test_replace_and_split_batch_every_record(generic):
    for pat in PATTERNS:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            recs = _records(utf8)
            text, off = b"".join(recs), _offsets(recs)
            o = O.OracleRegex(pat, only_utf8=utf8)
            per = [o.find_iter(l) for l in recs]
            r = cls(pat)
            r.force_generic(generic)
            tag = (pat, utf8, generic)
            for rep, expand, limit in [(b"<$0>", True, 0), (b"<$0>", True, 1), (b"${0}$$|", True, 3), (b"$0", False, 0), (b"", True, 2)]:
                ooff, out = r.replacen_batch(text, off, limit, rep, expand)
                assert ooff.shape == (len(recs) + 1,) and int(ooff[0]) == 0 and int(ooff[-1]) == out.size, tag
                fn = _rep_fn(rep) if expand else (lambda m, rep=rep: rep)
                for i, l in enumerate(recs):
                    assert out[int(ooff[i]):int(ooff[i + 1])].tobytes() == _replace_rec(l, per[i], limit, fn), (tag, rep, limit, i, l)
            for has_limit, limit in [(False, 0), (True, 0), (True, 1), (True, 2), (True, 5), (True, 10 ** 9)]:
                poff, pieces = r.splitn_batch(text, off, limit) if has_limit else r.split_batch(text, off)
                exp = _split_recs(recs, per, has_limit, limit)
                assert int(poff[-1]) == pieces.shape[0], tag
                for i in range(len(recs)):
                    got = [tuple(int(v) for v in x) for x in pieces[int(poff[i]):int(poff[i + 1])]]
                    assert got == exp[i], (tag, has_limit, limit, i, recs[i])


def test_sample_equals_single_haystack_calls():
    rng = np.random.Generator(np.random.PCG64(7))
    for pat in PATTERNS + LOOKS:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            recs = _records(utf8)
            text, off = b"".join(recs), _offsets(recs)
            r = cls(pat)
            ooff, out = r.replacen_batch(text, off, 2, b"[$0]")
            poff, pieces = r.splitn_batch(text, off, 3)
            moff, slots = r.captures_iter_batch(text, off)
            for i in [0, 1, 2, 3, 7, 17, len(recs) - 1] + rng.integers(0, len(recs), 12).tolist():
                l = recs[i]
                assert out[int(ooff[i]):int(ooff[i + 1])].tobytes() == r.replacen(l, 2, b"[$0]"), (pat, utf8, i)
                assert [l[int(a):int(b)] for a, b in pieces[int(poff[i]):int(poff[i + 1])]] == r.splitn(l, 3), (pat, utf8, i)
                assert (slots[int(moff[i]):int(moff[i + 1])] == r.captures_all(l)).all(), (pat, utf8, i)
                assert int(moff[i + 1] - moff[i]) == r.captures_all(l).shape[0], (pat, utf8, i)


def test_group_templates():
    recs = _records(False)
    text, off = b"".join(recs), _offsets(recs)
    o = O.OracleRegex(DATE)
    caps = [o.captures_iter(l) for l in recs]

    def expand(l, c, parts):
        return b"".join(p if isinstance(p, bytes) else (l[c[p][0]:c[p][1]] if c[p] else b"") for p in parts)

    for generic in (False, True):
        r = R.BytesRegex(DATE)
        r.force_generic(generic)
        for rep, parts in [(b"$3/$2/$1", [3, b"/", 2, b"/", 1]), (b"${1}x", [1, b"x"]), (b"<$9$nope>", [b"<>"]), (b"$0", [0])]:
            for limit in (0, 1):
                ooff, out = r.replacen_batch(text, off, limit, rep)
                for i, l in enumerate(recs):
                    exp, last = [], 0
                    for k, c in enumerate(caps[i]):
                        if limit and k >= limit:
                            break
                        exp += [l[last:c[0][0]], expand(l, c, parts)]
                        last = c[0][1]
                    assert out[int(ooff[i]):int(ooff[i + 1])].tobytes() == b"".join(exp) + l[last:], (rep, limit, i, l)
    # a named group; the template error of the single call
    r = R.BytesRegex(r"(?P<y>\d{4})-(?P<m>\d{2})")
    ooff, out = r.replace_all_batch(b"2014-01 x2015-02", [0, 7, 16], b"$m.$y")
    assert out.tobytes() == b"01.2014 x02.2015" and ooff.tolist() == [0, 7, 16]
    with pytest.raises(R.Error, match="too many parts"):
        r.replace_all_batch(b"2014-01", [0, 7], b"$y." * 20)


def test_captures_iter_batch_every_record():
    for pat in PATTERNS + LOOKS:
        for cls, utf8 in ((R.BytesRegex, False), (R.Regex, True)):
            recs = _records(utf8)
            if pat == DIVERGING[0]:
                recs = recs[:50] + [DIVERGING[1]] + recs[50:]
            text, off = b"".join(recs), _offsets(recs)
            o = O.OracleRegex(pat, only_utf8=utf8)
            r = cls(pat)
            g = r.captures_len()
            moff, slots = r.captures_iter_batch(text, off)
            assert slots.shape == (int(moff[-1]), g, 2), (pat, utf8)
            for i, l in enumerate(recs):
                exp = _pad(o.captures_iter(l, only_utf8=utf8), g)
                assert _rows(slots[int(moff[i]):int(moff[i + 1])], g) == exp, (pat, utf8, i, l)


def test_divergence_path_runs():
    pat, rec = DIVERGING
    o = O.OracleRegex(pat)
    assert [c[0] for c in o.captures_iter(rec)] != o.find_iter(rec)  # the pinned record does diverge
    r = R.BytesRegex(pat)
    recs = [b"ab", rec, b"", b"x\nab", rec, b"abab\n"]
    moff, slots = r.captures_iter_batch(b"".join(recs), _offsets(recs))
    for i, l in enumerate(recs):
        assert _rows(slots[int(moff[i]):int(moff[i + 1])], 1) == _pad(o.captures_iter(l), 1), (i, l)
    # capped device call on the same batch: complete offsets and total, the first rows stored
    import torch
    d_text = torch.frombuffer(bytearray(b"".join(recs)), dtype=torch.uint8).cuda()
    d_off = torch.from_numpy(_offsets(recs).astype(np.int64)).cuda()
    d_moff = torch.full((len(recs) + 1,), -1, dtype=torch.int64, device="cuda")
    d_slots = torch.full((3, 1, 2), -1, dtype=torch.int64, device="cuda")
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    assert r.captures_iter_batch_device(d_text, d_off, d_moff, d_slots) == slots.shape[0]
    assert (d_moff.cpu().numpy().astype(np.uint64) == moff).all()
    assert (d_slots.cpu().numpy().view(np.uint64) == slots[:3]).all()


def test_device_variants_caps_unaligned_and_empty():
    import torch
    recs = _records(False)[:700]
    text, off = b"".join(recs), _offsets(recs)
    r = R.BytesRegex(DATE)
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    buf = torch.frombuffer(bytearray(b"#" + text), dtype=torch.uint8).cuda()
    d_text = buf[1:]  # not 16-byte aligned: the generic iterator runs
    assert d_text.data_ptr() % 16 != 0
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    n1 = len(recs) + 1
    # replace: size only, then a short buffer (prefix stored, total and offsets exact), then everything
    ooff, out = r.replacen_batch(text, off, 0, b"$3/$2/$1")
    d_oo = torch.full((n1,), -1, dtype=torch.int64, device="cuda")
    assert r.replacen_batch_device(d_text, d_off, 0, b"$3/$2/$1", d_oo) == out.size
    assert (d_oo.cpu().numpy().astype(np.uint64) == ooff).all()
    short = torch.zeros(out.size // 2, dtype=torch.uint8, device="cuda")
    assert r.replacen_batch_device(d_text, d_off, 0, b"$3/$2/$1", d_oo, short) == out.size
    assert short.cpu().numpy().tobytes() == out[:out.size // 2].tobytes()
    full = torch.zeros(out.size, dtype=torch.uint8, device="cuda")
    assert r.replacen_batch_device(d_text, d_off, 0, b"$3/$2/$1", d_oo, full) == out.size
    assert full.cpu().numpy().tobytes() == out.tobytes()
    # split
    poff, pieces = r.split_batch(text, off)
    d_po = torch.full((n1,), -1, dtype=torch.int64, device="cuda")
    assert r.split_batch_device(d_text, d_off, d_po) == pieces.shape[0]
    d_p = torch.full((pieces.shape[0] // 3, 2), -1, dtype=torch.int64, device="cuda")
    assert r.split_batch_device(d_text, d_off, d_po, d_p) == pieces.shape[0]
    assert (d_po.cpu().numpy().astype(np.uint64) == poff).all()
    assert (d_p.cpu().numpy().astype(np.uint64) == pieces[:d_p.shape[0]]).all()
    poff2, pieces2 = r.splitn_batch(text, off, 2)
    d_p = torch.empty((pieces2.shape[0], 2), dtype=torch.int64, device="cuda")
    assert r.split_batch_device(d_text, d_off, d_po, d_p, limit=2) == pieces2.shape[0]
    assert (d_p.cpu().numpy().astype(np.uint64) == pieces2).all() and (d_po.cpu().numpy().astype(np.uint64) == poff2).all()
    # captures_iter
    moff, slots = r.captures_iter_batch(text, off)
    d_mo = torch.full((n1,), -1, dtype=torch.int64, device="cuda")
    d_s = torch.full((slots.shape[0] // 2, 4, 2), -1, dtype=torch.int64, device="cuda")
    assert r.captures_iter_batch_device(d_text, d_off, d_mo, d_s) == slots.shape[0]
    assert (d_mo.cpu().numpy().astype(np.uint64) == moff).all()
    assert (d_s.cpu().numpy().view(np.uint64) == slots[:d_s.shape[0]]).all()
    assert r.captures_iter_batch_device(d_text, d_off, d_mo) == slots.shape[0]
    # no records
    one = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    assert r.replacen_batch_device(d_text, d_off[:1], 0, b"x", one) == 0 and int(one[0]) == 0
    one.fill_(-1)
    assert r.split_batch_device(d_text, d_off[:1], one) == 0 and int(one[0]) == 0
    one.fill_(-1)
    assert r.captures_iter_batch_device(d_text, d_off[:1], one) == 0 and int(one[0]) == 0
    z = np.zeros(1, dtype=np.uint64)
    assert [x.tolist() for x in r.replace_all_batch(b"", z, b"x")] == [[0], []]
    assert r.split_batch(b"", z)[1].shape == (0, 2) and r.captures_iter_batch(b"", z)[1].shape == (0, 4, 2)
    # records that do not start at 0: results are record-relative and the bytes before offsets[0] are not read
    sub = off[100:201]
    ooff_s, out_s = r.replace_all_batch(text, sub, b"<date>", expand=False)
    for k in range(100):
        l = recs[100 + k]
        assert out_s[int(ooff_s[k]):int(ooff_s[k + 1])].tobytes() == R.BytesRegex(DATE).replace_all(l, b"<date>", expand=False), k


def test_sets_are_rejected():
    import ctypes
    s = R.BytesRegexSet([r"a", r"b"])
    off, o2, total = np.array([0, 2], dtype=np.uint64), np.zeros(2, dtype=np.uint64), ctypes.c_size_t()
    lib = R.lib()
    assert not lib.rure_b200_replace_batch(s._h, b"ab", off.ctypes.data, 1, b"x", 1, 1, 0, o2.ctypes.data, None, 0, ctypes.byref(total))
    assert "exactly one pattern" in R._last_error()
    assert not lib.rure_b200_split_batch(s._h, b"ab", off.ctypes.data, 1, 0, 0, o2.ctypes.data, None, 0, ctypes.byref(total))
    assert "exactly one pattern" in R._last_error()
    assert not lib.rure_b200_captures_iter_batch(s._h, b"ab", off.ctypes.data, 1, o2.ctypes.data, None, 0, ctypes.byref(total))
    assert "exactly one pattern" in R._last_error()


def test_c3_one_million_lines():
    """1 M C3 lines: a NoExpand redaction and a split on whitespace, offsets checked in full against the per-record
    find_iter, the bytes against the oracle on a seeded sample of lines."""
    import torch
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import corpus as C
    n_lines = 1_000_000
    d_text, d_off = C.log_lines(n_lines, torch.device("cuda", 0))
    host = d_text.cpu().numpy().tobytes()
    offs = d_off.cpu().numpy().astype(np.int64)
    lens = np.diff(offs)
    rng = np.random.Generator(np.random.PCG64(3))
    sample = np.unique(np.concatenate([np.arange(50), rng.integers(0, n_lines, 2000)]))
    for pat, kind in [(DATE, "replace"), (r"\s+", "split")]:
        r = R.BytesRegex(pat)
        r.set_stream(torch.cuda.current_stream().cuda_stream)
        d_m = torch.empty(n_lines + 1, dtype=torch.int64, device="cuda")
        m = r.find_iter_batch_device(d_text, d_off, d_m)
        d_sp = torch.empty((max(m, 1), 2), dtype=torch.int64, device="cuda")
        r.find_iter_batch_device(d_text, d_off, d_m, d_sp)
        moff, sp = d_m.cpu().numpy(), d_sp.cpu().numpy()[:m]
        cnt = np.diff(moff)
        d_res = torch.empty(n_lines + 1, dtype=torch.int64, device="cuda")
        o = O.OracleRegex(pat)
        if kind == "replace":
            rep = b"<date>"
            total = r.replacen_batch_device(d_text, d_off, 0, rep, d_res, expand=False)
            d_out = torch.empty(total, dtype=torch.uint8, device="cuda")
            assert r.replacen_batch_device(d_text, d_off, 0, rep, d_res, d_out, expand=False) == total
            matched = np.add.reduceat(np.concatenate([sp[:, 1] - sp[:, 0], [0]]), moff[:-1]) * (cnt > 0)
            exp_len = lens - matched + cnt * len(rep)
            res = d_res.cpu().numpy()
            assert res[0] == 0 and (np.diff(res) == exp_len).all() and res[-1] == total
            out = d_out.cpu().numpy().tobytes()
            for i in sample:
                l = host[offs[i]:offs[i + 1]]
                assert out[res[i]:res[i + 1]] == _replace_rec(l, o.find_iter(l), 0, lambda x: rep), i
        else:
            total = r.split_batch_device(d_text, d_off, d_res)
            d_p = torch.empty((total, 2), dtype=torch.int64, device="cuda")
            assert r.split_batch_device(d_text, d_off, d_res, d_p) == total
            last_end = np.where(cnt > 0, sp[np.maximum(moff[1:] - 1, 0), 1], 0)
            res = d_res.cpu().numpy()
            assert res[0] == 0 and (np.diff(res) == cnt + (last_end < lens)).all() and res[-1] == total
            pieces = d_p.cpu().numpy()
            for i in sample:
                l = host[offs[i]:offs[i + 1]]
                got = [l[a:b] for a, b in pieces[res[i]:res[i + 1]]]
                exp = [l[a:b] for a, b in _split_recs([l], [o.find_iter(l)], False, 0)[0]]
                assert got == exp, i
