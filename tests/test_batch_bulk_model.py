"""CPU model of the index arithmetic behind the batched replacen / splitn (engine.cu replace_batch_device,
split_batch_device; kernels.cu csr_counts, batch_keep_spans, batch_to_base, batch_replace_offsets,
batch_split_counts, batch_split_pieces).

The spans are the oracle's find_iter of every record alone, in the CSR form the per-record find_iter produces.
The model keeps the first `limit` spans of every record, makes them relative to offsets[0], scatters the
concatenated records as replace_gaps / replace_matches do, and cuts the output at
out_offsets[r] = (offsets[r] - offsets[0]) - L[K_r] + P[K_r].  Split counts its pieces per record and finds
each piece's record by a binary search.  Every record's result must equal the reference loop run on that
record alone (_model_replacen / _model_split of tests/test_gpu_bulk_ops.py)."""
import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_bulk_ops import _model_replacen, _model_split

EDGE = [b"", b"a", b"aaa", b"b", b"", b"abcab", b"  x  y  ", b"2014-01-02 and 2015-03-04", b"\n", b"aaaa aa a", b"xyz"]


def _exclusive(counts):
    return np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))]).astype(np.int64)


def _csr_row(csr, i):
    """The last record r with csr[r] <= i (kernels.cu csr_row; empty records are passed over)."""
    return np.searchsorted(csr[:-1], i, side="right") - 1


def batch_find_iter(pat, recs, utf8=False):
    o = O.OracleRegex(pat, only_utf8=utf8)
    per = [o.find_iter(r) for r in recs]
    spans = np.array([s for p in per for s in p], dtype=np.int64).reshape(-1, 2)
    return _exclusive([len(p) for p in per]), spans


def keep_first(moff, spans, limit):
    """csr_counts + scan + batch_keep_spans: the first `limit` spans of every record (0 = all)."""
    if not limit:
        return moff, spans
    koff = _exclusive(np.minimum(np.diff(moff), limit))
    kept = np.zeros((int(koff[-1]), 2), dtype=np.int64)
    j = np.arange(spans.shape[0])
    r = _csr_row(moff, j)
    i = j - moff[r]
    sel = i < koff[r + 1] - koff[r]
    kept[koff[r[sel]] + i[sel]] = spans[sel]
    return koff, kept


def replace_batch(recs, base, moff, spans, limit, rep_fn):
    """The concatenated records text[offsets[0], offsets[n]) (`base` = offsets[0]) are scattered once."""
    text = b"".join(recs)
    off = _exclusive([len(r) for r in recs]) + base
    koff, kept = keep_first(moff, spans, limit)
    m = kept.shape[0]
    # batch_to_base: relative to offsets[0]
    bs = kept + (off[_csr_row(koff, np.arange(m))] - off[0])[:, None] if m else kept
    reps = [rep_fn(text[s:e]) for s, e in bs]
    L = _exclusive(bs[:, 1] - bs[:, 0])          # lens_before, extended by the total
    P = _exclusive([len(x) for x in reps])       # reps_before, extended by the total
    n = len(text)
    out = bytearray(n - int(L[-1]) + int(P[-1]))
    for i, (s, e) in enumerate(bs):              # replace_matches
        o = s - L[i] + P[i]
        out[o:o + len(reps[i])] = reps[i]
    x = 0
    for i in range(m + 1):                       # replace_gaps: gap byte q in front of match i lands at q - L[i] + P[i]
        ms, me = (bs[i] if i < m else (n, n))
        out[x - L[i] + P[i]:ms - L[i] + P[i]] = text[x:ms]
        x = max(x, me)
    out_off = (off - off[0]) - L[koff] + P[koff]  # batch_replace_offsets
    return out_off, bytes(out)


def split_batch(recs, moff, spans, has_limit, limit):
    lens = np.array([len(r) for r in recs], dtype=np.int64)
    n = len(recs)
    if has_limit and limit == 0:
        return np.zeros(n + 1, dtype=np.int64), np.zeros((0, 2), dtype=np.int64)
    counts = []
    for r in range(n):                           # batch_split_counts
        c = int(moff[r + 1] - moff[r])
        last_end = int(spans[moff[r + 1] - 1, 1]) if c else 0
        p = c + (1 if last_end < lens[r] else 0)
        if has_limit and p + 1 >= limit:
            p = limit
        counts.append(p)
    poff = _exclusive(counts)
    pieces = np.zeros((int(poff[-1]), 2), dtype=np.int64)
    for i in range(pieces.shape[0]):             # batch_split_pieces (split_piece of its record)
        r = int(_csr_row(poff, i))
        np_, c, j = int(poff[r + 1] - poff[r]), int(moff[r + 1] - moff[r]), i - int(poff[r])
        sp = spans[moff[r]:moff[r + 1]]
        last_is_rest = has_limit and np_ == limit
        pieces[i, 0] = 0 if j == 0 else (sp[j - 1, 1] if j - 1 < c else lens[r])
        pieces[i, 1] = sp[j, 0] if (j < c and not (last_is_rest and j + 1 == np_)) else lens[r]
    return poff, pieces


def _records(seed, k):
    rng = np.random.Generator(np.random.PCG64(seed))
    alphabet = np.frombuffer(b"ab  x\n2-0", dtype=np.uint8)
    return EDGE + [bytes(alphabet[rng.integers(0, alphabet.size, int(rng.integers(0, 12)))]) for _ in range(k)]


PATS = [(r"a+", b"<$0>"), (r"", b"|"), (r"a*", b"-"), (r"\s+", b" "), (r"(?m)^", b"> "), (r"\d{4}-\d{2}-\d{2}", b"<date>"),
        (r"x|y", b"${0}${0}$$"), (r"q", b"Q")]


def _rep_fn(rep):
    return lambda m: rep.replace(b"${0}", b"\0M").replace(b"$$", b"\0D").replace(b"$0", b"\0M").replace(b"\0M", m).replace(b"\0D", b"$")


@pytest.mark.parametrize("utf8", [False, True])
@pytest.mark.parametrize("base", [0, 7])
def test_replacen_batch_model(utf8, base):
    recs = _records(3, 60)
    for pat, rep in PATS:
        moff, spans = batch_find_iter(pat, recs, utf8)
        for limit in (0, 1, 3):
            out_off, out = replace_batch(recs, base, moff, spans, limit, _rep_fn(rep))
            assert out_off[0] == 0 and out_off[-1] == len(out), (pat, limit)
            for r, rec in enumerate(recs):
                exp = _model_replacen(pat, rec, limit, _rep_fn(rep), utf8)
                assert out[out_off[r]:out_off[r + 1]] == exp, (pat, limit, r, rec)


def test_split_batch_model():
    recs = _records(5, 60)
    for pat, _ in PATS:
        moff, spans = batch_find_iter(pat, recs)
        for has_limit, limit in [(False, 0), (True, 0), (True, 1), (True, 2), (True, 5), (True, 10 ** 9)]:
            poff, pieces = split_batch(recs, moff, spans, has_limit, limit)
            assert poff[0] == 0 and poff[-1] == pieces.shape[0]
            for r, rec in enumerate(recs):
                got = [rec[s:e] for s, e in pieces[poff[r]:poff[r + 1]]]
                exp = _model_split(pat, rec, limit if has_limit else None)
                assert got == exp, (pat, has_limit, limit, r, rec)


def test_limit_compaction_keeps_record_order():
    recs = [b"aaaa", b"", b"a", b"aa", b"b"]
    moff, spans = batch_find_iter(r"a", recs)
    koff, kept = keep_first(moff, spans, 1)
    assert koff.tolist() == [0, 1, 1, 2, 3, 3]
    assert kept.tolist() == [[0, 1], [0, 1], [0, 1]]
    koff, kept = keep_first(moff, spans, 3)
    assert np.diff(koff).tolist() == [3, 0, 1, 2, 0]
