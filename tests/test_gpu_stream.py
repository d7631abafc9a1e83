"""Streams (include/rure_b200.h, Regex.stream): find_iter over text written in pieces through a
bounded device window must give exactly find_all on the whole resident text -- for every search
path, ragged writes, wrong reverse-scan guesses at piece edges, str mode with scalars split across
writes -- and find_all / count_all / rure_iter_next through the window (option "host_window")
must equal the resident search."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import regex_b200 as R
from helpers import tiled_corpus
from oracle import oracle as O

pytestmark = pytest.mark.gpu

N = 12 << 20
PATTERNS = [r"[a-zA-Z]+ing", r"\w+", r"a+", r"a*", r"(?m)^\w+", r"(?-u:\b)the(?-u:\b)", r"Holmes", r"Holmes.{0,40}Watson"]
WRITE_SIZES = [0, 1, 255, 257, 1 << 20, 3 << 20, 5 << 20]


def _corpora():
    corpus = tiled_corpus(N)
    special = bytearray(corpus)
    special[5_000_000:5_300_000] = b"a" * 300_000
    return {"corpus": corpus, "run": bytes(special)}


@pytest.fixture(scope="module")
def corpora():
    return _corpora()


def _compile(pat, utf8=False):
    r = (R.Regex if utf8 else R.BytesRegex)(pat)
    if pat == r"Holmes.{0,40}Watson":
        r.set_option("candidate_starts", 1)  # the path of patterns over the automaton budget
    return r


def _writes(data, rng):
    """data cut into writes of the sizes above, in random order, reading back in between."""
    pos = 0
    while pos < len(data):
        k = int(rng.choice(WRITE_SIZES))
        yield data[pos:pos + k]
        pos += k


def _stream(r, data, piece, seed, spans=True, hold=0):
    rng = np.random.Generator(np.random.PCG64(seed))
    parts = []
    with r.stream(piece=piece, hold=hold, spans=spans) as s:
        for i, w in enumerate(_writes(data, rng)):
            s.write(w if i % 3 else np.frombuffer(w, dtype=np.uint8))  # bytes and arrays
            if i % 2:
                parts.append(s.read())
        s.finish()
        parts.append(s.read())
        count = s.count
    got = np.concatenate(parts) if spans else np.empty((0, 2), dtype=np.uint64)
    return got, count


@pytest.mark.parametrize("name", ["corpus", "run"])
def test_stream_equals_find_all(corpora, name):
    data = corpora[name]
    for pat in PATTERNS:
        r = _compile(pat)
        plain = r.find_all(data, cap=4_000_000)
        for j, piece in enumerate((1 << 20, 3 << 20)):
            got, count = _stream(r, data, piece, seed=17 * j + len(pat))
            assert count == len(plain), (pat, piece)
            assert got.shape == plain.shape and np.array_equal(got, plain), (pat, piece)
        _, count = _stream(r, data, 1 << 20, seed=3, spans=False)
        assert count == len(plain), pat


def test_stream_against_oracle(corpora):
    prefix = corpora["corpus"][:3 << 20]
    for pat in (r"[a-zA-Z]+ing", r"(?m)^\w+"):
        got, _ = _stream(_compile(pat), prefix, 1 << 20, seed=5)
        exp = np.array(O.OracleRegex(pat).find_iter(prefix), dtype=np.uint64).reshape(-1, 2)
        assert got.shape == exp.shape and np.array_equal(got, exp), pat


def test_stream_researches_wrong_edge_guesses(corpora):
    """warm=64 makes the reverse scan guess the state at a piece's top from 64 bytes of halo, which
    is wrong where a match spans the edge: the pending piece is searched again."""
    for name, data in corpora.items():
        for pat in (r"[a-zA-Z]+ing", r"\w+", r"a+", r"(?m)^\w+"):
            r = _compile(pat)
            plain = r.find_all(data, cap=4_000_000)
            r.set_tuning(warm=64)
            got, count = _stream(r, data, 1 << 20, seed=11)
            assert count == len(plain) and np.array_equal(got, plain), (name, pat)


def test_stream_str_mode_split_scalars():
    words = "Шерлок Холмс и доктор Ватсон — ёж, щука, яблоко. ".encode("utf-8")
    text = (words * ((6 << 20) // len(words) + 1))[: 6 << 20]
    text = text[: len(text) - len(text.split(b" ")[-1])]  # end on a whole scalar
    for pat in (r"\w*", r"\w+", r"[а-я]+"):
        r = _compile(pat, utf8=True)
        plain = r.find_all(text, cap=4_000_000)
        got, count = _stream(r, text, 1 << 20, seed=7)  # odd write sizes split two-byte scalars
        assert count == len(plain) and np.array_equal(got, plain), pat


def _iter_all(r, data):
    """rure_iter_next over data; the first calls alternate between two copies of the buffer, so
    each of them searches again from the iterator's last end (find_all_host with start > 0)."""
    lib = R.lib()
    other = bytes(bytearray(data))
    bufs = [ctypes.c_char_p(data), ctypes.c_char_p(other)]
    it = lib.rure_iter_new(r._h)
    m = R._Match()
    out = []
    try:
        while True:
            b = bufs[len(out) % 2] if len(out) < 4 else bufs[0]
            if not lib.rure_iter_next(it, ctypes.cast(b, ctypes.c_void_p), len(data), ctypes.byref(m)):
                break
            out.append((m.start, m.end))
    finally:
        lib.rure_iter_free(it)
    return np.array(out, dtype=np.uint64).reshape(-1, 2)


def test_host_window_equals_resident(corpora):
    data = corpora["run"]
    for pat in (r"[a-zA-Z]+ing", r"a+", r"(?m)^\w+", r"Holmes"):
        r = _compile(pat)
        plain = r.find_all(data, cap=4_000_000)
        r.set_option("host_window", 4 << 20)  # pieces and hold of 512 KiB
        assert np.array_equal(r.find_all(data, cap=4_000_000), plain), pat
        assert np.array_equal(r.find_all(data), plain), pat  # too small a cap first, then the exact one
        assert r.count_all(data) == len(plain), pat
        assert np.array_equal(_iter_all(r, data), plain), pat


def test_stream_errors(corpora):
    r = _compile(r"a+")
    with r.stream(piece=1 << 20, hold=4096) as s:
        with pytest.raises(R.Error, match=r"a match is longer than the stream window \(4096 bytes\)"):
            s.write(corpora["run"])
        with pytest.raises(R.Error):
            s.write(b"more")  # a failed stream stays failed
    with r.stream() as s:
        s.write(b"aaa b aa")
        s.finish()
        assert s.read().tolist() == [[0, 3], [6, 8]]
        with pytest.raises(R.Error, match="write after finish"):
            s.write(b"a")
    with r.stream() as s:  # empty text
        s.finish()
        assert s.count == 0
    with _compile(r"a*").stream() as s:
        s.finish()
        assert s.read().tolist() == [[0, 0]]


def test_stream_c_example(corpora, tmp_path):
    """tests/capi/stream.c: fread in 1 MiB blocks into a stream, strict ANSI C."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_dir = os.path.join(root, "regex_b200")
    exe = str(tmp_path / "stream_example")
    subprocess.check_call(["gcc", "-ansi", "-Wall", "-Werror", os.path.join(root, "tests", "capi", "stream.c"), "-I" + os.path.join(root, "include"),
                           "-L" + lib_dir, "-lrure_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    path = tmp_path / "hay.txt"
    path.write_bytes(corpora["run"])
    for pat, piece in ((r"[a-zA-Z]+ing", 1 << 20), (r"a+", 3 << 20)):
        out = subprocess.run([exe, pat, str(path), str(piece)], capture_output=True, text=True, timeout=300, check=True).stdout.split("\n")
        assert out[-2] == f"count {len(out) - 2}"
        got = np.array([l.split() for l in out[:-2]], dtype=np.uint64).reshape(-1, 2)
        plain = R.BytesRegex(pat).find_all(corpora["run"], cap=4_000_000)
        assert np.array_equal(got, plain), pat
