"""Bounded fix-up work (north star: "per-chunk state maps are composed ... to resolve boundaries"):
automata whose state depends on far context, matches longer than many chunks, chains that never
meet again, and the early exits of is_match / shortest_match / RegexSet::matches
(src/dfa.rs:658-667, 675-682).  Results against the oracle on slices and against closed-form
expectations at full size; the fix-up counters must stay small."""
import random
import re as pyre

import numpy as np
import pytest

import regex_b200 as R
from helpers import tiled_corpus, xorshift_bytes
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _spans(a):
    return [tuple(int(v) for v in r) for r in np.asarray(a).reshape(-1, 2).tolist()]


def _device_repeat(base, reps):
    import torch
    return torch.frombuffer(bytearray(base), dtype=torch.uint8).cuda().repeat(reps)


def test_sticky_automaton_is_solved_by_state_map_composition():
    """`(?s)foo.*bar` over 256 MiB: the reverse scan's state is "a bar lies somewhere to the right" for
    the whole haystack, which no warm-up can guess; the single match covers ~260 000 chunks and is
    measured by the parallel long-run pass (state maps of the anchored automaton from `foo` on)."""
    import torch
    base = tiled_corpus(16 << 20)
    reps = 64
    d = _device_repeat(base, reps)
    n = d.numel()
    first_foo = base.find(b"foo")
    last_bar = (reps - 1) * len(base) + base.rfind(b"bar")
    assert 0 <= first_foo < last_bar
    r = R.BytesRegex(r"(?s)foo.*bar")
    out = torch.empty((16, 2), dtype=torch.int64, device="cuda")
    total = r.find_all_device(d, out)
    st = r.last_stats()
    assert total == 1 and _spans(out[:1].cpu().numpy()) == [(first_foo, last_bar + 3)]
    assert st["map_passes"] > 0 and st["scan_redo_rounds"] <= 6, st
    assert st["stitch_rounds"] <= 4 and st["sequential_passes"] == 0 and st["long_runs"] == 1, st
    assert st["total_ms"] < 2000, st
    # forward searches: the same stickiness left to right, plus the early exit
    assert r.shortest_match_device(d) == base.find(b"bar", first_foo + 3) + 3
    assert r.last_stats()["waves"] == 1
    # small haystack, tiny segments: the same machinery against the oracle
    small = base[:300000]
    r2 = R.BytesRegex(r"(?s)foo.*bar")
    r2.set_tuning(seg=64, chunk=256)
    assert _spans(r2.find_all(small)) == O.OracleRegex(r"(?s)foo.*bar").find_iter(small)
    assert r2.last_stats()["map_passes"] > 0


def test_state_map_composition_in_both_scan_directions():
    """`(?s)foo.*bar` with 2400 bytes between the `foo` and the `bar`: on 64-byte segments the warm-up guess
    is wrong for every segment between them, in both scan directions.  With no plain redo round allowed,
    the entry states are composed from state maps at once: in the reverse start scan (find_all, whole and
    in two shards) and in the forward scans (shortest_match, RegexSet::matches)."""
    import torch
    from test_gpu_parity import _run_gpu_shards
    filler = xorshift_bytes(5, 2800, b"xyz \n")
    text = filler[:200] + b"foo" + filler[200:2600] + b"bar" + filler[2600:]
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    pat = r"(?s)foo.*bar"
    oracle = O.OracleRegex(pat)
    exp = oracle.find_iter(text)
    assert len(exp) == 1

    def tuned(re_):
        re_.set_tuning(seg=64)
        re_.set_option("max_redo_rounds", 0)
        return re_

    r = tuned(R.BytesRegex(pat))
    assert _spans(r.find_all(text)) == exp
    assert r.last_stats()["map_passes"] > 0
    assert r.shortest_match_device(d) == oracle.shortest_match_at(text)
    assert r.last_stats()["map_passes"] > 0
    pats = [pat, r"zzzq"]
    s = tuned(R.BytesRegexSet(pats))
    assert s.matches_device(d) == list(O.OracleRegex(pats).set_matches(text))
    assert s.last_stats()["map_passes"] > 0
    stats = {}
    got = _run_gpu_shards(pat, text, d, 2, len(exp), halo=1 << 16, tuning={"seg": 64}, options={"max_redo_rounds": 0}, stats=stats)
    assert got == exp
    assert any(st["map_passes"] > 0 for st in stats.values()), stats


def test_matches_longer_than_the_run_cap_against_python_re():
    """Several multi-MiB matches next to short ones: each long one is one parallel long-run pass."""
    filler = tiled_corpus(5 << 20).replace(b"<<", b"< ").replace(b">>", b"> ")
    parts = []
    for i in range(3):
        parts += [b"x <<", filler[: (2 + i) << 20], b">> y <<short>> "]
    text = b"".join(parts) + filler[:70000]
    for pat in (r"(?s)<<.*?>>", r"(?s)<<(?:[^>]|>[^>])*>>", r"(?s)<<.*?>>|short"):
        exp = [m.span() for m in pyre.finditer(pat.encode(), text)]
        assert len(exp) >= 6
        r = R.BytesRegex(pat)
        assert _spans(r.find_all(text)) == exp, pat
        st = r.last_stats()
        assert st["long_runs"] == 3 and st["sequential_passes"] == 0, (pat, st)
    # an automaton too large for the long-run pass keeps the one-thread run (and stays exact)
    pat = r"(?s)<<.*?>>|" + "|".join("q%dz{3}w" % i for i in range(60))
    r = R.BytesRegex(pat)
    assert _spans(r.find_all(text[: 3 << 20])) == [m.span() for m in pyre.finditer(pat.encode(), text[: 3 << 20])]


def test_lazy_dotall_comments_spanning_many_chunks():
    import torch
    filler = tiled_corpus(3 << 20).replace(b"*/", b"* ").replace(b"/*", b"/ ")
    text = b"".join(b"code(); /* " + filler[i * 700000:(i + 1) * 700000] + b" */ more();\n" for i in range(4)) + filler[:100000]
    pat = r"(?s)/\*.*?\*/"
    exp = [m.span() for m in pyre.finditer(pat.encode(), text)]
    assert len(exp) == 4
    r = R.BytesRegex(pat)
    assert _spans(r.find_all(text)) == exp
    st = r.last_stats()
    assert st["scan_redo_rounds"] <= 6 and st["stitch_rounds"] <= 6, st
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for world in (2, 3):
        from test_gpu_parity import _run_gpu_shards
        try:
            got = _run_gpu_shards(pat, text, d, world, len(exp), halo=1 << 16)
        except R.Error as e:
            assert "enlarge the halo" in str(e)  # a 700 KB match cannot fit a 64 KiB halo: explicit error
            continue
        assert got == exp


@pytest.mark.parametrize("chunk,n", [(256, 200000), (4096, 3 << 20)])
def test_chains_that_never_meet_fall_back_to_one_sequential_pass(chunk, n):
    """`(?s).{7}` tiles the haystack out of phase with every chunk: each chunk's speculative chain is
    wrong and stays wrong, so re-walk rounds would cascade one chunk at a time."""
    text = xorshift_bytes(3, n, b"abcdefgh\n")
    r = R.BytesRegex(r"(?s-u).{7}")
    r.set_tuning(chunk=chunk)
    r.set_option("max_stitch_rounds", 6)
    got = r.find_all(text)
    k = n // 7
    exp = np.stack([np.arange(k) * 7, np.arange(k) * 7 + 7], axis=1)
    assert got.shape == exp.shape and (np.asarray(got, dtype=np.int64) == exp).all()
    st = r.last_stats()
    assert st["sequential_passes"] >= 1 and st["stitch_rounds"] <= 40, st
    # variable-length variant through the table runner
    r = R.BytesRegex(r"(?s-u).{6,7}?")
    r.set_tuning(chunk=chunk)
    r.set_option("max_stitch_rounds", 6)
    small = text[:100000]
    assert _spans(r.find_all(small)) == O.OracleRegex(r"(?s-u).{6,7}?").find_iter(small)


def test_sequential_pass_with_a_generic_table_over_48_kib():
    """The sequential pass stages the generic runner's table in shared memory as the chunk walks do: a tiling
    pattern whose anchored table is over the 48 KiB a kernel gets without opting in."""
    rng = random.Random(7)
    alphabet = "abcdefghijklmnopqrstuvwxyz0123456789ABCD"
    words = set()
    while len(words) < 250:
        words.add("".join(rng.choice(alphabet) for _ in range(6)))
    pat = r"(?s-u).{7}|" + "|".join(sorted(words))
    r = R.BytesRegex(pat)
    table = r.dfa(R.DFA_FWD_ANCHORED_LF)["trans"]
    assert 48 << 10 < table.nbytes <= 200 << 10, table.shape
    r.force_generic(True)
    r.set_tuning(chunk=256)
    r.set_option("max_stitch_rounds", 0)
    n = 200000
    text = xorshift_bytes(3, n, b"abcdefgh\n")
    got = r.find_all(text)
    k = n // 7  # the 3 bytes left over are too few for a word
    exp = np.stack([np.arange(k) * 7, np.arange(k) * 7 + 7], axis=1)
    assert got.shape == exp.shape and (np.asarray(got, dtype=np.int64) == exp).all()
    assert r.last_stats()["sequential_passes"] >= 1, r.last_stats()


def test_forward_search_waves_and_early_exit():
    import torch
    line = b"the quick brown fox jumps over the lazy dog 0123456789\n"
    a = line * ((40 << 20) // len(line))
    text = a + b"xx NEEDLE yy\n" + line * ((30 << 20) // len(line))
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for pat, exp in [(r"NEEDLE", len(a) + 3 + 6), (r"quick", text.find(b"quick") + 5), (r"zebra", None), (r"dog \d+\nxx", len(a) + 2)]:
        r = R.BytesRegex(pat)
        r.set_option("wave0", 32 << 20)
        assert r.shortest_match_device(d) == exp, pat
        waves = r.last_stats()["waves"]
        assert waves == (1 if pat == "quick" else 2), (pat, waves)
        r.set_option("wave0", 0)
        assert r.shortest_match_device(d) == exp, pat
    # every wave boundary state is exact: a match that straddles the first boundary, tiny waves
    r = R.BytesRegex(r"lazy dog \d+\nthe quick")
    r.set_option("wave0", 4096)
    small = text[:100000]
    small_d = d[:100000].clone()
    assert r.shortest_match_device(small_d) == O.OracleRegex(r"lazy dog \d+\nthe quick").shortest_match_at(small)
    for pat in (r"fox\s+jumps", r"\d{11}", r"(?m)^the lazy", r"9\n$"):
        r = R.BytesRegex(pat)
        r.set_option("wave0", 4096)
        assert r.shortest_match_device(small_d) == O.OracleRegex(pat).shortest_match_at(small), pat


def test_regex_set_narrowing_equals_the_product_automaton():
    import torch
    base = tiled_corpus(24 << 20)
    late = b" zyxwvut 987654 "
    text = base[:20 << 20] + late + base[20 << 20:]
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    pats = [r"\w+", r"\d+", r"Holmes", r"zyxwvut", r"9876\d+", r"qqqqqq", r"(?i)WATSON\s", r"^The", r"\.$", r"xyzzy|plugh", r"[A-Z][a-z]+ing"]
    exp = [i for i, p in enumerate(pats) if pyre.search(p.encode(), text, 0) is not None]
    exp_oracle = list(O.OracleRegex(pats).set_matches(text[:1 << 20]))
    for wave0, narrow in ((1 << 20, 1), (1 << 20, 0), (0, 1), (32 << 20, 1)):
        s = R.BytesRegexSet(pats)
        s.set_option("wave0", wave0)
        s.set_option("narrow_sets", narrow)
        assert s.matches_device(d) == exp, (wave0, narrow)
        assert s.matches(text[:1 << 20]) == exp_oracle
    s = R.BytesRegexSet(pats)
    s.set_option("wave0", 1 << 20)
    s.matches_device(d)
    assert s.last_stats()["waves"] >= 3
    # all patterns match early: one wave, no narrowing needed (dfa.rs:675-682)
    s = R.BytesRegexSet([r"\w+", r"Holmes", r"\s"])
    s.set_option("wave0", 1 << 20)
    assert s.matches_device(d) == [0, 1, 2] and s.last_stats()["waves"] == 1


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_forward_searches_on_the_gpu(world):
    """is_match / shortest_match / RegexSet::matches over byte-range shards driven through one GPU
    (one thread per shard, in-process collectives): first-end min and mask OR must equal the
    whole-haystack answers; sticky automata need the exact-state exchange."""
    import threading
    import torch
    from regex_b200 import sharded
    text = tiled_corpus(3 << 20) + b" NEEDLE " + tiled_corpus(1 << 20, seed=9)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()

    def run(make, fn_expected):
        comm = sharded.ThreadComm(world)
        out, errs = [None] * world, []

        def work(rank):
            try:
                re_ = make()
                re_.set_option("wave0", 1 << 18)
                geom = sharded.plan(len(text), world, rank, halo=256)
                buf = d_text[geom.buf_lo:geom.buf_hi].clone()
                out[rank] = sharded.forward_sharded(lambda io: re_.forward_shard_device(buf, io), geom, comm.view(rank))
            except Exception as e:  # noqa: BLE001
                errs.append(e)
                comm._barrier.abort()

        threads = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=120)
            assert not t.is_alive()
        assert not errs, errs
        assert all(o[:2] == out[0][:2] for o in out)
        return out[0]

    for pat in (r"NEEDLE", r"Holmes", r"qqqqqqqq", r"(?s)Sherlock.*NEEDLE", r"(?m)^NEEDLE", r"E \w+\s"):
        first, _, _ = run(lambda: R.BytesRegex(pat), None)
        assert first == O.OracleRegex(pat).shortest_match_at(text), pat
    pats = [r"\w+", r"NEEDLE", r"qqqqqq", r"(?s)NEEDLE.*Watson", r"(?s)Watson.*NEEDLE", r"\d{7}", r"(?i)needle "]
    _, masks, _ = run(lambda: R.BytesRegexSet(pats), None)
    exp = [i for i, p in enumerate(pats) if pyre.search(p.encode(), text) is not None]
    assert [i for i in range(len(pats)) if (masks[0] >> i) & 1] == exp


def test_scalar_find_searches_in_growing_windows():
    """rure_find on a host haystack uploads and searches windows from `start` (64 KiB, x8 each) and
    stops at the first span: the C idiom `while (rure_find(re, h, n, pos, &m)) pos = m.end;` must
    cost about one pass, not one pass per call; results equal the oracle's find_at everywhere,
    including look-around patterns whose windows start in the middle of the text."""
    import time
    text = tiled_corpus(48 << 20) + b" NEEDLE at the end\n"
    r = R.BytesRegex(r"Holmes|Watson")
    exp = O.OracleRegex(r"Holmes|Watson").find_iter(text[:4 << 20])
    t0 = time.perf_counter()
    pos, got = 0, []
    while len(got) < 1500:
        m = r.find_at(text, pos)
        got.append(m)
        pos = m[1]
    dt = time.perf_counter() - t0
    assert got == exp[:1500]
    assert dt < 30, dt  # the whole-haystack version of this loop moves 1500 x 48 MiB over PCIe
    # a match hundreds of windows away, and none at all
    r = R.BytesRegex(r"NEEDLE")
    assert r.find_at(text, 12345) == (text.find(b"NEEDLE"), text.find(b"NEEDLE") + 6)
    assert r.find_at(text, text.find(b"NEEDLE") + 1) is None
    assert r.is_match_at(text, 5) and not R.BytesRegex(r"NEEDLES").is_match(text)
    assert R.BytesRegex(r"Sherlock").shortest_match_at(text, 1000) == text.find(b"Sherlock", 1000) + 8
    small = text[:3 << 20]
    for pat in (r"(?m)^\w+$", r"(?-u:\b)the(?-u:\b)", r"\w*", r"(?m)^[ab]{2,}\w*?|(?m:$)", r"[^\n]{60,}", r"(?s)Gutenberg.*Gutenberg"):
        r, o = R.BytesRegex(pat), O.OracleRegex(pat)
        for start in (0, 1, 255, 256, 257, 65535, 65536, 65537, 131072, 600000, 2000001, len(small) - 3, len(small)):
            assert r.find_at(small, start) == o.find_at(small, start), (pat, start)
            assert r.shortest_match_at(small, start) == o.shortest_match_at(small, start), (pat, start)


def test_one_compiled_regex_from_several_threads():
    """rure.h:27-34: a compiled regex may be used from multiple threads simultaneously.  The engine's device
    scratch is per object; the scalar entry points lease an idle engine (a clone when the object is busy)."""
    import threading
    base = tiled_corpus(1 << 20)
    pats = [r"[a-zA-Z]+ing", r"(?i)holmes\s+\w+", r"\d{3,}"]
    regs = [R.BytesRegex(p) for p in pats]
    sets = R.BytesRegexSet([r"Holmes", r"Watson", r"zzzzqq", r"\d+"])
    hays = [base[i * 50000:(i + 3) * 50000 + 17 * i] for i in range(8)]
    exp = [[(m.span() if m else None) for m in (pyre.search(p.encode(), h) for h in hays)] for p in pats]
    exp_set = [[i for i, p in enumerate([rb"Holmes", rb"Watson", rb"zzzzqq", rb"\d+"]) if pyre.search(p, h)] for h in hays]
    errors = []

    def worker(tid):
        try:
            for rep in range(6):
                for j in range(len(hays)):
                    k = (j + tid + rep) % len(hays)
                    for pi, r in enumerate(regs):
                        got = r.find(hays[k])
                        assert (tuple(got) if got else None) == exp[pi][k], (pats[pi], k)
                        assert r.is_match(hays[k]) == (exp[pi][k] is not None)
                    assert list(sets.matches(hays[k])) == exp_set[k]
        except Exception as e:  # noqa: BLE001
            errors.append((tid, repr(e)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:3]
