#!/usr/bin/env python
"""RegexSets in pattern groups (DESIGN.md §2) on one GPU, with the product automaton as the reference point.

  sets              c4            the C4 64-pattern set: one product automaton (the reference point)
                    words1024     1 024 sherlock vocabulary words as literals (4 groups of 256)
                    over_budget   \\w+, \\d+, \\s+, [A-Z][a-z]+ and 60 `(?i)<word>\\s+\\w+`: the product is over the budget
                    c4_k16        C4 with set_group_patterns = 16 (4 groups)
  matches_device    over --gib GiB of C2 (sherlock lines): the first call (narrowing compiles a subset of the
                    patterns still open after two waves) and the steady state, with waves and groups
  matches_batch_device   over --lines C3 log lines (device-resident), lines/s
  compile           seconds to compile each set (host determinization, including a failed product attempt)

Oracle checks: set_matches on the first and last --window bytes of the C2 haystack (device slices; the oracle runs at
about 1 MB/s on these sets, so the windows are 8 MiB), and every
record of the first --check-lines C3 lines.  Prints one JSON line (and appends it to --out).
  python tools/bench_set_groups.py [--gib 16] [--lines 100000000] [--out profiles/<name>.json]
"""
import argparse
import json
import os
import re
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import corpus as C
import regex_b200 as R
from bench_batch_iter import card
from bench_configs import _frac, timed, use_torch_stream


def sets():
    text = open(os.path.join(ROOT, "tests", "golden", "sherlock.txt"), "rb").read()
    words = [w.decode() for w in sorted(set(re.findall(rb"[A-Za-z]{4,}", text)))]
    return {
        "c4": (C.c4_patterns(), 0),
        "words1024": (words[:1024], 0),
        "over_budget": ([r"\w+", r"\d+", r"\s+", r"[A-Z][a-z]+"] + [rf"(?i){w}\s+\w+" for w in words[200:260]], 0),
        "c4_k16": (C.c4_patterns(), 16),
    }


def rows(masks, n_pat):
    return [[i for i in range(n_pat) if (int(r[i // 64]) >> (i % 64)) & 1] for r in masks]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=16)
    ap.add_argument("--lines", type=int, default=100_000_000)
    ap.add_argument("--check-lines", type=int, default=20000)
    ap.add_argument("--window", type=int, default=8 << 20)  # the oracle runs at about 1 MB/s on these sets
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    from oracle import oracle as O
    pool = ThreadPoolExecutor(8)  # oracle checks (ctypes releases the GIL)
    res = {"compile_s": {}, "groups": {}}
    objs = {}
    for name, (pats, k) in sets().items():
        t0 = time.perf_counter()
        s = R.BytesRegexSet(pats)
        if k:
            s.set_option("set_group_patterns", k)
        res["compile_s"][name] = round(time.perf_counter() - t0, 3)
        res["groups"][name] = s.groups()
        objs[name] = (use_torch_stream(s), pats)

    # ---- C2: whole haystack ----
    nbytes = int(a.gib * (1 << 30))
    text = C.device_corpus(nbytes, C.SEED, dev)
    n = text.numel()
    w = min(a.window, n)
    for name, (s, pats) in objs.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        first = s.matches_device(text)
        first_ms = (time.perf_counter() - t0) * 1e3
        first_stats = s.last_stats()
        ms, got = timed(lambda: s.matches_device(text), steps=a.steps, warmup=1)
        assert got == first
        st = s.last_stats()
        checks = [(s.matches_device(text[lo:lo + w]), pats, text[lo:lo + w].cpu().numpy().tobytes()) for lo in (0, n - w)]
        bad = sum(pool.map(lambda c: c[0] != O.OracleRegex(c[1]).set_matches(c[2]), checks))
        gbs, frac = _frac(n, ms)
        res[f"c2_matches_device[{name}]"] = {
            "patterns": len(pats), "matched": len(first), "first_call_ms": round(first_ms, 3),
            "first_call_waves": int(first_stats["waves"]), "ms": round(ms, 3), "GB_s": gbs, "hbm_frac": frac,
            "waves": int(st["waves"]), "groups": int(st["groups"]), "oracle_checked_windows": 2, "oracle_mismatches": int(bad)}
    del text
    torch.cuda.empty_cache()

    # ---- C3: batched records ----
    text, offsets = C.log_lines(a.lines, dev)
    nl = a.lines
    k = min(a.check_lines, nl)
    host, offs = text[:int(offsets[k])].cpu().numpy().tobytes(), offsets[:k + 1].tolist()
    for name, (s, pats) in objs.items():
        mw = (len(pats) + 63) // 64
        out = torch.empty((nl, mw), dtype=torch.int64, device=dev)
        ms, _ = timed(lambda: s.matches_batch_device(text, offsets, out), steps=a.steps, warmup=1)
        got = rows(out[:k].cpu().numpy().view(np.uint64), len(pats))

        def check(lo, hi):  # one oracle object per thread
            o = O.OracleRegex(pats)
            return sum(got[i] != o.set_matches(host[offs[i]:offs[i + 1]]) for i in range(lo, hi))
        bad = sum(pool.map(lambda lo: check(lo, min(k, lo + 2500)), range(0, k, 2500)))
        gbs, frac = _frac(text.numel() + 8 * nl + 8 * mw * nl, ms)
        res[f"c3_matches_batch_device[{name}]"] = {"ms": round(ms, 3), "Mlines_s": round(nl / ms / 1e3, 1), "GB_s": gbs,
                                                   "groups": int(s.last_stats()["groups"]), "oracle_checked_lines": k,
                                                   "oracle_mismatches": int(bad)}
        del out

    line = json.dumps({
        "workload": f"C2 (sherlock lines, {a.gib} GiB) matches_device; C3 synthetic log lines ({a.lines}) matches_batch_device",
        "card": card(), "timing": f"CUDA events on torch's stream, mean of {a.steps} calls after one warm-up call; "
                                  "first_call_ms = host clock around the first call (includes narrowing's subset compile)",
        "results": res})
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    assert all(v.get("oracle_mismatches", 0) == 0 for v in res.values() if isinstance(v, dict)), "oracle mismatches"


if __name__ == "__main__":
    main()
