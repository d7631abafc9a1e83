#!/usr/bin/env python
"""Candidate-start mode (DESIGN.md §2) on one GPU: patterns whose unanchored automata exceed the table budget.

  find_all_device   `Holmes.{0,40}Watson`, `[a-z]+.{0,30}ing` over --gib GiB of C2 (sherlock lines), with
                    `Holmes|Watson` on the DFA path in the same run as the reference point
  find_iter_batch / is_match_batch   `[a-z]+.{0,30}ing` over --lines C3 log lines (device-resident)
  compile           seconds to compile each pattern (host determinization)

Oracle checks: find_iter on the first and last --window bytes of the C2 haystack (matches inside each window that
end at least 4 KiB before its edge), and every call on the first --check-lines C3 lines.  The candidate path's
speed is set by the candidate density times the anchored run length.  Prints one JSON line (and appends it to --out).
  python tools/bench_candidate.py [--gib 16] [--lines 100000000] [--out profiles/<name>.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch

import corpus as C
import regex_b200 as R
from bench_batch_iter import card
from bench_configs import _frac, timed, use_torch_stream

C2_PATTERNS = [r"Holmes.{0,40}Watson", r"[a-z]+.{0,30}ing", r"Holmes|Watson"]
C3_PATTERN = r"[a-z]+.{0,30}ing"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=16)
    ap.add_argument("--lines", type=int, default=100_000_000)
    ap.add_argument("--check-lines", type=int, default=20000)
    ap.add_argument("--window", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    from oracle import oracle as O
    res = {"compile_s": {}}
    objs = {}
    for pat in C2_PATTERNS:
        t0 = time.perf_counter()
        objs[pat] = use_torch_stream(R.BytesRegex(pat))
        res["compile_s"][pat] = round(time.perf_counter() - t0, 3)

    # ---- C2: whole haystack ----
    nbytes = int(a.gib * (1 << 30))
    text = C.device_corpus(nbytes, C.SEED, dev)
    n = text.numel()
    w = a.window
    heads = [(0, text[:w].cpu().numpy().tobytes()), (n - w, text[n - w:].cpu().numpy().tobytes())]
    for pat in C2_PATTERNS:
        r = objs[pat]
        total = r.find_all_device(text)
        out = torch.empty((total + 16, 2), dtype=torch.int64, device=dev)
        ms, got = timed(lambda: r.find_all_device(text, out), steps=a.steps, warmup=1)
        assert got == total
        path = int(r.last_stats()["path"])
        spans = out[:total].cpu().numpy()
        o, bad, checked = O.OracleRegex(pat), 0, 0
        for lo, h in heads:
            exp = [(s + lo, e + lo) for s, e in o.find_iter(h) if s >= (4096 if lo else 0) and e + 4096 <= len(h)]
            sel = spans[(spans[:, 0] >= exp[0][0]) & (spans[:, 1] <= exp[-1][1])] if exp else spans[:0]
            bad += [tuple(map(int, x)) for x in sel.tolist()] != exp
            checked += len(exp)
        gbs, frac = _frac(n, ms)
        res[f"c2_find_all[{pat}]"] = {"matches": total, "ms": round(ms, 3), "GB_s": gbs, "hbm_frac": frac, "path": path,
                                      "oracle_checked_matches": checked, "oracle_mismatches": int(bad)}
        del out
    del text
    torch.cuda.empty_cache()

    # ---- C3: batched records ----
    text, offsets = C.log_lines(a.lines, dev)
    nl = a.lines
    k = min(a.check_lines, nl)
    host, offs = text[:int(offsets[k])].cpu().numpy().tobytes(), offsets[:k + 1].tolist()
    t0 = time.perf_counter()
    r = use_torch_stream(R.BytesRegex(C3_PATTERN))
    res["compile_s"][C3_PATTERN + " (C3)"] = round(time.perf_counter() - t0, 3)
    o = O.OracleRegex(C3_PATTERN)
    per = [o.find_iter(host[offs[i]:offs[i + 1]]) for i in range(k)]
    moff = torch.empty(nl + 1, dtype=torch.int64, device=dev)
    m = r.find_iter_batch_device(text, offsets, moff)
    spans = torch.empty((m, 2), dtype=torch.int64, device=dev)
    ms, got = timed(lambda: r.find_iter_batch_device(text, offsets, moff, spans), steps=a.steps, warmup=1)
    assert got == m
    mo, sp = moff[:k + 1].tolist(), spans[:int(moff[k])].cpu().numpy().tolist()
    bad = sum([tuple(x) for x in sp[mo[i]:mo[i + 1]]] != per[i] for i in range(k))
    gbs, frac = _frac(text.numel() + 16 * nl + 16 * m, ms)
    res["c3_find_iter_batch"] = {"pattern": C3_PATTERN, "matches": m, "ms": round(ms, 3), "Mlines_s": round(nl / ms / 1e3, 1), "GB_s": gbs,
                                 "oracle_checked_lines": k, "oracle_mismatches": int(bad)}
    del spans
    bits = torch.empty((nl + 31) // 32 + 1, dtype=torch.int32, device=dev)
    ms, _ = timed(lambda: r.is_match_batch_device(text, offsets, bits), steps=a.steps, warmup=1)
    hb = bits.cpu().numpy().view("uint32")
    bad = sum(bool((hb[i >> 5] >> (i & 31)) & 1) != bool(per[i]) for i in range(k))
    res["c3_is_match_batch"] = {"pattern": C3_PATTERN, "ms": round(ms, 3), "Mlines_s": round(nl / ms / 1e3, 1),
                                "oracle_checked_lines": k, "oracle_mismatches": int(bad)}

    line = json.dumps({
        "workload": f"C2 (sherlock lines, {a.gib} GiB) find_all_device; C3 synthetic log lines ({a.lines}) find_iter_batch / is_match_batch",
        "card": card(), "timing": f"CUDA events on torch's stream, mean of {a.steps} calls after one warm-up call",
        "paths": "stats path 4 = candidate starts, 3 = literal prefilter, 0-2 = DFA scan", "results": res})
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    assert all(v.get("oracle_mismatches", 0) == 0 for v in res.values() if isinstance(v, dict)), "oracle mismatches"


if __name__ == "__main__":
    main()
