#!/usr/bin/env python
"""Match streams against the resident forward searches, on one GPU (DESIGN.md §8).

16 GiB of tools/corpus.py text in pinned host memory:
  (a) is_match of a pattern with no match (a full pass): resident rure_b200_is_match against a match stream fed in
      64 MiB writes;
  (b) RegexSet::matches of 64 patterns (56 of tools/corpus.py's C4 set and 8 that never match, so no leg can stop
      early): resident, a set match stream, and set_matches forced through the window (option "host_window" 256 MiB);
  (c) a set match stream over copies of the text written back to back until it is longer than the card's memory,
      its mask checked against the resident mask of one copy and of the seam between two copies;
  (d) early exit: one match planted at 1 GiB; the stream stops being fed once decided, against (a)'s full pass.
Every leg's answer must equal the resident one.  Rates are haystack bytes over wall time of a call that ends with its
answer on the host; the median of --steps runs.  Prints one JSON line (and writes it to --out).
  python tools/bench_match_stream.py [--gib 16] [--out profiles/r08_bench_match_stream.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import corpus as C
import regex_b200 as R
from bench_batch_iter import card

ABSENT = r"zqxwvj"
WRITE = 64 << 20
PLANT = 1 << 30


def timed(fn, steps):
    ts, out = [], None
    for _ in range(steps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def feed(stream, src, n, masks=False):
    """src in 64 MiB writes, stopping once the stream is decided; returns the stream's state"""
    with stream as s:
        for pos in range(0, n, WRITE):
            s.write(src[pos:pos + WRITE])
            if s.decided:
                break
        s.finish()
        return {"found": s.found, "end": s.end, "searched": s.searched, "mask": s.mask if masks else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=16)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    n = int(a.gib * (1 << 30)) // 256 * 256
    d = C.device_corpus(n, C.SEED, dev)
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(d)
    del d
    torch.cuda.empty_cache()
    res = {"bytes": n, "card": card()}
    legs = {}

    def leg(name, dt, size=n):
        legs[name] = {"seconds": dt, "gb_per_s": size / dt / 1e9}
        print(f"{name}: {dt:.3f} s, {size / dt / 1e9:.1f} GB/s", flush=True)

    # (a) a full pass
    r = R.BytesRegex(ABSENT)
    r.is_match(pinned[:1 << 30])  # warm-up
    feed(r.match_stream(), pinned, 1 << 30)
    dt, exp = timed(lambda: r.is_match(pinned), a.steps)
    leg("a_is_match_resident", dt)
    dt, got = timed(lambda: feed(r.match_stream(), pinned, n), a.steps)
    leg("a_is_match_stream", dt)
    res["a_equal"] = got["found"] == exp and got["searched"] == n
    full_pass = dt

    # (b) 64 patterns
    pats = C.c4_patterns()[:56] + [f"zqx{i}wvj" for i in range(8)]
    s = R.BytesRegexSet(pats)
    s.matches_mask(pinned[:1 << 30])
    feed(s.match_stream(), pinned, 1 << 30, masks=True)
    dt, exp_mask = timed(lambda: s.matches_mask(pinned), a.steps)
    leg("b_set_matches_resident", dt)
    dt, got = timed(lambda: feed(s.match_stream(), pinned, n, masks=True), a.steps)
    leg("b_set_matches_stream", dt)
    res["b_stream_equal"] = got["mask"] == exp_mask
    s.set_option("host_window", 256 << 20)
    dt, got_w = timed(lambda: s.matches_mask(pinned), a.steps)
    leg("b_set_matches_window", dt)
    res["b_window_equal"] = got_w == exp_mask
    s.set_option("host_window", 0)
    res["set_patterns"] = len(pats)
    res["set_matching"] = sum(bin(w).count("1") for w in exp_mask)

    # (d) early exit at 1 GiB
    saved = pinned[PLANT:PLANT + len(ABSENT)].clone()
    pinned[PLANT:PLANT + len(ABSENT)] = torch.frombuffer(bytearray(ABSENT.encode()), dtype=torch.uint8)
    dt_res, exp_end = timed(lambda: r.shortest_match(pinned), a.steps)
    dt, got = timed(lambda: feed(r.match_stream(), pinned, n), a.steps)
    pinned[PLANT:PLANT + len(ABSENT)] = saved
    res["d_early_exit"] = {"match_end": exp_end, "equal": got["end"] == exp_end, "searched": got["searched"], "seconds": dt,
                           "resident_seconds": dt_res, "full_pass_seconds": full_pass}
    print(f"d: end {got['end']}, searched {got['searched']} bytes in {dt:.3f} s (full pass {full_pass:.3f} s)", flush=True)
    # (c) longer than the card's memory
    dev_bytes = torch.cuda.get_device_properties(0).total_memory
    copies = dev_bytes // n + 1
    edge = 4096
    seam = bytes(pinned[n - edge:].numpy()) + bytes(pinned[:edge].numpy())
    expected = [x | y for x, y in zip(exp_mask, s.matches_mask(seam))]
    t0 = time.perf_counter()
    with s.match_stream() as st:
        for k in range(copies):
            for pos in range(0, n, WRITE):
                st.write(pinned[pos:pos + WRITE])
            print(f"c: copy {k + 1} of {copies} written, {time.perf_counter() - t0:.1f} s", flush=True)
        st.finish()
        dt = time.perf_counter() - t0
        got = {"searched": st.searched, "mask": st.mask}
    res["c_larger_than_device"] = {"device_bytes": dev_bytes, "text_bytes": copies * n, "copies": copies, "searched": got["searched"],
                                   "mask_equal": got["mask"] == expected, "seconds": dt, "gb_per_s": copies * n / dt / 1e9}
    print(f"c: {copies * n} bytes, {copies * n / dt / 1e9:.1f} GB/s", flush=True)

    res["legs"] = legs
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
