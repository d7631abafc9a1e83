#!/usr/bin/env python
"""Streams against the whole-haystack host search, on one GPU (DESIGN.md §8).

16 GiB of tools/corpus.py text in pinned host memory, `[a-zA-Z]+ing`, searched four ways:
  (a) rure_b200_find_all on the pinned buffer (uploaded in 64 MiB pieces, searched resident),
  (b) a stream fed in 64 MiB writes from the pinned buffer,
  (c) the same from pageable memory (every write copied through the stream's pinned staging),
  (d) rure_b200_find_all forced through the bounded window (option "host_window" = 256 MiB).
All four must give identical spans.  Then a count-only stream over copies of the buffer written
back to back until the text is longer than the card's memory.  Rates are haystack bytes over
wall time of a call that ends with its results on the host; the median of --steps runs.
Prints one JSON line (and writes it to --out).
  python tools/bench_stream.py [--gib 16] [--out profiles/r07_bench_stream.json]
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

PATTERN = r"[a-zA-Z]+ing"
WRITE = 64 << 20


def timed(fn, steps):
    ts, out = [], None
    for _ in range(steps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def stream_spans(r, src, n, total):
    """a stream fed `src` (a pinned tensor or a numpy array) in 64 MiB writes; spans into one array"""
    out = np.empty((total, 2), dtype=np.uint64)
    got = 0
    with r.stream() as s:
        for pos in range(0, n, WRITE):
            s.write(src[pos:pos + WRITE])
            k = s.read()
            out[got:got + len(k)] = k
            got += len(k)
        s.finish()
        k = s.read()
        out[got:got + len(k)] = k
        got += len(k)
    assert got == total, (got, total)
    return out


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
    pageable = np.empty(n, dtype=np.uint8)
    pageable[:] = pinned.numpy()
    r = R.BytesRegex(PATTERN)
    total = r.count_all(pinned)
    res = {"pattern": PATTERN, "bytes": n, "matches": total, "card": card()}
    print(f"{n} bytes, {total} matches", flush=True)

    # (a) warm up every path on a 1 GiB prefix first
    r.find_all(pinned[:1 << 30], cap=total)
    stream_spans(r, pinned[:1 << 30], 1 << 30, r.count_all(pinned[:1 << 30]))
    legs = {}

    def leg(name, dt):
        legs[name] = dt
        print(f"{name}: {dt:.3f} s, {n / dt / 1e9:.1f} GB/s", flush=True)

    dt, ref = timed(lambda: r.find_all(pinned, cap=total), a.steps)
    leg("a_find_all_pinned", dt)
    dt, got = timed(lambda: stream_spans(r, pinned, n, total), a.steps)
    leg("b_stream_pinned", dt)
    res["b_equal"] = bool(np.array_equal(got, ref))
    del got
    dt, got = timed(lambda: stream_spans(r, pageable, n, total), a.steps)
    leg("c_stream_pageable", dt)
    res["c_equal"] = bool(np.array_equal(got, ref))
    del got
    r.set_option("host_window", 256 << 20)
    dt, got = timed(lambda: r.find_all(pinned, cap=total), a.steps)
    leg("d_find_all_window", dt)
    res["d_equal"] = bool(np.array_equal(got, ref))
    r.set_option("host_window", 0)
    del got, ref
    res["seconds"] = legs
    res["gb_per_s"] = {k: n / v / 1e9 for k, v in legs.items()}

    # count-only stream over copies of the buffer until the text is longer than the card's memory
    dev_bytes = torch.cuda.get_device_properties(0).total_memory
    copies = dev_bytes // n + 1
    edge = 4096  # matches of this pattern never span more than a line
    ht = bytes(pinned[n - edge:].numpy()) + bytes(pinned[:edge].numpy())
    seam = r.count_all(ht) - r.count_all(ht[:edge]) - r.count_all(ht[edge:])
    t0 = time.perf_counter()
    with r.stream(spans=False) as s:
        for _ in range(copies):
            for pos in range(0, n, WRITE):
                s.write(pinned[pos:pos + WRITE])
        s.finish()
        big = s.count
    dt = time.perf_counter() - t0
    res["larger_than_device"] = {"device_bytes": dev_bytes, "text_bytes": copies * n, "copies": copies, "matches": big,
                                 "expected": copies * total + (copies - 1) * seam, "seconds": dt, "gb_per_s": copies * n / dt / 1e9}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
