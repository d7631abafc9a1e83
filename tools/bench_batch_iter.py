#!/usr/bin/env python
"""Per-record find_iter, match counts and captures over the C3 log lines, device-resident, on one GPU.

For each call: Mlines/s, GB/s on algorithmic bytes, the fraction of the measured HBM bandwidth, and an
oracle check of the first --check-lines lines (every span / every group).  find_batch on the same input is
measured in the same run as the reference point.  Prints one JSON line (and appends it to --out).
  python tools/bench_batch_iter.py [--lines 100000000] [--out profiles/<name>.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import corpus as C
import regex_b200 as R
from bench_configs import _frac, hbm_peak, timed, use_torch_stream

DATE = r"(\d{4})-(\d{2})-(\d{2})"
PATTERNS = [DATE, r"[a-z]+ing", r"\w+"]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number still stands with the card's name; say why the limit is missing
        q = f"unavailable ({e})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def check_iter(o, host, offs, moff, spans, k):
    bad = 0
    for i in range(k):
        exp = o.find_iter(host[offs[i]:offs[i + 1]])
        got = spans[moff[i]:moff[i + 1]]
        if len(exp) != got.shape[0] or (exp and not (got == np.array(exp, dtype=np.int64)).all()):
            bad += 1
    return bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=100_000_000)
    ap.add_argument("--check-lines", type=int, default=20000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    from oracle import oracle as O
    text, offsets = C.log_lines(a.lines, dev)
    n, nbytes = a.lines, text.numel()
    k = min(a.check_lines, n)
    host = text[:int(offsets[k])].cpu().numpy().tobytes()
    offs = offsets[:k + 1].tolist()
    res = {}
    for pat in PATTERNS:
        r = use_torch_stream(R.BytesRegex(pat))
        o = O.OracleRegex(pat)
        moff = torch.empty(n + 1, dtype=torch.int64, device=dev)
        ms_count, total = timed(lambda: r.find_iter_batch_device(text, offsets, moff), steps=a.steps, warmup=1)
        spans = torch.empty((total, 2), dtype=torch.int64, device=dev)
        ms_iter, total2 = timed(lambda: r.find_iter_batch_device(text, offsets, moff, spans), steps=a.steps, warmup=1)
        assert total2 == total
        bad = check_iter(o, host, offs, moff[:k + 1].tolist(), spans[:int(moff[k])].cpu().numpy(), k)
        gb_c, f_c = _frac(nbytes + 8 * (n + 1) + 8 * n, ms_count)
        gb_i, f_i = _frac(nbytes + 8 * (n + 1) + 8 * n + 16 * total, ms_iter)
        row = {"matches": total, "matches_per_line": round(total / n, 3),
               "find_iter_batch": {"ms": round(ms_iter, 3), "Mlines_s": round(n / ms_iter / 1e3, 1), "GB_s": gb_i, "hbm_frac": f_i},
               "count_batch": {"ms": round(ms_count, 3), "Mlines_s": round(n / ms_count / 1e3, 1), "GB_s": gb_c, "hbm_frac": f_c},
               "oracle_checked_lines": k, "oracle_mismatches": bad}
        del spans
        if pat == DATE:
            bits = torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev)
            first = torch.empty((n, 2), dtype=torch.int64, device=dev)
            ms_find, _ = timed(lambda: r.find_batch_device(text, offsets, first, bits), steps=a.steps, warmup=1)
            gb_f, f_f = _frac(nbytes + 8 * (n + 1) + n / 8 + 16 * n, ms_find)
            row["find_batch"] = {"ms": round(ms_find, 3), "Mlines_s": round(n / ms_find / 1e3, 1), "GB_s": gb_f, "hbm_frac": f_f}
            del first
            g = r.captures_len()
            slots = torch.empty(n * 2 * g, dtype=torch.int64, device=dev)
            ms_cap, _ = timed(lambda: r.captures_batch_device(text, offsets, slots, bits), steps=a.steps, warmup=1)
            sl = slots[:k * 2 * g].cpu().numpy().view(np.uint64).reshape(k, g, 2)
            bw = np.unpackbits(bits[:(k + 31) // 32].cpu().numpy().view(np.uint8), bitorder="little")
            cbad = 0
            for i in range(k):
                exp = o.captures_at(host[offs[i]:offs[i + 1]])
                got = None if not bw[i] else [None if int(x) == 2**64 - 1 else (int(x), int(y)) for x, y in sl[i]]
                cbad += got != exp
            gb_cap, f_cap = _frac(nbytes + 8 * (n + 1) + n / 8 + 16 * g * n, ms_cap)
            row["captures_batch"] = {"groups": g, "ms": round(ms_cap, 3), "Mlines_s": round(n / ms_cap / 1e3, 1), "GB_s": gb_cap, "hbm_frac": f_cap,
                                     "oracle_checked_lines": k, "oracle_mismatches": cbad}
            del slots, bits
        res[pat] = row
    out = {"workload": f"C3 per-line find_iter / count / captures over {n} synthetic log lines (tools/corpus.py log_lines), device-resident",
           "lines": n, "haystack_bytes": nbytes, "card": card(), "hbm_peak": hbm_peak()[1],
           "algorithmic_bytes": {"find_iter_batch": "line bytes + 8 B offsets + 8 B match offset per line + 16 B per span",
                                 "count_batch": "line bytes + 8 B offsets + 8 B count per line",
                                 "find_batch": "line bytes + 8 B offsets + 1 bit + 16 B span per line",
                                 "captures_batch": "line bytes + 8 B offsets + 1 bit + 16 B per group per line"},
           "timing": f"CUDA events on torch's stream, mean of {a.steps} calls after one warm-up call", "results": res}
    line = json.dumps(out)
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    assert all(v["oracle_mismatches"] == 0 and v.get("captures_batch", {}).get("oracle_mismatches", 0) == 0 for v in res.values()), "oracle mismatches"


if __name__ == "__main__":
    main()
