#!/usr/bin/env python
"""Per-record replace_all, split and captures_iter over the C3 log lines, device-resident, on one GPU.

  replace_all_batch  NoExpand redaction of the date pattern (`<date>`)   --lines (default 100 M)
  split_batch        on \\s+                                              --lines
  replace_all_batch  `$3/$2/$1` on the date pattern (Pike VM pass)       --pike-lines (default 1 M)
  captures_iter_batch on the date pattern (Pike VM pass)                 --pike-lines

For each call: ms, M lines/s, GB/s on algorithmic bytes (input bytes + output bytes + 8 B per offset entry,
+ 16 B per span / piece or per group slot pair), and the oracle mismatches on the first --check-lines lines.
find_iter_batch on the date pattern is measured in the same run as the reference point.  Prints one JSON line
(and appends it to --out).
  python tools/bench_batch_bulk.py [--lines 100000000] [--pike-lines 1000000] [--out profiles/<name>.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import corpus as C
import regex_b200 as R
from bench_batch_iter import card
from bench_configs import _frac, hbm_peak, timed, use_torch_stream

DATE = r"(\d{4})-(\d{2})-(\d{2})"
NONE = 2**64 - 1


def _replace_rec(l, caps, expand):
    out, last = [], 0
    for c in caps:
        out += [l[last:c[0][0]], expand(l, c)]
        last = c[0][1]
    return b"".join(out) + l[last:]


def _split_rec(l, spans):
    out, last = [], 0
    for s, e in spans:
        out.append((last, s))
        last = e
    if last < len(l):
        out.append((last, len(l)))
    return out


def _rate(n, alg, ms):
    gb, f = _frac(alg, ms)
    return {"ms": round(ms, 3), "Mlines_s": round(n / ms / 1e3, 1), "GB_s": gb, "hbm_frac": f}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=100_000_000)
    ap.add_argument("--pike-lines", type=int, default=1_000_000)
    ap.add_argument("--check-lines", type=int, default=20000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    from oracle import oracle as O
    res = {}

    def host_prefix(text, offsets, k):
        return text[:int(offsets[k])].cpu().numpy().tobytes(), offsets[:k + 1].tolist()

    # ---- streaming calls over --lines ----
    text, offsets = C.log_lines(a.lines, dev)
    n, nbytes = a.lines, text.numel()
    k = min(a.check_lines, n)
    host, offs = host_prefix(text, offsets, k)
    r = use_torch_stream(R.BytesRegex(DATE))
    o = O.OracleRegex(DATE)
    moff = torch.empty(n + 1, dtype=torch.int64, device=dev)
    m = r.find_iter_batch_device(text, offsets, moff)
    spans = torch.empty((m, 2), dtype=torch.int64, device=dev)
    ms_iter, _ = timed(lambda: r.find_iter_batch_device(text, offsets, moff, spans), steps=a.steps, warmup=1)
    res["find_iter_batch_date"] = {"matches": m, **_rate(n, nbytes + 8 * (n + 1) + 8 * n + 16 * m, ms_iter)}
    del spans
    rep = b"<date>"
    out_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    total = r.replacen_batch_device(text, offsets, 0, rep, out_off, expand=False)
    out = torch.empty(total, dtype=torch.uint8, device=dev)
    ms, t2 = timed(lambda: r.replacen_batch_device(text, offsets, 0, rep, out_off, out, expand=False), steps=a.steps, warmup=1)
    assert t2 == total
    oo, ob = out_off[:k + 1].tolist(), out[:int(out_off[k])].cpu().numpy().tobytes()
    bad = sum(ob[oo[i]:oo[i + 1]] != _replace_rec(host[offs[i]:offs[i + 1]], o.captures_iter(host[offs[i]:offs[i + 1]]), lambda l, c: rep)
              for i in range(k))
    res["replace_all_batch_noexpand"] = {"pattern": DATE, "rep": rep.decode(), "out_bytes": total, "matches": m,
                                         **_rate(n, nbytes + total + 8 * (n + 1) * 2 + 16 * m, ms), "oracle_checked_lines": k,
                                         "oracle_mismatches": int(bad)}
    del out
    rs = use_torch_stream(R.BytesRegex(r"\s+"))
    os_ = O.OracleRegex(r"\s+")
    poff = torch.empty(n + 1, dtype=torch.int64, device=dev)
    np_ = rs.split_batch_device(text, offsets, poff)
    pieces = torch.empty((np_, 2), dtype=torch.int64, device=dev)
    ms, t2 = timed(lambda: rs.split_batch_device(text, offsets, poff, pieces), steps=a.steps, warmup=1)
    assert t2 == np_
    po, pc = poff[:k + 1].tolist(), pieces[:int(poff[k])].cpu().numpy().tolist()
    bad = sum([tuple(p) for p in pc[po[i]:po[i + 1]]] != _split_rec(host[offs[i]:offs[i + 1]], os_.find_iter(host[offs[i]:offs[i + 1]]))
              for i in range(k))
    res["split_batch_whitespace"] = {"pattern": r"\s+", "pieces": np_, **_rate(n, nbytes + 8 * (n + 1) * 2 + 16 * np_, ms),
                                     "oracle_checked_lines": k, "oracle_mismatches": int(bad)}
    del pieces, poff, out_off, moff, text, offsets
    torch.cuda.empty_cache()

    # ---- the Pike VM pass over --pike-lines ----
    text, offsets = C.log_lines(a.pike_lines, dev)
    n, nbytes = a.pike_lines, text.numel()
    k = min(a.check_lines, n)
    host, offs = host_prefix(text, offsets, k)
    g = r.captures_len()
    out_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    tmpl = b"$3/$2/$1"
    total = r.replacen_batch_device(text, offsets, 0, tmpl, out_off)
    out = torch.empty(total, dtype=torch.uint8, device=dev)
    ms, t2 = timed(lambda: r.replacen_batch_device(text, offsets, 0, tmpl, out_off, out), steps=a.steps, warmup=1)
    assert t2 == total
    oo, ob = out_off[:k + 1].tolist(), out[:int(out_off[k])].cpu().numpy().tobytes()

    def swap(l, c):
        return l[c[3][0]:c[3][1]] + b"/" + l[c[2][0]:c[2][1]] + b"/" + l[c[1][0]:c[1][1]]

    bad = sum(ob[oo[i]:oo[i + 1]] != _replace_rec(host[offs[i]:offs[i + 1]], o.captures_iter(host[offs[i]:offs[i + 1]]), swap)
              for i in range(k))
    moff = torch.empty(n + 1, dtype=torch.int64, device=dev)
    m = r.captures_iter_batch_device(text, offsets, moff)
    res["replace_all_batch_groups"] = {"pattern": DATE, "rep": tmpl.decode(), "out_bytes": total, "matches": m,
                                       **_rate(n, nbytes + total + 8 * (n + 1) * 2 + 16 * g * m, ms), "oracle_checked_lines": k,
                                       "oracle_mismatches": int(bad)}
    slots = torch.empty((m, g, 2), dtype=torch.int64, device=dev)
    ms, t2 = timed(lambda: r.captures_iter_batch_device(text, offsets, moff, slots), steps=a.steps, warmup=1)
    assert t2 == m
    mo, sl = moff[:k + 1].tolist(), slots[:int(moff[k])].cpu().numpy().view(np.uint64)
    bad = 0
    for i in range(k):
        got = [[None if int(x) == NONE else (int(x), int(y)) for x, y in row] for row in sl[mo[i]:mo[i + 1]]]
        bad += got != o.captures_iter(host[offs[i]:offs[i + 1]])
    res["captures_iter_batch"] = {"pattern": DATE, "groups": g, "matches": m, **_rate(n, nbytes + 8 * (n + 1) * 2 + 16 * g * m, ms),
                                  "oracle_checked_lines": k, "oracle_mismatches": int(bad)}

    line = json.dumps({
        "workload": f"C3 synthetic log lines (tools/corpus.py log_lines), device-resident: replace_all / split over {a.lines} lines, "
                    f"the Pike VM calls over {a.pike_lines} lines",
        "card": card(), "hbm_peak": hbm_peak()[1],
        "algorithmic_bytes": "input bytes + output bytes + 8 B per offset entry (input and output offsets) + 16 B per span / piece "
                             "or per group slot pair",
        "timing": f"CUDA events on torch's stream, mean of {a.steps} calls after one warm-up call", "results": res})
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    assert all(v.get("oracle_mismatches", 0) == 0 for v in res.values()), "oracle mismatches"


if __name__ == "__main__":
    main()
