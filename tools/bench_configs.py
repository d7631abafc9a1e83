#!/usr/bin/env python
"""Secondary workloads of BASELINE.json (C1, C3, C4, C5) on one GPU, device-resident inputs.

bench.py measures the headline C2 metric and, at N=1, calls these functions to put the other
configs on the same JSON line ("configs": {...}), each with its size, throughput, fraction of
the measured HBM roofline on ALGORITHMIC bytes (SURVEY.md 8d) and a bounded oracle check.
Stand-alone:  python tools/bench_configs.py [--lines 100000000] [--gib 16] [--skip c1,c3,c4,c5]
prints one JSON line per config.  The full-size parity tests are tests/test_gpu_configs.py.
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

GIB = C.GIB
DNA_VARIANTS = C.DNA_VARIANTS
log_lines = C.log_lines
c4_patterns = C.c4_patterns


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def timed(fn, steps=5, warmup=3):
    """CUDA events on torch's current stream (the regex objects are told to launch there),
    device synchronize on both sides."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out


def use_torch_stream(r):
    r.set_stream(torch.cuda.current_stream().cuda_stream)
    return r


def _frac(alg_bytes, ms):
    peak, _ = hbm_peak()
    gbs = alg_bytes / ms / 1e6
    return round(gbs, 1), round(gbs / peak, 4)


def c1(dev):
    raw = open(os.path.join(ROOT, "tests", "golden", "regexdna-input.txt"), "rb").read()
    import re
    seq = re.sub(rb">[^\n]*\n|\n", b"", raw)
    expected = {}
    for line in open(os.path.join(ROOT, "tests", "golden", "regexdna-output.txt")):
        parts = line.split()
        if len(parts) == 2 and parts[1].isdigit() and not parts[0].isdigit():
            expected[parts[0]] = int(parts[1])
    d = torch.frombuffer(bytearray(seq), dtype=torch.uint8).to(dev)
    out = {}
    for v in DNA_VARIANTS:
        r = use_torch_stream(R.BytesRegex(v))
        ms, cnt = timed(lambda: r.find_all_device(d), steps=20)
        assert cnt == expected[v], (v, cnt, expected[v])
        out[v] = {"us": round(ms * 1e3, 1), "count": cnt}
    return {"workload": "C1 regex-dna: 9 variants, find_iter count over the cleaned 100 000 B input (latency; counts == regexdna-output.txt)",
            "haystack_bytes": len(seq), "us_per_variant_median": float(np.median([v["us"] for v in out.values()])), "results": out}


def c3(dev, n_lines, check_lines=20000):
    from oracle import oracle as O
    text, offsets = log_lines(n_lines, dev)
    nbytes = text.numel()
    res = {}
    for pat in (r"(\d{4})-(\d{2})-(\d{2})", r"(?-u)(\d{4})-(\d{2})-(\d{2})"):
        r = use_torch_stream(R.BytesRegex(pat))
        if os.environ.get("RB_BATCH_REFILL"):  # experiments: 0 batch_fast, 1 refill for is_match on large batches, 2 on any
            r.set_option("batch_refill", int(os.environ["RB_BATCH_REFILL"]))
        bits = torch.zeros((n_lines + 31) // 32, dtype=torch.int32, device=dev)
        spans = torch.empty((n_lines, 2), dtype=torch.int64, device=dev)
        ms_is, _ = timed(lambda: r.is_match_batch_device(text, offsets, bits))
        ms_find, _ = timed(lambda: r.find_batch_device(text, offsets, spans, bits))
        # every one of the first check_lines lines against the oracle
        o = O.OracleRegex([pat])
        k = min(check_lines, n_lines)
        host = text[:int(offsets[k])].cpu().numpy().tobytes()
        offs = offsets[:k + 1].tolist()
        sp = spans[:k].tolist()
        bw = np.unpackbits(bits[:(k + 31) // 32].cpu().numpy().view(np.uint8), bitorder="little")
        bad = 0
        for i in range(k):
            m = o.find_at(host[offs[i]:offs[i + 1]])
            if (m is None) != (not bw[i]) or (m is not None and tuple(m) != tuple(sp[i])):
                bad += 1
        assert bad == 0, (pat, bad)
        gb_is, f_is = _frac(nbytes + 8 * n_lines + n_lines / 8, ms_is)
        gb_find, f_find = _frac(nbytes + 8 * n_lines + n_lines / 8 + 16 * n_lines, ms_find)
        res[pat] = {"is_match_Mlines_s": round(n_lines / ms_is / 1e3, 1), "is_match_GB_s": gb_is, "is_match_roofline_frac": f_is,
                    "find_Mlines_s": round(n_lines / ms_find / 1e3, 1), "find_GB_s": gb_find, "find_roofline_frac": f_find,
                    "oracle_checked_lines": k, "oracle_mismatches": bad}
    del text, offsets
    return {"workload": f"C3 batched per-line is_match + find of (\\d{{4}})-(\\d{{2}})-(\\d{{2}}) over {n_lines} synthetic log lines",
            "lines": n_lines, "haystack_bytes": nbytes,
            "algorithmic_bytes": "line bytes + 8 B offsets + 1 bit per line (is_match); + 16 B span per line (find)", "results": res}


def c4(dev, text, check_bytes=8 << 20, per_line=True):
    """text: the C2 corpus already resident on the device."""
    from oracle import oracle as O
    n = text.numel()
    pats = c4_patterns()
    s = R.BytesRegexSet(pats)
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    ms, mask = timed(lambda: s.matches_mask_device(text))
    waves = s.last_stats()["waves"]
    s0 = R.BytesRegexSet(pats)
    s0.set_stream(torch.cuda.current_stream().cuda_stream)
    s0.set_option("narrow_sets", 0)
    s0.set_option("wave0", 0)
    ms0, mask0 = timed(lambda: s0.matches_mask_device(text), steps=2, warmup=1)
    assert list(mask0) == list(mask), (mask0, mask)
    # bounded check: every member alone (RegexSet::matches is per-pattern existence) on a slice
    sl = text[:check_bytes].cpu().numpy().tobytes()
    exp = sum(1 << i for i, p in enumerate(pats) if O.OracleRegex(p).is_match_at(sl))
    got = s.matches_mask_device(text[:check_bytes].contiguous())[0]
    assert got == exp, (hex(got), hex(exp))
    assert mask[0] & exp == exp
    gb, fr = _frac(n + 8, ms)
    gb0, fr0 = _frac(n + 8, ms0)
    res = {"n_patterns": len(pats), "whole_haystack_GB_s": gb, "whole_haystack_roofline_frac": fr, "whole_haystack_ms": round(ms, 3), "waves": waves,
           "mask": [hex(m) for m in mask], "product_automaton_only_GB_s": gb0, "product_automaton_only_roofline_frac": fr0,
           "oracle_checked_bytes": check_bytes}
    if per_line:
        nl = torch.nonzero(text == 10).flatten() + 1
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), nl])
        del nl
        n_lines = offsets.numel() - 1
        masks = torch.zeros((n_lines, (len(pats) + 63) // 64), dtype=torch.int64, device=dev)
        ms2, _ = timed(lambda: s.matches_batch_device(text, offsets, masks), steps=2, warmup=1)
        o = O.OracleRegex(pats)
        offs = offsets[:1001].tolist()
        hostl = text[:offs[-1]].cpu().numpy().tobytes()
        gotl = masks[:1000, 0].cpu().numpy().view(np.uint64)
        for i in range(1000):
            e = sum(1 << j for j in o.set_matches(hostl[offs[i]:offs[i + 1]]))
            assert int(gotl[i]) == e, (i, hex(int(gotl[i])), hex(e))
        gb2, fr2 = _frac(int(offsets[-1]) + 16 * n_lines, ms2)
        res.update({"per_line_GB_s": gb2, "per_line_roofline_frac": fr2, "per_line_Mlines_s": round(n_lines / ms2 / 1e3, 1), "lines": n_lines,
                    "per_line_oracle_checked_lines": 1000})
        del offsets, masks
    return {"workload": f"C4 RegexSet x{len(pats)} (bytes::RegexSet, Unicode \\w \\d \\s) over {n / GIB:g} GiB of the C2 corpus: one matches() over the "
                        "whole haystack, and one matches() per line", "haystack_bytes": n,
            "algorithmic_bytes": "haystack + 8 B (whole); haystack + 8 B offsets + 8 B mask per line (per line)", "results": res}


def c5(dev, gib, check_bytes=64 << 20):
    from oracle import oracle as O
    n = int(gib * GIB)
    text = C.device_dna(n, dev)
    host = text[:check_bytes].cpu().numpy().tobytes()
    res = {}
    for v in DNA_VARIANTS:
        r = use_torch_stream(R.BytesRegex(v))
        cnt = r.find_all_device(text)
        spans = torch.empty((cnt + 16, 2), dtype=torch.int64, device=dev)
        ms, c2 = timed(lambda: r.find_all_device(text, spans), steps=3, warmup=2)
        assert c2 == cnt
        exp = np.array(O.OracleRegex(v).find_iter(host[:check_bytes - 64]), dtype=np.int64).reshape(-1, 2)
        got = spans[:exp.shape[0]].cpu().numpy()
        assert (got == exp).all(), v
        gb, fr = _frac(n + 16 * cnt, ms)
        res[v] = {"GB_s": gb, "roofline_frac": fr, "matches": cnt, "density_per_byte": cnt / n, "oracle_checked_spans": int(exp.shape[0])}
    del text
    return {"workload": f"C5 regex-dna variants, find_iter spans over {gib:g} GiB of uniform acgt on one GPU (the multi-GPU form is bench.py --gpus N)",
            "haystack_bytes": n, "algorithmic_bytes": "haystack + 16 B per span",
            "GB_s_median": float(np.median([v["GB_s"] for v in res.values()])), "results": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=100_000_000)
    ap.add_argument("--gib", type=float, default=16.0)
    ap.add_argument("--skip", default="")
    a = ap.parse_args()
    skip = set(a.skip.split(","))
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    if "c1" not in skip:
        print(json.dumps(c1(dev)), flush=True)
    if "c3" not in skip:
        print(json.dumps(c3(dev, a.lines)), flush=True)
    if "c4" not in skip:
        text = C.device_corpus(int(a.gib * GIB), C.SEED, dev)
        print(json.dumps(c4(dev, text)), flush=True)
        del text
    if "c5" not in skip:
        print(json.dumps(c5(dev, a.gib)), flush=True)


if __name__ == "__main__":
    main()
