#!/usr/bin/env python3
"""Headline benchmark: haystack GB/s scanned by find_iter with bit-exact spans.

Contract (task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON
line from rank 0.  A "step" is one full find_iter pass (all spans written to HBM) over
this rank's resident haystack shard.

Workload at N=1 = BASELINE.json configs[1]: sherlock-style patterns over 16 GiB of
synthetic English text (lines of bench/src/data/sherlock.txt sampled with replacement,
SURVEY.md 8d C2), headline pattern `[a-zA-Z]+ing`.  At N>1 every rank holds its own
16 GiB shard of a 16*N GiB corpus (weak scaling, byte-range sharding); see
regex_b200/sharded.py for the boundary exchange.

Besides the contract's keys the line carries
  parity       span-exact comparison with the oracle on windows of the haystack (first and last
               256 MiB, random 16 MiB windows, both sides of every shard boundary)
  e2e          the same search through rure_b200_find_all on pinned HOST memory, whole shard
  cpu_baseline the oracle port of the reference's CPU engine on the whole shard, all host threads
  rg           ripgrep (a descendant of the reference engine) on a <= 4 GiB slice, counts cross-checked
  configs      the other BASELINE.json configs (C1, C3, C4, C5) at full size (N=1 only)
  also         the other C2 patterns

`--impl reference` times the CPU path (the oracle's restatement of the reference's lazy
DFA pipeline -- the reference itself is Rust and cannot be built here) on the box's
host cores over the SAME corpus (one 16 GiB shard, generated with the same seed).
"""
import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import corpus as C  # noqa: E402  (tools/corpus.py: the synthetic inputs)

PATTERN = r"[a-zA-Z]+ing"
ALSO = [r"Holmes|Watson", r"Sherlock|Holmes", r"Sher[a-z]+|Hol[a-z]+", r"(?i)Sherlock|Holmes|Watson", r"the\s+\w+", r"\w+"]
SEED = C.SEED
GIB = C.GIB
sherlock_lines, host_corpus, device_corpus = C.sherlock_lines, C.host_corpus, C.device_corpus
# ncu --set full, scan_rev_fast<1> on 1 GiB of this corpus (profiles/): dram bytes read + written per haystack byte
TRAFFIC_PER_BYTE = (1.779481e9 + 0.225388e9) / (1 << 30)  # profiles/r02_ncu_summaries.md section 1b
METRIC = "haystack GB/s scanned (find_iter, bit-exact spans)"
DUMP_SPANS = 1 << 21  # --dump-outputs: at most 2 Mi spans x (start, end, index) x 8 B = 48 MiB in all


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gib", type=float, default=16.0, help="haystack GiB per GPU")
    ap.add_argument("--pattern", default=PATTERN)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip parity windows beyond the shard edges, rg, the other configs and patterns")
    ap.add_argument("--lines", type=int, default=100_000_000, help="C3 log lines")
    ap.add_argument("--seg", type=int, default=0, help="scan segment bytes (0 = automatic)")
    ap.add_argument("--no-fuse", action="store_true")
    ap.add_argument("--no-tensor-tma", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64), to compare two "
                         "builds on the same inputs: match_counts [this rank's matches, matches on earlier ranks, matches on all "
                         "ranks]; the GPU search adds spans [k, 2] (all, or a fixed, seeded sample) and span_index [k]")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------ clocks ----
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(s[3 + j].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------- the CPU legs (oracle) ----
def _count_parallel_ptr(pattern, ptr, n, threads):
    """oracle.count_parallel on a raw host buffer (a 16 GiB haystack is not copied into a bytes object)."""
    from oracle import oracle as O
    p = pattern.encode("utf-8")
    return O.lib().oracle_count_parallel(p, len(p), O.FLAG_UNICODE, 0, ctypes.cast(ptr, ctypes.c_char_p), n, threads)


def cpu_reference_ptr(pattern, ptr, n, threads, steps, warmup):
    from oracle import oracle as O
    O.build()
    for _ in range(warmup):
        _count_parallel_ptr(pattern, ptr, min(n, 1 << 30), threads)
    t0 = time.perf_counter()
    count = 0
    for _ in range(steps):
        count = _count_parallel_ptr(pattern, ptr, n, threads)
    dt = (time.perf_counter() - t0) / steps
    return n / dt / 1e9, dt, count


def oracle_spans(o, data):
    """find_iter spans of `data` (bytes) as an int64 [k, 2] array."""
    import numpy as np
    from oracle import oracle as O
    total = O.lib().oracle_find_iter(o._h, O.ENGINE_DFA, data, len(data), None, 0)
    buf = np.empty((max(total, 1), 2), dtype=np.uint64)
    O.lib().oracle_find_iter(o._h, O.ENGINE_DFA, data, len(data), buf.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), total)
    return buf[:total].astype(np.int64)


def run_reference(args):
    """The reference's own CPU algorithm (oracle port; kind "port": no rustc in this image) on the
    arm's config: the same 16 GiB shard (same generator and seed), every step scans all of it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    n = int(args.gib * GIB)
    if torch.cuda.is_available():  # the same bytes the GPU arm scans (the generator runs on the device)
        torch.cuda.set_device(0)
        dev_text = device_corpus(n, SEED, torch.device("cuda", 0))
        host = torch.empty(n, dtype=torch.uint8)
        host.copy_(dev_text)
        del dev_text
        torch.cuda.empty_cache()
        how = "generated by the GPU arm's generator with the same seed, copied to host memory before timing"
    else:
        host = torch.frombuffer(bytearray(host_corpus(n)), dtype=torch.uint8)
        how = "host generator (no GPU visible)"
    steps = args.steps
    gbs, dt, count = cpu_reference_ptr(args.pattern, host.data_ptr(), n, threads, steps, min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 4),
        "unit": "GB/s", "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": round(dt * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"C2 sherlock-style find_iter `{args.pattern}` over {args.gib:g} GiB/GPU synthetic English text "
                               f"(reference arm: every step scans one whole {args.gib:g} GiB shard on the host cores; {how})",
                   "haystack_bytes_per_gpu": n, "sample_bytes": n, "matches": count},
        "cpu_baseline": {"value": round(gbs, 4), "unit": "GB/s", "cores": threads, "kind": "port",
                         "sample": f"the whole {args.gib:g} GiB shard, {threads} threads, byte ranges cut at newlines, oracle engine 'auto' "
                                   f"(DfaSuffix where the reference selects it, exec.rs:1176-1210); matches={count}"},
        "e2e": {"value": round(gbs, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:  # one process scans the whole shard: it is rank 0 of a world of one
        save_outputs(args.dump_outputs, {"match_counts": [count, 0, count]})
    print(json.dumps(line), flush=True)


# ------------------------------------------------------- parity windows ----
def check_window(o, text, spans_dev, n_spans, pos_shift, a, b):
    """Span-exact comparison on [a, b) of the buffer `text`: the oracle runs on the window cut at
    line starts (no match of these patterns contains a newline) and must reproduce exactly the
    GPU spans that lie inside it.  spans_dev holds buffer-relative positions + pos_shift."""
    import numpy as np
    import torch
    nl = torch.nonzero(text[a:min(b, a + (1 << 16))] == 10)
    a2 = a if a == 0 else a + int(nl[0]) + 1
    tail = torch.nonzero(text[max(a2, b - (1 << 16)):b] == 10)
    b2 = b if b == text.numel() else max(a2, b - (1 << 16)) + int(tail[-1]) + 1
    host = text[a2:b2].cpu().numpy().tobytes()
    exp = oracle_spans(o, host) + a2
    starts = spans_dev[:n_spans, 0].contiguous()
    lo = int(torch.searchsorted(starts, torch.tensor([a2 + pos_shift], device=starts.device))[0])
    hi = int(torch.searchsorted(starts, torch.tensor([b2 + pos_shift], device=starts.device))[0])
    got = spans_dev[lo:hi].cpu().numpy() - pos_shift
    ok = got.shape == exp.shape and bool((got == exp).all())
    return ok, int(exp.shape[0]), b2 - a2


# -------------------------------------------------------------------- ours ----
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import regex_b200 as R
    from regex_b200 import sharded

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (regex_b200 has no CPU path)"
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_near_gpu(local_rank) if world > 1 else None  # pinned host buffers next to this rank's GPU
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG=VERSION/INFO writes to stdout by default: the contract is ONE JSON line there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    n = int(args.gib * GIB)          # bytes owned per GPU (multiple of 256)
    total_len = n * world            # one haystack, byte-range sharded (weak scaling)
    halo = 1 << 16
    own = device_corpus(n, SEED + rank, dev)
    geom = sharded.plan(total_len, world, rank, halo=halo)
    assert geom.b - geom.a == n
    if world > 1:
        # replicate 256 B of left context and `halo` bytes of the right neighbour (NCCL p2p)
        left = torch.empty(geom.a - geom.buf_lo, dtype=torch.uint8, device=dev)
        right = torch.empty(geom.buf_hi - geom.b, dtype=torch.uint8, device=dev)
        ops = []
        if rank + 1 < world:
            ops += [dist.P2POp(dist.isend, own[-256:].contiguous(), rank + 1), dist.P2POp(dist.irecv, right, rank + 1)]
        if rank > 0:
            ops += [dist.P2POp(dist.isend, own[:halo].contiguous(), rank - 1), dist.P2POp(dist.irecv, left, rank - 1)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()
        text = torch.cat([left, own, right])
        del left, right
        comm = sharded.TorchDistComm(dev)
    else:
        text = own
        comm = sharded.SingleComm()
    del own

    re_ = R.BytesRegex(args.pattern)
    re_.set_stream(torch.cuda.current_stream().cuda_stream)  # so torch events bracket the kernels
    if args.seg:
        re_.set_tuning(seg=args.seg)
    if args.no_fuse:
        re_.set_fuse(False)
    if args.no_tensor_tma:
        re_.set_tensor_tma(False)
    info = re_.pattern_info()
    # count pass sizes the span buffer
    probe = sharded.GpuShardEngine(re_, text, cap=0)
    n_local, _, _, _ = sharded.find_all_sharded(probe, geom, comm, info["can_match_empty"], info["has_looks"])
    engine = sharded.GpuShardEngine(re_, text, cap=n_local + 1024)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return sharded.find_all_sharded(engine, geom, comm, info["can_match_empty"], info["has_looks"])

    scan_ms, walk_ms = [], []
    with ClockSampler(local_rank) as clk:  # samples cover the warm-up steps and the timed steps
        for _ in range(max(args.warmup, 3)):
            step()
        barrier()
        launches0 = R.kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            got, offset, grand_total, rounds = step()
            st = re_.last_stats()
            scan_ms.append(st["scan_ms"]); walk_ms.append(st["walk_ms"])
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
    launches = R.kernel_launches() - launches0
    assert got == n_local
    if args.dump_outputs:  # what the last timed step returned; with N > 1 every rank adds _rank<r> to the names
        idx, sample = span_sample(engine.spans, got, geom.buf_lo, world)
        sfx = f"_rank{rank}" if world > 1 else ""
        save_outputs(args.dump_outputs, {f"match_counts{sfx}": [got, offset, grand_total], f"spans{sfx}": sample, f"span_index{sfx}": idx})
    dev_s = e0.elapsed_time(e1) / 1e3
    t = torch.tensor([dev_s, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, wall = float(t[0]), float(t[1])
    ms_per_step = dev_s / args.steps * 1e3
    value = total_len / (dev_s / args.steps) / 1e9

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    result = None
    if rank == 0:
        scan = sum(scan_ms) / len(scan_ms)
        path = {0: "scan_rev_bitmap (generic scan)", 1: "scan_rev_fast<scan only>", 2: "scan_rev_fast<fused scan+walk>", 3: "literal_scan (prefilter)"}[int(st["path"])]
        emits = int(st["path"]) in (2, 3)
        # SURVEY.md 8(d): 1 byte read per haystack byte + 16 bytes written per emitted span; the start
        # bitmap, staging and stitch traffic are this design's overhead and earn no credit.  The fused
        # kernel (reverse scan + chain walk of each segment) emits the spans; without fusion the
        # dominant kernel is the scan alone and the spans belong to walk_chunks.
        alg_bytes = n + (16 * n_local if emits else 0)
        achieved = alg_bytes / (scan / 1e3) / 1e9
        result = {
            "metric": METRIC, "value": round(value, 2), "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"C2 sherlock-style find_iter `{args.pattern}` over {args.gib:g} GiB/GPU synthetic English text "
                                   f"({world} byte-range shard(s) of one {args.gib * world:g} GiB haystack)",
                       "haystack_bytes_per_gpu": n, "matches_rank0": n_local, "matches_total": grand_total,
                       "l2": "each shard (16 GiB) far exceeds the 126 MB L2; no flush needed",
                       "timing": "torch CUDA events on the stream the library launches on (set_stream), barrier + synchronize on both sides, "
                                 "max over ranks; includes the boundary all_gathers; wall clock %.3f s" % wall,
                       "boundary_fixup_rounds": rounds},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                         "traffic": TRAFFIC_PER_BYTE * n if int(st["path"]) == 2 and args.pattern == PATTERN else None,
                         "traffic_source": "ncu --set full dram__bytes_read+write of scan_rev_fast<1> on a 1 GiB haystack (profiles/), scaled per byte",
                         "kernel": path, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": round(scan, 4),
                         "other_kernels_ms": round(sum(walk_ms) / len(walk_ms), 4),
                         "step_frac": round((n + 16 * n_local) / (ms_per_step / 1e3) / 1e9 / peak, 4)},
            "clocks": clk.summary(),
            "fixups": {k: st[k] for k in ("scan_redo_rounds", "scan_redo_segments", "stitch_rounds", "stitch_dirty_chunks", "sequential_passes", "map_passes")},
        }

    # ---- parity: span-exact windows against the oracle (SURVEY.md 8d) ----
    from oracle import oracle as O
    O.build()
    o = O.OracleRegex(args.pattern)
    win = (256 << 20) if world == 1 else (64 << 20)
    win = min(win, n // 2)
    lo_o, hi_o = geom.own_lo, geom.own_lo + n
    windows = [("first", lo_o, lo_o + win), ("last", hi_o - win, hi_o)]
    if world == 1 and not args.no_extras:
        rng = np.random.Generator(np.random.PCG64(0x5EED))
        w16 = min(16 << 20, n // 4)
        for i in range(64 if n >= (4 << 30) else 8):
            a = int(rng.integers(0, n - w16)) // 256 * 256
            windows.append((f"random{i}", lo_o + a, lo_o + a + w16))
    par = {"windows": 0, "spans": 0, "bytes": 0, "mismatches": []}
    for name, a, b in windows:
        ok, k, nb = check_window(o, text, engine.spans, n_local, 0, a, b)
        par["windows"] += 1
        par["spans"] += k
        par["bytes"] += nb
        if not ok:
            par["mismatches"].append(f"rank{rank}:{name}")
    pt = torch.tensor([par["windows"], par["spans"], par["bytes"], len(par["mismatches"])], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(pt)
    assert int(pt[3]) == 0, ("span parity failed", par["mismatches"])
    if rank == 0:
        result["parity"] = {"windows": int(pt[0]), "spans_compared": int(pt[1]), "bytes_compared": int(pt[2]), "mismatches": 0,
                            "what": "GPU spans == oracle find_iter spans on the first and last %d MiB of every shard (both sides of every shard "
                                    "boundary)%s, windows cut at line starts" % (win >> 20, " and 64 random 16 MiB windows" if len(windows) > 2 else "")}

    # ---- N > 1: all spans in one buffer on rank 0 (global positions), checked and timed ----
    if world > 1:
        counts = sharded.find_all_sharded.last_counts
        # (a 16-span gather first: NCCL sets up its point-to-point channels on first use)
        sharded.gather_spans(engine.spans, min(n_local, 16), [min(c, 16) for c in counts], geom.buf_lo, rank, world)
        barrier()
        t0 = time.perf_counter()
        allspans = sharded.gather_spans(engine.spans, n_local, counts, geom.buf_lo, rank, world)
        barrier()
        gather_ms = (time.perf_counter() - t0) * 1e3
        if rank == 0:
            assert allspans.shape[0] == grand_total
            assert bool((allspans[1:, 0] >= allspans[:-1, 1]).all()) and bool((allspans[:, 0] < allspans[:, 1]).all())
            result["span_gather"] = {"ms": round(gather_ms, 2), "spans": int(grand_total), "bytes": int(grand_total) * 16,
                                     "note": "NCCL point-to-point gather of every rank's spans into one ordered buffer on rank 0 (outside the timed steps)"}
        del allspans

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ----
    host = None
    host_full = None
    if not args.no_e2e or (rank == 0 and not args.no_cpu):
        if world > 1:  # the whole shard buffer [left context | own bytes | halo], as the sharded search wants it
            host_full = torch.empty(text.numel(), dtype=torch.uint8, pin_memory=True)
            host_full.copy_(text)
            host = host_full[geom.own_lo:geom.own_lo + n]
        else:
            host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
            host.copy_(text[geom.own_lo:geom.own_lo + n])
        torch.cuda.synchronize()
    if not args.no_e2e:
        cap = n_local + 4096
        out_t = torch.empty((cap, 2), dtype=torch.int64, pin_memory=True)  # the caller's result buffer, pinned like the haystack
        out = out_t.numpy().view(np.uint64)
        tot = R.ctypes.c_size_t()
        if world == 1:
            def e2e_once():
                ok = R.lib().rure_b200_find_all(re_._h, host.data_ptr(), n, out.ctypes.data, cap, R.byref(tot))
                assert ok
                return tot.value
            how = ("rure_b200_find_all on pinned host memory, the whole haystack; H2D of the haystack and D2H of all spans inside the "
                   "timed region; the library pipelines upload, search and download in 64 MiB pieces; spans compared with the "
                   "device-resident search")
        else:
            def e2e_once():  # upload the shard, the sharded protocol (boundary all_gathers included), download this rank's spans
                text.copy_(host_full, non_blocking=True)
                got_, _, _, _ = step()
                out_t[:got_].copy_(engine.spans[:got_], non_blocking=True)
                torch.cuda.synchronize()
                return got_
            how = ("every rank uploads its shard buffer (own bytes + left context + halo) from pinned host memory, the ranks run the "
                   "sharded protocol of the timed steps (boundary all_gathers included), every rank downloads its spans into a pinned "
                   "host buffer; all inside the timed region, max over ranks")
        for _ in range(2):
            e2e_once()
        barrier()
        k = args.steps
        t0 = time.perf_counter()
        for _ in range(k):
            got_e2e = e2e_once()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / k
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mine = engine.spans[:n_local].cpu().numpy().astype(np.uint64)
        assert got_e2e == n_local and (out[:n_local] == mine).all(), "e2e spans differ from the device-resident search"
        if rank == 0:
            result["e2e"] = {"value": round(n * world / float(t[0]) / 1e9, 3), "unit": "GB/s",
                             "h2d_bytes_per_step": int(host_full.numel() if world > 1 else n),
                             "d2h_bytes_per_step": int(min(got_e2e, cap) * 16 + 8), "haystack_bytes": n, "note": how}
            if numa:
                result["e2e"]["host_cpus_rank0"] = f"{len(numa)} CPUs local to GPU {local_rank} (NVML affinity; pinned buffers first-touched there)"
        del out, out_t

    if rank == 0:
        threads = os.cpu_count() or 1
        if not args.no_cpu:
            os.sched_setaffinity(0, all_cpus)  # the CPU leg uses every host core again
            gbs, dt, count = cpu_reference_ptr(args.pattern, host.data_ptr(), n, threads, 1, 1)
            assert count == n_local, ("parity check failed: CPU count != GPU count", count, n_local)
            result["cpu_baseline"] = {"value": round(gbs, 4), "unit": "GB/s", "cores": threads, "kind": "port",
                                      "sample": f"rank 0's whole {args.gib:g} GiB shard, {threads} threads cut at newlines, oracle engine 'auto' "
                                                f"(DfaSuffix as the reference selects for this pattern, exec.rs:1176-1210), count {count} == GPU count"}
        if not args.no_extras and not args.no_cpu:
            result["rg"] = rg_leg(args.pattern, host, n, re_, text, geom)
    del host, host_full
    if rank == 0 and world == 1 and not args.no_extras:
        result["also"] = also_patterns(R, text, n, n_local, dev, peak)
        result["configs"] = other_configs(args, text, dev)
    if rank == 0:
        print(json.dumps(result), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def span_sample(spans, n_spans, pos_shift, world):
    """The spans --dump-outputs writes: all of them, or when there are more than DUMP_SPANS / world a
    fixed, seeded sample.  Returns their indices among this rank's spans and their [k, 2] start/end byte
    offsets in the whole haystack."""
    import numpy as np
    import torch
    k = DUMP_SPANS // world
    if n_spans <= k:
        idx = np.arange(n_spans, dtype=np.int64)
    else:
        idx = np.unique(np.random.Generator(np.random.PCG64(SEED)).integers(0, n_spans, size=k))
    return idx, (spans[torch.from_numpy(idx).to(spans.device)] + pos_shift).cpu().numpy()


def save_outputs(out_dir, arrays):
    """--dump-outputs: DIR/<name>.npy for every array, float64 throughout (exact for offsets below 2**53)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def rg_leg(pattern, host, n, re_, text, geom):
    """Independent data point (BASELINE.md 3.2): ripgrep, a descendant of the reference engine (lazy DFA +
    SIMD literals, newer Unicode tables), single thread, on a <= 4 GiB slice; count cross-checked."""
    rg = shutil.which("rg")
    if not rg:
        return {"unavailable": "rg not on PATH"}
    import numpy as np
    import torch
    k = min(n, 4 * GIB)
    arr = host[:k].numpy()
    k = int(np.flatnonzero(arr[max(0, k - 65536):k] == 10)[-1]) + max(0, k - 65536) + 1  # cut at a line end
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > k + (1 << 30) else "/tmp"
    path = os.path.join(tmpdir, f"rb200_rg_slice_{os.getpid()}.txt")
    try:
        arr[:k].tofile(path)
        t0 = time.perf_counter()
        out = subprocess.run([rg, "-U", "-a", "--count-matches", "-j1", "--no-config", "-e", pattern, path], capture_output=True, text=True, timeout=600)
        dt = time.perf_counter() - t0
        count = int(out.stdout.strip() or 0)
    finally:
        if os.path.exists(path):
            os.remove(path)
    gpu = re_.find_all_device(text[geom.own_lo:geom.own_lo + k].contiguous())
    ver = subprocess.run([rg, "--version"], capture_output=True, text=True).stdout.split("\n")[0]
    return {"value": round(k / dt / 1e9, 3), "unit": "GB/s", "threads": 1, "bytes": k, "count": count, "gpu_count_same_slice": gpu,
            "counts_equal": count == gpu, "version": ver, "note": "rg -U -a --count-matches -j1 on a file in %s (page cache); wall clock of the process" % tmpdir}


def also_patterns(R, text, n, n_local, dev, peak):
    import torch
    also = {}
    spans = torch.empty((min(int(n / 3.5), 1 << 30) + 4096, 2), dtype=torch.int64, device=dev)  # `\w+` finds more; the rest is counted, not stored
    for pat in ALSO:
        r2 = R.BytesRegex(pat)
        r2.set_stream(torch.cuda.current_stream().cuda_stream)
        c = r2.find_all_device(text)
        ms = []
        for _ in range(3):
            c = r2.find_all_device(text, spans)
            ms.append(r2.last_stats()["total_ms"])
        t = sorted(ms)[1]
        also[pat] = {"GB/s": round(n / (t / 1e3) / 1e9, 1), "matches": c, "roofline_frac_step": round((n + 16 * min(c, spans.shape[0])) / (t / 1e3) / 1e9 / peak, 4),
                     "path": int(r2.last_stats()["path"])}
    del spans
    return also


def other_configs(args, text, dev):
    """C1, C3, C4, C5 at the sizes BASELINE.json names (one GPU), each with a bounded oracle check;
    the full-size parity tests are tests/test_gpu_configs.py."""
    import torch
    import bench_configs as BC
    out = {}
    for name, fn in (("C1", lambda: BC.c1(dev)), ("C4", lambda: BC.c4(dev, text)), ("C3", lambda: BC.c3(dev, args.lines)),
                     ("C5", lambda: BC.c5(dev, args.gib))):
        try:
            t0 = time.perf_counter()
            out[name] = fn()
            out[name]["wall_s"] = round(time.perf_counter() - t0, 1)
        except Exception as e:  # a failed extra must not lose the headline line; it is reported as failed
            out[name] = {"failed": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()
    return out


def bind_near_gpu(index):
    """Run this process on the CPUs NVML reports as local to GPU `index`, so that the pinned host buffers it
    allocates (first touch) sit on that GPU's NUMA node: with several ranks uploading at once the e2e leg is
    otherwise limited by cross-socket traffic.  Returns the CPU list, or None when NVML cannot tell."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
