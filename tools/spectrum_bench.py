"""The k-mer spectrum and solid k-mers of an index (msbwt_kmer_spectrum, spectrum.cu), in one process:

  cfg3 : configs[2]'s index (10 M 150-bp reads, 1 % errors, 1.51 Gsymbols), k in {21, 31}, min_count in {1, 2},
         histogram only and with the list
  cfg2 : configs[1]'s index (1 M reads, no errors, 151 Msymbols), k = 31, beside the host path a user without the
         index takes: np.unique over the reads' 31-windows

One JSON line per run: the card and its power limit (read in the same run), the warmed-up wall time of the call,
n_kmers, the ranges the traversal expanded (1 + sum over d < k of n_kmers(d, min_count), from histogram-only calls at
each depth), kernel launches (msbwt_launch_count delta), the device time of the expand / emit kernels and of CUB's
compaction from a separate torch.profiler run, the block-fetch rate that implies (every expanded range fetches the one
or two 64-byte blocks holding l and h; which of the two is not counted, so both bounds are given) against
msbwt_gather_bench at 64 bytes in the same process, and the share of the wall time not spent in kernels (per-slice
launches, read-backs and copies).

    python tools/spectrum_bench.py [--out FILE] [--cases cfg3,cfg2]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import rust_msbwt_b200 as M  # noqa: E402
from oracle import spectrum as S  # noqa: E402


def card() -> dict:
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "not read"
    return out


def gather_rate_64() -> float:
    """random 64-byte reads per second over an 8 GB buffer (msbwt_gather_bench), best of three after a warm-up"""
    buf = torch.empty(8 << 30, dtype=torch.uint8, device="cuda")
    buf[::4096].zero_()
    sink = torch.zeros(1, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    n, best = 1 << 28, None
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        M.gather_bench(0, buf.data_ptr(), buf.numel(), 64, n, 5 + it, sink.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if it and (best is None or ms < best):
            best = ms
    del buf
    torch.cuda.empty_cache()
    return n / (best / 1e3)


def kernel_times(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    sums = {"expand_ms": 0.0, "emit_ms": 0.0, "compaction_ms": 0.0, "other_ms": 0.0, "kernels": 0}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        ms = ev.time_range.elapsed_us() / 1e3
        key = ("expand_ms" if "spectrum_expand" in ev.name else "emit_ms" if "spectrum_emit" in ev.name
               else "compaction_ms" if "DeviceSelect" in ev.name or "DeviceCompact" in ev.name else "other_ms")
        sums[key] += ms
        sums["kernels"] += 1
    return {k: round(v, 3) if isinstance(v, float) else v for k, v in sums.items()}


def timed(fn, reps: int = 2):
    fn()  # warm-up
    best = None
    for _ in range(reps):
        t = time.perf_counter()
        r = fn()
        dt = time.perf_counter() - t
        best = dt if best is None or dt < best else best
    return r, best


def run(g, key: str, k: int, t: int, with_list: bool, gather: float, crd: dict, depth_kmers: dict) -> dict:
    fn = (lambda: g.list_kmers(k, t)) if with_list else (lambda: g.kmer_spectrum(k, t, 10001))
    before = M.launch_count()
    r, wall = timed(fn)
    launches = (M.launch_count() - before) // 3
    n_kmers = int(r[0].size) if with_list else int(r.sum())
    for d in range(1, k):  # n_kmers(d, min_count), shared by the runs of one index
        if (d, t) not in depth_kmers:
            depth_kmers[(d, t)] = int(g.kmer_spectrum(d, t, 2)[1])
    expanded = 1 + sum(depth_kmers[(d, t)] for d in range(1, k))
    kt = kernel_times(fn)
    search_ms = kt["expand_ms"] + kt["emit_ms"]
    busy_ms = search_ms + kt["compaction_ms"] + kt["other_ms"]
    res = {"case": key, "k": k, "min_count": t, "list": with_list, "card": crd, "wall_s": round(wall, 4),
           "n_kmers": n_kmers, "expanded_ranges": expanded, "launches": launches, **kt,
           "expanded_ranges_per_s_in_search_kernels": round(expanded / (search_ms / 1e3)) if search_ms else None,
           "block_fetches_per_s_bounds": [round(expanded / (search_ms / 1e3)), round(2 * expanded / (search_ms / 1e3))]
           if search_ms else None,
           "gather64_reads_per_s": round(gather),
           "host_overhead_share": round(1 - busy_ms / 1e3 / wall, 3)}
    print(json.dumps(res), flush=True)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--cases", default="cfg3,cfg2")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    crd = card()
    gather = gather_rate_64()
    lines = []
    for key in args.cases.split(","):
        cfg = bench.WORKLOADS[key]
        torch.cuda.empty_cache()
        reads, rle, total = bench.build_reads_and_bwt(cfg, dev, True)
        g = M.RleBWT.new(devices=[0])
        g.load_vector(rle)
        runs = [(21, 1), (21, 2), (31, 1), (31, 2)] if key == "cfg3" else [(31, 1), (31, 2)]
        depth_kmers: dict = {}
        for k, t in runs:
            for with_list in (False, True):
                lines.append(run(g, key, k, t, with_list, gather, crd, depth_kmers))
        if key == "cfg2":
            host = reads.cpu().numpy()
            t0 = time.perf_counter()
            _, km, cn = S.from_reads(list(host), 31, 1)
            host_s = time.perf_counter() - t0
            dev_kmers, dev_counts = g.list_kmers(31, 1)
            res = {"case": key, "host_reference": "np.unique over the reads' 31-windows (oracle/spectrum.from_reads,"
                   " with the co-lexicographic sort)", "card": crd, "host_s": round(host_s, 3),
                   "n_kmers": int(km.size), "equal_to_device": bool((km == dev_kmers).all() and (cn == dev_counts).all())}
            print(json.dumps(res), flush=True)
            lines.append(res)
        del g, reads
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
