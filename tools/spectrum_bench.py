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

--canonical: msbwt_kmer_spectrum_canonical at k in {21, 31} and min_count in {1, 2, 5}, histogram only and with the
list, each beside the plain call in the same process, on two indexes of configs[2]'s reads, built and loaded one at a
time: the reads as synthesised (all from the forward strand, so nearly every reverse complement is absent), then with
every other read reverse-complemented (two-strand data, where both members of most pairs occur).  Per run: wall time
of both calls (best of three, the two calls alternating),
the device time of the walk (expand / emit + CUB's compaction), of the reverse-complement counts (the query path's
seed and count kernels) and of the resolve kernels from a separate torch.profiler run, the reverse-complement lookups
(the k-mers the walk lists at ceil(min_count / 2)) per second of their kernels against the query path's rate on
batches of 2^22 listed k-mers and of their reverse complements (msbwt_seed_kmers_u64_device +
msbwt_count_kmers_packed_device, the one-request kernel at k = 31) measured in the same process, and the share of the
wall time not spent in kernels.

    python tools/spectrum_bench.py --canonical [--out FILE]
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
from oracle import canonical_spectrum as CS  # noqa: E402
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


def canonical_kernel_times(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    sums = {"walk_ms": 0.0, "compaction_ms": 0.0, "rc_count_ms": 0.0, "resolve_ms": 0.0, "other_ms": 0.0, "kernels": 0}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        n = ev.name
        key = ("walk_ms" if "spectrum_expand" in n or "spectrum_emit" in n
               else "compaction_ms" if "DeviceSelect" in n or "DeviceCompact" in n
               else "resolve_ms" if "canonical_" in n
               else "rc_count_ms" if "seed" in n or "count_kmers" in n else "other_ms")
        sums[key] += ev.time_range.elapsed_us() / 1e3
        sums["kernels"] += 1
    return {k: round(v, 3) if isinstance(v, float) else v for k, v in sums.items()}


def lookup_rate(g, kmers: np.ndarray, k: int) -> float:
    """u64 k-mer lookups per second on the query path (seed + count kernels), batches of 2^22 listed k-mers, best of
    five after a warm-up"""
    n = min(1 << 22, kmers.size)
    d_km = torch.from_numpy(kmers[:n].view(np.int64)).cuda()
    d_packed = torch.empty(g.packed_bytes(k, n) // 8, dtype=torch.int64, device="cuda")
    d_out = torch.empty(n, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    best = None
    for it in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.seed_kmers_u64_device(d_km.data_ptr(), k, n, d_packed.data_ptr(), d_out.data_ptr(), stream)
        g.count_kmers_packed_device(d_packed.data_ptr(), k, n, d_out.data_ptr(), stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if it and (best is None or ms < best):
            best = ms
    return n / (best / 1e3)


def run_canonical(g, reads_label: str, k: int, t: int, with_list: bool, crd: dict, rates: dict) -> dict:
    def call(canonical):
        return (lambda: g.list_kmers(k, t, canonical=canonical)) if with_list else \
            (lambda: g.kmer_spectrum(k, t, 10001, canonical=canonical))
    call(False)()  # warm-up
    call(True)()
    plain_wall = wall = None
    for _ in range(3):  # alternating, best of three each
        (plain, dt_plain), (r, dt) = timed(call(False), 1, False), timed(call(True), 1, False)
        plain_wall = dt_plain if plain_wall is None else min(plain_wall, dt_plain)
        wall = dt if wall is None else min(wall, dt)
    n_kmers = int(r[0].size) if with_list else int(r.sum())
    walk_min = t // 2 + t % 2
    lookups = int(g.kmer_spectrum(k, walk_min, 2)[1])  # the k-mers the canonical walk lists and looks up
    if k not in rates:
        listed = g.list_kmers(k, 2)[0]
        rates[k] = (lookup_rate(g, listed, k), lookup_rate(g, CS.revcomp_u64(listed[: 1 << 22], k), k))
    kt = canonical_kernel_times(call(True))
    busy_ms = sum(v for key, v in kt.items() if key.endswith("_ms"))
    res = {"case": "cfg3", "reads": reads_label, "mode": "canonical", "k": k, "min_count": t, "list": with_list,
           "card": crd, "wall_s": round(wall, 4), "plain_wall_s": round(plain_wall, 4), "n_kmers": n_kmers,
           "plain_n_kmers": int(plain[0].size) if with_list else int(plain.sum()), "walk_min_count": walk_min,
           "rc_lookups": lookups, **kt,
           "rc_lookups_per_s_in_query_kernels": round(lookups / (kt["rc_count_ms"] / 1e3)) if kt["rc_count_ms"] else None,
           "query_path_lookups_per_s_batches_of_2p22_listed": round(rates[k][0]),
           "query_path_lookups_per_s_batches_of_2p22_their_rc": round(rates[k][1]),
           "host_overhead_share": round(1 - busy_ms / 1e3 / wall, 3)}
    print(json.dumps(res), flush=True)
    return res


def timed(fn, reps: int = 2, warm_up: bool = True):
    if warm_up:
        fn()
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
    ap.add_argument("--canonical", action="store_true")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    crd = card()
    if args.canonical:
        reads, rle, total = bench.build_reads_and_bwt(bench.WORKLOADS["cfg3"], dev, True)
        lines = []
        for label in ("forward strand only", "every other read reverse-complemented"):
            if label != "forward strand only":
                del g
                rc = torch.tensor([0, 5, 3, 2, 4, 1], dtype=torch.uint8, device=dev)  # $ A C G N T -> complements
                reads[::2] = rc[reads[::2].flip(1).long()]
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                rle, _ = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
            torch.cuda.empty_cache()
            g = M.RleBWT.new(devices=[0])
            g.load_vector(rle)
            rates: dict = {}
            for k in (21, 31):
                for t in (1, 2, 5):
                    for with_list in (False, True):
                        lines.append(run_canonical(g, label, k, t, with_list, crd, rates))
        if args.out:
            with open(args.out, "w") as f:
                for r in lines:
                    f.write(json.dumps(r) + "\n")
        return
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
