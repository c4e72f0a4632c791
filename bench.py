#!/usr/bin/env python
"""bench.py -- 31-mer count_kmer throughput (queries/s) on B200, per the driver contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload default|cfg2|cfg3|cfg5|tiny]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (pack/seed + backward-search kernels) over one batch of synthetic k-mer
queries.  Headline workload = BASELINE.json configs[2]: 10 M synthetic 150-bp reads with 1 % errors (1.51 Gsymbol
BWT), a FIXED batch of 100 M read-sampled 31-mers.  With N > 1 (torchrun, one rank per GPU) every rank holds a
replica of the index and the rank's contiguous slice of that batch (strong scaling, no data-path collective); the
only torch.distributed traffic is the barrier and the max-over-ranks of the timings.

  value : kernel-only -- the batch resident in HBM as symbol bytes, pack/seed + search timed with CUDA events
  e2e   : the drop-in C-ABI call (msbwt_count_kmers_fixed) on pinned HOST buffers, copies inside the timed region,
          through ONE handle created with devices = [0..N-1] on rank 0 -- the library's own multi-GPU dispatcher
          (the other ranks have released their replicas and sleep in a gloo barrier); the packed-integer entry
          points (8 bytes in, 8 or 4 bytes out per query) are timed beside it

Nested `other_workloads`: configs[1] (151 Msymbol BWT, N = 1 only) and configs[4] (3.02 Gsymbol BWT; one GPU's
125 M-query share at N = 1, the full 10^9 queries over 8 replicas at N = 8).

One JSON line on stdout (rank 0).  Everything else goes to stderr.

--dump-outputs DIR: rank 0 writes, per workload, the counts the last timed step returned for its queries
(DIR/<workload>_counts.npy, float64) and their positions in the batch (DIR/<workload>_query_index.npy); a batch larger
than DUMP_SAMPLE queries is sampled at fixed, seeded positions.  The inputs are seeded too, so two builds run with the
same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]
    "cfg2": dict(key="cfg2", reads=1_000_000, read_len=150, coverage=30.0, error=0.0, n_read=5_000_000, n_random=5_000_000, k=31,
                 scaling="strong",
                 name="configs[1]: 1M synthetic 150bp reads (151 Msymbol BWT), 5M random + 5M read-sampled 31-mers"),
    # BASELINE.json configs[2]: the headline
    "cfg3": dict(key="cfg3", reads=10_000_000, read_len=150, coverage=30.0, error=0.01, n_read=100_000_000, n_random=0, k=31,
                 scaling="strong",
                 name="configs[2]: 10M synthetic 150bp reads with 1% errors (1.51 Gsymbol BWT), 100M read-sampled 31-mers"),
    # BASELINE.json configs[4]: the 3.02 Gsymbol index is replicated, every GPU answers 125 M of the 10^9 queries
    "cfg5": dict(key="cfg5", reads=20_000_000, read_len=150, coverage=30.0, error=0.01, n_read=125_000_000, n_random=0, k=31,
                 scaling="weak",
                 name="configs[4]: 20M synthetic 150bp reads with 1% errors (3.02 Gsymbol BWT), 125M read-sampled 31-mers per GPU (1 B over 8)"),
    # small shape for plumbing checks
    "tiny": dict(key="tiny", reads=20_000, read_len=150, coverage=30.0, error=0.01, n_read=100_000, n_random=100_000, k=31,
                 scaling="strong",
                 name="tiny: 20k reads, 200k 31-mers (plumbing check, not a bench line)"),
}
HEADLINE = "cfg3"
METRIC = "count_kmer_31mer_queries_per_sec"
UNIT = "queries/s"
BLOCK_BYTES = 64      # layout.h: one 64-byte block per 128 symbols (one-step path)
BLOCK_SHIFT = 7
PAIR_BYTES = 128      # layout.h: one 128-byte line per 96 positions, two steps per line (pair path)
PAIR_SYMS = 96
QUAD_SECTOR_BYTES = 32  # layout.h: one 32-byte sector per 224 positions and 4-symbol code, four steps per sector (quad path)
QUAD_SYMS = 224
LINE_BYTES = 128      # what one L2 miss costs HBM whatever the request size (profiles/r1_gather_dram_bytes.csv)
DUMP_SAMPLE = 1 << 20  # --dump-outputs: queries kept per workload, 16 B each (count + index): 48 MB for the default run
DUMP_SEED = 0x5EED00D0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload_config(cfg: dict, total: int | None, world: int) -> dict:
    """The `config` object: names the workload.  Identical in both arms (`--impl ours` / `--impl reference`)."""
    n = cfg["n_read"] + cfg["n_random"]
    return {"workload": cfg["name"], "bwt_symbols": total, "k": cfg["k"],
            "queries": n if cfg["scaling"] == "strong" else n * world,
            "seeds": "torch Philox 0x5EED0001.. (harness/synth.py)"}


def ncu_traffic(workload_key: str, kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed
    `ncu --set full` capture of this same workload / kernel (profiles/ncu_traffic.json); None when none matches."""
    try:
        for e in json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["captures"]:
            if e["workload"] == workload_key and e.get("kernel") == kernel:
                return e["dram_bytes_per_launch"], e["source"]
    except Exception:
        pass
    return None, None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  nvidia-smi needs a few hundred
    milliseconds before its first line and the timed region of the headline workload is ~40 ms, so the sampler is
    started before the warm-up, the warm-up is extended until its first line is there (`has_sample`), it samples every
    20 ms, and `stop` keeps the samples whose own time stamps fall inside the timed region."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def has_sample(self) -> bool:
        try:
            return self.proc is None or os.path.getsize(self.path) > 0
        except OSError:
            return True

    @staticmethod
    def _epoch(stamp: str):
        import datetime
        try:
            return datetime.datetime.strptime(stamp.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0: float | None = None, t1: float | None = None) -> dict:
        """t0, t1: time.time() around the timed region; without them every sample counts"""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 10:
                    continue
                try:
                    rows.append((self._epoch(f[0]), float(f[2]), float(f[3]), [nm for nm, v in zip(names, f[6:10]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        window = "timed region"
        inside = [r for r in rows if t0 is not None and r[0] is not None and t0 <= r[0] <= t1]
        if not inside and t0 is not None:   # (a region shorter than the sampling period can fall between two samples)
            inside = [r for r in rows if r[0] is not None and t0 - 0.05 <= r[0] <= t1 + 0.05]
            window = "timed region +- 50 ms"
        if not inside:
            inside, window = rows, "warm-up + timed region"
        if inside:
            out = {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": max(r[2] for r in inside),
                   "reasons": sorted({nm for r in inside for nm in r[3]}), "samples": len(inside), "window": window}
        return out


def build_reads_and_bwt(cfg: dict, device, use_library: bool):
    """Synthetic reads -> BWT -> RLE bytes (host).  `use_library`: the product's device-side builder
    (bwt_build.cu; equals the harness builder and naive_bwt, tests/); otherwise the torch harness only, so that the
    reference arm never maps our library."""
    import torch
    from harness import bwt_build, synth
    reads = synth.make_reads(cfg["reads"], cfg["read_len"], cfg["coverage"], cfg["error"], device=device)
    if use_library and device.type == "cuda":
        import rust_msbwt_b200 as M
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        rle_host, total = M.build_rle_bwt(reads.data_ptr(), device.index or 0, reads.shape[0], reads.shape[1])
    else:
        rle, total = bwt_build.build_rle_bwt(reads)
        rle_host = rle.cpu().numpy()
        del rle
    return reads, rle_host, total


def build_workload(cfg: dict, device, rank: int, use_library: bool = True):
    """RLE bytes (host) and a query batch (device).  A strong-scaling workload has ONE batch, the same on every rank
    (the ranks then take slices of it); a weak-scaling one gives every rank its own batch (seed offset = rank)."""
    import torch
    from harness import synth
    t0 = time.time()
    reads, rle_host, total = build_reads_and_bwt(cfg, device, use_library)
    seed_offset = 0 if cfg["scaling"] == "strong" else 1000 * rank
    queries = synth.make_queries(reads, cfg["k"], cfg["n_read"], cfg["n_random"], seed_offset=seed_offset)
    reads_sample = reads[:100_000].cpu().numpy()   # for the pileup leg (count_read_kmers)
    del reads
    if device.type == "cuda":
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    log(f"[rank {rank}] workload built in {time.time() - t0:.1f}s: {total} symbols, {rle_host.size} RLE bytes, "
        f"{queries.shape[0]} queries")
    return rle_host, total, queries, reads_sample


def encode_u64(q, k: int):
    """[n, k] symbol bytes (all ACGT) on a torch device -> n int64: the k-mer as a 2k-bit integer, first symbol most
    significant, A,C,G,T = 0..3 (msbwt_count_kmers_u64's input format)."""
    import torch
    lut = torch.tensor([0, 0, 1, 2, 0, 3], dtype=torch.int64, device=q.device)
    out = torch.empty(q.shape[0], dtype=torch.int64, device=q.device)
    step = 1 << 24
    for a in range(0, q.shape[0], step):
        blk = q[a:a + step]
        acc = torch.zeros(blk.shape[0], dtype=torch.int64, device=q.device)
        for j in range(k):
            acc = (acc << 2) | lut[blk[:, j].long()]
        out[a:a + step] = acc
    return out


def dump_outputs(out_dir: str, key: str, counts, offset: int) -> None:
    """--dump-outputs: `counts` (u64, one per query of the batch slice starting at query `offset`) as float64, exact
    below 2^53, with the batch position of every entry kept; at most DUMP_SAMPLE entries, at seeded positions"""
    import numpy as np
    n = counts.shape[0]
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_SAMPLE, replace=False)) if n > DUMP_SAMPLE else np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{key}_counts.npy"), counts[idx].astype(np.float64))
    np.save(os.path.join(out_dir, f"{key}_query_index.npy"), (idx + offset).astype(np.float64))


def cpu_reference_leg(orc, q_host, k, threads, target_s, label):
    """Times the oracle's count_kmer loop on a bounded prefix of the batch."""
    n = q_host.shape[0]
    probe = min(n, 50_000)
    t0 = time.perf_counter()
    orc.count_kmers_fixed(q_host[:probe], k, threads=threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    m = int(min(n, max(probe, probe / dt * target_s)))
    t0 = time.perf_counter()
    counts = orc.count_kmers_fixed(q_host[:m], k, threads=threads)
    dt = time.perf_counter() - t0
    log(f"[cpu] {label}: {m} queries in {dt:.2f}s on {threads} thread(s) -> {m / dt:,.0f} q/s")
    return m / dt, m, counts


def reference_measure(args, cfg):
    """The reference's own CPU algorithm (oracle port; the Rust crate cannot be built in this image) on this box's
    host cores, all threads, bounded samples of the workload.  Inputs come from the torch harness alone."""
    import torch
    from oracle import oracle as O
    dev = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")  # GPU only manufactures the inputs
    rle_host, total, queries, _ = build_workload(cfg, dev, 0, use_library=False)
    q_host = queries.cpu().numpy()
    del queries
    orc = O.RleBWT()
    orc.load_vector(rle_host)
    cores = os.cpu_count() or 1
    k = cfg["k"]
    n = q_host.shape[0]
    probe = min(n, 100_000)
    t0 = time.perf_counter()
    orc.count_kmers_fixed(q_host[:probe], k, threads=cores)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    per_step = int(min(n, max(probe, rate * 4.0)))  # ~4 s of CPU work per step
    times = []
    for s in range(args.warmup + args.steps):
        a = (s * per_step) % max(1, n - per_step + 1)
        t0 = time.perf_counter()
        orc.count_kmers_fixed(q_host[a:a + per_step], k, threads=cores)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    total_t = sum(times)
    value = per_step * len(times) / total_t
    return {"value": value, "ms_per_step": 1e3 * total_t / len(times), "cores": cores, "per_step": per_step,
            "n": n, "total": total, "k": k}


def run_reference(args, cfgs):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    r = reference_measure(args, cfgs[0])
    sample = f"{r['per_step']} of the workload's {r['n']} queries per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": cfgs[0]["scaling"], "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(cfgs[0], r["total"], world),
        "queries_per_step": r["per_step"],
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    for extra in cfgs[1:]:
        x = reference_measure(args, extra)
        line.setdefault("other_workloads", []).append(
            {"config": workload_config(extra, x["total"], world), "value": x["value"], "unit": UNIT, "cores": x["cores"],
             "sample": f"{x['per_step']} of {x['n']} queries per step"})
    print(json.dumps(line), flush=True)


def time_host_calls(fn, steps: int, warm: int = 1) -> float:
    """seconds per call of a blocking host-buffer entry point (results are in host memory when it returns)"""
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    return (time.perf_counter() - t0) / steps


def e2e_legs(args, cfg, handle, lib, M, q_dev_list, k, reads_sample, n_devices, want_bytes_leg=True):
    """End-to-end legs through ONE handle (`n_devices` replicas) on pinned host buffers.  `q_dev_list`: the batch as
    device tensors (one per original rank for a weak workload) -- copied to pinned host memory here, outside the
    timed regions.  Returns (dict of legs, host arrays needed for the parity check)."""
    import ctypes

    import numpy as np
    import torch

    n = sum(int(q.shape[0]) for q in q_dev_list)
    steps = args.steps
    legs = {}
    vp = ctypes.c_void_p

    # the packed-integer batch: what a k-mer counter holds (8 bytes per 31-mer)
    km_pinned = torch.empty(n, dtype=torch.int64, pin_memory=True)
    at = 0
    for q in q_dev_list:
        km_pinned[at:at + q.shape[0]].copy_(encode_u64(q, k))
        at += q.shape[0]
    torch.cuda.synchronize()
    km_np = km_pinned.numpy().view(np.uint64)
    out64 = torch.empty(n, dtype=torch.int64, pin_memory=True)
    out32 = torch.empty(n, dtype=torch.int32, pin_memory=True)
    o64, o32 = out64.numpy().view(np.uint64), out32.numpy().view(np.uint32)

    def leg(name, what, fn, out_arr):
        dt = time_host_calls(fn, steps)
        h2d, d2h = M.last_transfer_bytes()
        legs[name] = {"value": n / dt, "unit": UNIT, "ms_per_step": 1e3 * dt, "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": d2h, "entry": what, "steps": steps}
        legs[name]["checksum"] = int(out_arr.astype(np.uint64).sum())
        log(f"[e2e] {name}: {n / dt / 1e9:.2f} G q/s ({1e3 * dt:.2f} ms per {n} queries, {h2d / n:.1f} B in, {d2h / n:.1f} B out per query)")

    def call(fn_name, *a):
        rc = getattr(lib, fn_name)(handle, *a)
        assert rc == 0, lib.msbwt_last_error()

    leg("u64", "msbwt_count_kmers_u64: k-mers as 2-bit-per-symbol integers in, u64 counts out",
        lambda: call("msbwt_count_kmers_u64", vp(km_np.ctypes.data), k, n, vp(o64.ctypes.data)), o64)
    leg("u64_out32", "msbwt_count_kmers_u64_u32: the same with u32 counts (index below 2^32 symbols)",
        lambda: call("msbwt_count_kmers_u64_u32", vp(km_np.ctypes.data), k, n, vp(o32.ctypes.data)), o32)
    assert legs["u64"]["checksum"] == legs["u64_out32"]["checksum"], "u64 and u32 counts differ"

    host = {"o64": o64, "q_np": None}
    if want_bytes_leg:
        q_pinned = torch.empty((n, k), dtype=torch.uint8, pin_memory=True)
        at = 0
        for q in q_dev_list:
            q_pinned[at:at + q.shape[0]].copy_(q)
            at += q.shape[0]
        torch.cuda.synchronize()
        q_np = q_pinned.numpy()
        host["q_np"] = q_np
        ob = torch.empty(n, dtype=torch.int64, pin_memory=True)
        ob_np = ob.numpy().view(np.uint64)
        leg("bytes", "msbwt_count_kmers_fixed: one symbol per byte in (the reference's &[u8] k-mers), u64 counts out",
            lambda: call("msbwt_count_kmers_fixed", vp(q_np.ctypes.data), k, n, vp(ob_np.ctypes.data)), ob_np)
        h2d = legs["bytes"]["h2d_bytes_per_step"]
        legs["bytes"]["route"] = ("symbol bytes H2D -> pack + search kernels -> D2H" if h2d >= n * k else
                                  "host threads pack 2 bit/symbol into pinned staging -> H2D -> seed + search kernels -> D2H"
                                  if h2d <= 8 * -(-k // 32) * n + 4096 else
                                  "hybrid: chunks packed 2 bit/symbol by the host pool, and raw symbol-byte chunks whenever the "
                                  "copy engine is idle -> seed / pack + search kernels -> D2H")
        legs["bytes"]["host_input_bytes_per_step"] = n * k
        assert legs["bytes"]["checksum"] == legs["u64"]["checksum"], "byte and integer entry points differ"
        host["o64"] = ob_np

    # pileup: count_kmer of every window of whole reads (msbwt_count_read_kmers): only the reads cross PCIe
    if reads_sample is not None:
        nr, rl = reads_sample.shape
        r_pinned = torch.empty((nr, rl), dtype=torch.uint8, pin_memory=True)
        r_pinned.copy_(torch.from_numpy(reads_sample))
        p_out = torch.empty((nr, rl - k + 1), dtype=torch.int64, pin_memory=True)
        r_np, p_np = r_pinned.numpy(), p_out.numpy().view(np.uint64)
        dt = time_host_calls(lambda: call("msbwt_count_read_kmers", vp(r_np.ctypes.data), rl, nr, k, 1, vp(p_np.ctypes.data)), steps)
        legs["pileup"] = {"value": nr * (rl - k + 1) / dt, "unit": UNIT, "reads_per_step": nr, "windows_per_read": rl - k + 1,
                          "h2d_bytes_per_step": nr * rl, "d2h_bytes_per_step": nr * (rl - k + 1) * 8, "ms_per_step": 1e3 * dt,
                          "entry": "msbwt_count_read_kmers on pinned host reads: every 31-mer window of every read, forward strand"}
        host["pile_counts"] = p_np[:64].copy()
    legs["host_pack_threads"] = M.host_pack_threads()
    legs["devices"] = n_devices
    return legs, host


def measure_ours(args, cfg, ctx, primary: bool):
    """One workload: kernel-only `value` (one replica + one slice per rank), end-to-end legs through one handle
    (rank 0), parity checks on every rank, CPU baseline and roofline accounting (rank 0)."""
    import numpy as np
    import torch

    import rust_msbwt_b200 as M
    from harness.dist import shard_bounds
    from oracle import oracle as O

    rank, world, local, dev = ctx["rank"], ctx["world"], ctx["local"], ctx["dev"]
    barrier, max_over_ranks, host_barrier = ctx["barrier"], ctx["max_over_ranks"], ctx["host_barrier"]
    k = cfg["k"]
    strong = cfg["scaling"] == "strong"
    rle_host, total, queries_all, reads_sample = build_workload(cfg, dev, rank)
    n_batch = queries_all.shape[0]
    lo, hi = shard_bounds(n_batch, rank, world) if strong else (0, n_batch)
    queries = queries_all[lo:hi]
    n = queries.shape[0]
    n_job = n_batch if strong else n_batch * world          # queries the whole job answers per step
    t0 = time.time()
    bwt = M.RleBWT.new(devices=[local])
    bwt.load_vector(rle_host)
    log(f"[rank {rank}] index resident: {bwt.index_bytes / 1e9:.2f} GB (suffix table s={bwt.suffix_table_s}, quad {bwt.quad_index}, "
        f"oct {bwt.oct_index} b={bwt.oct_bucket_shift}, final {bwt.final_index}) in {time.time() - t0:.1f}s")

    stream = torch.cuda.current_stream().cuda_stream
    table_s = bwt.suffix_table_s
    d_packed = torch.empty(bwt.packed_bytes(k, n) // 8, dtype=torch.int64, device=dev)  # pack -> search scratch
    d_out = torch.empty(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(1, dtype=torch.int32, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > L2: evicts index + queries between steps

    fused = bwt.oct_index and k <= 32 and os.environ.get("MSBWT_FUSED", "0") not in ("", "0")   # opt-in, slower

    def step(ev=None):
        d_status.zero_()
        if fused:   # one kernel from symbol bytes to counts (msbwt_count_kmers_fixed_device, fused_kernels.cu)
            if ev:
                ev[0].record()
            bwt.count_kmers_fixed_device(queries.data_ptr(), k, n, d_out.data_ptr(), d_status.data_ptr(), stream)
        else:
            bwt.pack_kmers_device(queries.data_ptr(), k, n, d_packed.data_ptr(), d_out.data_ptr(), d_status.data_ptr(), stream)
            if ev:
                ev[0].record()
            bwt.count_kmers_packed_device(d_packed.data_ptr(), k, n, d_out.data_ptr(), stream)
        if ev:
            ev[1].record()

    # ---- value: kernel-only, inputs resident in HBM ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        flush.fill_(1)
        step()
    if rank == 0:   # further untimed steps (the GPU stays under load) until nvidia-smi has printed its first line
        t_wait = time.time()
        while not sampler.has_sample() and time.time() - t_wait < 3.0:
            flush.fill_(1)
            step()
            torch.cuda.synchronize()
    barrier()
    launches0 = M.launch_count()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    t_epoch0 = time.time()
    for s in range(args.steps):
        flush.fill_(s & 1)               # L2 flush between timed iterations (not inside the event spans)
        ev[s][0].record()
        step((ev[s][1], ev[s][2]))
    barrier()
    t_epoch1 = time.time()
    wall = time.perf_counter() - t_wall0
    launches = M.launch_count() - launches0
    step_ms = [ev[s][0].elapsed_time(ev[s][2]) for s in range(args.steps)]
    kern_ms = [ev[s][1].elapsed_time(ev[s][2]) for s in range(args.steps)]
    total_ms = max_over_ranks(sum(step_ms))
    clocks = sampler.stop(t_epoch0, t_epoch1) if rank == 0 else None
    assert int(d_status.item()) == 0
    value = n_job * args.steps / (total_ms / 1e3)
    checksum = int(d_out.sum().item())
    got = d_out.cpu().numpy().view(np.uint64)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cfg["key"], got, lo)

    # ---- the same step with the k-mers resident as 2-bit-per-symbol integers (8 B per query instead of k): what a
    #      k-mer counter that keeps packed k-mers on the device would call (msbwt_seed_kmers_u64_device + search) ----
    packed_input = None
    if k <= 32 and not fused:
        keys = encode_u64(queries, k)
        d_out_p = torch.empty(n, dtype=torch.int64, device=dev)
        evp = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
        for s in range(args.steps + 1):
            flush.fill_(s & 1)
            if s:
                evp[s - 1][0].record()
            bwt.seed_kmers_u64_device(keys.data_ptr(), k, n, d_packed.data_ptr(), d_out_p.data_ptr(), stream)
            bwt.count_kmers_packed_device(d_packed.data_ptr(), k, n, d_out_p.data_ptr(), stream)
            if s:
                evp[s - 1][1].record()
        torch.cuda.synchronize()
        assert (d_out_p == d_out).all(), "packed-integer and symbol-byte inputs give different counts"
        p_ms = max_over_ranks(sum(e[0].elapsed_time(e[1]) for e in evp))
        packed_input = {"value": n_job * args.steps / (p_ms / 1e3), "unit": UNIT, "ms_per_step": p_ms / args.steps,
                        "what": "kernel-only with the k-mers resident in HBM as 2-bit-per-symbol integers (8 B per query in)"}
        del keys, d_out_p

    # ---- exact index traffic of one step (outside any timing): what the pack stage's one-request path fetched and
    #      left over (its own counters), and what the search then fetches (counting build of the oct kernel) ----
    stats = None
    pstats = None
    if bwt.oct_index and not fused:
        d_stats = torch.zeros(8, dtype=torch.int64, device=dev)
        d_out_s = torch.empty(n, dtype=torch.int64, device=dev)
        d_status.zero_()
        bwt.pack_kmers_device(queries.data_ptr(), k, n, d_packed.data_ptr(), d_out_s.data_ptr(), d_status.data_ptr(), stream)
        pstats = bwt.pack_stats(d_packed.data_ptr(), k, n)
        bwt.count_kmers_packed_stats_device(d_packed.data_ptr(), k, n, d_out_s.data_ptr(), d_stats.data_ptr(), stream)
        # (list B -- k-mers holding `$` / `N` -- is not walked by the counting build: compare where it has nothing to add)
        torch.cuda.synchronize()
        if pstats["live_b"] == 0:
            assert (d_out_s == d_out).all(), "the counting build of the search kernel returns different counts"
        stats = [int(v) for v in d_stats.cpu().tolist()]
        del d_stats, d_out_s
    del flush, d_packed

    # ---- parity, every rank: a sample of this rank's slice against the CPU oracle ----
    cores = os.cpu_count() or 1
    my_threads = max(1, cores // world)
    orc = O.RleBWT()
    orc.load_vector(rle_host)
    q_slice_host = None
    if world > 1:
        m = min(n, 200_000)
        q_slice_host = queries[:m].cpu().numpy()
        assert (got[:m] == orc.count_kmers_fixed(q_slice_host, k, threads=my_threads)).all(), \
            f"rank {rank}: GPU counts differ from the CPU oracle"
        log(f"[rank {rank}] parity: {m} queries of slice [{lo}, {hi}) equal the oracle's counts")

    res = {
        "value": value, "ms_per_step": total_ms / args.steps,
        "config": workload_config(cfg, total, world),
        "engine": {"index_bytes": bwt.index_bytes, "suffix_table_s": table_s, "pair_index": bwt.pair_index,
                   "quad_index": bwt.quad_index, "oct_index": bwt.oct_index, "oct_bucket_shift": bwt.oct_bucket_shift,
                   "final_index": bwt.final_index, "final_bucket_shift": bwt.final_bucket_shift,
                   "queries_per_gpu_per_step": n,
                   "parallelism": f"index replicated on {world} GPU(s), the batch cut into {world} contiguous slice(s), no collective",
                   "l2": "L2 flushed (512 MB fill) between timed iterations; the query batch (n*k bytes) exceeds L2"},
        "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall, "checksum": checksum,
        "parity": {"every_rank_checked_its_slice": world > 1},
        "packed_input": packed_input,
    }

    # ---- e2e: the drop-in C-ABI calls with HOST buffers (pinned), H2D + D2H inside, ONE handle over all the GPUs ----
    lib = M.load_library()
    want_bytes = True
    q_dev_list = [queries_all]
    if not strong and world > 1:
        # configs[4] at N GPUs: rank 0 regenerates every rank's share (same seeds) for the one-handle run; the batch
        # travels as packed integers only (a 10^9-query byte batch would be 31 GB of pinned host memory)
        want_bytes = False
    if world == 1:
        legs, host = e2e_legs(args, cfg, bwt.handle, lib, M, q_dev_list, k, reads_sample, 1, want_bytes)
        assert legs["u64"]["checksum"] == checksum, "host-path and device-path results differ"
        del bwt
    else:
        # every rank releases its replica; rank 0 alone then drives devices 0..N-1 through one handle while the
        # others sleep in a gloo barrier (an NCCL barrier would keep a kernel spinning on their GPUs)
        del bwt, d_out
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        host_barrier()
        legs, host = None, None
        if rank == 0:
            os.environ["MSBWT_HOST_THREADS"] = str(min(64, cores))
            if not strong:
                from harness import synth
                reads = synth.make_reads(cfg["reads"], cfg["read_len"], cfg["coverage"], cfg["error"], device=dev)   # same seeds: same reads
                q_dev_list = [synth.make_queries(reads, k, cfg["n_read"], cfg["n_random"], seed_offset=1000 * r) for r in range(world)]
                del reads
                torch.cuda.empty_cache()
            t0 = time.time()
            multi = M.RleBWT.new(devices=list(range(world)))
            multi.load_vector(rle_host)
            log(f"[rank 0] one handle over devices {multi.device_ordinals}: replicas built in {time.time() - t0:.1f}s")
            legs, host = e2e_legs(args, cfg, multi.handle, lib, M, q_dev_list, k, reads_sample, world, want_bytes)
            # parity of the dispatcher: this rank's slice equals what its own replica computed, and an evenly spread
            # sample of the whole batch equals the oracle
            if strong:
                assert (host["o64"][lo:hi] == got).all(), "one-handle dispatcher and per-rank replica differ on rank 0's slice"
            nq = host["o64"].shape[0]
            idx = np.linspace(0, nq - 1, 200_000).astype(np.int64)
            if host["q_np"] is not None:
                qs = host["q_np"][idx]
            else:
                allq = torch.cat([q[torch.from_numpy(idx[(idx >= o) & (idx < o + q.shape[0])] - o).to(q.device)]
                                  for o, q in zip(np.cumsum([0] + [int(q.shape[0]) for q in q_dev_list[:-1]]), q_dev_list)])
                qs = allq.cpu().numpy()
            assert (host["o64"][idx] == orc.count_kmers_fixed(qs, k, threads=cores)).all(), "dispatcher counts differ from the CPU oracle"
            res["parity"]["dispatcher_sample"] = int(idx.size)
            del multi
            os.environ.pop("MSBWT_HOST_THREADS", None)
        del q_dev_list
        torch.cuda.empty_cache()
        host_barrier()
    if rank == 0:
        main_leg = legs["bytes"] if "bytes" in legs else legs["u64"]
        res["e2e"] = {"value": main_leg["value"], "unit": UNIT, "h2d_bytes_per_step": main_leg["h2d_bytes_per_step"],
                      "d2h_bytes_per_step": main_leg["d2h_bytes_per_step"], "ms_per_step": main_leg["ms_per_step"],
                      "entry": main_leg["entry"], "route": main_leg.get("route"),
                      "handle": f"one msbwt_index over devices [0..{world - 1}] on rank 0 (the library's dispatcher: one host thread per device, host-side gather)",
                      "host_pack_threads": legs["host_pack_threads"],
                      "u64": legs["u64"], "u64_out32": legs["u64_out32"], "pileup": legs.get("pileup"),
                      "bytes": legs.get("bytes")}

    # ---- parity (full), CPU baseline and algorithmic bytes (rank 0, bounded samples) ----
    if rank == 0:
        q_host = host["q_np"] if host["q_np"] is not None else queries[: min(n, 2_000_000)].cpu().numpy()
        if "pile_counts" in host:
            pw = np.ascontiguousarray(np.lib.stride_tricks.sliding_window_view(reads_sample[:64], k, axis=1)).reshape(-1, k)
            assert (host["pile_counts"].reshape(-1) == orc.count_kmers_fixed(pw, k, threads=cores)).all(), "pileup counts differ from the CPU oracle"
        if world == 1:
            tgt = 8.0 if primary else 4.0
            v1, m1, c1 = cpu_reference_leg(orc, q_host, k, 1, tgt, "single thread")
            assert (got[:m1] == c1).all(), "GPU counts differ from the CPU oracle"
            vN, mN, cN = cpu_reference_leg(orc, q_host, k, cores, tgt, "all-core static split")
            assert (got[:mN] == cN).all(), "GPU counts differ from the CPU oracle"
            res["cpu_baseline"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                                   "sample": f"first {m1} of {n} queries, single thread (the reference's loop)",
                                   "allcore": {"value": vN, "cores": cores, "sample": f"first {mN} of {n} queries"},
                                   "parity_checked_queries": max(m1, mN)}
            res["parity"]["oracle_checked_queries"] = max(m1, mN)
        else:
            res["cpu_baseline"] = None
        # algorithmic bytes (SURVEY 8d): the index lines the implemented algorithm must touch -- counted EXACTLY by
        # the counting build of the search kernel on the first `ms` queries when the index has an oct image, else by
        # replaying the batch through the oracle -- plus the packed query and the result.  The no-table / one-step
        # figure (what the reference's 31 steps would cost on 64-B blocks) is reported beside it.
        mo = min(n, 1_000_000, q_host.shape[0])
        steps0, two0 = orc.count_kmers_stats(q_host[:mo], k, BLOCK_SHIFT)
        packed_q = 8 * (-(-k // 21) + 1) + 4   # symbol words + seed + index of the compacted live list
        bytes_per_query_no_table = (steps0 + two0) * BLOCK_BYTES / mo + packed_q + 8
        pair, quad, octi = res["engine"]["pair_index"], res["engine"]["quad_index"], res["engine"]["oct_index"]
        oct_lines = final_lines = final_overflowed = quad_steps = quad_lines = one_steps = one_blocks = pair_lines = 0
        hits = mo
        if stats is not None:
            oct_lines, final_lines, final_overflowed, quad_steps, quad_lines, one_steps, one_blocks, walked = stats
            denom = n
            ref_steps = M.oct_symbols() * oct_lines + 20 * (final_lines - final_overflowed) + 4 * quad_steps + one_steps
            source = f"counting build of the search kernel on this rank's {n} queries ({walked} reached the search)"
        elif quad:
            st = orc.count_kmers_stats_quad(q_host[:mo], k, table_s, QUAD_SYMS, LINE_BYTES // QUAD_SECTOR_BYTES, BLOCK_SHIFT, 0, M.oct_symbols(), 0)
            hits, quad_steps = st["table_hits"], st["quad_steps"]
            quad_lines = st["quad_steps"] + st["two_line_quad_steps"]
            one_steps, one_blocks = st["one_steps"], st["one_steps"] + st["two_block_one_steps"]
            denom, ref_steps = mo, 4 * st["quad_steps"] + st["one_steps"]
            source = f"oracle replay of the first {mo} of {n} queries"
        elif pair:
            st = orc.count_kmers_stats_pair(q_host[:mo], k, table_s, PAIR_SYMS, BLOCK_SHIFT)
            hits = st["table_hits"]
            pair_lines = st["pair_steps"] + st["two_line_pair_steps"]
            one_steps, one_blocks = st["one_steps"], st["one_steps"] + st["two_block_one_steps"]
            denom, ref_steps = mo, 2 * st["pair_steps"] + st["one_steps"]
            source = f"oracle replay of the first {mo} of {n} queries"
        else:
            steps, two, hits = orc.count_kmers_stats_skip(q_host[:mo], k, BLOCK_SHIFT, table_s)
            one_steps, one_blocks, denom, ref_steps = steps, steps + two, mo, steps
            source = f"oracle replay of the first {mo} of {n} queries"
        depth = M.load_library().msbwt_debug_table_depth(k, table_s, M.oct_symbols() if octi else (4 if quad else 2 if pair else 1))
        table_level_bytes = (4 ** depth) * 8 if depth > 0 else 0
        table_hit_bytes = 8 if table_level_bytes <= 64 << 20 else LINE_BYTES   # an L2-resident level costs its 8 bytes
        table_hits_q = (hits / mo) if depth > 0 else 0.0
        peak, peak_src = measured_peak_gbs()
        pack_s = statistics.mean(step_ms) / 1e3 - statistics.mean(kern_ms) / 1e3
        search_s = statistics.mean(kern_ms) / 1e3
        step_s = statistics.mean(step_ms) / 1e3
        # the two kernels of a step.  SEARCH: the index lines it fetches, the packed query (symbol word, seed range,
        # index) of every query that reaches it, the result.  PACK/SEED: k symbol bytes in, one suffix-table entry, and
        # either the packed query out (20 B) or -- on the one-request path (pack_seed_final_kernel: k = 31 / 32 with a
        # final-step image) -- one 128-B final-step line and the 8-B result, with only the leftovers written out.
        search_lines128 = oct_lines + final_lines + quad_lines + pair_lines
        search_queries = (pstats["live_a"] + pstats["live_b"]) if pstats else n
        search_bytes = search_lines128 * LINE_BYTES * (n / denom) + one_blocks * BLOCK_BYTES * (n / denom) + search_queries * (packed_q + 8)
        one_request = bool(pstats and pstats["final_lines"] > 0)
        if one_request:
            answered = n - pstats["live_a"] - pstats["live_b"]
            pack_bytes = n * (k + table_hit_bytes) + pstats["final_lines"] * LINE_BYTES + answered * 8 + (pstats["live_a"] + pstats["live_b"]) * packed_q
            pack_lines = pstats["final_lines"]
            pack_kernel = "pack_seed_final_kernel (pack + suffix-table entry + ONE final-step line per 31-mer)"
        else:
            pack_bytes = n * (k + table_hits_q * table_hit_bytes) + search_queries * packed_q + (n - search_queries) * 8
            pack_lines = 0
            pack_kernel = "pack_seed_kernel"
        search_kernel = ("count_kmers_oct_kernel<RAW> (fused: pack + table + search)" if fused else "count_kmers_oct_kernel" if octi
                         else "count_kmers_quad_kernel" if quad else ("count_kmers_pair_kernel" if pair else "count_kmers_packed_kernel"))
        if fused:   # the fused kernel reads the k symbol bytes itself and one 16-byte piece of the (L2-resident) table level
            search_bytes = search_lines128 * LINE_BYTES * (n / denom) + one_blocks * BLOCK_BYTES * (n / denom) + n * (16 + k + 8)
        dominant_is_pack = one_request and pack_s >= search_s
        dom_bytes, dom_s, dom_kernel = (pack_bytes, pack_s, pack_kernel) if dominant_is_pack else (search_bytes, search_s, search_kernel)
        achieved = dom_bytes / dom_s / 1e9
        hbm_requests = pack_lines + (search_lines128 + one_blocks) * (n / denom)   # line fills a step asks HBM for (table entries come from L2)
        if table_hit_bytes == LINE_BYTES:
            hbm_requests += table_hits_q * n
        traffic, traffic_src = ncu_traffic(cfg["key"], dom_kernel.split(" ")[0])
        res["roofline"] = {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src, "kernel": dom_kernel,
            "fused": bool(fused), "kernel_ms": 1e3 * dom_s, "algorithmic_bytes_per_launch": dom_bytes,
            "algorithmic_bytes_per_query": dom_bytes / n,
            "one_request_path": one_request, "pack_stage": pstats,
            "kernels": {"pack": {"kernel": pack_kernel, "ms": 1e3 * pack_s, "algorithmic_bytes": pack_bytes,
                                 "achieved": pack_bytes / max(pack_s, 1e-9) / 1e9, "hbm_line_requests": pack_lines},
                        "search": {"kernel": search_kernel, "ms": 1e3 * search_s, "algorithmic_bytes": search_bytes,
                                   "achieved": search_bytes / max(search_s, 1e-9) / 1e9, "queries": search_queries,
                                   "oct_lines": oct_lines * (n / denom), "final_step_lines": final_lines * (n / denom),
                                   "final_step_overflowed": final_overflowed * (n / denom), "quad_lines": quad_lines * (n / denom),
                                   "pair_lines": pair_lines * (n / denom), "one_step_blocks": one_blocks * (n / denom),
                                   "mean_reference_steps_per_query": ref_steps / max(1, denom), "accounting_source": source}},
            "hbm_line_requests_per_query": hbm_requests / n,
            "index_accesses_per_query": hbm_requests / n,
            "index_accesses_per_s": hbm_requests / step_s,
            "no_table": {"algorithmic_bytes_per_query": bytes_per_query_no_table, "mean_steps_per_query": steps0 / mo,
                         "achieved_if_counted_without_table": bytes_per_query_no_table * n / step_s / 1e9},
            "step": {"what": "pack/seed kernel + search kernel = value's timed region",
                     "ms": 1e3 * step_s, "algorithmic_bytes": pack_bytes + search_bytes,
                     "achieved": (pack_bytes + search_bytes) / step_s / 1e9, "frac": (pack_bytes + search_bytes) / step_s / 1e9 / peak,
                     "suffix_table_depth_used": depth, "suffix_table_level_bytes": table_level_bytes,
                     "hbm_line_requests_per_s": hbm_requests / step_s},
            "note": ("achieved counts every index line as a 128-B HBM line fill; where part of an image stays in L2 "
                     "the kernel runs above the HBM random-request rate and frac can exceed what DRAM alone would allow -- "
                     "`traffic` is the DRAM side.  The physical ceiling of this path is the random-read REQUEST rate "
                     "(gather_reads_per_s, K4 in the same run), not the copy bandwidth `peak`: see frac_of_gather128_request_rate"),
            "peak_source": peak_src}
        res["kernel_share_of_step"] = statistics.mean(kern_ms) / statistics.mean(step_ms)
    del queries, queries_all
    torch.cuda.empty_cache()
    return res


def gather_roofline(local, dev):
    """K4: what independent random 32/64/128-B reads sustain on this box (2 GiB buffer, DRAM)."""
    import torch

    import rust_msbwt_b200 as M
    stream = torch.cuda.current_stream().cuda_stream
    gb = torch.empty(2 << 30, dtype=torch.uint8, device=dev)
    sink = torch.zeros(1, dtype=torch.int64, device=dev)
    res = {}
    for gran in (32, 64, 128):
        ng = 1 << 27
        best = None
        for it in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            M.gather_bench(local, gb.data_ptr(), gb.numel(), gran, ng, 1234 + it, sink.data_ptr(), stream)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        res[str(gran)] = {"gb_per_s": ng * gran / (best / 1e3) / 1e9, "reads_per_s": ng / (best / 1e3)}
    del gb
    return res


def host_memory_bandwidth():
    """What the end-to-end path is bound by on the host side: one large memcpy per thread count (numpy releases the
    GIL), GB/s of bytes read + written."""
    import threading

    import numpy as np
    out = {}
    try:
        cores = os.cpu_count() or 1
        size = 256 << 20
        for th in sorted({1, min(8, cores), cores}):
            src = [np.ones(size, dtype=np.uint8) for _ in range(th)]
            dst = [np.empty(size, dtype=np.uint8) for _ in range(th)]
            def work(i):
                np.copyto(dst[i], src[i])
            for rep in range(2):
                ts = [threading.Thread(target=work, args=(i,)) for i in range(th)]
                t0 = time.perf_counter()
                for t in ts:
                    t.start()
                for t in ts:
                    t.join()
                dt = time.perf_counter() - t0
            out[str(th)] = 2 * size * th / dt / 1e9
    except Exception as e:  # measurement aid only
        out["error"] = str(e)
    return out


def run_ours(args, cfg_keys):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist = None
    gloo = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout at first use; stdout carries only the JSON line
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
            gloo = dist.new_group(backend="gloo")
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():   # CPU-side only: the waiting ranks leave their GPUs idle
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier(group=gloo)

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = dict(rank=rank, world=world, local=local, dev=dev, barrier=barrier, max_over_ranks=max_over_ranks,
               host_barrier=host_barrier)
    cfgs = [WORKLOADS[key] for key in cfg_keys]
    main_res = measure_ours(args, cfgs[0], ctx, primary=True)
    others = [measure_ours(args, c, ctx, primary=False) for c in cfgs[1:]]
    if rank == 0:
        gather = None
        try:
            gather = gather_roofline(local, dev)
        except Exception as e:  # measurement aid only
            log("gather microbench failed:", e)
        for r in [main_res] + others:
            rf = r.get("roofline")
            if rf and gather:
                rf["gather_gbs"] = {g: v["gb_per_s"] for g, v in gather.items()}
                rf["gather_reads_per_s"] = {g: v["reads_per_s"] for g, v in gather.items()}
                rf["frac_of_gather128_request_rate"] = rf["index_accesses_per_s"] / gather["128"]["reads_per_s"]
                # the random-read roofline in BYTES: what K4's independent random 128-byte reads move per second on this
                # box in this run -- the ceiling of any kernel whose traffic is line fills (the copy peak is not reachable
                # by random access: K4 itself sits at 0.77 of it)
                rf["random_read_roofline_gbs"] = gather["128"]["gb_per_s"]
                rf["frac_of_random_read_roofline"] = rf["achieved"] / gather["128"]["gb_per_s"]
                for kn in ("pack", "search"):
                    kk = rf["kernels"][kn]
                    if kn == "pack":
                        kk["line_requests_per_s"] = kk["hbm_line_requests"] / max(kk["ms"] / 1e3, 1e-9)
                    else:
                        kk["line_requests_per_s"] = (kk["oct_lines"] + kk["final_step_lines"] + kk["quad_lines"] + kk["pair_lines"] + kk["one_step_blocks"]) / max(kk["ms"] / 1e3, 1e-9)
                    kk["frac_of_gather128_request_rate"] = kk["line_requests_per_s"] / gather["128"]["reads_per_s"]
        line = {
            "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": cfgs[0]["scaling"], "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        }
        for key in ("config", "engine", "e2e", "packed_input", "gpu_launches", "clocks", "roofline", "cpu_baseline", "parity",
                    "wall_s_timed_region", "checksum", "kernel_share_of_step"):
            line[key] = main_res.get(key)
        line["host_memory_gbs_by_threads"] = host_memory_bandwidth()
        if others:
            line["other_workloads"] = [
                {key: r.get(key) for key in ("value", "ms_per_step", "config", "engine", "e2e", "packed_input", "gpu_launches", "roofline",
                                             "cpu_baseline", "parity", "checksum")} | {"scaling": c["scaling"]}
                for r, c in zip(others, cfgs[1:])]
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS) + ["default"],
                    default=os.environ.get("MSBWT_BENCH_WORKLOAD", "default"),
                    help="default = configs[2] as the bench line; configs[1] (N = 1) and configs[4] (N = 1 and 8) nested beside it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the counts of the last timed step of every workload to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "default":
        keys = [HEADLINE]
        if args.impl == "ours":
            if world == 1:
                keys.append("cfg2")
            # configs[4] is specified at 8 GPUs (and measured as one GPU's share at N = 1); MSBWT_BENCH_CFG5_ANY_N=1 runs
            # its N-GPU code path at any N (plumbing checks on smaller boxes)
            if (world in (1, 8) or os.environ.get("MSBWT_BENCH_CFG5_ANY_N", "0") not in ("", "0")) and \
                    os.environ.get("MSBWT_BENCH_SKIP_CFG5", "0") in ("", "0"):
                keys.append("cfg5")
    else:
        keys = [args.workload]
    if args.impl == "reference":
        run_reference(args, [WORKLOADS[key] for key in keys])
    else:
        run_ours(args, keys)


if __name__ == "__main__":
    main()
