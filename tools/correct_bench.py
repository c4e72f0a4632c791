"""Read correction against an index (msbwt_correct_reads, correct.cu) on configs[2]'s index (10 M 150-bp reads of
a 50 Mbp genome, 1 % substitutions, 1.51 Gsymbols, forward strand).  The genome is regenerated from harness/synth.py's
seed with the same generator on the same device; reads to correct are sampled from it, from either strand, with
substitutions, insertions and deletions in equal parts: 10 kbp long reads at 1 %, 5 % and 10 % error and 150 bp short
reads at 1 %.  Each set is corrected at k = 21 and 31 (min_count 5, frac_permille 100, branch_limit 4).
One JSON line per run: the card and its power limit (read in the same run), the best-of-three wall time and bases per
second, the call's stats, the kernel launches (msbwt_launch_count delta), the peak device memory above the level before
the call (cudaMemGetInfo sampled every millisecond), accuracy on a sample of the reads (fraction identical to the truth,
edit distance to the truth before and after), and, from a separate torch.profiler run, BFS rounds (expand launches)
and the device time of the query kernels, of the correction kernels, of CUB and of copies, with the host's share
(wall time not covered by device time).  A last line times oracle/correct.py on a few reads, its count2 taken from
the same index one k-mer pair per call, and checks that it equals the device.
    python tools/correct_bench.py [--out profiles/correct_bench.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import rust_msbwt_b200 as M  # noqa: E402
from harness import synth  # noqa: E402
from oracle import correct as OC  # noqa: E402
from unitig_bench import PeakMemory, card  # noqa: E402

LUT = np.array([1, 2, 3, 5], np.uint8)
RC_SYM = np.array([0, 5, 3, 2, 4, 1], np.uint8)
PARAMS = (5, 100, 4)  # min_count, frac_permille, branch_limit


def sample(rng, genome, n, length, rate):
    """(reads with errors, their truths): a third of `rate` each as substitutions, insertions and deletions"""
    reads, truths = [], []
    for _ in range(n):
        a = int(rng.integers(0, genome.size - length + 1))
        t = LUT[genome[a:a + length]]
        if rng.random() < 0.5:
            t = RC_SYM[t[::-1]]
        kind = np.digitize(rng.random(t.size), [rate / 3, 2 * rate / 3, rate])  # 0 sub, 1 ins, 2 del, 3 keep
        r = t.copy()
        r[kind == 0] = LUT[(np.searchsorted(LUT, r[kind == 0]) + rng.integers(1, 4, int((kind == 0).sum()))) % 4]
        rep = np.where(kind == 1, 2, np.where(kind == 2, 0, 1))
        out = np.repeat(r, rep)
        out[np.cumsum(rep)[kind == 1] - 1] = LUT[rng.integers(0, 4, int((kind == 1).sum()))]
        reads.append(out)
        truths.append(t)
    return reads, truths


def edit_distance(a: np.ndarray, b: np.ndarray) -> int:
    """Levenshtein distance, one numpy pass per row: an insertion chain is a running minimum of t[j] - j"""
    ar = np.arange(b.size + 1)
    prev = ar.copy()
    for i in range(1, a.size + 1):
        t = np.empty(b.size + 1, np.int64)
        t[0] = i
        t[1:] = np.minimum(prev[1:] + 1, prev[:-1] + (b != a[i - 1]))
        prev = np.minimum.accumulate(t - ar) + ar
    return int(prev[-1])


def phase_times(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    sums = {"query_ms": 0.0, "correct_ms": 0.0, "cub_ms": 0.0, "copy_ms": 0.0, "other_ms": 0.0}
    rounds = 0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        n, ms = ev.name, ev.time_range.elapsed_us() / 1e3
        if "correct_expand_kernel" in n:
            rounds += 1
        if "Memcpy" in n or "Memset" in n:
            sums["copy_ms"] += ms
        elif "correct_" in n and "_kernel" in n and "cub" not in n:
            sums["correct_ms"] += ms
        elif "cub" in n or "Device" in n:
            sums["cub_ms"] += ms
        elif any(s in n for s in ("seed", "count", "oct", "pair", "quad", "final", "pack", "one_step", "search")):
            sums["query_ms"] += ms
        else:
            sums["other_ms"] += ms
    return {"bfs_rounds": rounds, **{k: round(v, 3) for k, v in sums.items()}}


def run(g, label: str, reads, truths, k: int, crd: dict, n_acc: int) -> dict:
    L = M.load_library()
    bases = int(sum(r.size for r in reads))
    wall, out, stats, launches, mem = None, None, None, 0, None
    for _ in range(3):
        before = L.msbwt_launch_count()
        with PeakMemory() as pm:
            t0 = time.perf_counter()
            out, stats = g.correct_reads(reads, k, *PARAMS)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        launches = L.msbwt_launch_count() - before
        mem = pm.peak if mem is None else max(mem, pm.peak)
        wall = dt if wall is None else min(wall, dt)
    idx = range(min(n_acc, len(reads)))
    before_d = [edit_distance(reads[i], truths[i]) for i in idx]
    after_d = [edit_distance(out[i], truths[i]) for i in idx]
    prof = phase_times(lambda: g.correct_reads(reads, k, *PARAMS))
    dev_ms = sum(v for key, v in prof.items() if key.endswith("_ms"))
    res = {"reads": label, "n_reads": len(reads), "bases": bases, "k": k, "min_count": PARAMS[0],
           "frac_permille": PARAMS[1], "branch_limit": PARAMS[2], "card": crd, "wall_s": round(wall, 4),
           "bases_per_s": round(bases / wall, 1), "stats": [int(x) for x in stats], "launches": int(launches),
           "peak_device_bytes": int(mem), "accuracy_sample": len(idx),
           "identical_to_truth": round(float(np.mean([d == 0 for d in after_d])), 4),
           "identical_to_truth_before": round(float(np.mean([d == 0 for d in before_d])), 4),
           "edit_distance_before": int(sum(before_d)), "edit_distance_after": int(sum(after_d)),
           **prof, "device_ms_total": round(dev_ms, 3),
           "host_share_of_wall": round(max(0.0, 1 - dev_ms / 1e3 / wall), 4)}
    print(json.dumps(res), flush=True)
    return res


def oracle_run(g, reads, k: int, crd: dict) -> dict:
    """oracle/correct.py with count2 from the index, one k-mer pair per call, against the device on the same reads"""
    cache = {}

    def count2(x):
        if x not in cache:
            c = g.count_kmers_u64(np.array([x, OC.revcomp(x, k)], np.uint64), k)
            cache[x] = int(c[0]) + int(c[1])
        return cache[x]

    t0 = time.perf_counter()
    want, wstats = OC.correct_reads([r.tolist() for r in reads], k, *PARAMS, count2)
    dt = time.perf_counter() - t0
    got, gstats = g.correct_reads(reads, k, *PARAMS)
    same = gstats.tolist() == wstats and all(a.tolist() == b for a, b in zip(got, want))
    res = {"reads": "oracle/correct.py on the host, count2 one k-mer pair per library call", "n_reads": len(reads),
           "bases": int(sum(r.size for r in reads)), "k": k, "card": crd, "wall_s": round(dt, 3),
           "bases_per_s": round(sum(r.size for r in reads) / dt, 1), "count2_calls": len(cache),
           "stats": wstats, "device_equals_oracle": bool(same)}
    print(json.dumps(res), flush=True)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "correct_bench.jsonl"))
    ap.add_argument("--long-reads", type=int, default=200)
    ap.add_argument("--short-reads", type=int, default=200000)
    ap.add_argument("--accuracy-sample", type=int, default=10)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    crd = card()
    cfg = bench.WORKLOADS["cfg3"]
    reads, rle, _ = bench.build_reads_and_bwt(cfg, dev, True)
    del reads
    torch.cuda.empty_cache()
    glen = max(cfg["read_len"], int(cfg["reads"] * cfg["read_len"] / cfg["coverage"]))
    genome = torch.randint(0, 4, (glen,), generator=synth._gen(dev, synth.SEED_GENOME), device=dev,
                           dtype=torch.uint8).cpu().numpy()
    g = M.RleBWT.new(devices=[0])
    g.load_vector(rle)
    del rle
    rng = np.random.default_rng(2026)
    sets = [(f"10 kbp at {int(e * 100)} %", *sample(rng, genome, args.long_reads, 10000, e)) for e in (0.01, 0.05, 0.10)]
    sets.append(("150 bp at 1 %", *sample(rng, genome, args.short_reads, 150, 0.01)))
    g.correct_reads(sets[0][1][:4], 21, *PARAMS)  # warm-up: module load, CUB's first calls
    results = []
    for label, rs, ts in sets:
        for k in (21, 31):
            results.append(run(g, label, rs, ts, k, crd, args.accuracy_sample))
    small = sets[3][1][:20] + sets[0][1][:1]
    for k in (21, 31):
        results.append(oracle_run(g, small, k, crd))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in results:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
