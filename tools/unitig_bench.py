"""The unitigs of an index's solid k-mers (msbwt_unitigs, unitigs.cu) on configs[2]'s index (10 M 150-bp reads, 1 %
errors, 1.51 Gsymbols).  Plain mode runs on the reads as synthesised (one strand); canonical mode on the same reads
with every other read reverse-complemented (two-strand data, as tools/spectrum_bench.py --canonical uses), the two
indexes built and loaded one at a time.  k in {21, 31}, min_count in {1, 2, 5}.
One JSON line per run: the card and its power limit (read in the same run), the best-of-three wall time of the call,
n_nodes (|V|), n_unitigs, the total symbols, the N50 of the unitig lengths, the peak device memory above the level
before the call (cudaMemGetInfo sampled every millisecond), the kernel launches (msbwt_launch_count delta) and, from
a separate torch.profiler run, the device time of each phase: walk (spectrum expand / emit, both passes), walk_rc
(canonical: the query path's reverse-complement counts and the resolve kernels), select (CUB compactions), sort
(CUB radix sort), link, cycles, ranking, emission (tail / emit kernels and the scans) and copy (device-to-host).
    python tools/unitig_bench.py [--out profiles/unitig_bench.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import rust_msbwt_b200 as M  # noqa: E402


def card() -> dict:
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "not read"
    return out


class PeakMemory:
    """device bytes in use above the level at start, sampled with cudaMemGetInfo while the call runs"""

    def __enter__(self):
        torch.cuda.synchronize()
        self.base = torch.cuda.mem_get_info(0)[0]
        self.low = self.base
        self.stop = False
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def _run(self):
        while not self.stop:
            self.low = min(self.low, torch.cuda.mem_get_info(0)[0])
            time.sleep(0.001)

    def __exit__(self, *exc):
        self.stop = True
        self.t.join()
        self.peak = self.base - self.low


def phase(name: str, kind) -> str:
    if kind == torch.autograd.DeviceType.CUDA and "Memcpy DtoH" in name:
        return "copy_ms"
    n = name
    if "spectrum_expand" in n or "spectrum_emit" in n:
        return "walk_ms"
    if "canonical_" in n or "seed" in n or "count_kmers" in n:
        return "walk_rc_ms"
    if "DeviceSelect" in n or "DeviceCompact" in n:
        return "select_ms"
    if "Radix" in n or "Onesweep" in n:
        return "sort_ms"
    if any(s in n for s in ("unitig_link", "unitig_prev", "unitig_next", "unitig_revcomp")):
        return "link_ms"
    if "unitig_cycle" in n or "unitig_cut" in n:
        return "cycles_ms"
    if "unitig_rank" in n:
        return "ranking_ms"
    if "unitig_tail" in n or "unitig_emit" in n or "DeviceScan" in n:
        return "emission_ms"
    if "Memcpy DtoH" in n:
        return "copy_ms"
    return "other_ms"


def phase_times(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    keys = ("walk_ms", "walk_rc_ms", "select_ms", "sort_ms", "link_ms", "cycles_ms", "ranking_ms", "emission_ms",
            "copy_ms", "other_ms")
    sums = dict.fromkeys(keys, 0.0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        sums[phase(ev.name, ev.device_type)] += ev.time_range.elapsed_us() / 1e3
    return {k: round(v, 3) for k, v in sums.items()}


def n50(lens: np.ndarray) -> int:
    s = np.sort(lens)[::-1]
    c = np.cumsum(s)
    return int(s[np.searchsorted(c, (c[-1] + 1) // 2)]) if s.size else 0


def run(g, reads_label: str, k: int, t: int, canonical: bool, crd: dict) -> dict:
    L = M.load_library()
    g.unitigs(k, t, canonical)  # warm-up
    wall = None
    for _ in range(3):
        before = L.msbwt_launch_count()
        with PeakMemory() as mem:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            syms, offs, sums = g.unitigs(k, t, canonical)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        launches = L.msbwt_launch_count() - before
        wall = dt if wall is None else min(wall, dt)
    lens = np.diff(offs).astype(np.int64)
    n_nodes = int(g.kmer_spectrum(k, t, 2, canonical=canonical)[1])
    if canonical:  # both members of each pair, a palindrome once (none at odd k)
        n_nodes *= 2
    res = {"reads": reads_label, "mode": "canonical" if canonical else "plain", "k": k, "min_count": t, "card": crd,
           "wall_s": round(wall, 4), "n_nodes": n_nodes, "n_unitigs": int(lens.size), "total_symbols": int(lens.sum()),
           "n50": n50(lens), "windows": int((lens - k + 1).sum()), "peak_device_bytes": int(mem.peak),
           "peak_device_bytes_per_node": round(mem.peak / max(n_nodes, 1), 2), "launches": int(launches),
           **phase_times(lambda: g.unitigs(k, t, canonical))}
    del syms, offs, sums
    print(json.dumps(res), flush=True)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "unitig_bench.jsonl"))
    ap.add_argument("--ks", default="21,31")
    ap.add_argument("--min-counts", default="1,2,5")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    crd = card()
    ks = [int(x) for x in args.ks.split(",")]
    ts = [int(x) for x in args.min_counts.split(",")]
    results = []
    reads, rle, _ = bench.build_reads_and_bwt(bench.WORKLOADS["cfg3"], dev, True)
    for label, canonical in (("one strand", False), ("every other read reverse-complemented", True)):
        if canonical:
            rc = torch.tensor([0, 5, 3, 2, 4, 1], dtype=torch.uint8, device=dev)  # $ A C G N T -> complements
            reads[::2] = rc[reads[::2].flip(1).long()]
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            rle, _ = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
        torch.cuda.empty_cache()
        g = M.RleBWT.new(devices=[0])
        g.load_vector(rle)
        for k in ks:
            for t in ts:
                results.append(run(g, label, k, t, canonical, crd))
        del g
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in results:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
