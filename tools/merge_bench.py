"""Device merge of two multi-string BWTs (msbwt_merge_rle_bwts, bwt_merge.cu) at two sizes, in one process:

  cfg3_halves : configs[2]'s read set (10 M 150-bp reads, 1 % errors, 1.51 Gsymbols) built as 5 M + 5 M and merged;
                the device builder's time for all 10 M reads is measured beside it
  wide_halves : 15 M + 15 M reads of the same kind, each half built on its own (2.27 Gsymbols each), merged into
                4.53 Gsymbols -- beyond what the builder does in one call

One JSON line per case: the card and its power limit (read in the same run), passes, end-to-end merge time (host RLE
in -> host RLE out, the call returns after a device synchronise) and per pass, the kernel time per pass from a
separate torch.profiler run, the modelled bytes per pass and their rate against the copy peak, and the device memory
the merge held at its peak (cudaMemGetInfo sampled every millisecond while it ran).

    python tools/merge_bench.py [--out FILE] [--cases cfg3_halves,wide_halves]
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

import rust_msbwt_b200 as M  # noqa: E402
from harness import synth  # noqa: E402

COPY_PEAK_GBS = 6452.8  # DESIGN.md section 4: the project's measured device copy rate on B200
CASES = {"cfg3_halves": 5_000_000, "wide_halves": 15_000_000}

# Modelled DRAM bytes per merged row and pass (not measured):
#   interleave pass : the two inputs' bit-planes + checkpoints (64 B per 128 rows, each row in one input) 0.5,
#                     read I_t 1/8, write I_{t+1} 1/8
#   zeroing I_{t+1} : 1/8
#   count pass      : read I_{t+1} and I_t, 2/8
PASS_KERNEL_BYTES_PER_ROW = 0.5 + 0.125 + 0.125
ITERATION_BYTES_PER_ROW = PASS_KERNEL_BYTES_PER_ROW + 0.125 + 0.25


def card() -> dict:
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "not read"
    return out


def copy_peak() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            v = json.load(f).get("hbm_gbs")
        if v:
            return float(v), "MEASURED_PEAKS.json hbm_gbs"
    return COPY_PEAK_GBS, "DESIGN.md section 4 (6452.8 GB/s)"


class PeakMemory:
    """device bytes in use above the level at start, sampled with cudaMemGetInfo while the merge runs"""

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


def build_half(reads, lo, hi):
    part = reads[lo:hi]
    return M.build_rle_bwt(part.data_ptr(), 0, part.shape[0], part.shape[1])


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t


def kernel_times(rle_a, rle_b) -> dict:
    """sum of each kernel's device time over one merge (separate run, torch.profiler with CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        M.merge_rle_bwts(rle_a, rle_b)
        torch.cuda.synchronize()
    sums: dict[str, list] = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            s = sums.setdefault(ev.name, [0.0, 0])
            s[0] += ev.time_range.elapsed_us() / 1e3
            s[1] += 1
    return sums


def run_case(key: str, half: int) -> dict:
    torch.cuda.empty_cache()
    reads = synth.make_reads(2 * half, read_len=150, coverage=30.0, error_rate=0.01, device="cuda")
    (rle_a, n_a), build_a_s = timed(lambda: build_half(reads, 0, half))
    (rle_b, n_b), build_b_s = timed(lambda: build_half(reads, half, 2 * half))
    res = {"case": key, "reads": 2 * half, "read_len": 150, "error_rate": 0.01,
           "symbols_a": n_a, "symbols_b": n_b, "rle_bytes_a": int(rle_a.size), "rle_bytes_b": int(rle_b.size),
           "build_half_s": [round(build_a_s, 3), round(build_b_s, 3)]}
    whole = None
    if key == "cfg3_halves":   # the union still fits the builder
        (whole, _), res["build_union_s"] = timed(lambda: M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1]))
    del reads
    torch.cuda.empty_cache()

    with PeakMemory() as mem:
        (merged, total, iterations), merge_s = timed(lambda: M.merge_rle_bwts(rle_a, rle_b))
    res.update(total=total, iterations=iterations, merged_rle_bytes=int(merged.size), merge_s=round(merge_s, 4),
               merge_ms_per_iteration_end_to_end=round(1e3 * merge_s / iterations, 3),
               peak_device_bytes=int(mem.peak), peak_device_bytes_per_symbol=round(mem.peak / total, 3))
    if whole is not None:
        res["equals_union_build"] = bool(whole.size == merged.size and (whole == merged).all())
    del whole, merged

    ks = kernel_times(rle_a, rle_b)
    pass_ms = sum(v[0] for k, v in ks.items() if "merge_pass_kernel<false>" in k or "merge_pass_kernelILb0E" in k)
    zeros_ms = sum(v[0] for k, v in ks.items() if "tile_zeros_kernel" in k)
    other_ms = sum(v[0] for v in ks.values()) - pass_ms - zeros_ms
    peak, peak_src = copy_peak()
    pass_bytes = PASS_KERNEL_BYTES_PER_ROW * total
    iter_bytes = ITERATION_BYTES_PER_ROW * total
    per_pass_ms = pass_ms / iterations
    if not pass_ms:
        res["kernel_times"] = "not measured: the profiler recorded no interleave kernel"
        return res
    res.update(
        kernel_ms_total=round(sum(v[0] for v in ks.values()), 3),
        interleave_kernel_ms_per_iteration=round(per_pass_ms, 4),
        count_kernel_ms_per_iteration=round(zeros_ms / iterations, 4),
        other_device_ms_total=round(other_ms, 3),
        modelled_bytes_per_iteration=int(iter_bytes),
        modelled_interleave_kernel_bytes=int(pass_bytes),
        interleave_kernel_gbs=round(pass_bytes / per_pass_ms / 1e6, 1),
        interleave_kernel_share_of_copy_peak=round(pass_bytes / per_pass_ms / 1e6 / peak, 4),
        copy_peak_gbs=peak, copy_peak_source=peak_src,
        kernels={k: {"ms": round(v[0], 3), "launches": v[1]} for k, v in sorted(ks.items(), key=lambda kv: -kv[1][0])[:12]},
    )
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--cases", default=",".join(CASES))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the merge runs on the GPU only"
    torch.cuda.set_device(0)
    info = card()
    # warm-up: module load, first launches, the profiler's first start
    small = np.random.default_rng(1).choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(20_000, 150))
    a, _ = M.build_rle_bwt(small[:10_000])
    b, _ = M.build_rle_bwt(small[10_000:])
    M.merge_rle_bwts(a, b)
    kernel_times(a, b)
    lines = []
    for key in args.cases.split(","):
        res = {"card": info, **run_case(key, CASES[key])}
        line = json.dumps(res)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
