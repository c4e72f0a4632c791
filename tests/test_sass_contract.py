"""What the shipped SASS must contain, checked with cuobjdump (no GPU needed).

Kernels whose lanes exchange data after divergent code -- shuffles, ballots, shared memory + __syncwarp() -- need the
warp back together at those points.  ptxas 12.9 can "prove" that it is, drop every __syncwarp() and issue the
collectives without a WARPSYNC; on B200 that assumption failed under load in the oct search kernel (50-100 M-query
batches of k = 43 / 53 / 63: unanswered queries, warps that never finished; profiles/r2t_convergence.md).
`warp_sync_guard` (kernel_common.cuh) makes ptxas compile those kernels conservatively.  This test pins the outcome,
not the trick: every such kernel of libmsbwt_b200.so carries WARPSYNC instructions, at least one per collective for the
oct kernel -- a toolchain that changes its mind fails here instead of at 3 a.m. on somebody's read set."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")


@pytest.fixture(scope="module")
def sass_counts():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(LIB):
        pytest.skip("library not built (python rust-msbwt_b200/build.py)")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    demangle = shutil.which("cu++filt") or "/usr/local/cuda/bin/cu++filt"
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = {"WARPSYNC": 0, "SHFL": 0, "VOTE": 0}
            continue
        if cur:
            for op in ("WARPSYNC", "SHFL", "VOTE"):
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    names = list(counts)
    nice = subprocess.run([demangle], input="\n".join(names), capture_output=True, text=True).stdout.splitlines() \
        if os.path.exists(demangle) else names
    return {n: counts[m] for n, m in zip(nice, names)}


def test_every_warp_cooperative_search_kernel_keeps_its_warp_syncs(sass_counts):
    def pick(pred):
        got = {k: v for k, v in sass_counts.items() if pred(k)}
        assert got, "no such kernel in the library"
        return got

    # the oct search kernel: packed, counting (STATS) and WIDE instantiations -- per iteration a ballot, the
    # line requests exchanged through shared memory, cp.async rows read by other lanes, four __syncwarp(), the warp-wide
    # scan of the final-step lines (vote + reduce); ptxas's conservative build carries a WARPSYNC.COLLECTIVE for each
    oct_kernels = pick(lambda k: "count_kmers_oct_kernel<" in k)
    assert len(oct_kernels) == 3
    for name, c in oct_kernels.items():
        assert c["VOTE"] >= 4 and c["WARPSYNC"] >= 8, (name, c)
    # quads of lanes (pair image) and lane pairs (one-step blocks, LANES = 2) combine their parts through shuffles
    for name, c in pick(lambda k: "count_kmers_pair_kernel<" in k).items():
        assert c["SHFL"] >= 4 and c["WARPSYNC"] >= 1, (name, c)
    for name, c in pick(lambda k: re.search(r"count_kmers_packed_kernel<\(bool\)[01], \(int\)2,", k) is not None).items():
        assert c["SHFL"] >= 3 and c["WARPSYNC"] >= 1, (name, c)
    # the pack / seed kernels: append_live's ballots (one atomic per CTA and list) follow a divergent table lookup
    for name, c in pick(lambda k: re.search(r"(pack_seed_kernel|seed_packed_kernel|seed_u64_kernel)<", k) is not None).items():
        assert c["VOTE"] >= 2 and c["WARPSYNC"] >= 1, (name, c)
    # the one-request kernel (ptxas keeps these on its own; pinned all the same)
    for name, c in pick(lambda k: "pack_seed_final_kernel<" in k).items():
        assert c["WARPSYNC"] >= 24, (name, c)
