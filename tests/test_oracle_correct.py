"""oracle/correct.py -- the CPU restatement of msbwt_correct_reads -- on hand-built reads of a repeat-free random
genome whose counts come from error-free reads tiling both strands, and the shipped SASS of the correction kernels (no
GPU needed)."""
import os
import random
import re
import shutil
import subprocess

import pytest

from oracle import correct as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")
K = 15
_RC = str.maketrans("ACGT", "TGCA")


def rc(s):
    return s.translate(_RC)[::-1]


def sy(s):
    return ["$ACGNT".index(c) for c in s]


def text(syms):
    return "".join("$ACGNT"[s] for s in syms)


def tiles(g, length=80, step=5):
    """error-free reads tiling both strands of g"""
    out = []
    for i in list(range(0, len(g) - length + 1, step)) + [len(g) - length]:
        out += [g[i:i + length], rc(g[i:i + length])]
    return out


def genome(n, seed, k=K):
    """a random genome whose k-mers occur once on both strands together"""
    rng = random.Random(seed)
    while True:
        g = "".join(rng.choice("ACGT") for _ in range(n))
        seen = [g[i:i + k] for i in range(n - k + 1)]
        if len(set(seen + [rc(x) for x in seen])) == 2 * len(seen):
            return g


@pytest.fixture(scope="module")
def ref():
    g = genome(2000, 11)
    return g, C.window_count2([sy(t) for t in tiles(g)], K)


def correct(reads, count2, k=K, min_count=2, frac=100, branch_limit=4):
    out, stats = C.correct_reads([sy(r) for r in reads], k, min_count, frac, branch_limit, count2)
    return [text(o) for o in out], stats


def sub(s, i):
    return s[:i] + ("A" if s[i] != "A" else "C") + s[i + 1:]


def ins(s, i):
    """a base inserted before s[i] that differs from both neighbours (next to an equal base the run is one window
    short: the read then holds one base more than X and Y leave room for, which no E can remove)"""
    return s[:i] + min(set("ACGT") - {s[i - 1], s[i]}) + s[i:]


def site(s, i, n, new=""):
    """the first j >= i where replacing s[j:j+n] by `new` makes every window over the edit weak (the first and last
    base of the edit differ from the bases they displace: otherwise the run is shorter and may not be eligible)"""
    while (new or s[i + n:])[0] == s[i] or (s[:i] + new)[-1] == s[i + n - 1]:
        i += 1
    return i


def test_isolated_substitution_insertion_and_deletion_are_restored(ref):
    g, c2 = ref
    true = g[200:700]
    read = ins(true, 60)                           # insertion (L0 = 1)
    read = sub(read, 160)                          # substitution (L0 = 1)
    j = site(read, 360, 2)
    read = read[:j] + read[j + 2:]                 # two-base deletion (E of Emax = 2)
    j = site(read, 260, 1)
    read = read[:j] + read[j + 1:]                 # deletion (L0 = 0)
    got, stats = correct([read], c2)
    assert got == [true]
    assert stats == [4, 4, 4, 0, 0]


def test_two_close_errors_make_one_longer_run(ref):
    g, c2 = ref
    true = g[300:600]
    read = sub(sub(true, 100), 100 + K // 2)
    got, stats = correct([read], c2)
    assert got == [true] and stats == [1, 1, 1, 0, 0]


def test_an_n_in_p_is_replaced(ref):
    g, c2 = ref
    true = g[100:400]
    read = true[:150] + "N" + true[151:]
    got, stats = correct([read], c2)
    assert got == [true] and stats == [1, 1, 1, 0, 0]


def test_runs_touching_either_end_are_left(ref):
    g, c2 = ref
    true = g[500:800]
    read = sub(sub(true, 3), len(true) - 4)
    got, stats = correct([read], c2)
    assert got == [read] and stats == [2, 0, 0, 0, 0]


def test_a_run_shorter_than_k_minus_1_is_left(ref):
    g, c2 = ref
    true = g[500:800]
    low = {C.encode(sy(true[w:w + K])) for w in (120, 121, 122)}
    got, stats = correct([true], lambda x: 0 if x in low else c2(x))
    assert got == [true] and stats == [1, 0, 0, 0, 0]


def test_a_read_with_no_counted_window_is_left(ref):
    _, c2 = ref
    other = genome(300, 99)
    got, stats = correct([other, "N" * 40], c2)
    assert got == [other, "N" * 40] and stats == [0] * 5


def test_reads_shorter_than_k_plus_2_are_left(ref):
    g, c2 = ref
    short = sub(g[1000:1000 + K + 1], K // 2)
    got, stats = correct([short, "", "A"], c2)
    assert got == [short, "", "A"] and stats == [0] * 5


def test_a_solid_bubble_pins_the_tie_rules():
    """two alleles of one SNP, both solid: a read with the third base there has two bridges at distance 1 and the
    same length, and takes the lexicographically smaller; a read with an allele is left alone"""
    g = genome(600, 7)
    i = 300
    alleles = sorted({"A", "C", "G", "T"} - {g[i]})[:2]
    haps = [g[:i] + a + g[i + 1:] for a in alleles]
    c2 = C.window_count2([sy(t) for h in haps for t in tiles(h)], K)
    third = (set("ACGT") - set(alleles)).pop()
    read = g[100:500][:i - 100] + third + g[i + 1:500]
    got, stats = correct([read], c2)
    assert got == [haps[0][100:500]] and stats == [1, 1, 1, 0, 0]
    got, stats = correct([haps[1][100:500]], c2)
    assert got == [haps[1][100:500]] and stats == [0] * 5


def test_a_tandem_repeat_is_abandoned_over_a_budget_of_one():
    g = genome(400, 5)
    unit = "ACGTTGCAT"
    g2 = g[:200] + unit * 8 + g[200:]
    c2 = C.window_count2([sy(t) for t in tiles(g2)], K)
    true = g2[60:360]
    read = sub(true, 200 + 7 * len(unit) - 60)
    got, stats = correct([read], c2, branch_limit=1)
    assert got == [read] and stats[3] == 1 and stats[2] == 0
    got, stats = correct([read], c2, branch_limit=8)
    assert got == [true] and stats[3] == 0


@pytest.mark.parametrize("L0, removed", [(0, 2), (10, 15)])
def test_a_true_e_of_emax_is_found_and_one_longer_is_not(ref, L0, removed):
    """Emax = floor(13 L0 / 10) + 2: `removed` true bases replaced by L0 others are restored; one more are not"""
    g, c2 = ref
    assert removed == 13 * L0 // 10 + 2
    other = genome(L0 + 40, 3)[:L0]
    true = g[600:900]
    for extra, fixed in ((0, True), (1, False)):
        j = site(true, 150, removed + extra, other)
        read = true[:j] + other + true[j + removed + extra:]
        got, stats = correct([read], c2)
        assert (got == [true]) == fixed
        assert stats == ([1, 1, 1, 0, 0] if fixed else [1, 1, 0, 0, 1])


def test_threshold_is_the_upper_median_in_integers():
    assert C.threshold([0, 5, 3, 0, 9, 7], 1, 1000) == 7
    assert C.threshold([0, 5, 3, 0, 9], 1, 500) == 2
    assert C.threshold([0, 5, 3, 0, 9], 4, 100) == 4
    assert C.threshold([0, 0], 1, 100) is None


def test_levenshtein_treats_n_as_a_mismatch():
    assert C.levenshtein(sy("ACGT"), sy("ACGT")) == 0
    assert C.levenshtein(sy("ACGT"), sy("ANGT")) == 1
    assert C.levenshtein(sy(""), sy("NN")) == 2
    assert C.levenshtein(sy("ACGTA"), sy("CGT")) == 2


def _tool(name):
    p = shutil.which(name) or f"/usr/local/cuda/bin/{name}"
    if not os.path.exists(p):
        pytest.skip(f"{name} not available")
    return p


NKERNELS = 14
KERNEL = re.compile(r"\dcorrect_[a-z0-9_]+_kernel")  # a mangled correct_*_kernel (CUB's kernels carry the file's name)


def test_correct_kernels_use_no_warp_collectives():
    """the correction kernels exchange nothing between lanes: no shuffle, vote, match or reduction (their per-CTA
    counts go through shared memory).  A collective added to one must come with warp_sync_guard and a WARPSYNC pinned
    here."""
    cuobjdump = _tool("cuobjdump")
    if not os.path.exists(LIB):
        pytest.skip("library not built (python rust-msbwt_b200/build.py)")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if KERNEL.search(m.group(1)) else None
            if cur:
                counts[cur] = {op: 0 for op in ("VOTE", "REDUX", "MATCH", "SHFL")}
            continue
        if cur:
            for op in counts[cur]:
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    assert len(counts) == NKERNELS, list(counts)
    for name, c in counts.items():
        assert not any(c.values()), (name, c)


def test_correct_kernels_do_not_spill(tmp_path):
    nvcc = _tool("nvcc")
    src = os.path.join(ROOT, "rust-msbwt_b200", "csrc", "correct.cu")
    res = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                          "-c", src, "-o", str(tmp_path / "correct.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = res.stderr.splitlines()
    at = [i for i, ln in enumerate(lines) if "Function properties for" in ln and KERNEL.search(ln)]
    assert len(at) == NKERNELS
    for i in at:
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", lines[i + 1]), lines[i:i + 2]
