"""oracle/unitigs.py -- the CPU restatement of msbwt_unitigs -- on hand-made graphs, against its independent property
checker on random k-mer sets and on an error-free tiling of a genome, and the shipped SASS of the unitig kernels (no
GPU needed)."""
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import spectrum as S
from oracle import unitigs as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")
_RC = str.maketrans("ACGT", "TGCA")


def enc(s):
    v = 0
    for c in s:
        v = (v << 2) | "ACGT".index(c)
    return v


def text(syms):
    return "".join("$ACGNT"[s] for s in syms)


def kmer_set(seqs, k, circular=False):
    """(kmers, counts) of every k-window of the strings (wrapping around with `circular`)"""
    c = {}
    for s in seqs:
        t = s + s[:k - 1] if circular else s
        for i in range(len(t) - k + 1):
            c[enc(t[i:i + k])] = c.get(enc(t[i:i + k]), 0) + 1
    km = np.array(sorted(c), np.uint64)
    return km, np.array([c[int(x)] for x in km], np.uint64)


def canonical_set(seqs, k):
    """the canonical list of the strings: min(X, rc X) with count(X) + count(rc X) (palindromes once)"""
    km, cn = kmer_set(seqs, k)
    by = dict(zip(km.tolist(), cn.tolist()))
    out = {}
    for x, c in by.items():
        r = U.revcomp(x, k)
        out[min(x, r)] = c + (by.get(r, 0) if r != x else 0)
    keys = np.array(sorted(out), np.uint64)
    return keys, np.array([out[int(x)] for x in keys], np.uint64)


def run(km, cn, k, canonical=False):
    res = U.unitigs(km, cn, k, canonical)
    U.check_unitigs(*res, km, cn, k, canonical)
    syms, offs, sums = res
    return [text(syms[offs[i]:offs[i + 1]]) for i in range(offs.size - 1)], sums.tolist()


def test_revcomp():
    assert U.revcomp(enc("ACGT"), 4) == enc("ACGT") and U.revcomp(enc("AAC"), 3) == enc("GTT")


def test_path():
    assert run(*kmer_set(["ACGTT"], 3), 3) == (["ACGTT"], [3])


def test_fork_and_join():
    # ACG -> CGA and ACG -> CGT: a fork; ACG -> CGA and TCG -> CGA: a join
    assert run(*kmer_set(["ACGA", "ACGT"], 3), 3)[0] == ["ACG", "CGA", "CGT"]
    assert run(*kmer_set(["ACGA", "TCGA"], 3), 3)[0] == ["ACG", "CGA", "TCG"]


def test_bubble():
    got, sums = run(*kmer_set(["GAACTGC", "GAAGTGC"], 3), 3)
    assert got == ["AACTG", "AAGTG", "GAA", "TGC"] and sums == [3, 3, 2, 2]


def test_tip():
    assert run(*kmer_set(["ACGTTG", "CGTA"], 3), 3)[0] == ["ACGT", "GTA", "GTTG"]


def test_self_loop():
    assert run(*kmer_set(["AAAA"], 4), 4) == (["AAAA"], [1])
    assert run(*kmer_set(["AAAAAA"], 4), 4) == (["AAAA"], [3])  # the loop counts toward the degrees
    assert run(*kmer_set(["AAAAC"], 4), 4)[0] == ["AAAA", "AAAC"]
    assert run(*kmer_set(["AAAA"], 4), 4, canonical=True)[0] == ["AAAA"]  # TTTT is its reverse complement


def test_two_cycle():
    assert run(*kmer_set(["ACAC"], 3), 3) == (["ACAC"], [2])  # ACA -> CAC -> ACA: cut before ACA
    assert run(*kmer_set(["ACA"], 2), 2)[0] == ["ACA"]


def test_circular_genome_is_one_unitig_cut_at_its_minimum():
    rng = random.Random(3)
    for k in (7, 9, 11):
        while True:  # no (k-1)-mer twice on the circle and its reverse complement: two cycles, no branch
            g = "".join(rng.choice("ACGT") for _ in range(60))
            both = [c + c[:k - 2] for c in (g, g.translate(_RC)[::-1])]
            if len({c[i:i + k - 1] for c in both for i in range(len(g))}) == 2 * len(g):
                break
        got, sums = run(*kmer_set([g], k, circular=True), k)
        windows = [(g + g)[i:i + k] for i in range(len(g))]
        start = min(range(len(g)), key=lambda i: enc(windows[i]))
        assert got == [(g + g)[start:start + len(g) + k - 1]] and sums == [len(g)]
        # canonical mode: the cycle whose minimum is the smaller of the two
        rc = g.translate(_RC)[::-1]
        cgot, csums = run(*canonical_set([g + g[:k - 1]], k), k, canonical=True)
        rwin = [(rc + rc)[i:i + k] for i in range(len(g))]
        assert len(cgot) == 1 and csums == [len(g)]
        if enc(min(windows, key=enc)) < enc(min(rwin, key=enc)):
            assert cgot == got
        else:
            r0 = min(range(len(g)), key=lambda i: enc(rwin[i]))
            assert cgot == [(rc + rc)[r0:r0 + len(g) + k - 1]]


def test_palindromes_and_a_hairpin_at_even_k():
    assert run(*canonical_set(["ACGT"], 4), 4, canonical=True) == (["ACGT"], [1])
    assert run(*kmer_set(["ACGT"], 4), 4) == (["ACGT"], [1])
    # AAACGTTT is its own reverse complement: one unitig through the palindrome ACGT, kept once
    got, sums = run(*canonical_set(["AAACGTTT"], 4), 4, canonical=True)
    assert got == ["AAACGTTT"] and sums == [2 + 2 + 1 + 2 + 2]
    # plain mode of the same reads on both strands: the same single unitig (it is its own reverse complement)
    assert run(*kmer_set(["AAACGTTT", "AAACGTTT"], 4), 4)[0] == ["AAACGTTT"]


def test_k1_and_k2():
    assert run(*kmer_set(["A"], 1), 1) == (["A"], [1])  # a self-loop
    assert run(*kmer_set(["AC"], 1), 1)[0] == ["A", "C"]  # every node links to every node
    assert run(*kmer_set(["ACG"], 2), 2)[0] == ["ACG"]
    assert run(*canonical_set(["A"], 1), 1, canonical=True)[0] == ["A"]  # A and T: degrees 2 each
    assert run(*canonical_set(["AC"], 2), 2, canonical=True)[0] == ["AC"]  # AC / GT: no edge, GT dropped


def test_random_kmer_sets_pass_the_checker():
    rng = np.random.default_rng(11)
    for k in (1, 2, 3, 4, 5, 6, 7, 9, 12):
        for density in (0.05, 0.3, 0.8):
            universe = min(4 ** k, 4000)
            n = max(1, int(universe * density))
            km = np.unique(rng.integers(0, 4 ** k, n, dtype=np.uint64))
            cn = rng.integers(1, 9, km.size).astype(np.uint64)
            for canonical in (False, True):
                if canonical:
                    r = np.array([U.revcomp(int(x), k) for x in km], np.uint64)
                    km_c, first = np.unique(np.minimum(km, r), return_index=True)
                    res = U.unitigs(km_c, cn[first], k, True)
                    U.check_unitigs(*res, km_c, cn[first], k, True)
                else:
                    res = U.unitigs(km, cn, k)
                    U.check_unitigs(*res, km, cn, k)


def test_checker_rejects_broken_results():
    km, cn = kmer_set(["GAACTGC", "GAAGTGC"], 3)
    syms, offs, sums = U.unitigs(km, cn, 3)
    bad = [(syms, offs, sums + np.uint64(1)),                       # a count sum
           (syms, offs[[0, 2, 3, 4]], sums[[0, 2, 3]]),             # a unitig missing
           (np.concatenate([syms[5:], syms[:5]]), offs - offs + np.array([0, 5, 10, 12, 15], np.uint64), sums)]
    for b in bad:
        with pytest.raises(AssertionError):
            U.check_unitigs(*b, km, cn, 3)


def test_error_free_tiling_of_a_repeat_free_genome_gives_the_genome():
    rng = random.Random(5)
    k = 21
    g = "".join(rng.choice("ACGT") for _ in range(3000))
    assert len({g[i:i + k - 1] for i in range(len(g) - k + 2)}) == len(g) - k + 2
    reads = [g[a:a + 100] for a in range(0, len(g) - 100 + 1, 37)] + [g[-100:]]
    arrs = [np.array(["$ACGNT".index(c) for c in r], np.uint8) for r in reads]
    _, km, cn = S.from_reads(arrs, k, 1)
    order = np.argsort(km)
    got, sums = run(km[order], cn[order], k)
    assert got == [g] and sums[0] == int(cn.sum())
    # canonical: the genome or its reverse complement, whichever the keep rule picks
    rc = g.translate(_RC)[::-1]
    cgot, _ = run(*canonical_set(reads, k), k, canonical=True)
    assert cgot == [g if enc(g[:k]) <= enc(rc[:k]) else rc]


def _tool(name):
    p = shutil.which(name) or f"/usr/local/cuda/bin/{name}"
    if not os.path.exists(p):
        pytest.skip(f"{name} not available")
    return p


def test_unitig_kernels_use_no_warp_collectives():
    """the unitig kernels exchange nothing between lanes: no shuffle, vote, match or reduction (their per-CTA counts
    go through shared memory).  A collective added to one must come with warp_sync_guard and a WARPSYNC pinned here."""
    cuobjdump = _tool("cuobjdump")
    if not os.path.exists(LIB):
        pytest.skip("library not built (python rust-msbwt_b200/build.py)")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if "unitig_" in m.group(1) else None
            if cur:
                counts[cur] = {op: 0 for op in ("VOTE", "REDUX", "MATCH", "SHFL")}
            continue
        if cur:
            for op in counts[cur]:
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    assert len(counts) == 11, list(counts)
    for name, c in counts.items():
        assert not any(c.values()), (name, c)


def test_unitig_kernels_do_not_spill(tmp_path):
    nvcc = _tool("nvcc")
    src = os.path.join(ROOT, "rust-msbwt_b200", "csrc", "unitigs.cu")
    res = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                          "-c", src, "-o", str(tmp_path / "unitigs.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = res.stderr.splitlines()
    at = [i for i, ln in enumerate(lines) if "Function properties for" in ln and "unitig_" in ln]
    assert len(at) == 11
    for i in at:
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", lines[i + 1]), lines[i:i + 2]
