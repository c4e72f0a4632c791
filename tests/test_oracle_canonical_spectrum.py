"""oracle/canonical_spectrum.py -- the two CPU restatements of msbwt_kmer_spectrum_canonical -- against each other,
against brute force and against the properties the definition promises (strand invariance, the sum of windows, an
index that holds both strands), and the shipped SASS of the resolve kernel (no GPU needed)."""
import itertools
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import canonical_spectrum as CS
from oracle import naive
from oracle import oracle as O
from oracle import spectrum as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")
KS = (1, 2, 4, 5, 12, 21, 31, 32)
MIN_COUNTS = (1, 2, 3, 5)
NBINS = 9
_RC = str.maketrans("ACGTN", "TGCAN")


def _syms(s):
    return np.array(["$ACGNT".index(c) for c in s], np.uint8)


def _rc(s):
    return s.translate(_RC)[::-1]


def _same(a, b):
    for x, y in zip(a, b):
        assert x.dtype == y.dtype == np.uint64 and x.shape == y.shape and (x == y).all(), (x, y)


def _two_strand_reads(rng, n_sets):
    """seeded read sets from both strands of a random genome, with errors, N, duplicate and empty reads"""
    for t in range(n_sets):
        genome = "".join(rng.choice("ACGT") for _ in range(rng.randint(20, 200)))
        reads = []
        for _ in range(rng.randint(1, 40)):
            a = rng.randint(0, len(genome) - 1)
            r = list(genome[a:a + rng.randint(0, 40)])
            for i in range(len(r)):
                x = rng.random()
                if x < 0.03:
                    r[i] = rng.choice("ACGT")
                elif x < 0.05 and t % 2:
                    r[i] = "N"
            r = "".join(r)
            reads.append(_rc(r) if rng.random() < 0.5 else r)
        reads += reads[: rng.randint(0, 3)]  # duplicate reads
        yield reads


def test_revcomp():
    assert CS.revcomp_u64([0b00011011], 4).tolist() == [0b00011011]  # ACGT is its own reverse complement
    assert CS.revcomp_u64([0b0001], 2).tolist() == [0b1011]          # AC -> GT
    v = np.random.default_rng(1).integers(0, 1 << 62, 1000, dtype=np.uint64)
    for k in (1, 7, 31, 32):
        x = v & np.uint64((1 << (2 * k)) - 1)
        assert (CS.revcomp_u64(CS.revcomp_u64(x, k), k) == x).all()


def test_reference_two_string(two_string_npy):
    # ["ACGT", "TGCA"]: AC/GT, CG/CG (a palindrome), TG/CA and GC/GC pair up
    o = O.RleBWT()
    o.load_numpy_file(two_string_npy)
    rle = o.rle_bytes()
    reads = [_syms("ACGT"), _syms("TGCA")]
    hist, kmers, counts = CS.canonical_from_rle(rle, 2, 1, 4)
    _same((hist, kmers, counts), CS.canonical_from_reads(reads, 2, 1, 4))
    # AC (count 1 + GT 1), CA (1 + TG 1), CG (palindrome, 1), GC (palindrome, 1)
    assert kmers.tolist() == [0b0001, 0b0100, 0b0110, 0b1001] and counts.tolist() == [2, 2, 1, 1]
    assert hist.tolist() == [0, 2, 2, 0]
    for k in KS:
        for t in MIN_COUNTS:
            _same(CS.canonical_from_rle(rle, k, t, 3), CS.canonical_from_reads(reads, k, t, 3))


def test_two_strand_read_sets_with_errors_n_duplicates_and_empty_reads():
    rng = random.Random(23)
    for reads in _two_strand_reads(rng, 16):
        reads.append("")
        rle = O.convert_to_vec(naive.naive_bwt(reads))
        arrs = [_syms(r) for r in reads]
        walk = S.walk_rle(rle, 32, 1)
        for k in KS:
            for t in MIN_COUNTS:
                want = CS.canonical_from_reads(arrs, k, t, NBINS)
                _same(CS.canonical_from_walk(*walk[k - 1], k, t, NBINS), want)
                assert want[0][:t].sum() == 0


def test_golden_index():
    """the golden index's reads, regenerated as tests/golden/make_golden.py made them"""
    from harness import synth
    z = np.load(os.path.join(ROOT, "tests", "golden", "reads30x_k31.npz"))
    reads = synth.np_make_reads(3000, 100, 30.0, 0.01, seed=20261018)
    reads[11, 50:52] = 4
    walk = S.walk_rle(z["rle"], 32, 1)
    for k in KS:
        for t in MIN_COUNTS:
            _same(CS.canonical_from_walk(*walk[k - 1], k, t, 50), CS.canonical_from_reads(list(reads), k, t, 50))


def _brute(o, k):
    """(k-mers, canonical counts) of all 4^k k-mers, each pair once, from count_kmer alone"""
    allk = np.array(list(itertools.product((1, 2, 3, 5), repeat=k)), np.uint8)
    counts = o.count_kmers_fixed(allk, k)
    code = np.array([0, 0, 1, 2, 0, 3], np.uint64)
    vals = np.zeros(allk.shape[0], np.uint64)
    for j in range(k):
        vals = (vals << np.uint64(2)) | code[allk[:, j]]
    by_val = dict(zip(vals.tolist(), counts.tolist()))
    rc = CS.revcomp_u64(vals, k)
    canon = vals <= rc
    c = np.array([by_val[v] + (by_val[r] if v != r else 0) for v, r in zip(vals.tolist(), rc.tolist())], np.uint64)
    return vals[canon], c[canon]


def test_tiny_indexes_against_every_kmer():
    """BWTs from reads and BWTs that do not come from reads, k up to 6 (even k: palindromes)"""
    rng = np.random.default_rng(8)
    rles = [O.convert_to_vec(naive.naive_bwt(r)) for r in _two_strand_reads(random.Random(9), 4)]
    for _ in range(8):
        n_runs = int(rng.integers(1, 60))
        syms = np.repeat(rng.integers(0, 6, n_runs).astype(np.uint8), rng.integers(1, 9, n_runs))
        rles.append(O.convert_to_vec(O.convert_itos(syms)))
    for rle in rles:
        o = O.RleBWT()
        o.load_vector(rle)
        walk = S.walk_rle(rle, 6, 1)
        for k in range(1, 7):
            vals, c = _brute(o, k)
            for t in MIN_COUNTS:
                keep = c >= t
                _same(CS.canonical_from_walk(*walk[k - 1], k, t, 6), (S.histogram(c[keep], 6), vals[keep], c[keep]))


def test_strand_invariance_and_sum_of_windows():
    rng = random.Random(31)
    for reads in _two_strand_reads(rng, 10):
        flipped = [_rc(r) if rng.random() < 0.5 else r for r in reads]
        a = O.convert_to_vec(naive.naive_bwt(reads))
        b = O.convert_to_vec(naive.naive_bwt(flipped))
        wa, wb = S.walk_rle(a, 32, 1), S.walk_rle(b, 32, 1)
        for k in KS:
            windows = S.pack_windows([_syms(r) for r in reads], k).size
            for t in MIN_COUNTS:
                ra = CS.canonical_from_walk(*wa[k - 1], k, t, 200)
                _same(ra, CS.canonical_from_walk(*wb[k - 1], k, t, 200))
            nbins = sum(map(len, reads)) + 2  # above the largest count
            hist = CS.canonical_from_walk(*wa[k - 1], k, 1, nbins)[0]
            assert hist[-1] == 0 and int((np.arange(nbins, dtype=np.uint64) * hist).sum()) == windows


def test_index_of_both_strands():
    """the plain min_count 1 list of an index of the reads and their reverse complements, reduced to canonical members
    (palindromes' counts halved), is the canonical list of the reads alone"""
    for reads in _two_strand_reads(random.Random(37), 10):
        both = O.convert_to_vec(naive.naive_bwt(reads + [_rc(r) for r in reads]))
        alone = O.convert_to_vec(naive.naive_bwt(reads))
        wb, wa = S.walk_rle(both, 32, 1), S.walk_rle(alone, 32, 1)
        for k in KS:
            km, cn = wb[k - 1]
            rc = CS.revcomp_u64(km, k)
            keep = km <= rc
            km, cn = km[keep], np.where(km[keep] == rc[keep], cn[keep] // np.uint64(2), cn[keep])
            order = np.argsort(km)
            _same((km[order], cn[order]), CS.canonical_from_walk(*wa[k - 1], k, 1)[1:])


def _tool(name):
    p = shutil.which(name) or f"/usr/local/cuda/bin/{name}"
    if not os.path.exists(p):
        pytest.skip(f"{name} not available")
    return p


def test_resolve_kernel_sass():
    """canonical_resolve_kernel exchanges nothing between lanes: no shuffle, match or reduction, and at most the one
    vote ptxas emits itself to elect the lane of the per-CTA atomic (as in spectrum_emit_kernel,
    tests/test_oracle_spectrum.py).  A collective added to it must come with warp_sync_guard and a WARPSYNC pinned here."""
    cuobjdump = _tool("cuobjdump")
    if not os.path.exists(LIB):
        pytest.skip("library not built (python rust-msbwt_b200/build.py)")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if "canonical_" in m.group(1) else None
            if cur:
                counts[cur] = {op: 0 for op in ("WARPSYNC", "VOTE", "REDUX", "MATCH", "SHFL")}
            continue
        if cur:
            for op in counts[cur]:
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    assert sum("canonical_resolve_kernel" in n for n in counts) == 1, list(counts)
    for name, c in counts.items():
        assert c["SHFL"] == c["MATCH"] == c["REDUX"] == 0, (name, c)
        assert c["VOTE"] <= (1 if "resolve" in name else 0), (name, c)


def test_resolve_kernel_does_not_spill(tmp_path):
    nvcc = _tool("nvcc")
    src = os.path.join(ROOT, "rust-msbwt_b200", "csrc", "spectrum.cu")
    res = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                          "-c", src, "-o", str(tmp_path / "spectrum.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = res.stderr.splitlines()
    at = [i for i, ln in enumerate(lines) if "Function properties for" in ln and "canonical_resolve_kernel" in ln]
    assert len(at) == 1
    assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", lines[at[0] + 1]), lines[at[0] + 1]
