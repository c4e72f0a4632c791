"""oracle/spectrum.py -- the two CPU restatements of msbwt_kmer_spectrum -- against each other and against brute force,
and the shipped SASS of the device kernels (no GPU needed)."""
import itertools
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import naive
from oracle import oracle as O
from oracle import spectrum as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")


def _syms(s):
    return np.array(["$ACGNT".index(c) for c in s], np.uint8)


def _same(a, b):
    for x, y in zip(a, b):
        assert x.dtype == y.dtype == np.uint64 and x.shape == y.shape and (x == y).all(), (x, y)


def test_reference_two_string(two_string_npy):
    # test_data/two_string.npy holds the BWT of ["ACGT", "TGCA"]: six distinct 2-mers, each once
    o = O.RleBWT()
    o.load_numpy_file(two_string_npy)
    rle = o.rle_bytes()
    reads = [_syms("ACGT"), _syms("TGCA")]
    hist, kmers, counts = S.from_rle(rle, 2, 1, 4)
    _same((hist, kmers, counts), S.from_reads(reads, 2, 1, 4))
    assert hist.tolist() == [0, 6, 0, 0] and counts.tolist() == [1] * 6
    # co-lexicographic: CA (last symbol A) first, then AC, GC, CG, TG, GT
    assert kmers.tolist() == [0b0100, 0b0001, 0b1001, 0b0110, 0b1110, 0b1011]
    for k in (1, 3, 4, 5):
        _same(S.from_rle(rle, k, 1, 3), S.from_reads(reads, k, 1, 3))
    assert S.from_rle(rle, 5)[1].size == 0


def test_read_sets_with_errors_n_and_duplicates():
    rng = random.Random(21)
    for t in range(25):
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
            reads.append("".join(r))
        reads += reads[: rng.randint(0, 3)]  # duplicate reads
        rle = O.convert_to_vec(naive.naive_bwt(reads))
        arrs = [_syms(r) for r in reads]
        walks = {t_: S.walk_rle(rle, 12, t_) for t_ in (1, 2, 3)}
        for k in range(1, 13):
            for min_count in (1, 2, 3):
                want = S.from_reads(arrs, k, min_count, 7)
                km, cn = walks[min_count][k - 1]
                _same((S.histogram(cn, 7), km, cn), want)
                assert want[0][:min_count].sum() == 0


def test_random_rle_streams_against_every_kmer():
    """BWTs that do not come from reads: the walk lists exactly the k-mers whose count_kmer is >= min_count"""
    rng = np.random.default_rng(6)
    for _ in range(12):
        n_runs = int(rng.integers(1, 60))
        syms = np.repeat(rng.integers(0, 6, n_runs).astype(np.uint8), rng.integers(1, 9, n_runs))
        rle = O.convert_to_vec(O.convert_itos(syms))
        o = O.RleBWT()
        o.load_vector(rle)
        for k in range(1, 7):
            allk = np.array(list(itertools.product((1, 2, 3, 5), repeat=k)), np.uint8)
            counts = o.count_kmers_fixed(allk, k)
            code = np.array([0, 0, 1, 2, 0, 3], np.uint64)
            vals = np.zeros(allk.shape[0], np.uint64)
            for j in range(k):
                vals = (vals << np.uint64(2)) | code[allk[:, j]]
            for min_count in (1, 2, 5):
                keep = counts >= min_count
                order = np.argsort(S.colex_key(vals[keep], k), kind="stable")
                hist, km, cn = S.from_rle(rle, k, min_count, 6)
                _same((km, cn), (vals[keep][order], counts[keep][order]))
                assert (hist == S.histogram(counts[keep], 6)).all()


@pytest.fixture(scope="module")
def spectrum_kernel_sass():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(LIB):
        pytest.skip("library not built (python rust-msbwt_b200/build.py)")
    out = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            cur = name if re.search(r"spectrum_(expand|emit)_kernel", name) and "cub" not in name else None
            if cur:
                counts[cur] = {op: 0 for op in ("WARPSYNC", "VOTE", "REDUX", "MATCH", "SHFL")}
            continue
        if cur:
            for op in counts[cur]:
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    return counts


def test_spectrum_kernels_use_no_warp_collectives(spectrum_kernel_sass):
    """The expand and emit kernels exchange nothing between lanes, so the convergence guard (warp_sync_guard,
    DESIGN.md section 4a) has nothing to protect: no shuffle, match or reduction, and at most the one vote ptxas emits
    itself to elect the lane of a per-CTA atomic (computed over the lanes actually active).  A collective added to
    these kernels must come with the guard and a WARPSYNC pinned here."""
    assert len(spectrum_kernel_sass) == 8, list(spectrum_kernel_sass)  # expand / emit x WIDE x LIST
    for name, c in spectrum_kernel_sass.items():
        assert c["SHFL"] == c["MATCH"] == c["REDUX"] == 0, (name, c)
        assert c["VOTE"] <= (1 if "emit" in name else 0), (name, c)
