"""oracle/merge.py -- the numpy restatement of the Holt-McMillan merge (src/bwt_util.rs:108-141) -- against the
definition it must meet on BWTs built from reads: merging the BWTs of two read sets gives naive_bwt of their union
(src/bwt_util.rs:154-171).  Also the shipped SASS of the device merge's warp-cooperative pass (no GPU needed)."""
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import merge as OM
from oracle import naive
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rust-msbwt_b200", "libmsbwt_b200.so")


def _rle(strings):
    return O.convert_to_vec(naive.naive_bwt(list(strings)))


def _check_pair(a, b):
    got, total, iterations = OM.merge_rle(_rle(a), _rle(b))
    assert total == sum(len(s) + 1 for s in a + b)
    assert (got == _rle(a + b)).all(), (a, b)
    longest = max([len(s) for s in a + b], default=0)
    assert iterations <= 2 * longest + 2, (a, b, iterations)
    back, _, _ = OM.merge_rle(_rle(b), _rle(a))
    assert (back == got).all(), (a, b)
    return iterations


def test_rle_codec_round_trip_matches_the_reference_encoder():
    rng = np.random.default_rng(3)
    syms = np.repeat(rng.integers(0, 6, 400).astype(np.uint8), rng.integers(1, 40_000, 400))
    rle = OM.symbols_to_rle(syms)
    assert (rle == O.convert_to_vec(O.convert_itos(syms))).all()
    assert (OM.rle_to_symbols(rle) == syms).all()
    # digits are little-endian base 32, a zero digit included: 1 + 0 * 32 + 1 * 1024
    assert (OM.rle_to_symbols(np.array([1 | 3 << 3, 2 | 1 << 3, 2 | 0 << 3, 2 | 1 << 3], np.uint8)) ==
            np.array([1, 1, 1] + [2] * 1025, np.uint8)).all()
    with pytest.raises(ValueError):
        OM.rle_to_symbols(np.array([6], np.uint8))


def test_reference_sets():
    # test_data/two_string.npy holds the BWT of ["ACGT", "TGCA"] (src/rle_bwt.rs:76-79)
    got, total, _ = OM.merge_rle(_rle(["ACGT"]), _rle(["TGCA"]))
    o = O.RleBWT()
    o.load_numpy_file(os.path.join(ROOT, "tests", "golden", "two_string.npy"))
    assert total == 10 and (got == o.rle_bytes()).all()
    # the bwt_util.rs doc-test set, split across the two inputs
    got, total, _ = OM.merge_rle(_rle(["CCGT", "N"]), _rle(["ACG"]))
    assert O.convert_itos(OM.rle_to_symbols(got)) == "GTN$$ACCC$G"
    _check_pair(["CCGT", "N"], ["ACG"])


def test_random_ragged_sets_with_empty_reads_n_and_duplicates():
    rng = random.Random(108)
    for _ in range(250):
        def reads():
            alphabet = "ACGNT" if rng.random() < 0.3 else "ACGT"
            return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, 14))) for _ in range(rng.randint(0, 9))]
        a, b = reads(), reads()
        if a and rng.random() < 0.4:
            b.append(rng.choice(a))           # a duplicate across the two sets
        if a and rng.random() < 0.3:
            a.append(a[0])                    # and within one
        if rng.random() < 0.2:
            b.append("")
        _check_pair(a, b)


def test_reads_that_are_prefixes_or_suffixes_of_reads_in_the_other_set():
    rng = random.Random(141)
    for _ in range(120):
        a = ["".join(rng.choice("ACGT") for _ in range(rng.randint(1, 16))) for _ in range(rng.randint(1, 5))]
        b = []
        for s in a:
            cut = rng.randint(0, len(s))
            b += [s[:cut], s[cut:]]
        b.append(a[0] * 2)
        _check_pair(a, b)


def test_empty_inputs_and_self_merge():
    one = ["ACCA", "GT", "ACCA"]
    got, total, iterations = OM.merge_rle(_rle(one), np.zeros(0, np.uint8))
    assert (got == _rle(one)).all() and total == 13 and iterations == 1
    got, total, iterations = OM.merge_rle(np.zeros(0, np.uint8), np.zeros(0, np.uint8))
    assert got.size == 0 and total == 0 and iterations == 0
    _check_pair(one, one)


def test_arbitrary_streams_reach_a_fixed_point():
    """Any RLE stream is a legal index; the iteration must still end (within N_A + N_B passes) and the output is a
    permutation of the two inputs' symbols."""
    rng = np.random.default_rng(9)
    for _ in range(60):
        a = rng.integers(0, 6, int(rng.integers(0, 60))).astype(np.uint8)
        b = rng.integers(0, 6, int(rng.integers(0, 60))).astype(np.uint8)
        syms, iterations = OM.merge_symbols(a, b)
        assert iterations <= max(a.size + b.size, 1)
        assert (np.bincount(syms, minlength=6) == np.bincount(a, minlength=6) + np.bincount(b, minlength=6)).all()


@pytest.fixture(scope="module")
def merge_kernel_sass():
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
            cur = m.group(1) if "merge_pass_kernel" in m.group(1) else None
            if cur:
                counts[cur] = {op: 0 for op in ("WARPSYNC", "VOTE", "REDUX", "MATCH")}
            continue
        if cur:
            for op in counts[cur]:
                if re.search(r"\b" + op, line):
                    counts[cur][op] += 1
    return counts


def test_merge_pass_keeps_its_warp_syncs(merge_kernel_sass):
    """The interleave pass ballots the rows' symbol bit-planes and gathers every symbol's bits (six reductions) after
    a divergent symbol fetch: warp_sync_guard must leave a WARPSYNC before each of those collectives."""
    interleave = {k: v for k, v in merge_kernel_sass.items() if "ILb0E" in k}
    assert len(interleave) == 1, list(merge_kernel_sass)
    (c,) = interleave.values()
    assert c["REDUX"] >= 6 and c["VOTE"] >= 3, c
    assert c["WARPSYNC"] >= 9, c  # one before each of the three ballots and the six reductions
