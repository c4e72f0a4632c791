"""Read correction on the device (correct.cu, `msbwt_correct_reads`): byte for byte against oracle/correct.py, stats
included, across k, the parameters and the index layouts; isolated errors in long reads corrected to the truth; the
result independent of chunking and of the number of devices; empty input, bad arguments and concurrent queries."""
import ctypes as C
import threading

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import correct as OC

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KS = (5, 12, 21, 31, 32)
# (min_count, frac_permille, branch_limit): every value of each parameter appears
PARAMS = ((1, 0, 4), (2, 100, 1), (5, 500, 4), (2, 100, 4), (1, 500, 1), (5, 0, 1))
LAYOUTS = {
    "default": dict(),
    "one_request": dict(oct_index=1, final_index=1, suffix_table_s=12),  # 31/32-mers on the one-request kernel
    "no_oct_no_final": dict(final_index=0, oct_index=0),
    "superblocks": dict(superblock_shift=3),  # 64-bit position kernels (WIDE)
}
EINVAL = 1  # MSBWT_EINVAL, include/msbwt_gpu.h
LUT = np.array([1, 2, 3, 5], np.uint8)
RC_SYM = np.array([0, 5, 3, 2, 4, 1], np.uint8)


def _index(reads, **layout):
    g = M.RleBWT(**layout)
    g.load_vector(M.build_rle_bwt_ragged(reads)[0])
    return g


def _mutate(rng, r, rate, n_rate=0.0):
    """substitutions, single-base insertions and deletions at `rate` each, and N at n_rate"""
    kind = np.digitize(rng.random(r.size), [rate, 2 * rate, 3 * rate])  # 0 sub, 1 ins, 2 del, 3 keep
    r = r.copy()
    r[kind == 0] = LUT[rng.integers(0, 4, int((kind == 0).sum()))]
    rep = np.where(kind == 1, 2, np.where(kind == 2, 0, 1))
    out = np.repeat(r, rep)
    out[np.cumsum(rep)[kind == 1] - 1] = LUT[rng.integers(0, 4, int((kind == 1).sum()))]
    out[rng.random(out.size) < n_rate] = 4
    return out


def _sample(rng, g, lengths, rate=0.0, n_rate=0.0):
    reads = []
    for ln in lengths:
        a = int(rng.integers(0, g.size - ln + 1))
        r = LUT[g[a:a + ln]]
        if rng.random() < 0.5:
            r = RC_SYM[r[::-1]]
        reads.append(_mutate(rng, r, rate, n_rate) if rate or n_rate else r.copy())
    return reads


@pytest.fixture(scope="module")
def read_sets():
    """an index of 25x reads with 0.3 % errors of a 3 kbp genome, and reads to correct with 1 % of each error kind"""
    rng = np.random.default_rng(7)
    g = rng.integers(0, 4, 3000)
    index_reads = _sample(rng, g, [100] * 750, rate=0.001)
    queries = _sample(rng, g, rng.integers(20, 400, 40), rate=0.01, n_rate=0.003)
    queries += [np.zeros(0, np.uint8), LUT[g[:3]].copy()]
    return index_reads, queries


_COUNT2 = {}


def _oracle(index_reads, queries, k, params):
    if (id(index_reads), k) not in _COUNT2:
        _COUNT2[id(index_reads), k] = OC.window_count2([r.tolist() for r in index_reads], k)
    return OC.correct_reads([q.tolist() for q in queries], k, *params, _COUNT2[id(index_reads), k])


def _same(got, want):
    (gr, gs), (wr, ws) = got, want
    assert gs.tolist() == ws
    assert len(gr) == len(wr)
    for i, (a, b) in enumerate(zip(gr, wr)):
        assert a.dtype == np.uint8 and a.tolist() == b, i


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("k", KS)
def test_device_equals_the_oracle(read_sets, layout, k):
    index_reads, queries = read_sets
    g = _index(index_reads, **LAYOUTS[layout])
    bridged = 0
    for params in PARAMS:
        want = _oracle(index_reads, queries, k, params)
        _same(g.correct_reads(queries, k, *params), want)
        bridged += want[1][2]
    assert bridged > 0 or k == 5  # every 5-mer of the 3 kbp genome is solid: no weak runs at k = 5


def test_device_equals_the_oracle_with_the_general_kernels(read_sets, monkeypatch):
    """MSBWT_FINAL_FAST=0: 31-mers take the general query kernels on an index with final-step lines"""
    index_reads, queries = read_sets
    g = _index(index_reads, **LAYOUTS["one_request"])
    monkeypatch.setenv("MSBWT_FINAL_FAST", "0")
    _same(g.correct_reads(queries, 31, 2, 100, 4), _oracle(index_reads, queries, 31, (2, 100, 4)))


def _clean_genome(rng, n, k):
    """a random genome whose k-mers occur once on both strands together"""
    while True:
        g = rng.integers(0, 4, n)
        w = np.lib.stride_tricks.sliding_window_view(g, k) @ (4 ** np.arange(k - 1, -1, -1))
        r = np.lib.stride_tricks.sliding_window_view(3 - g[::-1], k) @ (4 ** np.arange(k - 1, -1, -1))
        if np.unique(np.concatenate([w, r])).size == 2 * w.size:
            return g


def test_isolated_errors_in_long_reads_are_corrected_to_the_truth():
    """5-20 kbp reads of a repeat-free genome with a substitution, insertion or deletion every 100-200 bases: every
    read comes back as the genome it was taken from (the index: error-free 100 bp reads tiling both strands)"""
    rng = np.random.default_rng(3)
    k = 21
    g = _clean_genome(rng, 60000, k)
    tiles = []
    for a in range(0, g.size - 100 + 1, 7):
        t = LUT[g[a:a + 100]]
        tiles += [t, RC_SYM[t[::-1]]]
    idx = _index(tiles)
    truths, reads, n_err = [], [], 0
    for _ in range(12):
        ln = int(rng.integers(5000, 20001))
        a = int(rng.integers(0, g.size - ln + 1))
        true = LUT[g[a:a + ln]]
        read = list(true)
        p = ln - 100
        while p > 100:  # from the back, so earlier positions stay put
            kind = int(rng.integers(0, 3))
            # the edit's first and last base differ from what they displace, so every window over it is weak
            if kind == 0:
                c = [s for s in LUT if s != read[p]][int(rng.integers(0, 3))]
                read[p] = c
            elif kind == 1:
                c = [s for s in LUT if s != read[p] and s != read[p - 1]][0]
                read.insert(p, c)
            elif read[p - 1] != read[p] and read[p] != read[p + 1]:
                del read[p]
            else:
                read[p] = [s for s in LUT if s != read[p]][0]
            n_err += 1
            p -= int(rng.integers(100, 201))
        truths.append(true)
        reads.append(np.array(read, np.uint8))
    got, stats = idx.correct_reads(reads, k, 5, 100, 4)
    assert stats[2] == n_err and stats[1] == n_err and stats[3] == 0 and stats[4] == 0
    for a, b in zip(got, truths):
        assert np.array_equal(a, b)


def test_the_result_does_not_depend_on_chunking():
    """one call over about 6 M symbols (two internal chunks and a read across their boundary) equals the
    concatenation of calls over a random partition of the reads"""
    rng = np.random.default_rng(11)
    g = rng.integers(0, 4, 200000)
    idx = _index(_sample(rng, g, [150] * 30000, rate=0.002))
    reads = _sample(rng, g, rng.integers(1000, 20000, 600), rate=0.02, n_rate=0.001)
    assert sum(r.size for r in reads) > (1 << 22)
    whole, stats = idx.correct_reads(reads, 21, 3, 100, 4)
    assert stats[2] > 1000
    cuts = np.sort(rng.choice(np.arange(1, len(reads)), 5, replace=False)).tolist()
    parts, total = [], np.zeros(5, np.uint64)
    for a, b in zip([0] + cuts, cuts + [len(reads)]):
        out, st = idx.correct_reads(reads[a:b], 21, 3, 100, 4)
        parts += out
        total += st
    assert total.tolist() == stats.tolist()
    assert len(parts) == len(whole) and all(np.array_equal(a, b) for a, b in zip(parts, whole))


def test_two_devices_give_the_same_result(read_sets):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    index_reads, queries = read_sets
    rle = M.build_rle_bwt_ragged(index_reads)[0]
    one, two = M.RleBWT(devices=[0]), M.RleBWT(devices=[1, 0])
    one.load_vector(rle)
    two.load_vector(rle)
    a, b = one.correct_reads(queries, 21, 2, 100, 4), two.correct_reads(queries, 21, 2, 100, 4)
    assert a[1].tolist() == b[1].tolist() and all(np.array_equal(x, y) for x, y in zip(a[0], b[0]))


def test_empty_batch_and_empty_reads(read_sets):
    index_reads, _ = read_sets
    g = _index(index_reads)
    out, stats = g.correct_reads([], 21)
    assert out == [] and stats.tolist() == [0] * 5
    out, stats = g.correct_reads([np.zeros(0, np.uint8)] * 3, 21)
    assert [o.size for o in out] == [0, 0, 0] and stats.tolist() == [0] * 5


def test_bad_arguments_are_einval(read_sets):
    index_reads, queries = read_sets
    g = _index(index_reads)
    L = M.load_library()
    flat = np.concatenate(queries[:3])
    offs = np.concatenate([[0], np.cumsum([q.size for q in queries[:3]])]).astype(np.uint64)
    s, o, st = C.c_void_p(0), C.c_void_p(0), np.zeros(5, np.uint64)

    def call(h=g.handle, syms=flat, offsets=offs, n=3, k=21, mc=5, fr=100, bl=4, out_s=True, out_o=True):
        sp = None if syms is None else C.c_void_p(syms.ctypes.data)
        op = None if offsets is None else C.c_void_p(offsets.ctypes.data)
        return L.msbwt_correct_reads(h, sp, op, n, k, mc, fr, bl, C.byref(s) if out_s else None,
                                     C.byref(o) if out_o else None, C.c_void_p(st.ctypes.data))

    assert call() == 0
    L.msbwt_buffer_free(s)
    L.msbwt_buffer_free(o)
    s.value = o.value = None
    bad_sym = flat.copy()
    bad_sym[5] = 0
    bad_sym6 = flat.copy()
    bad_sym6[7] = 6
    dec = offs.copy()
    dec[1], dec[2] = dec[2], dec[1]
    for kw in (dict(h=None), dict(k=0), dict(k=33), dict(mc=0), dict(fr=1001), dict(bl=0), dict(out_s=False),
               dict(out_o=False), dict(syms=None), dict(offsets=None), dict(offsets=dec), dict(syms=bad_sym),
               dict(syms=bad_sym6)):
        assert call(**kw) == EINVAL, kw
        assert s.value is None and o.value is None, kw
    with pytest.raises(M.MsbwtError):
        g.correct_reads(["ACGT$ACGTACGT" * 3], 5)


def test_concurrent_with_count_kmers(read_sets):
    index_reads, queries = read_sets
    g = _index(index_reads)
    want = g.correct_reads(queries, 21, 2, 100, 4)
    km = np.stack([r[:21] for r in index_reads[:500]])
    counts = g.count_kmers_fixed(km, 21)
    errors = []

    def counting():
        for _ in range(20):
            if not np.array_equal(g.count_kmers_fixed(km, 21), counts):
                errors.append("count_kmers")

    th = threading.Thread(target=counting)
    th.start()
    try:
        for _ in range(5):
            got = g.correct_reads(queries, 21, 2, 100, 4)
            if got[1].tolist() != want[1].tolist() or not all(np.array_equal(a, b) for a, b in zip(got[0], want[0])):
                errors.append("correct_reads")
    finally:
        th.join()
    assert not errors, errors
