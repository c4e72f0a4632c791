"""The device merge of two multi-string BWTs (bwt_merge.cu, `msbwt_merge_rle_bwts`): Holt and McMillan's interleave
(pairwise_bwt_merge, src/bwt_util.rs:108-141).  On BWTs built from reads it must give, byte for byte, what the builder
makes from all the reads at once; on any RLE streams, what oracle/merge.py computes (bytes and iteration count)."""
import ctypes as C

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import merge as OM
from oracle import naive
from oracle import oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _merge_checked(rle_a, rle_b):
    """device merge == oracle merge (bytes, total, iterations); returns the device result"""
    got, total, iterations = M.merge_rle_bwts(rle_a, rle_b)
    want, want_total, want_iterations = OM.merge_rle(rle_a, rle_b)
    assert total == want_total and iterations == want_iterations
    assert got.size == want.size and (got == want).all()
    return got, total, iterations


def _read_sets(a, b):
    rle_a, _ = M.build_rle_bwt_ragged(a)
    rle_b, _ = M.build_rle_bwt_ragged(b)
    got, total, iterations = _merge_checked(rle_a, rle_b)
    union, union_total = M.build_rle_bwt_ragged(list(a) + list(b))
    assert total == union_total and (got == union).all()
    assert (M.merge_rle_bwts(rle_b, rle_a)[0] == got).all()
    longest = max([len(r) for r in list(a) + list(b)], default=0)
    assert iterations <= 2 * longest + 2
    return got


def test_reference_sets():
    got = _read_sets(["ACGT"], ["TGCA"])
    o = O.RleBWT()
    o.load_vector(O.convert_to_vec(naive.naive_bwt(["ACGT", "TGCA"])))
    assert (got == o.rle_bytes()).all()
    got = _read_sets(["CCGT", "N"], ["ACG"])
    assert (got == O.convert_to_vec("GTN$$ACCC$G")).all()


def test_random_ragged_sets_prefixes_and_duplicates():
    rng = np.random.default_rng(108)
    for t in range(40):
        def reads(n):
            alphabet = np.array([1, 2, 3, 4, 5] if t % 3 == 0 else [1, 2, 3, 5], dtype=np.uint8)
            return [rng.choice(alphabet, size=int(rng.integers(0, 40))) for _ in range(n)]
        a, b = reads(int(rng.integers(3, 300))), reads(int(rng.integers(1, 300)))
        b += [a[0], a[1][: len(a[1]) // 2], a[2][len(a[2]) // 3:]]   # a duplicate, a prefix and a suffix of A's reads
        a.append(a[0])
        _read_sets(a, b)


def test_empty_inputs_and_self_merge():
    rng = np.random.default_rng(5)
    reads = rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(3000, 60))
    rle, total = M.build_rle_bwt(reads)
    empty = np.zeros(0, np.uint8)
    for a, b in ((rle, empty), (empty, rle)):
        got, n, iterations = _merge_checked(a, b)
        assert n == total and iterations == 1 and (got == rle).all()
    got, n, iterations = M.merge_rle_bwts(empty, empty)
    assert got.size == 0 and n == 0 and iterations == 0
    got, n, _ = _merge_checked(rle, rle)
    assert n == 2 * total and (got == M.build_rle_bwt(np.concatenate([reads, reads]))[0]).all()


def test_runs_of_three_or_more_digits_in_both_inputs():
    a = [np.full(6, 1, np.uint8)] * 2000 + [np.array([2, 3], np.uint8)] * 40
    b = [np.full(6, 1, np.uint8)] * 1500 + [np.full(4, 5, np.uint8)] * 1200
    for rle in (M.build_rle_bwt_ragged(a)[0], M.build_rle_bwt_ragged(b)[0]):
        syms = rle & 7
        digits = np.diff(np.flatnonzero(np.r_[True, syms[1:] != syms[:-1], True]))
        assert digits.max() >= 3
    _read_sets(a, b)


def test_arbitrary_streams_match_the_oracle():
    """RLE streams no builder made (random runs, several tiles of the interleave, non-canonical digits): the loader
    accepts them as indexes, so the merge must reach the oracle's fixed point in as many passes."""
    rng = np.random.default_rng(141)
    for n_a, n_b, longest in ((300, 200, 3000), (5000, 7000, 2), (1, 40_000, 50), (0, 700, 9000)):
        rle = []
        for n in (n_a, n_b):
            syms = (np.cumsum(rng.integers(1, 6, n)) % 6).astype(np.uint8)   # no two neighbouring runs share a symbol
            rle.append(O.encode_runs(syms, rng.integers(1, longest, n).astype(np.uint64)) if n else np.zeros(0, np.uint8))
        _merge_checked(*rle)
    # a run with a zero middle digit: 1 + 0 * 32 + 1 * 1024 symbols
    _merge_checked(np.array([1 | 3 << 3, 2 | 1 << 3, 2 | 0 << 3, 2 | 1 << 3, 0 | 2 << 3], np.uint8),
                   np.array([5 | 7 << 3, 2 | 4 << 3, 5 | 1 << 3, 0 | 1 << 3], np.uint8))


def test_errors():
    good = O.convert_to_vec("GTN$$ACCC$G")
    bad = good.copy()
    bad[3] = (int(bad[3]) & 0xF8) | 6
    for a, b in ((bad, good), (good, bad)):
        with pytest.raises(M.MsbwtError) as e:
            M.merge_rle_bwts(a, b)
        assert e.value.code == 3  # EFORMAT
    L = M.load_library()
    p = C.c_void_p(good.ctypes.data)
    out, n, total, it = C.c_void_p(0), C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
    assert L.msbwt_merge_rle_bwts(p, good.size, p, good.size, 0, None, C.byref(n), C.byref(total), C.byref(it)) == 1
    assert L.msbwt_merge_rle_bwts(p, good.size, p, good.size, 0, C.byref(out), None, C.byref(total), None) == 1
    assert L.msbwt_merge_rle_bwts(p, good.size, p, good.size, 0, C.byref(out), C.byref(n), None, None) == 1
    assert L.msbwt_merge_rle_bwts(None, 5, p, good.size, 0, C.byref(out), C.byref(n), C.byref(total), C.byref(it)) == 1
    assert not out.value
    # iterations may be NULL
    assert L.msbwt_merge_rle_bwts(p, good.size, p, good.size, 0, C.byref(out), C.byref(n), C.byref(total), None) == 0
    assert total.value == 2 * 11
    L.msbwt_buffer_free(out)


def _build_half(reads, lo, hi):
    part = reads[lo:hi]
    return M.build_rle_bwt(part.data_ptr(), 0, part.shape[0], part.shape[1])


def test_headline_size_equals_building_all_the_reads():
    """configs[2]'s read set (10 M 150-bp reads, 1 % errors, 1.51 Gsymbols) built as two halves and merged."""
    from harness import synth
    torch.cuda.empty_cache()
    reads = synth.make_reads(10_000_000, read_len=150, coverage=30.0, error_rate=0.01, device="cuda")
    rle_a, n_a = _build_half(reads, 0, 5_000_000)
    rle_b, n_b = _build_half(reads, 5_000_000, 10_000_000)
    whole, n = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
    del reads
    torch.cuda.empty_cache()
    got, total, iterations = M.merge_rle_bwts(rle_a, rle_b)
    assert total == n == n_a + n_b == 10_000_000 * 151
    assert iterations <= 2 * 150 + 2
    assert got.size == whole.size and (got == whole).all()
    back, _, back_iterations = M.merge_rle_bwts(rle_b, rle_a)
    assert back_iterations <= 2 * 150 + 2 and (back == whole).all()


def test_merge_beyond_2_pow_32_symbols():
    """15 M + 15 M reads, each half built on its own (2.27 Gsymbols each); the merged 4.53 Gsymbol BWT is beyond what
    the builder does in one call.  Totals and symbol counts add up, the merge is symmetric, k-mer counts add up, and
    the merged index answers as the CPU oracle does on a sample.  The merged BWT then takes part in one more merge, as
    an input wider than 2^32 symbols."""
    from harness import synth
    torch.cuda.empty_cache()
    half = 15_000_000
    reads = synth.make_reads(2 * half, read_len=150, coverage=30.0, error_rate=0.01, device="cuda")
    queries = synth.make_queries(reads, 31, 600_000, 500_000).cpu().numpy()   # read-sampled and random 31-mers
    rle_a, n_a = _build_half(reads, 0, half)
    rle_b, n_b = _build_half(reads, half, 2 * half)
    del reads
    torch.cuda.empty_cache()
    merged, total, iterations = M.merge_rle_bwts(rle_a, rle_b)
    assert total == n_a + n_b == 2 * half * 151 and total > (1 << 32)
    assert iterations <= 2 * 150 + 2
    back, _, _ = M.merge_rle_bwts(rle_b, rle_a)
    assert back.size == merged.size and (back == merged).all()
    del back
    # chaining: the 4.53 Gsymbol result (two superblocks, 64-bit positions) is itself an input
    more = synth.make_reads(200_000, read_len=150, coverage=30.0, error_rate=0.01, device="cuda", seed_offset=7)
    rle_c, n_c = _build_half(more, 0, more.shape[0])
    del more
    chained, total_c, iterations_c = M.merge_rle_bwts(merged, rle_c)
    assert total_c == total + n_c and iterations_c <= 2 * 150 + 2

    counts, syms = [], []
    for rle in (rle_a, rle_b, merged, rle_c, chained):   # one index at a time
        g = M.RleBWT(pair_index=0, quad_index=0, oct_index=0, final_index=0)
        g.load_vector(rle)
        counts.append(g.count_kmers_fixed(queries, 31))
        syms.append([g.get_symbol_count(s) for s in range(6)])
        g.close()
        torch.cuda.empty_cache()
    assert syms[2] == [x + y for x, y in zip(syms[0], syms[1])] and syms[2][0] == 2 * half
    assert (counts[2] == counts[0] + counts[1]).all()
    assert int((counts[2] > 0).sum()) >= 600_000
    assert syms[4] == [x + y for x, y in zip(syms[2], syms[3])]
    assert (counts[4] == counts[2] + counts[3]).all()

    g = M.RleBWT(pair_index=0, quad_index=0, oct_index=0, final_index=0)
    g.load_vector(merged)
    o = O.RleBWT()
    o.load_vector(merged)
    assert o.get_total_size() == total
    rng = np.random.default_rng(453)
    m = 20_000
    sym = rng.integers(0, 6, m).astype(np.uint8)
    lo = rng.integers(0, total + 1, m).astype(np.uint64)
    hi = np.minimum(lo + rng.choice(np.array([0, 1, 77, 1 << 20, 1 << 33], dtype=np.uint64), m), np.uint64(total))
    lo[:3], hi[:3] = [0, (1 << 32) - 5, total], [total, (1 << 32) + 5, total]
    gl, gh = g.constrain_ranges(sym, lo, hi)
    for i in range(m):
        assert (int(gl[i]), int(gh[i])) == o.constrain_range(int(sym[i]), int(lo[i]), int(hi[i])), i
    sample = queries[::50]
    assert (counts[2][::50] == o.count_kmers_fixed(sample, 31, threads=8)).all()
    g.close()
    torch.cuda.empty_cache()
