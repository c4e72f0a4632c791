"""The canonical k-mer spectrum on the device (spectrum.cu, `msbwt_kmer_spectrum_canonical`): histogram, canonical
k-mers and canonical counts against the CPU restatements of oracle/canonical_spectrum.py -- from the reads where the
BWT was built from reads (sampled from both strands), from a walk over the C oracle's constrain_range otherwise --
under every image layout the reverse-complement lookups can take."""
import ctypes as C
import threading

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import canonical_spectrum as CS
from oracle import oracle as O
from oracle import spectrum as S

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KS = (1, 2, 5, 12, 21, 31, 32)
MIN_COUNTS = (1, 2, 3, 5)
NBINS = 40
EINVAL = 1  # MSBWT_EINVAL, include/msbwt_gpu.h
RC_SYM = np.array([0, 5, 3, 2, 4, 1], np.uint8)  # $ A C G N T -> their complements ($ and N stay)


def _index(rle, sb_shift=0, **kw):
    g = M.RleBWT(superblock_shift=sb_shift, **kw)
    g.load_vector(rle)
    return g


def _sorted(kmers, counts):
    order = np.argsort(kmers, kind="stable")
    return kmers[order], counts[order]


def _check(g, k, want_kmers, want_counts):
    """device == oracle for every min_count, given the oracle's min_count-1 canonical list (ascending)"""
    full = g.kmer_spectrum(k, 1, NBINS, canonical=True)
    for t in MIN_COUNTS:
        keep = want_counts >= t
        km, cn = want_kmers[keep], want_counts[keep]
        hist = g.kmer_spectrum(k, t, NBINS, canonical=True)
        gk, gc = g.list_kmers(k, t, canonical=True)
        assert gk.dtype == gc.dtype == np.uint64
        gk, gc = _sorted(gk, gc)
        assert gk.shape == km.shape and (gk == km).all() and (gc == cn).all(), (k, t)
        assert (hist == S.histogram(cn, NBINS)).all(), (k, t)
        # a min_count t run is the min_count 1 run with the bins below t zeroed
        zeroed = full.copy()
        zeroed[:t] = 0
        assert (hist == zeroed).all()
        if gk.size:
            rc = CS.revcomp_u64(gk, k)
            assert (gk <= rc).all() and (gk[1:] > gk[:-1]).all()  # canonical members, each once
            c, c_rc = g.count_kmers_u64(gk, k), g.count_kmers_u64(rc, k)
            assert (gc == np.where(gk == rc, c, c + c_rc)).all()  # through the query path
    return full


def _revcomp_reads(reads, pick):
    return [RC_SYM[r[::-1]] if p else r for r, p in zip(reads, pick)]


def _read_set(rng, lengths, error=0.01, n_rate=0.0):
    """reads of a random genome, each from either strand"""
    genome = rng.integers(0, 4, 3000)
    lut = np.array([1, 2, 3, 5], np.uint8)
    reads = []
    for ln in lengths:
        a = int(rng.integers(0, genome.size - ln + 1))
        r = lut[genome[a:a + ln]].copy()
        hit = rng.random(ln) < error
        r[hit] = lut[rng.integers(0, 4, int(hit.sum()))]
        r[rng.random(ln) < n_rate] = 4
        reads.append(r)
    return _revcomp_reads(reads, rng.random(len(reads)) < 0.5)


def _same_result(g, h, k, t):
    """identical canonical histogram and (sorted) list on two indexes"""
    assert (g.kmer_spectrum(k, t, NBINS, canonical=True) == h.kmer_spectrum(k, t, NBINS, canonical=True)).all()
    a, b = _sorted(*g.list_kmers(k, t, canonical=True)), _sorted(*h.list_kmers(k, t, canonical=True))
    assert all(x.shape == y.shape and (x == y).all() for x, y in zip(a, b))


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_two_strand_equal_length_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(41)
    reads = _read_set(rng, [60] * 500, n_rate=0.002)
    reads += reads[:20]  # duplicate reads
    rle, _ = M.build_rle_bwt(np.stack(reads))
    g = _index(rle, sb_shift)
    for k in KS:
        _, km, cn = CS.canonical_from_reads(reads, k)
        _check(g, k, km, cn)
    # strand invariance: another strand for a random subset of the reads, the same result
    flipped, _ = M.build_rle_bwt(np.stack(_revcomp_reads(reads, rng.random(len(reads)) < 0.5)))
    h = _index(flipped, sb_shift)
    for k, t in ((12, 1), (31, 2), (32, 1)):
        _same_result(g, h, k, t)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_two_strand_ragged_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(42)
    reads = _read_set(rng, rng.integers(0, 90, 700), n_rate=0.005)
    rle, _ = M.build_rle_bwt_ragged(reads)
    g = _index(rle, sb_shift)
    for k in KS:
        _, km, cn = CS.canonical_from_reads(reads, k)
        _check(g, k, km, cn)


@pytest.fixture(scope="module")
def golden_walk(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    return z["rle"], S.walk_rle(z["rle"], 32, 1)


def _want(walk, k):
    return CS.canonical_from_walk(*walk[k - 1], k)[1:]


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_golden_index_matches_the_oracle(golden_walk, sb_shift):
    rle, walk = golden_walk
    g = _index(rle, sb_shift)
    for k in KS:
        _check(g, k, *_want(walk, k))


@pytest.mark.parametrize("layout", [
    dict(oct_index=1, final_index=1, suffix_table_s=12),  # the one-request kernel answers the rc lookups of 31/32-mers
    dict(oct_index=1, final_index=0),
    dict(pair_index=1, quad_index=0, oct_index=0),
    dict(oct_index=1, final_index=1, superblock_shift=4),  # 64-bit positions: the WIDE oct and one-request kernels
])
def test_golden_index_under_every_layout(golden_walk, layout):
    rle, walk = golden_walk
    g = M.RleBWT(**layout)
    g.load_vector(rle)
    if layout.get("final_index") and "superblock_shift" not in layout:
        assert g.final_index and g.table_depth_for_k(31) == 11 and g.table_depth_for_k(32) == 12
    for k in (12, 21, 31, 32):
        _check(g, k, *_want(walk, k))


def test_golden_index_with_the_general_kernels(golden_walk, monkeypatch):
    """MSBWT_FINAL_FAST=0: the rc lookups of 31-mers take the general query kernels"""
    rle, walk = golden_walk
    g = _index(rle, oct_index=1, final_index=1, suffix_table_s=12)
    monkeypatch.setenv("MSBWT_FINAL_FAST", "0")
    for k in (31, 32):
        _check(g, k, *_want(walk, k))


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_random_rle_streams_match_the_oracle(sb_shift):
    rng = np.random.default_rng(43)
    for _ in range(6):
        n_runs = int(rng.integers(50, 3000))
        syms = np.repeat(rng.choice(np.array([0, 1, 2, 3, 4, 5], np.uint8), n_runs, p=[.05, .22, .22, .22, .07, .22]),
                         rng.integers(1, 12, n_runs))
        rle = O.convert_to_vec(O.convert_itos(syms))
        walk = S.walk_rle(rle, 32, 1)
        g = _index(rle, sb_shift)
        for k in KS:
            _check(g, k, *_want(walk, k))


def test_many_slices_and_several_staging_batches(monkeypatch):
    """small slices (MSBWT_SPECTRUM_SLICE) over more than 10^7 expanded ranges, and more listed k-mers than one
    staging buffer (2^22) holds, so that several batches are resolved"""
    from harness import synth
    reads = synth.make_reads(240_000, read_len=100, coverage=20.0, error_rate=0.01, device="cuda:0")
    flip = torch.arange(reads.shape[0], device=reads.device) % 2 == 1
    rc = torch.from_numpy(RC_SYM).to(reads.device)[reads.flip(1).long()]
    reads = torch.where(flip[:, None], rc, reads).contiguous()
    rle, _ = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
    reads = reads.cpu().numpy()
    g = _index(rle)
    k = 31
    expanded = 1 + sum(int(g.kmer_spectrum(d, 1, 2)[1]) for d in range(1, k))
    assert expanded >= 10_000_000, expanded
    assert g.list_kmers(k, 1)[0].size > 1 << 22  # what the canonical walk stages at min_count 1 and 2
    _, km, cn = CS.canonical_from_reads(list(reads), k)
    want_hist = S.histogram(cn, NBINS)
    default = _sorted(*g.list_kmers(k, 1, canonical=True))
    assert (default[0] == km).all() and (default[1] == cn).all()
    monkeypatch.setenv("MSBWT_SPECTRUM_SLICE", "4096")
    for t in (1, 2):
        gk, gc = _sorted(*g.list_kmers(k, t, canonical=True))
        keep = cn >= t
        assert (gk == km[keep]).all() and (gc == cn[keep]).all()
        hist = g.kmer_spectrum(k, t, NBINS, canonical=True)
        want = want_hist.copy()
        want[:t] = 0
        assert (hist == want).all()


def test_bad_arguments_and_edge_cases(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    for kw in (dict(k=0), dict(k=33), dict(k=5, min_count=0), dict(k=5, nbins=1), dict(k=5, nbins=(1 << 20) + 1)):
        with pytest.raises(M.MsbwtError):
            g.kmer_spectrum(canonical=True, **kw)
    with pytest.raises(M.MsbwtError):
        g.list_kmers(33, canonical=True)
    L = M.load_library()
    km, n = C.c_void_p(0), C.c_uint64(7)
    hist = np.zeros(4, np.uint64)
    assert L.msbwt_kmer_spectrum_canonical(g.handle, 5, 1, None, 0, C.byref(km), None, C.byref(n)) == EINVAL
    assert L.msbwt_kmer_spectrum_canonical(g.handle, 5, 1, None, 4, None, None, C.byref(n)) == EINVAL
    assert L.msbwt_kmer_spectrum_canonical(g.handle, 5, 1, hist.ctypes.data, 4, None, None, None) == EINVAL
    assert L.msbwt_kmer_spectrum_canonical(g.handle, 0, 1, hist.ctypes.data, 4, None, None, C.byref(n)) == EINVAL
    assert L.msbwt_kmer_spectrum_canonical(g.handle, 5, 0, hist.ctypes.data, 4, None, None, C.byref(n)) == EINVAL
    assert n.value == 7 and not km.value and not hist.any()  # nothing written
    assert g.kmer_spectrum(5, 1, 2**20, canonical=True).size == 2**20
    # k longer than every read, a min_count above N, an index of $ and N only: no k-mer, an all-zero histogram
    rle, total = M.build_rle_bwt(np.full((50, 20), 2, np.uint8))
    short = _index(rle)
    assert not short.kmer_spectrum(21, 1, 8, canonical=True).any()
    assert short.list_kmers(21, 1, canonical=True)[0].size == 0
    # the one 20-mer CCC...C (whose reverse complement GGG...G does not occur) is canonical and counted 50 times
    assert short.kmer_spectrum(20, 1, 8, canonical=True).tolist() == [0] * 7 + [1]
    km1, cn1 = short.list_kmers(20, 1, canonical=True)
    assert km1.tolist() == [int("01" * 20, 2)] and cn1.tolist() == [50]
    assert not short.kmer_spectrum(3, total + 1, 8, canonical=True).any()
    for t in (total + 1, 2**64 - 1):  # the walk's threshold ceil(t / 2) must not wrap at the top of the range
        assert not short.kmer_spectrum(3, t, 8, canonical=True).any() and short.list_kmers(3, t, canonical=True)[0].size == 0
    dn = _index(O.convert_to_vec("NN$N$$N"))
    assert not dn.kmer_spectrum(1, 1, 8, canonical=True).any() and dn.list_kmers(1, 1, canonical=True)[0].size == 0


def test_counts_above_the_shared_memory_bins():
    """canonical counts of 4096 and more land in the global-atomic bins of the resolve kernel (the first 4096 bins of
    each CTA are kept in shared memory)"""
    rng = np.random.default_rng(44)
    base = _read_set(rng, [50] * 300)
    hot = np.array([1, 2, 3, 5, 5, 3, 1, 2, 2, 1] * 3, np.uint8)  # 30 symbols, read 5000 times on either strand
    reads = base + _revcomp_reads([hot] * 5000, rng.random(5000) < 0.5)
    rle, _ = M.build_rle_bwt_ragged(reads)
    g = _index(rle)
    nbins = 10001
    for k in (5, 12, 21):
        hist_want, km, cn = CS.canonical_from_reads(reads, k, 1, nbins)
        assert cn.max() >= 5000 and hist_want[4096:].sum() > 0
        for t in (1, 3):
            hist = g.kmer_spectrum(k, t, nbins, canonical=True)
            want = hist_want.copy()
            want[:t] = 0
            assert (hist == want).all(), (k, t)
        gk, gc = _sorted(*g.list_kmers(k, 1, canonical=True))
        assert (gk == km).all() and (gc == cn).all()


def test_two_calls_return_identical_arrays(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    for k in (12, 31):
        a, b = g.list_kmers(k, 1, canonical=True), g.list_kmers(k, 1, canonical=True)
        assert all(x.shape == y.shape and (x == y).all() for x, y in zip(a, b))


def test_two_devices_give_the_same_result(golden_dir):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    one, two = _index(z["rle"]), _index(z["rle"], devices=[1, 0])
    for k in (12, 31):
        assert (one.kmer_spectrum(k, canonical=True) == two.kmer_spectrum(k, canonical=True)).all()
        a, b = one.list_kmers(k, 1, canonical=True), two.list_kmers(k, 1, canonical=True)
        assert all((x == y).all() for x, y in zip(a, b))


def test_concurrent_count_kmers_on_the_same_handle(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    q, want = z["queries"], z["counts"]
    qq, ww = np.tile(q, (200, 1)), np.tile(want, 200)
    ref = g.list_kmers(31, 1, canonical=True)
    errors = []

    def counter():
        try:
            for _ in range(20):
                if not (g.count_kmers_fixed(qq, 31) == ww).all():
                    errors.append("count_kmers_fixed")
        except Exception as e:  # noqa: BLE001 -- surfaced below
            errors.append(repr(e))

    th = threading.Thread(target=counter)
    th.start()
    try:
        for _ in range(20):
            km, cn = g.list_kmers(31, 1, canonical=True)
            if not ((km == ref[0]).all() and (cn == ref[1]).all()):
                errors.append("list_kmers")
    finally:
        th.join()
    assert not errors, errors


def _windows(reads, k):
    n = 0
    for a in range(0, reads.shape[0], 1 << 20):
        n_in = torch.cumsum(torch.nn.functional.pad((reads[a:a + (1 << 20)] == 4).int(), (1, 0)), dim=1)
        n += int(((n_in[:, k:] - n_in[:, :-k]) == 0).sum().item())
    return n


def _device_sorted(km, cn, dev):
    d_km = torch.from_numpy(km.view(np.int64)).to(dev)  # k <= 31: every value fits an int64 unchanged
    d_km, order = torch.sort(d_km)
    return d_km, torch.from_numpy(cn.view(np.int64)).to(dev)[order]


def test_config3_full_size():
    """configs[2]: 10 M reads x 150 bp with 1 % errors, the 1.51 Gsymbol index of bench.py, k = 31"""
    import bench
    if torch.cuda.get_device_properties(0).total_memory < 150e9:
        pytest.skip("needs the 180 GB of a B200")
    cfg = bench.WORKLOADS["cfg3"]
    dev = torch.device("cuda:0")
    torch.cuda.empty_cache()
    reads, rle, total = bench.build_reads_and_bwt(cfg, dev, True)
    k = 31
    g = M.RleBWT.new(devices=[0])
    g.load_vector(rle)
    assert g.get_total_size() == total

    # sum of c * hist[c] = every N-free 31-window of the reads
    hist = g.kmer_spectrum(k, 1, 1 << 20, canonical=True)
    assert hist[-1] == 0
    assert int((np.arange(hist.size, dtype=np.uint64) * hist).sum()) == _windows(reads, k)
    km, cn = g.list_kmers(k, 2, canonical=True)
    want = hist.copy()
    want[:2] = 0
    assert km.size == int(want.sum()) and (S.histogram(cn, hist.size) == want).all()

    # a 100 k sample of the list against the C oracle's count_kmer of x and of rc x
    pick = np.random.default_rng(5).choice(km.size, 100_000, replace=False)
    code = np.array([1, 2, 3, 5], np.uint8)

    def syms(v):
        return np.ascontiguousarray(np.stack([code[(v >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)]
                                              for j in range(k)], axis=1))
    x, rx = km[pick], CS.revcomp_u64(km[pick], k)
    orc = O.RleBWT()
    orc.load_vector(rle)
    c, c_rc = orc.count_kmers_fixed(syms(x), k, threads=16), orc.count_kmers_fixed(syms(rx), k, threads=16)
    del orc
    assert (x <= rx).all() and (cn[pick] == np.where(x == rx, c, c + c_rc)).all()
    ref_km, ref_cn = _device_sorted(km, cn, dev)
    assert bool((ref_km[1:] > ref_km[:-1]).all())
    del g, km, cn, rle

    # every other read reverse-complemented (on the device), one index built and loaded at a time: the same result
    rc = torch.from_numpy(RC_SYM).to(dev)
    reads[::2] = rc[reads[::2].flip(1).long()]
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    rle2, total2 = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
    assert total2 == total
    del reads
    torch.cuda.empty_cache()
    h = M.RleBWT.new(devices=[0])
    h.load_vector(rle2)
    assert (h.kmer_spectrum(k, 1, 1 << 20, canonical=True) == hist).all()
    km2, cn2 = _device_sorted(*h.list_kmers(k, 2, canonical=True), dev)
    assert km2.shape == ref_km.shape and bool((km2 == ref_km).all()) and bool((cn2 == ref_cn).all())
