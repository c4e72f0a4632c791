"""The k-mer spectrum of an index and its solid k-mers on the device (spectrum.cu, `msbwt_kmer_spectrum`): histogram,
k-mer list, counts and co-lexicographic order against the CPU restatements of oracle/spectrum.py -- from the reads
where the BWT was built from reads, from a walk over the C oracle's constrain_range otherwise."""
import ctypes as C
import threading

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import oracle as O
from oracle import spectrum as S

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KS = (1, 2, 5, 12, 21, 31, 32)
MIN_COUNTS = (1, 2, 5)
NBINS = 40
EINVAL = 1  # MSBWT_EINVAL, include/msbwt_gpu.h


def _index(rle, sb_shift=0, **kw):
    g = M.RleBWT(superblock_shift=sb_shift, **kw)
    g.load_vector(rle)
    return g


def _check(g, k, want_kmers, want_counts):
    """device == oracle for every min_count, given the oracle's min_count-1 list of k-mers of length k"""
    full = g.kmer_spectrum(k, 1, NBINS)
    for t in MIN_COUNTS:
        keep = want_counts >= t
        km, cn = want_kmers[keep], want_counts[keep]
        hist = g.kmer_spectrum(k, t, NBINS)
        gk, gc = g.list_kmers(k, t)
        assert gk.dtype == gc.dtype == np.uint64
        assert gk.shape == km.shape and (gk == km).all() and (gc == cn).all(), (k, t)
        assert (hist == S.histogram(cn, NBINS)).all(), (k, t)
        # a min_count t run is the min_count 1 run with the bins below t zeroed
        zeroed = full.copy()
        zeroed[:t] = 0
        assert (hist == zeroed).all()
        if gk.size:
            assert (g.count_kmers_u64(gk, k) == gc).all()       # round trip through the query path
            key = S.colex_key(gk, k)
            assert (key[1:] > key[:-1]).all()                    # strictly increasing in co-lexicographic order
    return full


def _read_set(rng, lengths, error=0.01, n_rate=0.0):
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
    return reads


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_equal_length_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(31)
    reads = _read_set(rng, [60] * 500, n_rate=0.002)
    reads += reads[:20]  # duplicate reads
    rle, _ = M.build_rle_bwt(np.stack(reads))
    g = _index(rle, sb_shift)
    for k in KS:
        _, km, cn = S.from_reads(reads, k)
        _check(g, k, km, cn)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_ragged_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(32)
    reads = _read_set(rng, rng.integers(0, 90, 700), n_rate=0.005)
    rle, _ = M.build_rle_bwt_ragged(reads)
    g = _index(rle, sb_shift)
    for k in KS:
        _, km, cn = S.from_reads(reads, k)
        _check(g, k, km, cn)


@pytest.fixture(scope="module")
def golden_walk(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    return z["rle"], S.walk_rle(z["rle"], 32, 1)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_golden_index_matches_the_oracle(golden_walk, sb_shift):
    rle, walk = golden_walk
    g = _index(rle, sb_shift)
    for k in KS:
        _check(g, k, *walk[k - 1])
    # every image policy: the call reads only the one-step blocks, so the large-index images change nothing
    for kw in (dict(pair_index=1, quad_index=0, oct_index=0), dict(oct_index=1)):
        h = _index(rle, sb_shift, **kw)
        for k in (12, 31):
            assert all((a == b).all() for a, b in zip(h.list_kmers(k, 1), g.list_kmers(k, 1)))


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_random_rle_streams_match_the_oracle(sb_shift):
    rng = np.random.default_rng(33)
    for _ in range(6):
        n_runs = int(rng.integers(50, 3000))
        syms = np.repeat(rng.choice(np.array([0, 1, 2, 3, 4, 5], np.uint8), n_runs, p=[.05, .22, .22, .22, .07, .22]),
                         rng.integers(1, 12, n_runs))
        rle = O.convert_to_vec(O.convert_itos(syms))
        walk = S.walk_rle(rle, 32, 1)
        g = _index(rle, sb_shift)
        for k in KS:
            _check(g, k, *walk[k - 1])


def test_many_slices_at_several_depths(monkeypatch):
    """small slices (MSBWT_SPECTRUM_SLICE) over a read set that expands more than 10^7 ranges"""
    from harness import synth
    reads = synth.make_reads(60_000, read_len=100, coverage=20.0, error_rate=0.01, device="cuda:0")
    rle, _ = M.build_rle_bwt(reads.data_ptr(), 0, reads.shape[0], reads.shape[1])
    reads = reads.cpu().numpy()
    g = _index(rle)
    k = 31
    expanded = 1 + sum(int(g.kmer_spectrum(d, 1, 2)[1]) for d in range(1, k))
    assert expanded >= 10_000_000, expanded
    _, km, cn = S.from_reads(list(reads), k)
    want_hist = S.histogram(cn, NBINS)
    default = g.list_kmers(k, 1)
    monkeypatch.setenv("MSBWT_SPECTRUM_SLICE", "4096")
    for t in (1, 2):
        gk, gc = g.list_kmers(k, t)
        keep = cn >= t
        assert (gk == km[keep]).all() and (gc == cn[keep]).all()
        hist = g.kmer_spectrum(k, t, NBINS)
        want = want_hist.copy()
        want[:t] = 0
        assert (hist == want).all()
    monkeypatch.delenv("MSBWT_SPECTRUM_SLICE")
    assert (default[0] == km).all() and (default[1] == cn).all()


def test_bad_arguments_and_edge_cases(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    for kw in (dict(k=0), dict(k=33), dict(k=5, min_count=0), dict(k=5, nbins=1), dict(k=5, nbins=(1 << 20) + 1)):
        with pytest.raises(M.MsbwtError):
            g.kmer_spectrum(**kw)
    with pytest.raises(M.MsbwtError):
        g.list_kmers(33)
    L = M.load_library()
    km, n = C.c_void_p(0), C.c_uint64(7)
    hist = np.zeros(4, np.uint64)
    assert L.msbwt_kmer_spectrum(g.handle, 5, 1, None, 0, C.byref(km), None, C.byref(n)) == EINVAL
    assert L.msbwt_kmer_spectrum(g.handle, 5, 1, None, 4, None, None, C.byref(n)) == EINVAL
    assert L.msbwt_kmer_spectrum(g.handle, 5, 1, hist.ctypes.data, 4, None, None, None) == EINVAL
    assert n.value == 7 and not km.value  # nothing written
    assert g.kmer_spectrum(5, 1, 2**20).size == 2**20
    # k longer than every read, a min_count above N, an index of $ and N only: no k-mer, an all-zero histogram
    rle, total = M.build_rle_bwt(np.full((50, 20), 2, np.uint8))
    short = _index(rle)
    assert not short.kmer_spectrum(21, 1, 8).any() and short.list_kmers(21, 1)[0].size == 0
    assert short.kmer_spectrum(20, 1, 8).tolist() == [0] * 7 + [1]
    assert not short.kmer_spectrum(3, total + 1, 8).any()
    dn = _index(O.convert_to_vec("NN$N$$N"))
    assert not dn.kmer_spectrum(1, 1, 8).any() and dn.list_kmers(1, 1)[0].size == 0


def test_two_devices_give_the_same_result(golden_dir):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    one, two = _index(z["rle"]), _index(z["rle"], devices=[1, 0])
    for k in (12, 31):
        assert (one.kmer_spectrum(k) == two.kmer_spectrum(k)).all()
        assert all((a == b).all() for a, b in zip(one.list_kmers(k, 1), two.list_kmers(k, 1)))


def test_concurrent_count_kmers_on_the_same_handle(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    q, want = z["queries"], z["counts"]
    qq, ww = np.tile(q, (200, 1)), np.tile(want, 200)
    ref = g.list_kmers(31, 1)
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
            km, cn = g.list_kmers(31, 1)
            if not ((km == ref[0]).all() and (cn == ref[1]).all()):
                errors.append("list_kmers")
    finally:
        th.join()
    assert not errors, errors


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

    # sum of c * hist[c] = every N-free 31-window of the reads, counted on the device from the reads
    hist = g.kmer_spectrum(k, 1, 1 << 20)
    assert hist[-1] == 0
    windows = 0
    for a in range(0, reads.shape[0], 1 << 20):
        n_in = torch.cumsum(torch.nn.functional.pad((reads[a:a + (1 << 20)] == 4).int(), (1, 0)), dim=1)
        windows += int(((n_in[:, k:] - n_in[:, :-k]) == 0).sum().item())
    assert int((np.arange(hist.size, dtype=np.uint64) * hist).sum()) == windows

    # the solid list (min_count 2): strictly increasing in co-lexicographic order, its histogram is hist's
    km, cn = g.list_kmers(k, 2)
    want = hist.copy()
    want[:2] = 0
    assert km.size == int(want.sum()) and (S.histogram(cn, hist.size) == want).all()
    d_km = torch.from_numpy(km.view(np.int64)).to(dev)
    key = torch.zeros_like(d_km)
    for j in range(k):
        key |= ((d_km >> (2 * j)) & 3) << (2 * (k - 1 - j))
    assert bool((key[1:] > key[:-1]).all())

    # a 1 M-window sample of the reads: count >= 2 <=> listed, with count_kmers_u64's count
    gen = torch.Generator(device=dev).manual_seed(11)
    r = torch.randint(0, reads.shape[0], (1 << 20,), generator=gen, device=dev)
    o = torch.randint(0, reads.shape[1] - k + 1, (1 << 20,), generator=gen, device=dev)
    win = reads[r[:, None], o[:, None] + torch.arange(k, device=dev)]
    sample = bench.encode_u64(win, k)
    counts = torch.from_numpy(g.count_kmers_u64(sample.cpu().numpy().view(np.uint64), k).view(np.int64)).to(dev)
    skey = torch.zeros_like(sample)
    for j in range(k):
        skey |= ((sample >> (2 * j)) & 3) << (2 * (k - 1 - j))
    pos = torch.searchsorted(key, skey).clamp(max=key.numel() - 1)
    found = key[pos] == skey
    d_cn = torch.from_numpy(cn.view(np.int64)).to(dev)
    assert bool((found == (counts >= 2)).all())
    assert bool((d_cn[pos][found] == counts[found]).all())

    # the counts of a 100 k sample of the list against the oracle
    pick = np.random.default_rng(5).choice(km.size, 100_000, replace=False)
    code = np.array([1, 2, 3, 5], np.uint8)
    syms = np.stack([code[(km[pick] >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)] for j in range(k)], axis=1)
    orc = O.RleBWT()
    orc.load_vector(rle)
    assert (orc.count_kmers_fixed(np.ascontiguousarray(syms), k, threads=16) == cn[pick]).all()
