"""The unitigs of the compacted de Bruijn graph on the device (unitigs.cu, `msbwt_unitigs`): byte for byte against
oracle/unitigs.py built from the node list the spectrum gives, every result through the oracle's property checker, and
the semantic properties the definition promises (strand invariance, both-strand indexes, circular genomes, tiling)."""
import ctypes as C
import threading

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import oracle as O
from oracle import unitigs as U

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KS = (1, 2, 5, 12, 21, 31, 32)
MIN_COUNTS = (1, 2, 3, 5)
EINVAL = 1  # MSBWT_EINVAL, include/msbwt_gpu.h
RC_SYM = np.array([0, 5, 3, 2, 4, 1], np.uint8)  # $ A C G N T -> their complements ($ and N stay)
LUT = np.array([1, 2, 3, 5], np.uint8)


def _index(rle, sb_shift=0, **kw):
    g = M.RleBWT(superblock_shift=sb_shift, **kw)
    g.load_vector(rle)
    return g


def _same(a, b):
    assert len(a) == len(b) == 3
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape and (x == y).all()


def _check(g, k, t, canonical, oracle=True):
    """device == oracle (from the device's own node list, which the spectrum tests pin) and the property checker"""
    got = g.unitigs(k, t, canonical)
    km, cn = g.list_kmers(k, t, canonical=canonical)
    order = np.argsort(km)
    km, cn = km[order], cn[order]
    if oracle:
        _same(got, U.unitigs(km, cn, k, canonical))
    U.check_unitigs(*got, km, cn, k, canonical)
    return got


def _revcomp_reads(reads, pick):
    return [RC_SYM[r[::-1]] if p else r for r, p in zip(reads, pick)]


def _read_set(rng, lengths, error=0.01, n_rate=0.0, genome=600):
    """reads of a random genome, each from either strand"""
    g = rng.integers(0, 4, genome)
    reads = []
    for ln in lengths:
        a = int(rng.integers(0, g.size - ln + 1))
        r = LUT[g[a:a + ln]].copy()
        hit = rng.random(ln) < error
        r[hit] = LUT[rng.integers(0, 4, int(hit.sum()))]
        r[rng.random(ln) < n_rate] = 4
        reads.append(r)
    return _revcomp_reads(reads, rng.random(len(reads)) < 0.5)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_equal_length_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(51)
    reads = _read_set(rng, [60] * 200, n_rate=0.002)
    reads += reads[:10]  # duplicate reads
    g = _index(M.build_rle_bwt(np.stack(reads))[0], sb_shift)
    for k in KS:
        for t in MIN_COUNTS:
            for canonical in (False, True):
                _check(g, k, t, canonical)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_ragged_reads_match_the_oracle(sb_shift):
    rng = np.random.default_rng(52)
    reads = _read_set(rng, rng.integers(0, 90, 250), n_rate=0.005)
    g = _index(M.build_rle_bwt_ragged(reads)[0], sb_shift)
    for k in KS:
        for t in MIN_COUNTS:
            for canonical in (False, True):
                _check(g, k, t, canonical)


def test_golden_index_matches_the_oracle(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    for k in KS:
        for t in MIN_COUNTS:
            for canonical in (False, True):
                _check(g, k, t, canonical, oracle=t > 1 or k < 12)


@pytest.mark.parametrize("sb_shift", [0, 3])
def test_random_rle_streams_match_the_oracle(sb_shift):
    rng = np.random.default_rng(53)
    for _ in range(4):
        n_runs = int(rng.integers(50, 1500))
        syms = np.repeat(rng.choice(np.array([0, 1, 2, 3, 4, 5], np.uint8), n_runs, p=[.05, .22, .22, .22, .07, .22]),
                         rng.integers(1, 12, n_runs))
        g = _index(O.convert_to_vec(O.convert_itos(syms)), sb_shift)
        for k in KS:
            for t in MIN_COUNTS:
                for canonical in (False, True):
                    _check(g, k, t, canonical)


@pytest.mark.parametrize("layout", [
    dict(oct_index=1, final_index=1, suffix_table_s=12),
    dict(oct_index=1, final_index=0),
    dict(pair_index=1, quad_index=0, oct_index=0),
    dict(oct_index=1, final_index=1, superblock_shift=4),
])
def test_canonical_mode_under_every_layout(golden_dir, layout):
    """the rc counts of the canonical node list come from the query path, which each layout routes differently"""
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    ref = _index(z["rle"])
    g = M.RleBWT(**layout)
    g.load_vector(z["rle"])
    for k, t in ((21, 2), (31, 2), (32, 3)):
        _same(_check(g, k, t, True), ref.unitigs(k, t, True))


def test_canonical_strand_invariance():
    rng = np.random.default_rng(54)
    reads = _read_set(rng, [70] * 300)
    flipped = _revcomp_reads(reads, rng.random(len(reads)) < 0.5)
    g, h = _index(M.build_rle_bwt(np.stack(reads))[0]), _index(M.build_rle_bwt(np.stack(flipped))[0])
    for k in (5, 12, 21, 31, 32):
        for t in (1, 2, 3):
            _same(g.unitigs(k, t, True), h.unitigs(k, t, True))


def test_both_strand_index_filtered_by_the_keep_rule_is_canonical_mode():
    """odd k: the plain unitigs of an index of reads + their reverse complements, kept by the canonical rule, are the
    canonical unitigs of the reads alone, counts included"""
    rng = np.random.default_rng(55)
    reads = _read_set(rng, [70] * 300)
    both = _index(M.build_rle_bwt(np.stack(reads + _revcomp_reads(reads, [True] * len(reads))))[0])
    alone = _index(M.build_rle_bwt(np.stack(reads))[0])
    for k in (5, 13, 21, 31):
        for t in (1, 2, 4):
            syms, offs, sums = both.unitigs(k, t)
            V = set(both.list_kmers(k, t)[0].tolist())
            keep = []
            for i in range(offs.size - 1):
                w = U.windows(syms[offs[i]:offs[i + 1]], k)
                cycle = len(w) > 1 and U._succs(w[-1], k, V) == [w[0]] and U._preds(w[0], k, V) == [w[-1]]
                keep.append(min(w) <= min(U.revcomp(x, k) for x in w) if cycle else w[0] <= U.revcomp(w[-1], k))
            keep = np.array(keep, bool)
            lens = np.diff(offs)
            want_offs = np.concatenate([[0], np.cumsum(lens[keep])]).astype(np.uint64)
            want_syms = np.concatenate([syms[offs[i]:offs[i + 1]] for i in np.flatnonzero(keep)] or
                                       [np.zeros(0, np.uint8)])
            _same(alone.unitigs(k, t, True), (want_syms, want_offs, sums[keep]))


def _tiled(genome, read_len, step, circular=False):
    g = np.concatenate([genome, genome[:read_len]]) if circular else genome
    last = genome.size if circular else genome.size - read_len + 1
    starts = list(range(0, last, step)) + ([] if circular else [genome.size - read_len])
    return np.stack([LUT[g[a:a + read_len]] for a in starts])


def _repeat_free(rng, n, k, circular=False):
    while True:
        g = rng.integers(0, 4, n)
        s = np.concatenate([g, g[:k - 2]]) if circular else g
        v = np.zeros(s.size - k + 2, np.uint64)
        for j in range(k - 1):
            v = (v << np.uint64(2)) | s[j:j + v.size].astype(np.uint64)
        if np.unique(v).size == v.size:
            return g


def test_circular_genome_is_one_unitig():
    rng = np.random.default_rng(56)
    k = 31
    genome = _repeat_free(rng, 5000, k, circular=True)
    g = _index(M.build_rle_bwt(_tiled(genome, 100, 20, circular=True))[0])
    syms, offs, sums = _check(g, k, 1, False)
    assert offs.tolist() == [0, genome.size + k - 1]
    text = np.tile(genome, 3)
    start = np.flatnonzero([(LUT[text[i:i + genome.size + k - 1]] == syms).all() for i in range(genome.size)])
    assert start.size == 1


def test_error_free_tiling_of_a_repeat_free_genome_gives_the_genome(monkeypatch):
    """a 300 kbp genome: one unitig of 300 k nodes (19 pointer-jumping rounds), walked in small slices"""
    rng = np.random.default_rng(57)
    k = 31
    genome = _repeat_free(rng, 300_000, k)
    g = _index(M.build_rle_bwt(_tiled(genome, 150, 50))[0])
    monkeypatch.setenv("MSBWT_SPECTRUM_SLICE", "256")
    syms, offs, sums = g.unitigs(k, 1)
    assert offs.tolist() == [0, genome.size] and (syms == LUT[genome]).all()
    assert int(sums[0]) == int(g.list_kmers(k, 1)[1].sum())
    monkeypatch.delenv("MSBWT_SPECTRUM_SLICE")
    _same(g.unitigs(k, 1), (syms, offs, sums))


def test_bad_arguments_empty_results_and_repeats(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    L = M.load_library()
    s, o, c, n = C.c_void_p(7), C.c_void_p(7), C.c_void_p(7), C.c_uint64(7)
    args = (C.byref(s), C.byref(o), C.byref(c), C.byref(n))
    assert L.msbwt_unitigs(None, 5, 1, 0, *args) == EINVAL
    assert L.msbwt_unitigs(g.handle, 0, 1, 0, *args) == EINVAL
    assert L.msbwt_unitigs(g.handle, 33, 1, 0, *args) == EINVAL
    assert L.msbwt_unitigs(g.handle, 5, 0, 0, *args) == EINVAL
    assert L.msbwt_unitigs(g.handle, 5, 1, 2, *args) == EINVAL
    assert L.msbwt_unitigs(g.handle, 5, 1, -1, *args) == EINVAL
    for i in range(4):
        a = list(args)
        a[i] = None
        assert L.msbwt_unitigs(g.handle, 5, 1, 0, *a) == EINVAL
    assert s.value == o.value == c.value == 7 and n.value == 7  # nothing written
    with pytest.raises(M.MsbwtError):
        g.unitigs(33)
    # no node: n = 0 and NULL buffers
    assert L.msbwt_unitigs(g.handle, 5, 1 << 40, 1, *args) == 0
    assert not s.value and not o.value and not c.value and n.value == 0
    short = _index(M.build_rle_bwt(np.full((50, 20), 2, np.uint8))[0])
    for canonical in (False, True):
        syms, offs, sums = short.unitigs(21, 1, canonical)
        assert syms.size == 0 and offs.tolist() == [0] and sums.size == 0
    # repeat calls: identical arrays and an equal, positive launch count
    deltas = []
    for canonical in (False, True):
        for _ in range(2):
            before = L.msbwt_launch_count()
            got = g.unitigs(31, 2, canonical)
            deltas.append(L.msbwt_launch_count() - before)
            if _ == 0:
                first = got
        _same(first, got)
    assert deltas[0] == deltas[1] > 0 and deltas[2] == deltas[3] > 0


def test_concurrent_count_kmers_on_the_same_handle(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = _index(z["rle"])
    q, want = z["queries"], z["counts"]
    qq, ww = np.tile(q, (100, 1)), np.tile(want, 100)
    ref = g.unitigs(31, 1, True)
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
        for _ in range(10):
            got = g.unitigs(31, 1, True)
            if not all((x == y).all() for x, y in zip(got, ref)):
                errors.append("unitigs")
    finally:
        th.join()
    assert not errors, errors


def test_two_devices_give_the_same_result(golden_dir):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    one, two = _index(z["rle"]), _index(z["rle"], devices=[1, 0])
    for canonical in (False, True):
        _same(one.unitigs(31, 2, canonical), two.unitigs(31, 2, canonical))


def test_config3_full_size():
    """configs[2]: 10 M reads x 150 bp with 1 % errors from one 50 Mbp genome, k = 31, min_count 5"""
    import bench
    from harness import synth
    if torch.cuda.get_device_properties(0).total_memory < 150e9:
        pytest.skip("needs the 180 GB of a B200")
    cfg = bench.WORKLOADS["cfg3"]
    dev = torch.device("cuda:0")
    torch.cuda.empty_cache()
    reads, rle, total = bench.build_reads_and_bwt(cfg, dev, True)
    del reads
    k, t = 31, 5
    g = M.RleBWT.new(devices=[0])
    g.load_vector(rle)
    del rle
    syms, offs, sums = g.unitigs(k, t)
    lens = np.diff(offs).astype(np.int64)
    assert (lens >= k).all()
    assert int((lens - k + 1).sum()) == int(g.kmer_spectrum(k, t, 2)[1])

    # the genome, regenerated from the harness's seed, and the position of each of its 31-mers
    glen = max(cfg["read_len"], int(cfg["reads"] * cfg["read_len"] / cfg["coverage"]))
    gen = torch.Generator(device=dev)
    gen.manual_seed(synth.SEED_GENOME)
    genome = torch.randint(0, 4, (glen,), generator=gen, device=dev, dtype=torch.uint8)
    val = torch.zeros(glen - k + 1, dtype=torch.int64, device=dev)
    for j in range(k):
        val = (val << 2) | genome[j:j + val.numel()].long()
    sval, spos = torch.sort(val)
    # every unitig's first k-mer is a genome k-mer, and the unitig is the genome from there
    d_syms = torch.from_numpy(syms).to(dev)
    d_offs = torch.from_numpy(offs.view(np.int64)).to(dev)
    first = torch.zeros(lens.size, dtype=torch.int64, device=dev)
    code = torch.tensor([0, 0, 1, 2, 0, 3], dtype=torch.int64, device=dev)
    for j in range(k):
        first = (first << 2) | code[d_syms[d_offs[:-1] + j].long()]
    at = torch.searchsorted(sval, first).clamp(max=sval.numel() - 1)
    d_lens = torch.from_numpy(lens).to(dev)
    unitig_of = torch.repeat_interleave(torch.arange(lens.size, device=dev), d_lens)
    pos = spos[at][unitig_of] + torch.arange(int(lens.sum()), device=dev) - d_offs[:-1][unitig_of]
    lut = torch.tensor([1, 2, 3, 5], dtype=torch.uint8, device=dev)
    differs = lut[genome[pos.clamp(max=glen - 1)].long()] != d_syms
    wrong = torch.zeros(lens.size, dtype=torch.int64, device=dev).index_add_(0, unitig_of, differs.long())
    bad = ((sval[at] != first) | (wrong > 0)).cpu().numpy()
    # The exceptions are sequencing errors repeated at least min_count times: each such unitig holds a k-mer that is not
    # in the genome, and they are few.
    assert bad.sum() <= max(20, lens.size // 1000), (int(bad.sum()), lens.size)
    for i in np.flatnonzero(bad):
        w = torch.tensor(U.windows(syms[offs[i]:offs[i + 1]], k), dtype=torch.int64, device=dev)
        hit = torch.searchsorted(sval, w).clamp(max=sval.numel() - 1)
        assert not bool((sval[hit] == w).all()), i

    # a sample of the compaction conditions through count_kmers_u64: inside a unitig outdeg = indeg = 1
    rng = np.random.default_rng(6)
    mask = (1 << 62) - 1
    inner = np.flatnonzero(lens > k)
    pick = rng.choice(inner, min(2000, inner.size), replace=False)
    xs, ys = [], []
    for i in pick:
        w = U.windows(syms[offs[i]:offs[i] + k + 1], k)
        xs.append(w[0])
        ys.append(w[1])
    xs, ys = np.array(xs, np.uint64), np.array(ys, np.uint64)
    succ = np.stack([((xs << np.uint64(2)) & np.uint64(mask)) | np.uint64(c) for c in range(4)], 1)
    pred = np.stack([(ys >> np.uint64(2)) | np.uint64(c << 60) for c in range(4)], 1)
    assert ((g.count_kmers_u64(succ.reshape(-1), k).reshape(-1, 4) >= t).sum(1) == 1).all()
    assert ((g.count_kmers_u64(pred.reshape(-1), k).reshape(-1, 4) >= t).sum(1) == 1).all()
