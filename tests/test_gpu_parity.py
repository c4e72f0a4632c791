"""Parity tests proper: the CUDA path, called through the C ABI (include/msbwt_gpu.h via
the RleBWT mirror), against the CPU oracle on the same inputs -- bit-exact (u64 counts /
positions).  The cases follow the reference's own tests (file:line in the reference, rust-msbwt)."""
import itertools

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import naive
from oracle import oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def both(rle, **kw):
    g = M.RleBWT(**kw)
    g.load_vector(rle)
    o = O.RleBWT()
    o.load_vector(rle)
    return g, o


def from_strings(strings, **kw):
    return both(O.convert_to_vec(naive.naive_bwt(strings)), **kw)


def test_library_is_the_cuda_one_and_device_present():
    assert torch.cuda.is_available()
    assert M.load_library().msbwt_abi_version() == 4


# ---- test_data/two_string.npy (config 1): rle_bwt.rs:76-79, README.md:62-70 ----
def test_config1_two_string_all_kmers(two_string_npy):
    g = M.RleBWT.new()
    g.load_numpy_file(two_string_npy)
    o = O.RleBWT()
    o.load_numpy_file(two_string_npy)
    assert g.get_total_size() == o.get_total_size() == 10
    for s in range(6):
        assert g.get_symbol_count(s) == o.get_symbol_count(s)
    assert g.count_kmer(M.convert_stoi("ACGT")) == 1
    assert g.count_kmer(M.convert_stoi("TGCA")) == 1
    assert g.count_kmer(M.convert_stoi("$")) == 2
    launches0 = M.launch_count()
    nonzero, total = [], 0
    for k in range(1, 9):
        qs = np.array(list(itertools.product([1, 2, 3, 5], repeat=k)), dtype=np.uint8)
        got = g.count_kmers_fixed(qs, k)
        assert (got == o.count_kmers_fixed(qs, k)).all()
        nonzero.append(int((got > 0).sum()))
        total += len(qs)
    assert total == 87380 and nonzero == [4, 6, 4, 2, 0, 0, 0, 0]
    assert M.launch_count() > launches0  # the answers came from kernel launches
    # k-mers through $ and N, every 6-ary 1..3-mer
    for k in range(1, 4):
        qs = np.array(list(itertools.product(range(6), repeat=k)), dtype=np.uint8)
        assert (g.count_kmers_fixed(qs, k) == o.count_kmers_fixed(qs, k)).all()


# ---- rle_bwt.rs:601-675 ----
@pytest.mark.parametrize("sb_shift", [0, 1])
def test_constrain_range_every_position(sb_shift):
    g, o = from_strings(["CCGT", "N", "ACG"], superblock_shift=sb_shift)
    n = g.get_total_size()
    assert n == 11
    for sym in range(6):
        r = g.constrain_range(sym, M.BWTRange(0, n))
        assert (r.l, r.h) == (o.start_index(sym), o.end_index(sym))
    sym, lo, hi = [], [], []
    for s in range(6):
        for ind in range(n + 1):
            sym += [s, s]
            lo += [0, ind]
            hi += [ind, n]
    gl, gh = g.constrain_ranges(sym, lo, hi)
    for i in range(len(sym)):
        assert (int(gl[i]), int(gh[i])) == o.constrain_range(sym[i], lo[i], hi[i])


# ---- rle_bwt.rs:677-710, dynamic_bwt.rs:702-773, msbwt_core.rs:110-122 ----
def test_count_kmer_kats():
    data = ["CCGTACGTA", "GGTACAGTA", "ACGACGACG"]
    g, _ = from_strings(data)
    for c in range(6):
        assert g.count_kmer([c]) == g.get_symbol_count(c)
    for s in data:
        assert g.count_kmer(M.convert_stoi(s)) == 1
    assert g.count_kmer(M.convert_stoi("ACG")) == 4
    assert g.count_kmer(M.convert_stoi("CC")) == 1
    assert g.count_kmer(M.convert_stoi("TAC")) == 2
    g4, _ = from_strings(data + ["AAGTCATAT"])
    assert g4.count_kmer(M.convert_stoi("AA")) == 1
    assert g4.count_kmer(M.convert_stoi("GT")) == 5
    d, _ = both(O.convert_to_vec("TG$$CAGCCG"))
    assert d.get_total_size() == 10 and d.get_symbol_count(0) == 2
    assert d.count_kmer([1, 2, 3, 5]) == 1
    assert d.count_kmer([2, 3]) == 2
    assert d.count_kmer([]) == 10  # empty k-mer -> total_size


def test_invalid_symbol_is_refused_like_the_reference_assert():
    g, _ = from_strings(["ACGT", "TGCA"])
    with pytest.raises(M.MsbwtError) as e:
        g.count_kmer([1, 6])
    assert e.value.code == 1
    with pytest.raises(M.MsbwtError):
        g.count_kmers([[1, 2], [7]])
    with pytest.raises(M.MsbwtError):
        g.constrain_ranges([6], [0], [1])
    with pytest.raises(M.MsbwtError):
        g.constrain_ranges([1], [3], [2])
    with pytest.raises(M.MsbwtError):
        g.constrain_ranges([1], [0], [11])
    with pytest.raises(M.MsbwtError) as e:
        M.RleBWT().load_vector([9, 14])
    assert e.value.code == 3
    assert g.count_kmer([1, 2]) == 1  # handle still healthy


def _random_rle(rng, nruns, choices):
    syms, counts, prev = [], [], -1
    for _ in range(nruns):
        s = int(rng.choice(6, p=[0.05, 0.27, 0.25, 0.25, 0.03, 0.15]))
        if s == prev:
            continue
        prev = s
        syms.append(s)
        counts.append(int(rng.choice(choices)))
    return O.encode_runs(syms, counts)


@pytest.mark.parametrize("sb_shift", [0, 1, 4])
def test_random_streams_ranges_and_ragged_kmers(sb_shift):
    rng = np.random.default_rng(4242 + sb_shift)
    rle = _random_rle(rng, 30000, [1, 1, 1, 2, 3, 5, 9, 31, 32, 33, 255, 256, 257, 1025, 3104])
    g, o = both(rle, superblock_shift=sb_shift)
    n = o.get_total_size()
    assert g.get_total_size() == n
    m = 50000
    sym = rng.integers(0, 6, m).astype(np.uint8)
    a = rng.integers(0, n + 1, m)
    b = rng.integers(0, n + 1, m)
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    hi[:1000] = np.minimum(lo[:1000] + rng.integers(0, 40, 1000), n)  # narrow ranges: same-block path
    lo[-5:], hi[-5:] = [0, n, 0, n - 1, 255], [0, n, n, n, 256]
    gl, gh = g.constrain_ranges(sym, lo, hi)
    for i in range(m):
        assert (int(gl[i]), int(gh[i])) == o.constrain_range(int(sym[i]), int(lo[i]), int(hi[i])), i
    # ragged batch incl. empty k-mers and symbols $ / N
    kmers = [rng.integers(0, 6, int(rng.integers(0, 70))).astype(np.uint8) for _ in range(4000)]
    kmers[0] = np.zeros(0, np.uint8)
    kmers[-1] = np.zeros(0, np.uint8)
    assert (g.count_kmers(kmers) == o.count_kmers(kmers)).all()
    assert (g.count_kmers([]) == np.zeros(0, np.uint64)).all()


@pytest.mark.parametrize("table_s", [0, 1, 2, 3, 5, 7])
def test_suffix_table_depths_are_bit_exact(table_s):
    """The suffix table (the reference's planned kmer_cache, msbwt_core.rs:133-146) must not change a
    single count: k < s, k == s, k > s, k-mers with $ / N inside and outside the last s symbols."""
    rng = np.random.default_rng(77)
    reads = rng.choice(np.array([1, 2, 3, 4, 5], dtype=np.uint8), size=(300, 40), p=[0.28, 0.22, 0.22, 0.03, 0.25])
    from harness import bwt_build
    rle, _ = bwt_build.build_rle_bwt(torch.from_numpy(reads).cuda())
    for sb in (0, 2):
        g, o = both(rle.cpu().numpy(), suffix_table_s=table_s, superblock_shift=sb)
        assert g.suffix_table_s == table_s
        for k in (1, 2, 3, 4, 5, 6, 7, 8, 9, 22, 30):
            a = reads[rng.integers(0, 300, 400)][:, 5:5 + k] if k <= 30 else None
            b = rng.integers(0, 6, (300, k)).astype(np.uint8)
            q = np.concatenate([a, b, rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), (300, k))])
            assert (g.count_kmers_fixed(q, k) == o.count_kmers_fixed(q, k)).all(), (table_s, sb, k)
        kmers = [rng.integers(0, 6, int(rng.integers(0, 12))).astype(np.uint8) for _ in range(500)]
        assert (g.count_kmers(kmers) == o.count_kmers(kmers)).all()


def test_automatic_suffix_table_is_on_for_real_sizes(midsize):
    reads, g, o = midsize
    assert g.suffix_table_s == 8  # ceil(log4(2.02e6 / 32))


@pytest.mark.parametrize("lanes", [1, 2])
def test_both_kernel_mappings_are_bit_exact(lanes, monkeypatch, midsize, golden_dir):
    """LANES=1 (thread per query) and LANES=2 (lane pair per query) over the same block image."""
    from harness import synth
    reads, _, o = midsize
    monkeypatch.setenv("MSBWT_LANES", str(lanes))
    for sb, ts in ((0, -1), (3, 5), (0, 0)):
        g = M.RleBWT(superblock_shift=sb, suffix_table_s=ts)
        g.load_vector(o.rle_bytes())
        assert g.kernel_lanes == lanes
        for k in (1, 12, 31, 50):
            q = synth.make_queries(reads, k, 20001, 20000).cpu().numpy()
            q[5, 0] = 4
            q[7, k - 1] = 0
            assert (g.count_kmers_fixed(q, k) == o.count_kmers_fixed(q, k, threads=8)).all(), (lanes, sb, ts, k)
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g = M.RleBWT()
    g.load_vector(z["rle"])
    assert (g.count_kmers_fixed(z["queries"], 31) == z["counts"]).all()


def test_empty_bwt():
    g, o = both(np.zeros(0, np.uint8))
    assert g.get_total_size() == 0
    assert g.count_kmer([]) == 0 and g.count_kmer([1, 2, 3]) == 0
    r = g.constrain_range(1, M.BWTRange(0, 0))
    assert (r.l, r.h) == o.constrain_range(1, 0, 0)


@pytest.fixture(scope="module")
def midsize():
    from harness import bwt_build, synth
    reads = synth.make_reads(20000, read_len=100, coverage=25.0, error_rate=0.01, device="cuda")
    reads[17, 40:43] = 4  # a few N
    rle, n = bwt_build.build_rle_bwt(reads)
    rle = rle.cpu().numpy()
    g, o = both(rle)
    assert g.get_total_size() == n == 20000 * 101
    return reads, g, o


@pytest.mark.parametrize("k", [1, 15, 21, 22, 31, 42, 43, 63, 100])
def test_midsize_synthetic_fixed_k(midsize, k):
    from harness import synth
    reads, g, o = midsize
    q = synth.make_queries(reads, k, 30000, 30000).cpu().numpy()
    got = g.count_kmers_fixed(q, k)
    want = o.count_kmers_fixed(q, k, threads=8)
    assert (got == want).all()
    assert (got > 0).sum() >= 30000  # every read-sampled k-mer is present


def test_device_pointer_entry_matches_host_entry(midsize):
    from harness import synth
    reads, g, o = midsize
    k = 31
    q = synth.make_queries(reads, k, 50000, 50000)
    want = g.count_kmers_fixed(q.cpu().numpy(), k)
    out = torch.zeros(q.shape[0], dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    g.count_kmers_fixed_device(q.data_ptr(), k, q.shape[0], out.data_ptr(), status.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    assert (out.cpu().numpy().astype(np.uint64) == want).all()
    q[123, 5] = 6
    g.count_kmers_fixed_device(q.data_ptr(), k, q.shape[0], out.data_ptr(), status.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert int(status.item()) != 0


def test_golden_fixture(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    g, _ = both(z["rle"])
    assert g.get_total_size() == int(z["total"])
    assert (g.count_kmers_fixed(z["queries"], int(z["k"])) == z["counts"]).all()
    assert (g.count_kmers_fixed(z["queries_k12"], 12) == z["counts_k12"]).all()


def test_built_bwt_saved_as_npy_loads_back_with_the_requested_layout(midsize, tmp_path):
    """N1: the product writes msbwt2's container itself (codec.cpp, src/bwt_converter.rs:102-130) and
    load_numpy_file honours the layout knobs (msbwt_index_create_from_npy_opts)"""
    from harness import synth
    reads, g, o = midsize
    p = str(tmp_path / "built.npy")
    M.save_bwt_numpy(o.rle_bytes(), p)
    o2 = O.RleBWT()
    o2.load_numpy_file(p)                      # the oracle's reader accepts the file
    assert o2.get_total_size() == o.get_total_size()
    q = synth.make_queries(reads, 31, 20001, 10000).cpu().numpy()
    want = o.count_kmers_fixed(q, 31, threads=8)
    for opts in (dict(), dict(pair_index=1, suffix_table_s=5), dict(oct_index=1, final_index=0), dict(oct_index=1, keep_quad_index=0)):
        b = M.RleBWT(**opts)
        b.load_numpy_file(p)
        assert b.get_total_size() == o.get_total_size()
        if "pair_index" in opts:
            assert b.pair_index and b.suffix_table_s == 5
        if "oct_index" in opts:
            assert b.oct_index and b.final_index == (opts.get("final_index", -1) != 0)
            assert b.quad_index == (opts.get("keep_quad_index", 1) != 0)
        assert (b.count_kmers_fixed(q, 31) == want).all(), opts


def test_multi_device_split_matches_single(midsize):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from harness import synth
    reads, g, o = midsize
    q = synth.make_queries(reads, 31, 40001, 20000).cpu().numpy()
    g2 = M.RleBWT(devices=[0, 1])
    g2.load_vector(o.rle_bytes())
    assert g2.device_ordinals == [0, 1]
    assert (g2.count_kmers_fixed(q, 31) == g.count_kmers_fixed(q, 31)).all()


def test_full_size_config1_properties():
    """BASELINE.json configs[1] at full size (1 M x 150-bp reads, 151 Msymbol BWT, 31-mers): properties that
    need no oracle at scale, plus an oracle comparison on a sample.
      * partition: count(Q) == sum over the six symbols c of count(cQ)   (constrain_range splits a range)
      * every read-sampled k-mer occurs at least once; counts are permutation-equivariant
      * host-buffer path == device-buffer path (checksum of checksums)"""
    from harness import bwt_build, synth
    reads = synth.make_reads(1_000_000, 150, 30.0, 0.0, device="cuda")
    rle, total = bwt_build.build_rle_bwt(reads)
    rle = rle.cpu().numpy()
    g = M.RleBWT.new()
    g.load_vector(rle)
    assert g.get_total_size() == total == 151_000_000
    # 219 MB of one-step blocks + depth-12 table exceed L2: the loader builds the quad and oct images and deepens
    # the table (to 14 under the oct image: levels 11..14 are kept, a 31-mer starts from the L2-resident depth 11)
    assert g.quad_index and g.oct_index and g.suffix_table_s == 14
    k = 30
    q = synth.make_queries(reads, k, 600_000, 400_000)
    base = g.count_kmers_fixed(q.cpu().numpy(), k)
    assert int((base > 0).sum()) >= 600_000
    ext_sum = np.zeros_like(base)
    for c in range(6):
        ext = torch.cat([torch.full((q.shape[0], 1), c, dtype=torch.uint8, device=q.device), q], dim=1).contiguous()
        ext_sum += g.count_kmers_fixed(ext.cpu().numpy(), k + 1)
    assert (ext_sum == base).all()
    perm = torch.randperm(q.shape[0], device=q.device)
    assert (g.count_kmers_fixed(q[perm].contiguous().cpu().numpy(), k) == base[perm.cpu().numpy()]).all()
    out = torch.zeros(q.shape[0], dtype=torch.int64, device="cuda")
    g.count_kmers_fixed_device(q.data_ptr(), k, q.shape[0], out.data_ptr(), 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert int(out.sum().item()) == int(base.astype(np.int64).sum())
    o = O.RleBWT()
    o.load_vector(rle)
    m = 200_000
    assert (base[:m] == o.count_kmers_fixed(q[:m].cpu().numpy(), k, threads=8)).all()
    for s in range(6):
        assert g.get_symbol_count(s) == o.get_symbol_count(s)


def _kmers_that_occur(o, syms, ends, rng, k, m):
    """m k-mers with count >= 1 in ANY symbol stream: the symbols B[j], B[LF j], .. of a walk from a random position j
    are what count_kmer consumes, last symbol first (src/msbwt_core.rs:148-155), so reversed they are a k-mer whose
    range still holds the walk's end.  LF from the oracle's constrain_range; walks that meet `$` / N are dropped."""
    n = int(ends[-1])
    out = []
    while len(out) < m:
        p = int(rng.integers(0, n))
        walk = []
        for _ in range(k):
            s = int(syms[np.searchsorted(ends, np.int64(p), side="right")])  # (`ends` is int64: no per-call conversion)
            if s in (0, 4):
                break
            walk.append(s)
            p = o.constrain_range(s, p, p)[0]
        if len(walk) == k:
            out.append(walk[::-1])
    return np.array(out, dtype=np.uint8)


def test_wide_index_beyond_2_pow_32_symbols():
    """Maximum-size edge: N > 2^32 (u64 positions, two default-size superblocks).  Any RLE stream is a legal
    index, so a 4.6 Gsymbol one is made from ~4.6 M long runs; ranges and k-mer counts must match the
    oracle at positions on both sides of 2^32.  The index lives in HBM, so the automatic layout is the oct and
    final-step images with 40-bit checkpoints, built by walking LF through the one-step blocks and searched by the
    WIDE instantiation of the oct kernel (VERDICT r1 item 7); the pair image it replaced is checked beside it."""
    torch.cuda.empty_cache()
    rng = np.random.default_rng(2032)
    nruns = 4_600_000
    syms = rng.choice(np.array([0, 1, 2, 3, 4, 5], dtype=np.uint8), size=nruns, p=[0.02, 0.26, 0.24, 0.24, 0.02, 0.22])
    keep = np.ones(nruns, dtype=bool)
    keep[1:] = syms[1:] != syms[:-1]
    syms = syms[keep]
    counts = rng.integers(1, 2800, size=syms.size).astype(np.uint64)
    rle = O.encode_runs(syms, counts)
    g, o = both(rle)
    n = o.get_total_size()
    assert n > (1 << 32) and g.get_total_size() == n
    assert g.oct_index and g.final_index and not g.quad_index and not g.pair_index and g.suffix_table_s == 14
    m = 200_000
    sym = rng.integers(0, 6, m).astype(np.uint8)
    lo = rng.integers(0, n + 1, m).astype(np.uint64)
    width = rng.choice(np.array([0, 1, 5, 100, 4000, 1 << 20, 1 << 33], dtype=np.uint64), m)
    hi = np.minimum(lo + width, np.uint64(n))
    lo[:4], hi[:4] = [0, (1 << 32) - 1, 1 << 32, n], [n, (1 << 32) + 1, (1 << 32) + 7, n]
    gl, gh = g.constrain_ranges(sym, lo, hi)
    for i in range(0, m, 37):
        assert (int(gl[i]), int(gh[i])) == o.constrain_range(int(sym[i]), int(lo[i]), int(hi[i])), i
    for i in range(4):
        assert (int(gl[i]), int(gh[i])) == o.constrain_range(int(sym[i]), int(lo[i]), int(hi[i])), i
    pair = M.RleBWT(oct_index=0)  # the layout of such an index before the wide oct image existed
    pair.load_vector(rle)
    assert pair.pair_index and not pair.oct_index
    for k in (3, 9, 24):
        q = rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(100_000, k))
        q[::97, 0] = 4
        want = o.count_kmers_fixed(q, k, threads=8)
        assert (g.count_kmers_fixed(q, k) == want).all(), k
        assert (pair.count_kmers_fixed(q, k) == want).all(), k
    # k-mers that occur (walks of LF from random positions: half of them start beyond 2^32), through every kind of
    # step of the wide kernel: oct lines (k = 24, 44), a final-step line (31..34), both (45, 63, 70), remainders
    ends = np.cumsum(counts.astype(np.int64))
    for k in (24, 31, 32, 34, 44, 45, 63, 70):
        q = np.concatenate([_kmers_that_occur(o, syms, ends, rng, k, 600),
                            rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(500, k))])
        want = o.count_kmers_fixed(q, k, threads=8)
        assert int((want[:600] > 0).sum()) == 600
        got = g.count_kmers_fixed(q, k)
        assert (got == want).all(), (k, np.flatnonzero(got != want)[:5])
        assert (pair.count_kmers_fixed(q, k) == want).all(), k
    ragged = [rng.integers(0, 6, int(rng.integers(0, 9))).astype(np.uint8) for _ in range(3000)]
    assert (g.count_kmers(ragged) == o.count_kmers(ragged)).all()
    del g, pair
    torch.cuda.empty_cache()


@pytest.mark.parametrize("sb_shift", [0, 2])
def test_device_built_image_equals_host_built_image(sb_shift):
    """The GPU builder (builder.cu: scan / select / fill / stamp) must produce exactly the block image the
    serial host builder (loader.cu) produces: words, $/N side array and superblock bases."""
    rng = np.random.default_rng(515 + sb_shift)
    streams = [
        _random_rle(rng, 40000, [1, 1, 1, 2, 3, 5, 9, 31, 32, 33, 255, 256, 257, 1025, 3104, 40000]),
        O.encode_runs([1, 2, 1, 0, 4, 5], [128, 128, 1, 127, 3104, 5]),
        np.array([1, 9, 25, 10, 2, 2, 10, 11, 0, 8], dtype=np.uint8),  # zero low digits and zero-length runs
        O.convert_to_vec("A"),
        np.zeros(0, np.uint8),
    ]
    from harness import bwt_build, synth
    reads = synth.make_reads(3000, 80, 20.0, 0.02, device="cuda")
    streams.append(bwt_build.build_rle_bwt(reads)[0].cpu().numpy())
    for rle in streams:
        hb, ha, hc = M.debug_build_image(rle, sb_shift)
        g = M.RleBWT(superblock_shift=sb_shift)
        g.load_vector(rle)
        db, da, dc = g.device_image()
        assert db.shape == hb.shape and (db == hb).all()
        assert (da == ha).all()
        assert dc.shape == hc.shape and (dc == hc).all()
        o = O.RleBWT()
        o.load_vector(rle)
        assert g.get_total_size() == o.get_total_size()
        assert [g.get_symbol_count(s) for s in range(6)] == [o.get_symbol_count(s) for s in range(6)]
        assert [g.start_index(s) for s in range(6)] == [o.start_index(s) for s in range(6)]
