"""Exact kernel-launch counts (`msbwt_launch_count`) of every public entry point, under every image layout, and the
verbatim messages of device-side input errors.

bench.py reports the launch count beside its rates, and a launch that a call forgets to count, or counts twice, goes
unnoticed anywhere else.  Each entry point runs once on a small seeded index of each layout, with pageable host
inputs (a pinned input would let the hybrid route pick its lanes by timing), and the host-pack switch set explicitly,
so that the route of every call, and with it the number of kernels it launches, is fixed."""
import contextlib
import os

import numpy as np
import pytest

import rust_msbwt_b200 as M
from harness import synth

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

K = 31
LAYOUTS = {
    "default": dict(),
    "pair": dict(pair_index=1, suffix_table_s=8),
    "quad": dict(quad_index=1, oct_index=0, suffix_table_s=9),
    "oct_final": dict(oct_index=1, final_index=1, suffix_table_s=12),
    "wide": dict(oct_index=1, final_index=1, superblock_shift=4, suffix_table_s=12),
}

# msbwt_launch_count() delta of creating the index of each layout, from RLE bytes or from a .npy file
EXPECTED_CREATE = {"default": 7, "pair": 27, "quad": 290, "oct_final": 312, "wide": 31}
# ... of each call of measure() below on it: the same under every layout (the search runs one kernel per live list,
# whichever image serves list A, and the one-request kernel replaces the pack kernel)
EXPECTED_CALLS = {
    "count_kmers": 1,
    "count_kmers_fixed": 3,
    "count_kmers_fixed_u32": 4,
    "count_kmers_fixed_k21": 3,
    "count_kmers_fixed_host_packed": 2,
    "count_kmers_fixed_u32_host_packed": 3,
    "count_kmers_u64": 2,
    "count_kmers_u64_u32": 3,
    "constrain_ranges": 1,
    "constrain_ranges_fanout": 1,
    "count_read_kmers": 4,
    "count_read_kmers_both_strands": 5,
    "kmer_spectrum": 34,
    "kmer_spectrum_canonical": 42,
    "list_kmers": 38,
    "list_kmers_canonical": 46,
    "count_kmers_fixed_device": 3,
    "pack_kmers_device": 1,
    "debug_pack_stats": 0,
    "count_kmers_packed_device": 2,
    "seed_kmers_u64_device": 1,
    "count_kmers_packed_device_after_seed": 2,
    "constrain_ranges_device": 1,
    "constrain_ranges_fanout_device": 1,
}
# the counting build of the oct kernel (count_kmers_packed_stats_device): oct images with 32-bit positions only
EXPECTED_STATS = {"oct_final": 1}
# the calls of measure_standalone() below, which build no index
EXPECTED_STANDALONE = {"build_rle_bwt": 25, "build_rle_bwt_ragged": 25, "merge_rle_bwts": 314, "gather_bench": 1}


@contextlib.contextmanager
def _env(name, value):
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        yield
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


def _data():
    reads = synth.np_make_reads(3000, 100, 20.0, 0.01, seed=11)
    q = synth.np_make_queries(reads, K, 4000, 2000, seed=12)  # 6000 queries: the host-pack route takes them
    q21 = synth.np_make_queries(reads, 21, 1500, 500, seed=13)
    code = np.zeros(6, np.uint64)
    code[[1, 2, 3, 5]] = [0, 1, 2, 3]
    u64 = np.zeros(q.shape[0], np.uint64)
    for j in range(K):
        u64 = (u64 << np.uint64(2)) | code[q[:, j]]
    rng = np.random.default_rng(14)
    varlen = [q[i, : int(rng.integers(0, K + 1))] for i in range(500)]
    return reads, q, q21, u64, varlen


def _last_error():
    return (M.load_library().msbwt_last_error() or b"").decode()


def _delta(fn):
    before = M.launch_count()
    fn()
    torch.cuda.synchronize()
    return M.launch_count() - before


def measure(layout, rle, data, npy_path):
    """{call: launches} of every entry point that takes an index, on an index of `layout`; returns (counts, index)"""
    reads, q, q21, u64, varlen = data
    L = M.load_library()
    g = M.RleBWT(devices=[0], **LAYOUTS[layout])
    got = {"create": _delta(lambda: g.load_vector(rle))}
    h = M.RleBWT(devices=[0], **LAYOUTS[layout])
    got["create_from_npy"] = _delta(lambda: h.load_numpy_file(npy_path))
    h.close()
    n = q.shape[0]
    lo = np.zeros(1000, np.uint64)
    hi = np.full(1000, g.get_total_size(), np.uint64)
    sym = np.resize(np.array([1, 2, 3, 5, 4, 0], np.uint8), 1000)
    with _env("MSBWT_HOST_PACK", "0"):
        got["count_kmers"] = _delta(lambda: g.count_kmers(varlen))
        got["count_kmers_fixed"] = _delta(lambda: g.count_kmers_fixed(q, K))
        got["count_kmers_fixed_u32"] = _delta(lambda: g.count_kmers_fixed(q, K, counts32=True))
        got["count_kmers_fixed_k21"] = _delta(lambda: g.count_kmers_fixed(q21, 21))
    with _env("MSBWT_HOST_PACK", "1"):
        got["count_kmers_fixed_host_packed"] = _delta(lambda: g.count_kmers_fixed(q, K))
        got["count_kmers_fixed_u32_host_packed"] = _delta(lambda: g.count_kmers_fixed(q, K, counts32=True))
    got["count_kmers_u64"] = _delta(lambda: g.count_kmers_u64(u64, K))
    got["count_kmers_u64_u32"] = _delta(lambda: g.count_kmers_u64(u64, K, counts32=True))
    got["constrain_ranges"] = _delta(lambda: g.constrain_ranges(sym, lo, hi))
    got["constrain_ranges_fanout"] = _delta(lambda: g.constrain_ranges_fanout(lo, hi))
    got["count_read_kmers"] = _delta(lambda: g.count_read_kmers(reads[:200], K))
    got["count_read_kmers_both_strands"] = _delta(lambda: g.count_read_kmers(reads[:200], K, both_strands=True))
    got["kmer_spectrum"] = _delta(lambda: g.kmer_spectrum(12, 1, 50))
    got["kmer_spectrum_canonical"] = _delta(lambda: g.kmer_spectrum(12, 1, 50, canonical=True))
    got["list_kmers"] = _delta(lambda: g.list_kmers(12, 2))
    got["list_kmers_canonical"] = _delta(lambda: g.list_kmers(12, 2, canonical=True))

    d_syms = torch.from_numpy(q).cuda().contiguous()
    d_kmers = torch.from_numpy(u64.view(np.int64)).cuda()
    d_out = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_status = torch.zeros(1, dtype=torch.int32, device="cuda")
    d_packed = torch.zeros(g.packed_bytes(K, n) // 8 + 1, dtype=torch.int64, device="cuda")
    d_l = torch.from_numpy(lo.view(np.int64)).cuda()
    d_h = torch.from_numpy(hi.view(np.int64)).cuda()
    d_sym = torch.from_numpy(sym).cuda()
    d_out_l = torch.zeros(4 * lo.size, dtype=torch.int64, device="cuda")
    d_out_h = torch.zeros(4 * lo.size, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    got["count_kmers_fixed_device"] = _delta(lambda: g.count_kmers_fixed_device(d_syms.data_ptr(), K, n, d_out.data_ptr()))
    got["pack_kmers_device"] = _delta(lambda: g.pack_kmers_device(d_syms.data_ptr(), K, n, d_packed.data_ptr(),
                                                                  d_out.data_ptr(), d_status.data_ptr()))
    got["debug_pack_stats"] = _delta(lambda: g.pack_stats(d_packed.data_ptr(), K, n))
    got["count_kmers_packed_device"] = _delta(lambda: g.count_kmers_packed_device(d_packed.data_ptr(), K, n, d_out.data_ptr()))
    got["seed_kmers_u64_device"] = _delta(lambda: g.seed_kmers_u64_device(d_kmers.data_ptr(), K, n, d_packed.data_ptr(),
                                                                          d_out.data_ptr()))
    got["count_kmers_packed_device_after_seed"] = _delta(
        lambda: g.count_kmers_packed_device(d_packed.data_ptr(), K, n, d_out.data_ptr()))
    if g.oct_index and layout != "wide":
        d_stats = torch.zeros(8, dtype=torch.int64, device="cuda")
        g.pack_kmers_device(d_syms.data_ptr(), K, n, d_packed.data_ptr(), d_out.data_ptr(), d_status.data_ptr())
        got["count_kmers_packed_stats_device"] = _delta(lambda: g.count_kmers_packed_stats_device(
            d_packed.data_ptr(), K, n, d_out.data_ptr(), d_stats.data_ptr()))
    got["constrain_ranges_device"] = _delta(lambda: g.constrain_ranges_device(
        d_sym.data_ptr(), d_l.data_ptr(), d_h.data_ptr(), lo.size, d_out_l.data_ptr(), d_out_h.data_ptr()))
    rc = []
    got["constrain_ranges_fanout_device"] = _delta(lambda: rc.append(L.msbwt_constrain_ranges_fanout_device(
        g.handle, 0, d_l.data_ptr(), d_h.data_ptr(), lo.size, d_out_l.data_ptr(), d_out_h.data_ptr(), None)))
    assert rc == [0], _last_error()
    return got, g


def measure_standalone(reads):
    """{call: launches} of the entry points that build no index"""
    ragged = [r[: 50 + i % 50] for i, r in enumerate(reads[:1000])]
    half = reads.shape[0] // 2
    rle_a, _ = M.build_rle_bwt(reads[:half])
    rle_b, _ = M.build_rle_bwt(reads[half:])
    buf = torch.zeros(1 << 22, dtype=torch.uint8, device="cuda")
    sink = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    return {
        "build_rle_bwt": _delta(lambda: M.build_rle_bwt(reads)),
        "build_rle_bwt_ragged": _delta(lambda: M.build_rle_bwt_ragged(ragged)),
        "merge_rle_bwts": _delta(lambda: M.merge_rle_bwts(rle_a, rle_b)),
        "gather_bench": _delta(lambda: M.gather_bench(0, buf.data_ptr(), buf.numel(), 128, 1 << 16, 5, sink.data_ptr())),
    }


@pytest.fixture(scope="module")
def index_data(tmp_path_factory):
    data = _data()
    rle, _ = M.build_rle_bwt(data[0])
    npy = str(tmp_path_factory.mktemp("launch_counts") / "index.npy")
    M.save_bwt_numpy(rle, npy)
    return rle, data, npy


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_every_entry_point_counts_its_launches(index_data, layout):
    rle, data, npy = index_data
    got, g = measure(layout, rle, data, npy)
    images = (g.pair_index, g.quad_index, g.oct_index, g.final_index)
    assert images == {"default": (False, False, False, False), "pair": (True, False, False, False),
                      "quad": (False, True, False, False), "oct_final": (False, True, True, True),
                      "wide": (False, False, True, True)}[layout]
    assert _last_error() == ""
    want = {"create": EXPECTED_CREATE[layout], "create_from_npy": EXPECTED_CREATE[layout], **EXPECTED_CALLS}
    if layout in EXPECTED_STATS:
        want["count_kmers_packed_stats_device"] = EXPECTED_STATS[layout]
    assert got == want


def test_standalone_entry_points_count_their_launches(index_data):
    assert measure_standalone(index_data[1][0]) == EXPECTED_STANDALONE


def test_merge_with_a_bad_input_b_names_it():
    rle_a, _ = M.build_rle_bwt(synth.np_make_reads(20, 30, 2.0, 0.0, seed=15))
    with pytest.raises(M.MsbwtError) as e:
        M.merge_rle_bwts(rle_a, np.array([9, 14], np.uint8))  # 14 = symbol 6
    assert e.value.code == 3
    assert _last_error() == "input B: RLE stream has a symbol >= 6 or a run longer than 2^60 symbols"
    M.merge_rle_bwts(rle_a, rle_a)
    assert _last_error() == ""


def test_bwt_build_of_a_read_holding_a_terminator_says_so():
    reads = np.full((4, 10), 2, np.uint8)
    reads[2, 5] = 0
    with pytest.raises(M.MsbwtError) as e:
        M.build_rle_bwt(reads)
    assert e.value.code == 1
    assert _last_error() == "bwt build: a read holds '$' (0) or a symbol >= 6"
