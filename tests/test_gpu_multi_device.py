"""The in-library multi-GPU dispatcher (SURVEY §8e, north_star item 4): ONE handle created with `devices=[0, 1]`
replicates the index on both devices, cuts every batch into contiguous slices, and gathers the results on the
host into disjoint slices of the caller's output -- no collective.  `RleBWT` queries borrow `&self`
(src/rle_bwt.rs:14-24: only owned Vec fields, immutable after load), so every route must return exactly what a
one-device handle and the CPU oracle return.  Needs two GPUs; skipped on a machine with one."""
import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

CODE = np.zeros(6, dtype=np.uint64)
CODE[[1, 2, 3, 5]] = [0, 1, 2, 3]


def encode(syms: np.ndarray) -> np.ndarray:
    out = np.zeros(syms.shape[0], dtype=np.uint64)
    for j in range(syms.shape[1]):
        out = (out << np.uint64(2)) | CODE[syms[:, j]]
    return out


@pytest.fixture(scope="module")
def two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from harness import bwt_build, synth
    reads = synth.make_reads(20000, read_len=100, coverage=25.0, error_rate=0.01, device="cuda:0")
    reads[17, 40:43] = 4
    rle, total = bwt_build.build_rle_bwt(reads)
    o = O.RleBWT()
    o.load_vector(rle.cpu().numpy())
    return reads, o, total


OPTS = [dict(), dict(pair_index=1), dict(quad_index=1), dict(oct_index=1), dict(suffix_table_s=0)]


@pytest.mark.parametrize("opts", OPTS)
@pytest.mark.parametrize("host_pack", ["0", "1"])
def test_fixed_routes_two_devices(two_gpus, monkeypatch, opts, host_pack):
    """byte route (MSBWT_HOST_PACK=0) and packed route (=1) over two replicas, several chunks per device, with
    exceptions ($/N) sprinkled in; k straddles the 32-symbol word boundary"""
    from harness import synth
    reads, o, _ = two_gpus
    monkeypatch.setenv("MSBWT_HOST_THREADS", "4")
    monkeypatch.setenv("MSBWT_HOST_PACK", host_pack)
    g2 = M.RleBWT(devices=[0, 1], **opts)
    g2.load_vector(o.rle_bytes())
    assert g2.device_ordinals == [0, 1]
    for k, n in ((31, 1_300_003), (12, 50_001), (33, 70_000), (1, 17), (100, 20_001)):
        q = synth.make_queries(reads, k, n - n // 3, n // 3).cpu().numpy()
        q[5, 0] = 4
        q[min(7, n - 1), k - 1] = 0
        m = min(n, 200_000)
        got = g2.count_kmers_fixed(q, k)
        assert got.shape == (n,)
        assert (got[:m] == o.count_kmers_fixed(q[:m], k, threads=8)).all(), (opts, k)
        assert (got[-m:] == o.count_kmers_fixed(q[-m:], k, threads=8)).all(), (opts, k)


def test_two_devices_equal_one_device_on_every_entry_point(two_gpus, monkeypatch):
    from harness import synth
    reads, o, total = two_gpus
    g1 = M.RleBWT(devices=[1], oct_index=1)
    g1.load_vector(o.rle_bytes())
    g2 = M.RleBWT(devices=[0, 1], oct_index=1)
    g2.load_vector(o.rle_bytes())
    assert g1.device_ordinals == [1]
    k = 31
    q = synth.make_queries(reads, k, 700_001, 300_000).cpu().numpy()
    want = g1.count_kmers_fixed(q, k)
    assert (want[:100_000] == o.count_kmers_fixed(q[:100_000], k, threads=8)).all()
    assert (g2.count_kmers_fixed(q, k) == want).all()
    # hybrid route: the caller's buffer is pinned, raw and packed chunks interleave
    monkeypatch.setenv("MSBWT_HOST_PACK", "1")
    qp = torch.from_numpy(q).pin_memory()
    assert (g2.count_kmers_fixed(qp.numpy(), k) == want).all()
    monkeypatch.delenv("MSBWT_HOST_PACK")
    # ragged entry (count_kmers(&[Vec<u8>])): uniform lengths take the fixed-k routes, mixed lengths the byte kernel
    kmers = [q[i] for i in range(5000)] + [q[i, : 1 + i % 31] for i in range(5000)] + [np.zeros(0, np.uint8)]
    rag = g2.count_kmers(kmers)
    assert (rag[:5000] == want[:5000]).all()
    assert rag[-1] == total
    for i in (5000, 5001, 5030, 7777, 9999):
        assert rag[i] == o.count_kmer(kmers[i])
    # u64 entry
    acgt = np.isin(q, (1, 2, 3, 5)).all(axis=1)
    qa = q[acgt][:600_001]
    assert (g2.count_kmers_u64(encode(qa), k) == want[acgt][:600_001]).all()
    # constrain_ranges + fan-out
    rng = np.random.default_rng(7)
    n = 300_001
    l = rng.integers(0, total + 1, n).astype(np.uint64)
    h = rng.integers(0, total + 1, n).astype(np.uint64)
    l, h = np.minimum(l, h), np.maximum(l, h)
    sym = rng.integers(0, 6, n).astype(np.uint8)
    a = g1.constrain_ranges(sym, l, h)
    b = g2.constrain_ranges(sym, l, h)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    for i in range(0, n, 30011):
        assert (int(b[0][i]), int(b[1][i])) == o.constrain_range(int(sym[i]), int(l[i]), int(h[i]))
    fa = g1.constrain_ranges_fanout(l, h)
    fb = g2.constrain_ranges_fanout(l, h)
    assert (fa[0] == fb[0]).all() and (fa[1] == fb[1]).all()
    # pileup
    r = reads[:3000].cpu().numpy()
    pa = g1.count_read_kmers(r, k, both_strands=True)
    pb = g2.count_read_kmers(r, k, both_strands=True)
    assert (pa == pb).all()
    win = np.ascontiguousarray(np.lib.stride_tricks.sliding_window_view(r[:40], k, axis=1)).reshape(-1, k)
    fwd = o.count_kmers_fixed(win, k)
    rev = o.count_kmers_fixed(np.stack([M.reverse_complement_i(w) for w in win]), k)
    assert (pb[:40].reshape(-1) == fwd + rev).all()


def test_invalid_symbol_on_second_device_slice(two_gpus):
    """validation happens before any output is produced, wherever the bad k-mer sits"""
    from harness import synth
    reads, o, _ = two_gpus
    g2 = M.RleBWT(devices=[0, 1])
    g2.load_vector(o.rle_bytes())
    q = synth.make_queries(reads, 31, 900_000, 100_000).cpu().numpy()
    q[-3, 4] = 9
    with pytest.raises(M.MsbwtError) as e:
        g2.count_kmers_fixed(q, 31)
    assert e.value.code == 1
    q[-3, 4] = 1
    assert (g2.count_kmers_fixed(q, 31)[-1000:] == o.count_kmers_fixed(q[-1000:], 31)).all()
