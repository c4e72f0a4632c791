"""Every entry point where a 32-bit quantity reaches 2^32.

Below 2^32 symbols with one superblock the kernels run on 32-bit positions (Pos<false>: u32 suffix-table entries,
checkpoints, C and counts); everything else runs on 64-bit ones.  Two indexes straddle that switch:

  * N1 = 2^32 - 1, the largest 32-bit index: its one superblock is exactly full, u32 counts are accepted and the empty
    k-mer counts 0xFFFFFFFF;
  * N2 = 2^32, the smallest 64-bit index: its second superblock holds position N alone and u32 counts are refused.

Both come from one seeded generator of run tables: an A run longer than 2^31 inside the A range (so that A^k counts
pass 2^31 for small k), about 4 M short random runs, and a last run that crosses 2^32 - 128 and ends at N.  Ranges are
checked against a rank reference computed from the run table alone in exact integers; counts against the C oracle,
which the CPU test below first checks against that reference at this size.

Also here, at their own 2^32 edges: the BWT builder's 64-bit suffix ids (a ragged read set whose
n_reads * (longest + 1) reaches 2^32), and the pileup of one read whose expanded windows pass 2^32 bytes.

The GPU tests need the 180 GB of a B200; they keep one large index alive at a time."""
import ctypes as C
import re

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import canonical_spectrum as CS
from oracle import oracle as O
from oracle import spectrum as S
from oracle import unitigs as U

N1 = (1 << 32) - 1
N2 = 1 << 32
LONG_A = (1 << 31) + (1 << 29)   # the A run: count(A^k) stays above 2^31 for small k
TAIL = 300                       # the last run: crosses 2^32 - 128 and ends at N
EINVAL = 1
RC_SYM = np.array([0, 5, 3, 2, 4, 1], np.uint8)  # $ A C G N T -> their complements ($ and N stay)
ACGT = np.array([1, 2, 3, 5], np.uint8)
CODE = np.full(256, 255, np.uint8)
CODE[ACGT] = [0, 1, 2, 3]


# ---------------------------------------------------------------- inputs and the run-table reference

def make_runs(n: int, seed: int) -> tuple[np.ndarray, np.ndarray]:
    """(syms u8, counts u64) of a run table of exactly n symbols with no two neighbouring runs of one symbol:
    ~200 k short random runs, the long A run, short random runs up to N - TAIL, then the last run"""
    rng = np.random.default_rng(seed)

    def short(m):
        return (rng.choice(6, size=m, p=[0.02, 0.26, 0.24, 0.24, 0.02, 0.22]).astype(np.uint8),
                rng.integers(1, 800, size=m, dtype=np.int64))

    s1, c1 = short(200_000)   # ~80 M symbols, more than C[A] (~30 M): the long run starts inside the A range
    s2, c2 = short(4_200_000)
    fill = n - LONG_A - TAIL - int(c1.sum())
    cum = np.cumsum(c2)
    j = int(np.searchsorted(cum, fill))
    assert j < cum.size
    s2, c2 = s2[:j + 1], c2[:j + 1].copy()
    c2[j] -= int(cum[j]) - fill
    syms = np.concatenate([s1, [1], s2, [3]]).astype(np.uint8)
    counts = np.concatenate([c1, [LONG_A], c2, [TAIL]]).astype(np.int64)
    head = np.flatnonzero(np.r_[True, syms[1:] != syms[:-1]])
    syms, counts = syms[head], np.add.reduceat(counts, head)
    assert int(counts.sum()) == n
    return syms, counts.astype(np.uint64)


class RunRank:
    """rank(s, p) = occurrences of s in B[0, p), from the run table alone: per-symbol run starts and cumulative
    lengths, searchsorted, exact int64.  Independent of the C oracle and of the device."""

    def __init__(self, syms, counts):
        c = counts.astype(np.int64)
        self.syms = syms
        self.ends = np.cumsum(c)
        self.n = int(self.ends[-1])
        starts = self.ends - c
        self.start, self.len, self.cum = [], [], []
        for s in range(6):
            m = syms == s
            self.start.append(starts[m])
            self.len.append(c[m])
            self.cum.append(np.concatenate([[0], np.cumsum(c[m])]))
        self.count = [int(x[-1]) for x in self.cum]
        self.C = [sum(self.count[:s]) for s in range(6)]
        assert all(self.count)

    def rank(self, s: int, p) -> np.ndarray:
        p = np.asarray(p, np.int64)
        j = np.searchsorted(self.start[s], p, side="left") - 1   # the last s-run that starts before p
        jj = np.maximum(j, 0)
        r = self.cum[s][jj] + np.minimum(self.len[s][jj], p - self.start[s][jj])
        return np.where(j >= 0, r, 0)

    def constrain(self, sym, l, h) -> tuple[np.ndarray, np.ndarray]:
        sym, l, h = np.asarray(sym), np.asarray(l, np.int64), np.asarray(h, np.int64)
        out_l, out_h = np.empty_like(l), np.empty_like(h)
        for s in range(6):
            m = sym == s
            out_l[m] = self.C[s] + self.rank(s, l[m])
            out_h[m] = self.C[s] + self.rank(s, h[m])
        return out_l, out_h

    def walks(self, starts, length: int) -> np.ndarray:
        """[m, length]: B[p], B[LF p], .. from every start, reversed -- strings whose count is at least 1
        (count_kmer consumes a k-mer last symbol first, src/msbwt_core.rs:148-155)"""
        p = np.asarray(starts, np.int64)
        out = np.empty((p.size, length), np.uint8)
        for t in range(length):
            s = self.syms[np.searchsorted(self.ends, p, side="right")]
            out[:, length - 1 - t] = s
            p, _ = self.constrain(s, p, p)
        return out


def edge_ranges(n: int, rng, m: int = 200_000):
    """(sym, l, h): endpoints at the 2^31 and 2^32 edges crossed with widths on both sides, then m random ranges"""
    ends = [0, (1 << 31) - 1, 1 << 31, (1 << 31) + 1, (1 << 32) - 129, (1 << 32) - 128, (1 << 32) - 2, n - 1, n]
    widths = [0, 1, 5, 100, 4000, 1 << 20, 1 << 31, n]
    lo, hi = [], []
    for p in ends:
        for w in widths:
            lo += [p, max(p - w, 0)]
            hi += [min(p + w, n), p]
    lo, hi = np.array(lo * 6, np.uint64), np.array(hi * 6, np.uint64)
    sym = np.repeat(np.arange(6, dtype=np.uint8), lo.size // 6)
    rl = rng.integers(0, n + 1, m).astype(np.uint64)
    rw = rng.choice(np.array(widths, np.uint64), m)
    rh = np.minimum(rl + rw, np.uint64(n))
    return (np.concatenate([sym, rng.integers(0, 6, m).astype(np.uint8)]), np.concatenate([lo, rl]),
            np.concatenate([hi, rh]))


def stream(n: int, seed: int):
    syms, counts = make_runs(n, seed)
    ref = RunRank(syms, counts)
    rle = O.encode_runs(syms, counts)
    return rle, ref


@pytest.fixture(scope="module")
def n1():
    return stream(N1, 4_294_967)


@pytest.fixture(scope="module")
def n2():
    return stream(N2, 4_294_968)


def _oracle(rle):
    o = O.RleBWT()
    o.load_vector(rle)
    return o


@pytest.mark.parametrize("which", ["n1", "n2"])
def test_stream_shape_and_oracle_equals_run_table(which, request):
    """The generator makes what the GPU tests rely on, and the C oracle's constrain_range equals the run-table reference
    at this size, with a run longer than 2^31 -- before the oracle is trusted for k-mer counts."""
    rle, ref = request.getfixturevalue(which)
    n = N1 if which == "n1" else N2
    assert ref.n == n
    starts = ref.ends - np.diff(np.r_[0, ref.ends])
    long_run = int(np.argmax(np.diff(np.r_[0, ref.ends])))
    ls, le = int(starts[long_run]), int(ref.ends[long_run])
    assert ref.syms[long_run] == 1 and le - ls > (1 << 31)
    assert ref.C[1] <= ls and le <= ref.C[1] + ref.count[1]               # inside the A range
    for edge in (1 << 31, (1 << 32) - 128):                               # runs that cross both edges
        r = int(np.searchsorted(ref.ends, edge, side="right"))
        assert starts[r] < edge < ref.ends[r]
    assert ref.n - int(starts[-1]) >= TAIL and 1_000_000 < ref.syms.size < 10_000_000
    o = _oracle(rle)
    assert o.get_total_size() == n
    assert [o.get_symbol_count(s) for s in range(6)] == ref.count
    assert [o.start_index(s) for s in range(6)] == ref.C
    rng = np.random.default_rng(7)
    sym, lo, hi = edge_ranges(n, rng, 20_000)
    want_l, want_h = ref.constrain(sym, lo, hi)
    for i in range(sym.size):
        assert o.constrain_range(int(sym[i]), int(lo[i]), int(hi[i])) == (int(want_l[i]), int(want_h[i])), i


# ---------------------------------------------------------------- GPU checks shared by both indexes

def _need_b200():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available() or torch.cuda.get_device_properties(0).total_memory < 150e9:
        pytest.skip("needs the 180 GB of a B200")
    torch.cuda.empty_cache()
    return torch


def _image_sizes(g) -> tuple[int, int]:
    nb, ns = C.c_uint64(0), C.c_uint32(0)
    assert M.load_library().msbwt_debug_copy_image(g.handle, 0, C.byref(nb), C.byref(ns), None, None, None) == 0
    return nb.value, ns.value


def check_ranges(torch, g, ref, rng):
    """constrain_ranges, _device, _fanout and _fanout_device: every range equals the run-table reference"""
    sym, lo, hi = edge_ranges(ref.n, rng)
    want_l, want_h = ref.constrain(sym, lo, hi)
    gl, gh = g.constrain_ranges(sym, lo, hi)
    assert (gl.astype(np.int64) == want_l).all() and (gh.astype(np.int64) == want_h).all()
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    d_sym = torch.from_numpy(sym).to(dev)
    d_lo, d_hi = (torch.from_numpy(x.view(np.int64)).to(dev) for x in (lo, hi))
    d_ol, d_oh = torch.full_like(d_lo, -1), torch.full_like(d_hi, -1)
    g.constrain_ranges_device(d_sym.data_ptr(), d_lo.data_ptr(), d_hi.data_ptr(), sym.size, d_ol.data_ptr(),
                              d_oh.data_ptr(), stream)
    torch.cuda.synchronize()
    assert (d_ol.cpu().numpy() == want_l).all() and (d_oh.cpu().numpy() == want_h).all()
    fl, fh = g.constrain_ranges_fanout(lo, hi)
    d_fl = torch.full((lo.size, 4), -1, dtype=torch.int64, device=dev)
    d_fh = torch.full_like(d_fl, -1)
    assert M.load_library().msbwt_constrain_ranges_fanout_device(g.handle, 0, d_lo.data_ptr(), d_hi.data_ptr(), lo.size,
                                                                 d_fl.data_ptr(), d_fh.data_ptr(), None) == 0
    torch.cuda.synchronize()
    dfl, dfh = d_fl.cpu().numpy(), d_fh.cpu().numpy()
    for c, s in enumerate(ACGT):
        wl, wh = ref.constrain(np.full(lo.size, s), lo, hi)
        assert (fl[:, c].astype(np.int64) == wl).all() and (fh[:, c].astype(np.int64) == wh).all(), s
        assert (dfl[:, c] == wl).all() and (dfh[:, c] == wh).all(), s


def kmer_batch(ref, rng, k: int) -> np.ndarray:
    """k-mers that occur (LF walks from [2^31, N), $ and N included), A^k, random ACGT k-mers, and k-mers holding
    $ or N; more than 4096 so that the host-packed route is taken when asked for"""
    occ = ref.walks(rng.integers(1 << 31, ref.n, 3000), k)
    rnd = rng.choice(ACGT, size=(3000, k))
    dn = rng.choice(ACGT, size=(1000, k))
    dn[np.arange(1000), rng.integers(0, k, 1000)] = rng.choice(np.array([0, 4], np.uint8), 1000)
    return np.concatenate([occ, np.ones((4, k), np.uint8), rnd, dn])


def encode_u64(q: np.ndarray) -> np.ndarray:
    v = np.zeros(q.shape[0], np.uint64)
    for j in range(q.shape[1]):
        v = (v << np.uint64(2)) | CODE[q[:, j]].astype(np.uint64)
    return v


def check_counts(torch, g, o, ref, rng, monkeypatch, narrow: bool, ks) -> int:
    """Every k-mer entry point against the C oracle; returns how many compared counts lie in (2^31, 2^32) for
    k = 1, 2, 3"""
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    big = 0
    for k in ks:
        q = kmer_batch(ref, rng, k)
        n = q.shape[0]
        want = o.count_kmers_fixed(q, k, threads=8)
        assert (want[:3000] >= 1).all() and (want[3000:3004] == want[3000]).all()
        if k <= 3:
            big += int(((want > (1 << 31)) & (want < (1 << 32))).sum())
        for host_pack in ("0", "1"):
            monkeypatch.setenv("MSBWT_HOST_PACK", host_pack)
            got = g.count_kmers_fixed(q, k)
            assert (got == want).all(), (k, host_pack, np.flatnonzero(got != want)[:5])
            if narrow:
                assert (g.count_kmers_fixed(q, k, counts32=True) == want).all(), (k, host_pack)
        monkeypatch.delenv("MSBWT_HOST_PACK")
        d_q = torch.from_numpy(q).to(dev)
        d_out = torch.full((n,), -1, dtype=torch.int64, device=dev)
        d_status = torch.zeros(1, dtype=torch.int32, device=dev)
        g.count_kmers_fixed_device(d_q.data_ptr(), k, n, d_out.data_ptr(), d_status.data_ptr(), stream)
        torch.cuda.synchronize()
        assert int(d_status.item()) == 0 and (d_out.cpu().numpy().view(np.uint64) == want).all(), k
        d_packed = torch.empty(g.packed_bytes(k, n) // 8, dtype=torch.int64, device=dev)
        d_out.fill_(-1)
        g.pack_kmers_device(d_q.data_ptr(), k, n, d_packed.data_ptr(), d_out.data_ptr(), d_status.data_ptr(), stream)
        g.count_kmers_packed_device(d_packed.data_ptr(), k, n, d_out.data_ptr(), stream)
        torch.cuda.synchronize()
        assert int(d_status.item()) == 0 and (d_out.cpu().numpy().view(np.uint64) == want).all(), k
        if k <= 32:
            acgt = np.flatnonzero((CODE[q] != 255).all(axis=1))
            keys, w = encode_u64(q[acgt]), want[acgt]
            assert (g.count_kmers_u64(keys, k) == w).all(), k
            if narrow:
                assert (g.count_kmers_u64(keys, k, counts32=True) == w).all(), k
            d_keys = torch.from_numpy(keys.view(np.int64)).to(dev)
            d_packed = torch.empty(g.packed_bytes(k, keys.size) // 8, dtype=torch.int64, device=dev)
            d_o = torch.full((keys.size,), -1, dtype=torch.int64, device=dev)
            g.seed_kmers_u64_device(d_keys.data_ptr(), k, keys.size, d_packed.data_ptr(), d_o.data_ptr(), stream)
            g.count_kmers_packed_device(d_packed.data_ptr(), k, keys.size, d_o.data_ptr(), stream)
            torch.cuda.synchronize()
            assert (d_o.cpu().numpy().view(np.uint64) == w).all(), k
        del d_q, d_out, d_packed
    ragged = [rng.integers(0, 6, int(rng.integers(0, 12))).astype(np.uint8) for _ in range(3000)]
    ragged += [np.zeros(0, np.uint8), np.ones(7, np.uint8), np.ones(1, np.uint8)]
    want = o.count_kmers(ragged)
    assert (want[-3] == ref.n) and want[-2] > (1 << 31)
    assert (g.count_kmers(ragged) == want).all()
    return big


def check_pileup(g, o, ref, rng):
    """count_read_kmers on reads made of LF walks and an all-A read, on both strands: the oracle on the same windows"""
    reads = np.concatenate([ref.walks(rng.integers(0, ref.n, 400), 80), np.ones((1, 80), np.uint8)])
    for k in (1, 3, 31):
        win = np.lib.stride_tricks.sliding_window_view(reads, k, axis=1).reshape(-1, k)
        fwd = o.count_kmers_fixed(win, k, threads=8)
        rev = o.count_kmers_fixed(RC_SYM[win[:, ::-1]], k, threads=8)
        assert (g.count_read_kmers(reads, k).reshape(-1) == fwd).all(), k
        assert (g.count_read_kmers(reads, k, both_strands=True).reshape(-1) == fwd + rev).all(), k
        assert fwd[-1] > (1 << 31) if k <= 3 else fwd[-1] >= 1


def check_spectrum_and_unitigs(g, o, ref):
    """kmer_spectrum, list_kmers, their canonical forms and unitigs (both modes) from the oracle's counts of all 4^k
    k-mers, at thresholds 1, 2^31, N and N + 1"""
    for k in (1, 2, 3, 6):
        allk = np.arange(4 ** k, dtype=np.uint64)
        syms = ACGT[((allk[:, None] >> (2 * np.arange(k - 1, -1, -1, dtype=np.uint64))) & np.uint64(3)).astype(np.int64)]
        cnt = o.count_kmers_fixed(syms, k, threads=8)
        occ = cnt > 0
        for t in (1, 1 << 31, ref.n, ref.n + 1):
            keep = cnt >= t
            order = np.argsort(S.colex_key(allk[keep], k), kind="stable")
            want_km, want_cn = allk[keep][order], cnt[keep][order]
            assert (g.kmer_spectrum(k, t, nbins=64) == S.histogram(want_cn, 64)).all(), (k, t)
            km, cn = g.list_kmers(k, t)
            assert (km == want_km).all() and (cn == want_cn).all(), (k, t)
            ch, ckm, ccn = CS.canonical_from_walk(allk[occ], cnt[occ], k, t, 64)
            assert (g.kmer_spectrum(k, t, nbins=64, canonical=True) == ch).all(), (k, t)
            km, cn = g.list_kmers(k, t, canonical=True)
            order = np.argsort(km)
            assert (km[order] == ckm).all() and (cn[order] == ccn).all(), (k, t)
            assert keep.any() == (t <= (1 << 31))    # A^k passes 2^31; no k-mer reaches N
            for canonical, (vk, vc) in ((False, (want_km, want_cn)), (True, (ckm, ccn))):
                order = np.argsort(vk)
                got = g.unitigs(k, t, canonical)
                want = U.unitigs(vk[order], vc[order], k, canonical)
                for x, y in zip(got, want):
                    assert x.dtype == y.dtype and x.shape == y.shape and (x == y).all(), (k, t, canonical)
        assert int(cnt[0]) > (1 << 31)   # A^k


def check_image(g, rle):
    hb, ha, hc = M.debug_build_image(rle)
    db, da, dc = g.device_image()
    assert db.shape == hb.shape and (db == hb).all()
    assert (da == ha).all()
    assert dc.shape == hc.shape and (dc == hc).all()


KS = (1, 2, 3, 9, 24, 31, 32, 45)


def _ks(g):
    s = g.suffix_table_s
    return KS + ((s,) if s and s not in KS else ())


# ---------------------------------------------------------------- N1 = 2^32 - 1

N1_LAYOUTS = {
    "auto": {},
    "no_pair_no_table": dict(pair_index=0, suffix_table_s=0),
    "no_pair_one_lane_table5": dict(pair_index=0, kernel_lanes=1, suffix_table_s=5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(N1_LAYOUTS))
def test_largest_32bit_index(layout, n1, monkeypatch):
    torch = _need_b200()
    rle, ref = n1
    o = _oracle(rle)
    g = M.RleBWT(**N1_LAYOUTS[layout])
    g.load_vector(rle)
    try:
        assert g.get_total_size() == N1
        assert [g.get_symbol_count(s) for s in range(6)] == ref.count
        assert [g.start_index(s) for s in range(6)] == ref.C
        assert _image_sizes(g)[1] == 1                          # narrow: one superblock
        assert not g.quad_index and not g.oct_index
        if layout == "auto":
            assert g.pair_index and g.suffix_table_s == 15 and g.kernel_lanes == 2, \
                (g.pair_index, g.suffix_table_s, g.kernel_lanes)
            assert g.pair_image()[1].shape[0] == 0              # no c2base rows below 2^32
        else:
            assert not g.pair_index
            assert g.suffix_table_s == N1_LAYOUTS[layout]["suffix_table_s"]
            if "kernel_lanes" in N1_LAYOUTS[layout]:
                assert g.kernel_lanes == 1
        rng = np.random.default_rng(101)
        check_ranges(torch, g, ref, rng)
        assert check_counts(torch, g, o, ref, rng, monkeypatch, True, _ks(g)) > 0
        if layout == "auto":
            check_pileup(g, o, ref, rng)
            check_spectrum_and_unitigs(g, o, ref)
            check_image(g, rle)
    finally:
        g.close()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------- N2 = 2^32

@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["auto", "pair"])
def test_smallest_64bit_index(layout, n2, monkeypatch):
    torch = _need_b200()
    rle, ref = n2
    o = _oracle(rle)
    g = M.RleBWT(**({} if layout == "auto" else dict(oct_index=0)))
    g.load_vector(rle)
    try:
        assert g.get_total_size() == N2
        assert [g.get_symbol_count(s) for s in range(6)] == ref.count
        assert _image_sizes(g)[1] == 2                          # wide: position N alone in the second superblock
        if layout == "auto":
            assert g.oct_index and g.final_index and not g.quad_index and not g.pair_index
        else:
            assert g.pair_index and not g.oct_index
        for call in (lambda: g.count_kmers_fixed(np.ones(31, np.uint8), 31, counts32=True),
                     lambda: g.count_kmers_u64(np.zeros(1, np.uint64), 31, counts32=True)):
            with pytest.raises(M.MsbwtError) as e:
                call()
            assert e.value.code == EINVAL
            assert "32-bit counts need an index below 2^32 symbols (a count can reach total_size)" in str(e.value)
        rng = np.random.default_rng(202)
        check_ranges(torch, g, ref, rng)
        assert check_counts(torch, g, o, ref, rng, monkeypatch, False, _ks(g)) > 0
        if layout == "auto":
            check_pileup(g, o, ref, rng)
            check_spectrum_and_unitigs(g, o, ref)
            check_image(g, rle)
    finally:
        g.close()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------- the BWT builder's 64-bit suffix ids

def _count_in_reads(joined: bytes, w: np.ndarray) -> int:
    return sum(1 for _ in re.finditer(b"(?=" + re.escape(w.tobytes()) + b")", joined))


@pytest.mark.gpu
@pytest.mark.parametrize("n_reads,longest", [(65_537, 65_534), (65_536, 65_535)])
def test_ragged_build_at_the_suffix_id_switch(n_reads, longest):
    """Suffix ids are u32 while n_reads * (longest + 1) < 2^32 and u64 from there (bwt_build.cu); the two sets
    straddle that switch exactly (2^32 - 1 = 65537 * 65535).  The whole set must build to exactly the BWT the merge of
    two parts below the switch gives, and the result must count sampled windows as the reads hold them."""
    torch = _need_b200()
    assert n_reads * (longest + 1) == N1 + (n_reads == 65_536)
    rng = np.random.default_rng(n_reads)
    lens = rng.integers(20, 151, n_reads)
    lens[0] = longest
    reads = [rng.choice(np.array([1, 2, 3, 4, 5], np.uint8), int(n), p=[0.25, 0.25, 0.25, 0.01, 0.24]) for n in lens]
    whole, total = M.build_rle_bwt_ragged(reads)
    assert total == int(lens.sum()) + n_reads
    a, _ = M.build_rle_bwt_ragged(reads[:200])
    b, _ = M.build_rle_bwt_ragged(reads[200:])
    merged, mtotal, _ = M.merge_rle_bwts(a, b)
    assert mtotal == total and merged.shape == whole.shape and (merged == whole).all()
    o = _oracle(whole)
    assert o.get_total_size() == total
    joined = b"\x09".join(r.tobytes() for r in reads)
    for k in (1, 12, 40):
        wins = [reads[0][p:p + k] for p in rng.integers(0, longest - k, 60)]
        wins += [reads[int(i)][:k] for i in rng.integers(1, n_reads, 60) if lens[int(i)] >= k]
        for w in wins:
            assert o.count_kmer(w) == _count_in_reads(joined, w), (k, w)
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- pileup of one read beyond 2^32 window bytes

@pytest.mark.gpu
@pytest.mark.parametrize("k,strands", [(100, 2), (200, 1)])
def test_pileup_of_one_read_past_2_pow_32_window_bytes(k, strands):
    """One 22 Mbp read at k = 100 on both strands (and k = 200 on one) lays out (windows * strands * k) > 2^32 bytes
    on the device; every window's count must equal count_kmers_fixed of the same window laid out on the host.  The
    index is 60x coverage of a random 100 kbp circle and the read walks that circle, so windows occur with counts
    that differ from window to window: a window copied from the wrong place would not go unnoticed."""
    torch = _need_b200()
    rng = np.random.default_rng(k)
    circle = rng.choice(ACGT, 100_003)
    ring = np.concatenate([circle, circle[:400]])
    starts = rng.integers(0, circle.size, 20_000)
    idx_reads = ring[starts[:, None] + np.arange(300)]
    rle, _ = M.build_rle_bwt(idx_reads)
    g = M.RleBWT()
    g.load_vector(rle)
    try:
        read = np.resize(circle, 22_000_000)
        read[rng.integers(0, read.size, 20)] = 4
        got = g.count_read_kmers(read[None, :], k, both_strands=strands == 2).reshape(-1)
        windows = read.size - k + 1
        assert got.size == windows and windows * strands * k > (1 << 32)
        first_far = ((1 << 32) - (1 << 20)) // (strands * k)
        sample = np.union1d(np.arange(first_far, windows), rng.choice(first_far, 1_000_000, replace=False))
        view = np.lib.stride_tricks.sliding_window_view(read, k)

        def counts(w):
            q = np.ascontiguousarray(view[w])
            c = g.count_kmers_fixed(q, k)
            return c + g.count_kmers_fixed(RC_SYM[q[:, ::-1]], k) if strands == 2 else c

        want = np.concatenate([counts(sample[i:i + 500_000]) for i in range(0, sample.size, 500_000)])
        bad = np.flatnonzero(got[sample] != want)
        assert bad.size == 0, (bad.size, sample[bad[:5]], got[sample[bad[:5]]], want[bad[:5]])
        assert np.unique(want).size > 10                        # counts differ from window to window
        o = _oracle(rle)
        few = rng.choice(sample, 50_000, replace=False)
        q = np.ascontiguousarray(view[few])
        ow = o.count_kmers_fixed(q, k, threads=8)
        if strands == 2:
            ow = ow + o.count_kmers_fixed(RC_SYM[q[:, ::-1]], k, threads=8)
        assert (got[few] == ow).all()
    finally:
        g.close()
        torch.cuda.empty_cache()
