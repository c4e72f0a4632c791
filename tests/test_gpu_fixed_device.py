"""The fixed-k device entry point (msbwt_count_kmers_fixed_device) on an index with an oct image: symbol bytes in
device memory, counts out.  It takes the one-request kernel (final_kernels.cu) where that applies -- 31- and
32-mers in a 16-byte aligned buffer with a final-step image -- and pack / seed + the search kernel (oct_kernel.cuh)
for every other k, table depth and alignment; k-mers holding `$` / `N` are seeded one symbol at a time.
Every count must equal BWT::count_kmer (src/msbwt_core.rs:125-161) as restated by the CPU oracle."""
import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def readset():
    from harness import bwt_build, synth
    reads = synth.make_reads(20000, read_len=100, coverage=25.0, error_rate=0.01, device="cuda")
    reads[17, 40:43] = 4
    rle, n = bwt_build.build_rle_bwt(reads)
    o = O.RleBWT()
    o.load_vector(rle.cpu().numpy())
    return reads, o


def run_device(g, q):
    n, k = q.shape
    out = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    g.count_kmers_fixed_device(q.data_ptr(), k, n, out.data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint64), int(status.item())


@pytest.mark.parametrize("table_s", [-1, 0, 3, 11, 12])
def test_fixed_device_counts_equal_the_oracle(readset, table_s):
    from harness import synth
    reads, o = readset
    g = M.RleBWT(suffix_table_s=table_s, oct_index=1)
    g.load_vector(o.rle_bytes())
    assert g.oct_index
    for k in (1, 2, 3, 4, 5, 7, 9, 10, 11, 12, 13, 14, 15, 19, 20, 21, 24, 29, 30, 31, 32):
        q = synth.make_queries(reads, k, 12001, 8000)          # read-sampled + random (mostly absent for large k)
        q[5, 0] = 4
        q[7, k - 1] = 0
        q[11, k // 2] = 4
        q[4000:4100, 0] = 4                                       # a run of exceptions
        got, status = run_device(g, q)
        want = o.count_kmers_fixed(q.cpu().numpy(), k, threads=8)
        assert status == 0
        assert (got == want).all(), (table_s, k, np.flatnonzero(got != want)[:5])
    # an unaligned batch takes pack / seed + search rather than the one-request kernel: same counts
    q = synth.make_queries(reads, 31, 5000, 5000)
    got, _ = run_device(g, q[1:])
    assert (got == o.count_kmers_fixed(q[1:].cpu().numpy(), 31, threads=8)).all()


def test_fixed_device_over_many_chunks_and_bad_symbols(readset):
    from harness import synth
    reads, o = readset
    g = M.RleBWT(oct_index=1)
    g.load_vector(o.rle_bytes())
    q = synth.make_queries(reads, 31, 1_500_000, 700_003)
    got, status = run_device(g, q)
    assert status == 0
    sel = np.random.default_rng(3).choice(q.shape[0], 300_000, replace=False)
    assert (got[sel] == o.count_kmers_fixed(q.cpu().numpy()[sel], 31, threads=8)).all()
    assert int((got > 0).sum()) >= 1_500_000                      # every read-sampled 31-mer occurs
    q[123, 4] = 6                                                  # not a symbol: flagged, as count_kmer panics
    _, status = run_device(g, q[:1000])
    assert status != 0
    # tiny batches
    for n in (1, 31, 32, 33, 511, 513):
        got, _ = run_device(g, q[200:200 + n])
        assert (got == o.count_kmers_fixed(q[200:200 + n].cpu().numpy(), 31)).all()
