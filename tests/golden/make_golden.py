"""Regenerates the committed golden fixtures.  Run from the repo root:

    python tests/golden/make_golden.py

two_string.npy    -- byte-identical to the reference fixture test_data/two_string.npy
                     (strings ACGT, TGCA; payload [13,9,10,8,11,9,13,10,11,8]); produced
                     with the oracle's own naive_bwt -> convert_to_vec -> save_bwt_numpy.
                     tests/test_oracle_kat.py pins its SHA-256.
reads30x_k31.npz  -- 3000 synthetic 100-bp reads (30x, 1% substitutions, one read with N),
                     their msbwt RLE stream, 3000 31-mers + 3000 12-mers (half read-sampled,
                     half random) and the counts the pinned CPU oracle gives for them.
                     The reference itself cannot run here (Rust-only, no cargo), so these
                     vectors are oracle outputs; the oracle is pinned by tests/test_oracle_kat.py.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from harness import bwt_build, synth  # noqa: E402
from oracle import naive  # noqa: E402
from oracle import oracle as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    p = os.path.join(HERE, "two_string.npy")
    O.save_bwt_numpy(O.convert_to_vec(naive.naive_bwt(["ACGT", "TGCA"])), p)

    reads = synth.np_make_reads(3000, 100, 30.0, 0.01, seed=20261018)
    reads[11, 50:52] = 4
    rle, total = bwt_build.build_rle_bwt(torch.from_numpy(reads))
    rle = rle.numpy()
    q31 = synth.np_make_queries(reads, 31, 1500, 1500, seed=1)
    q12 = synth.np_make_queries(reads, 12, 1500, 1500, seed=2)
    b = O.RleBWT()
    b.load_vector(rle)
    assert b.get_total_size() == total
    c31 = b.count_kmers_fixed(q31, 31)
    c12 = b.count_kmers_fixed(q12, 12)
    assert (c31 > 0).sum() >= 1500
    np.savez_compressed(os.path.join(HERE, "reads30x_k31.npz"), rle=rle, total=np.uint64(total), k=np.uint32(31),
                        queries=q31, counts=c31, queries_k12=q12, counts_k12=c12)
    print("reads30x_k31.npz:", total, "symbols,", rle.size, "RLE bytes, checksum", int(c31.sum()), int(c12.sum()))


if __name__ == "__main__":
    main()
