"""CPU restatements of msbwt_kmer_spectrum_canonical (TEST INFRASTRUCTURE ONLY): the canonical k-mers of an index, their
canonical counts and the histogram of those counts, in the library's encoding.

  rc(X)    : the k 2-bit groups of X reversed, each code c mapped to 3 - c;
  canon(X) : min(X, rc(X));
  C(X)     : count_kmer(X) + count_kmer(rc(X)), or count_kmer(X) alone when X == rc(X) (a palindrome, even k only).

  * canonical_from_reads: the definition for a BWT built from reads -- canon of every N-free length-k window, then
    np.unique (each window adds 1 to exactly one canonical k-mer);
  * canonical_from_rle: the definition for any BWT -- oracle.spectrum.walk_rle at min_count 1, with the count of each
    k-mer's reverse complement looked up in the same walk (an absent one counts 0).

Both return (hist, kmers, counts) with the k-mers ascending; the library promises no order, so tests compare sets."""
from __future__ import annotations

import numpy as np

from oracle import spectrum as S


def revcomp_u64(kmers, k: int) -> np.ndarray:
    v = np.asarray(kmers, dtype=np.uint64)
    r = np.zeros_like(v)
    for j in range(k):
        r |= (np.uint64(3) - ((v >> np.uint64(2 * j)) & np.uint64(3))) << np.uint64(2 * (k - 1 - j))
    return r


def _finish(kmers, counts, min_count: int, nbins: int):
    keep = counts >= np.uint64(min_count)
    kmers, counts = kmers[keep], counts[keep]
    order = np.argsort(kmers, kind="stable")
    return S.histogram(counts, nbins), kmers[order], counts[order]


def canonical_from_reads(reads, k: int, min_count: int = 1, nbins: int = 0):
    """(hist, kmers, counts) from the reads themselves"""
    w = S.pack_windows(reads, k)
    kmers, counts = np.unique(np.minimum(w, revcomp_u64(w, k)), return_counts=True)
    return _finish(kmers, counts.astype(np.uint64), min_count, nbins)


def canonical_from_walk(kmers, counts, k: int, min_count: int = 1, nbins: int = 0):
    """(hist, kmers, counts) from every k-mer of count >= 1 and its count (walk_rle's output at min_count 1)"""
    kmers = np.asarray(kmers, dtype=np.uint64)
    counts = np.asarray(counts, dtype=np.uint64)
    order = np.argsort(kmers)
    kmers, counts = kmers[order], counts[order]
    rc = revcomp_u64(kmers, k)
    pos = np.searchsorted(kmers, rc).clip(max=max(kmers.size - 1, 0))
    c_rc = np.where(kmers[pos] == rc, counts[pos], np.uint64(0)) if kmers.size else counts
    pal = kmers == rc
    total = np.where(pal, counts, counts + c_rc)
    # one member per pair: the canonical one, or the other when the canonical one does not occur
    stands = (kmers <= rc) | (c_rc == 0)
    return _finish(np.minimum(kmers, rc)[stands], total[stands], min_count, nbins)


def canonical_from_rle(rle, k: int, min_count: int = 1, nbins: int = 0):
    """(hist, kmers, counts) from any RLE stream"""
    kmers, counts = S.walk_rle(rle, k, 1)[k - 1]
    return canonical_from_walk(kmers, counts, k, min_count, nbins)
