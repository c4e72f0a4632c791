"""CPU restatements of msbwt_kmer_spectrum (TEST INFRASTRUCTURE ONLY): the k-mers of an index with count >= min_count,
their counts and the histogram of those counts, in the library's encoding and order.

  * from_reads: the definition for a BWT built from reads -- count every length-k window of the reads that holds no N
    (numpy, np.unique);
  * walk_rle / from_rle: the definition for any BWT -- a depth-first backward search over the C oracle's
    constrain_range (src/rle_bwt.rs:202-287) from [0, N), extending by A, C, G, T and dropping ranges narrower than
    min_count, so it covers BWTs that do not come from reads.

Encoding: A,C,G,T = 0..3, the first symbol in the most significant of the 2k bits (msbwt_count_kmers_u64's input).
Order: co-lexicographic -- ascending by the last symbol, then by the one before it, and so on."""
from __future__ import annotations

import numpy as np

from oracle import oracle as O

ACGT = (1, 2, 3, 5)
_CODE = np.full(256, 255, dtype=np.uint8)
_CODE[[1, 2, 3, 5]] = [0, 1, 2, 3]


def colex_key(kmers, k: int) -> np.ndarray:
    """the value with its k 2-bit groups reversed: ascending key = co-lexicographic order"""
    v = np.asarray(kmers, dtype=np.uint64)
    key = np.zeros_like(v)
    for j in range(k):
        key |= ((v >> np.uint64(2 * j)) & np.uint64(3)) << np.uint64(2 * (k - 1 - j))
    return key


def histogram(counts, nbins: int) -> np.ndarray:
    hist = np.zeros(nbins, dtype=np.uint64)
    if nbins:
        np.add.at(hist, np.minimum(np.asarray(counts, dtype=np.uint64), nbins - 1).astype(np.int64), 1)
    return hist


def pack_windows(reads, k: int) -> np.ndarray:
    """every length-k window of the reads (uint8 symbol arrays, any lengths) without N, packed as u64; reads of one
    length are packed together"""
    by_len: dict[int, list] = {}
    for r in reads:
        r = np.asarray(r, dtype=np.uint8).reshape(-1)
        if r.size >= k:
            by_len.setdefault(r.size, []).append(r)
    out = []
    for ln, group in by_len.items():
        codes = _CODE[np.stack(group)]
        w = ln - k + 1
        v = np.zeros((codes.shape[0], w), dtype=np.uint64)
        bad = np.zeros((codes.shape[0], w), dtype=bool)
        for j in range(k):
            c = codes[:, j:j + w]
            bad |= c == 255
            v = (v << np.uint64(2)) | (c & 3).astype(np.uint64)
        out.append(v[~bad])
    return np.concatenate(out) if out else np.zeros(0, np.uint64)


def from_reads(reads, k: int, min_count: int = 1, nbins: int = 0):
    """(hist, kmers, counts) from the reads themselves"""
    kmers, counts = np.unique(pack_windows(reads, k), return_counts=True)
    counts = counts.astype(np.uint64)
    keep = counts >= np.uint64(min_count)
    kmers, counts = kmers[keep], counts[keep]
    order = np.argsort(colex_key(kmers, k), kind="stable")
    return histogram(counts, nbins), kmers[order], counts[order]


def walk_rle(rle, kmax: int, min_count: int = 1):
    """[(kmers, counts) for k = 1..kmax]: one depth-first walk over constrain_range, emitting at every depth"""
    o = O.RleBWT()
    o.load_vector(rle)
    found = [([], []) for _ in range(kmax)]
    stack = [(0, 0, o.get_total_size(), 0)]  # (depth, l, h, value); children pushed T..A so that A pops first
    while stack:
        d, l, h, v = stack.pop()
        if d:
            found[d - 1][0].append(v)
            found[d - 1][1].append(h - l)
        if d == kmax:
            continue
        kids = []
        for code, sym in enumerate(ACGT):
            cl, ch = o.constrain_range(sym, l, h)
            if ch - cl >= min_count:
                kids.append((d + 1, cl, ch, v | code << (2 * d)))
        stack.extend(reversed(kids))
    return [(np.array(km, dtype=np.uint64), np.array(cn, dtype=np.uint64)) for km, cn in found]


def from_rle(rle, k: int, min_count: int = 1, nbins: int = 0):
    """(hist, kmers, counts) from any RLE stream"""
    kmers, counts = walk_rle(rle, k, min_count)[k - 1]
    return histogram(counts, nbins), kmers, counts
