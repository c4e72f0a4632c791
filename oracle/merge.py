"""Holt-McMillan merge of two multi-string BWTs, restated in numpy (TEST INFRASTRUCTURE ONLY).

The reference's pairwise_bwt_merge (src/bwt_util.rs:108-141) interleaves the rows of two BWTs until the interleave
stops changing:

    I_0     = all of A's rows (0), then all of B's (1)
    I_{t+1} = walk I_t in order, take each row's symbol from its source (the next unread symbol of that input) and
              append the row's source bit to that symbol's bucket; bucket c starts at C_A[c] + C_B[c]

i.e. one stable bucket pass (a stable sort of I_t by the rows' symbols) per iteration.  At the fixed point the merged
BWT is each row's symbol taken in that order.  `iterations` counts every pass, the last one (which changed nothing)
included, as msbwt_merge_rle_bwts does; it is 0 when both inputs are empty.  This is what the device merge
(rust-msbwt_b200/csrc/bwt_merge.cu) is checked against.
"""
from __future__ import annotations

import numpy as np


def rle_to_symbols(rle) -> np.ndarray:
    """msbwt RLE bytes (byte = sym | digit << 3; consecutive bytes of one symbol are little-endian base-32 digits of
    one run, src/bwt_converter.rs:52-56) -> one uint8 symbol per BWT row."""
    b = np.asarray(rle, dtype=np.uint8).reshape(-1)
    if b.size == 0:
        return np.zeros(0, dtype=np.uint8)
    sym = b & 7
    if (sym >= 6).any():
        raise ValueError("RLE byte with a symbol >= 6")
    head = np.ones(b.size, dtype=bool)
    head[1:] = sym[1:] != sym[:-1]
    first = np.flatnonzero(head)
    digit = np.arange(b.size) - first[np.cumsum(head) - 1]
    if digit.max() >= 12:
        raise ValueError("run of 2^60 symbols or more")
    lengths = np.add.reduceat((b >> 3).astype(np.uint64) << (5 * digit).astype(np.uint64), first)
    return np.repeat(sym[first], lengths.astype(np.int64))


def symbols_to_rle(syms) -> np.ndarray:
    """The canonical encoding: one run per maximal block of equal symbols, its length in the fewest base-32 digits."""
    s = np.asarray(syms, dtype=np.uint8).reshape(-1)
    if s.size == 0:
        return np.zeros(0, dtype=np.uint8)
    head = np.ones(s.size, dtype=bool)
    head[1:] = s[1:] != s[:-1]
    first = np.flatnonzero(head)
    lengths = np.diff(np.append(first, s.size))
    out = []
    for sym, n in zip(s[first].tolist(), lengths.tolist()):
        while n:
            out.append(sym | ((n & 31) << 3))
            n >>= 5
    return np.array(out, dtype=np.uint8)


def merge_symbols(a, b) -> tuple[np.ndarray, int]:
    """(merged symbols, iterations) of two BWTs given as one symbol per row."""
    a = np.asarray(a, dtype=np.uint8).reshape(-1)
    b = np.asarray(b, dtype=np.uint8).reshape(-1)
    n = a.size + b.size
    if n == 0:
        return np.zeros(0, dtype=np.uint8), 0
    src = np.concatenate([np.zeros(a.size, dtype=np.uint8), np.ones(b.size, dtype=np.uint8)])
    rows = np.empty(n, dtype=np.uint8)
    iterations = 0
    while True:
        rows[src == 0] = a
        rows[src == 1] = b
        nxt = src[np.argsort(rows, kind="stable")]
        iterations += 1
        if np.array_equal(nxt, src):
            return rows.copy(), iterations
        src = nxt


def merge_rle(rle_a, rle_b) -> tuple[np.ndarray, int, int]:
    """(merged RLE bytes, total symbols, iterations): msbwt_merge_rle_bwts's outputs."""
    syms, iterations = merge_symbols(rle_to_symbols(rle_a), rle_to_symbols(rle_b))
    return symbols_to_rle(syms), int(syms.size), iterations
