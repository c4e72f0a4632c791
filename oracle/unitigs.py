"""CPU restatement of msbwt_unitigs (TEST INFRASTRUCTURE ONLY): the unitigs of the node-centric compacted de Bruijn
graph of a k-mer set, in the library's encoding, order and alphabet.

  * unitigs: builds the graph from the k-mer list with dicts and follows include/msbwt_gpu.h's definitions word for
    word: edges, compacted edges, linear paths from their heads, cycles cut before their smallest node, and in
    canonical mode the keep rule first(U) <= first(U'), U' the unitig holding rc(first(U)).
  * check_unitigs: an independent property check of a result that does not rebuild the graph: every node is a window
    of exactly one unitig (in canonical mode on one of its strands), consecutive windows are compacted edges, the ends
    are maximal, cycles start at their minimum, the keep rule, the order and the count sums.

K-mers: A,C,G,T = 0..3, first symbol in the most significant of the 2k bits (msbwt_count_kmers_u64's encoding).
Symbols of the output: A,C,G,T = 1,2,3,5."""
from __future__ import annotations

import numpy as np

SYM = np.array([1, 2, 3, 5], np.uint8)
_CODE = {1: 0, 2: 1, 3: 2, 5: 3}


def revcomp(v: int, k: int) -> int:
    r = 0
    for _ in range(k):
        r = (r << 2) | (3 - (v & 3))
        v >>= 2
    return r


def nodes(kmers, counts, k: int, canonical: bool) -> dict:
    """V with its counts: the list itself, or in canonical mode the list of canonical members and their rc"""
    cnt = {int(x): int(c) for x, c in zip(np.asarray(kmers).tolist(), np.asarray(counts).tolist())}
    if canonical:
        for x, c in list(cnt.items()):
            cnt.setdefault(revcomp(x, k), c)
    return cnt


def _succs(x, k, cnt):
    mask = (1 << (2 * k)) - 1
    return [y for y in (((x << 2) & mask) | c for c in range(4)) if y in cnt]


def _preds(y, k, cnt):
    return [x for x in ((y >> 2) | (c << (2 * (k - 1))) for c in range(4)) if x in cnt]


def encode(windows_first: int, path: list[int], k: int) -> np.ndarray:
    codes = [(windows_first >> (2 * (k - 1 - j))) & 3 for j in range(k)] + [x & 3 for x in path[1:]]
    return SYM[np.array(codes, np.int64)]


def _result(units, cnt, k):
    """(syms u8, offsets u64[n + 1], count_sums u64[n]) of node paths, ascending by first node"""
    units = sorted(units, key=lambda p: p[0])
    seqs = [encode(p[0], p, k) for p in units]
    offsets = np.zeros(len(units) + 1, np.uint64)
    if units:
        offsets[1:] = np.cumsum([s.size for s in seqs])
    syms = np.concatenate(seqs) if seqs else np.zeros(0, np.uint8)
    sums = np.array([sum(cnt[x] for x in p) for p in units], np.uint64)
    return syms.astype(np.uint8), offsets, sums


def unitigs(kmers, counts, k: int, canonical: bool = False):
    """msbwt_unitigs from V's list: `kmers` / `counts` as msbwt_kmer_spectrum (canonical: _canonical) lists them"""
    cnt = nodes(kmers, counts, k, canonical)
    succ = {x: _succs(x, k, cnt) for x in cnt}
    pred = {y: _preds(y, k, cnt) for y in cnt}
    nxt, prv = {}, {}
    for x in cnt:  # the compacted edges
        if len(succ[x]) == 1:
            y = succ[x][0]
            if len(pred[y]) == 1 and x != y:
                nxt[x], prv[y] = y, x
    units, seen = [], set()
    for x in sorted(cnt):  # linear paths, from their heads
        if x not in prv:
            p = [x]
            while p[-1] in nxt:
                p.append(nxt[p[-1]])
            units.append(p)
            seen.update(p)
    for x in sorted(cnt):  # what is left lies on cycles: cut each before its smallest node
        if x in seen:
            continue
        cyc = [x]
        while nxt[cyc[-1]] != x:
            cyc.append(nxt[cyc[-1]])
        m = cyc.index(min(cyc))
        units.append(cyc[m:] + cyc[:m])
        seen.update(cyc)
    if canonical:
        first_of = {x: p[0] for p in units for x in p}
        units = [p for p in units if p[0] <= first_of[revcomp(p[0], k)]]
    return _result(units, cnt, k)


def windows(seq: np.ndarray, k: int) -> list[int]:
    codes = [_CODE[int(s)] for s in seq]
    out, v, mask = [], 0, (1 << (2 * k)) - 1
    for i, c in enumerate(codes):
        v = ((v << 2) | c) & mask
        if i + 1 >= k:
            out.append(v)
    return out


def check_unitigs(syms, offsets, count_sums, kmers, counts, k: int, canonical: bool = False) -> None:
    """asserts that (syms, offsets, count_sums) are the unitigs msbwt_unitigs promises for V's list"""
    cnt = nodes(kmers, counts, k, canonical)
    offsets = np.asarray(offsets, np.uint64)
    n = offsets.size - 1
    assert offsets[0] == 0 and offsets[-1] == len(syms) and np.asarray(count_sums).size == n
    assert (np.diff(offsets.astype(np.int64)) >= k).all()
    outdeg = lambda x: len(_succs(x, k, cnt))  # noqa: E731
    indeg = lambda y: len(_preds(y, k, cnt))  # noqa: E731
    compacted = lambda x, y: outdeg(x) == 1 and indeg(y) == 1 and x != y and ((x << 2) & ((1 << 2 * k) - 1)) == (y & ~3)  # noqa: E731
    covered: dict[int, int] = {}
    firsts = []
    for i in range(n):
        w = windows(np.asarray(syms[int(offsets[i]):int(offsets[i + 1])]), k)
        assert len(set(w)) == len(w), f"unitig {i} repeats a window"
        assert all(x in cnt for x in w), f"unitig {i} has a window outside V"
        assert all(compacted(a, b) for a, b in zip(w, w[1:])), f"unitig {i} crosses an edge that is not compacted"
        assert int(count_sums[i]) == sum(cnt[x] for x in w), f"count sum of unitig {i}"
        f, last = w[0], w[-1]
        closes = compacted(last, f)
        if closes:  # a cycle: cut before its smallest node
            assert f == min(w), f"cycle {i} does not start at its minimum"
        else:  # maximal: nothing compacted enters the first window or leaves the last
            assert not any(compacted(p, f) for p in _preds(f, k, cnt)), f"unitig {i} extends to the left"
            assert not any(compacted(last, s) for s in _succs(last, k, cnt)), f"unitig {i} extends to the right"
        if canonical:
            rw = [revcomp(x, k) for x in w]
            assert (min(w) <= min(rw)) if closes else (f <= revcomp(last, k)), f"unitig {i} breaks the keep rule"
            strands = set(w) | set(rw)
        else:
            strands = set(w)
        for x in strands:
            covered[x] = covered.get(x, 0) + 1
        firsts.append(f)
    assert all(a < b for a, b in zip(firsts, firsts[1:])), "not strictly ascending by first k-mer"
    assert set(covered) == set(cnt) and all(c == 1 for c in covered.values()), "a node is not in exactly one unitig"
