"""CPU restatement of msbwt_correct_reads (include/msbwt_gpu.h), step by step.

`count2(x)` gives count_kmer(x) + count_kmer(rc x) of a k-mer x in msbwt_count_kmers_u64's encoding (A,C,G,T = 0..3,
first symbol most significant).  For an index built from reads, count_kmer(x) is the number of k-windows of the reads
equal to x (oracle/spectrum.py argues why), so `window_count2` builds count2 from a dict of the reads' windows.
Reads and results are sequences of symbol codes $,A,C,G,N,T = 0..5."""
from collections import Counter

CODE = {1: 0, 2: 1, 3: 2, 5: 3}  # A C G T -> 2-bit code
SYM = (1, 2, 3, 5)               # 2-bit code -> symbol


def revcomp(x, k):
    r = 0
    for _ in range(k):
        r = (r << 2) | (3 - (x & 3))
        x >>= 2
    return r


def encode(window):
    """the k-mer of a window of symbols, or None when it holds a symbol outside ACGT"""
    v = 0
    for s in window:
        if s not in CODE:
            return None
        v = (v << 2) | CODE[s]
    return v


def window_count2(reads, k):
    """count2 for an index built from `reads`: every k-window counted on both strands"""
    c = Counter()
    for r in reads:
        for i in range(len(r) - k + 1):
            x = encode(r[i:i + k])
            if x is not None:
                c[x] += 1
    return lambda x: c.get(x, 0) + c.get(revcomp(x, k), 0)


def levenshtein(e, p):
    """unit-cost edit distance over symbol codes; an N (4) in p matches nothing"""
    prev = list(range(len(p) + 1))
    for i, a in enumerate(e, 1):
        cur = [i] + [0] * len(p)
        for j, b in enumerate(p, 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (0 if a == b and b != 4 else 1))
        prev = cur
    return prev[-1]


def threshold(c2, min_count, frac_permille):
    """T of a read from its window counts, or None when no window counts (step 2)"""
    v = sorted(c for c in c2 if c)
    if not v:
        return None
    return max(min_count, v[len(v) // 2] * frac_permille // 1000)


def weak_runs(c2, T):
    """the maximal runs [a, b) of windows with count2 < T (step 3)"""
    runs, w = [], 0
    while w < len(c2):
        if c2[w] < T:
            a = w
            while w < len(c2) and c2[w] < T:
                w += 1
            runs.append((a, w))
        else:
            w += 1
    return runs


def bridges(X, Y, k, T, Emax, budget, count2):
    """Step 4: (the bridges' E as lists of codes in the order found, abandoned).  Breadth-first over walks from X, one
    symbol per round, children of each walk in A < C < G < T order: bridges of one round come out lexicographically."""
    mask = (1 << (2 * k)) - 1
    frontier = [(X, [])]  # (newest window, symbols appended so far)
    found, work = [], 0
    for t in range(1, k + Emax + 1):
        nxt = []
        for z, path in frontier:
            for c in range(4):
                y = ((z << 2) | c) & mask
                if count2(y) < T:
                    continue
                work += 1
                walk = path + [c]
                if t >= k and y == Y:
                    found.append(walk[:t - k])
                else:
                    nxt.append((y, walk))
        if work > budget:
            return found, True
        frontier = nxt
        if not frontier:
            break
    return found, False


def correct_read(read, k, min_count, frac_permille, branch_limit, count2, stats):
    read = list(read)
    n = len(read)
    if n < k + 2:
        return read
    nwin = n - k + 1
    c2 = []
    for w in range(nwin):
        x = encode(read[w:w + k])
        c2.append(0 if x is None else count2(x))
    T = threshold(c2, min_count, frac_permille)
    if T is None:
        return read
    edits = []
    for a, b in weak_runs(c2, T):
        stats[0] += 1
        if not (1 <= a and b <= nwin - 1 and b - a >= k - 1):
            continue
        stats[1] += 1
        X, Y = encode(read[a - 1:a - 1 + k]), encode(read[b:b + k])
        P = read[a - 1 + k:b]
        L0 = len(P)
        Emax = 13 * L0 // 10 + 2
        found, abandoned = bridges(X, Y, k, T, Emax, branch_limit * (k + Emax), count2)
        if abandoned:
            stats[3] += 1
            continue
        if not found:
            stats[4] += 1
            continue
        best = min(found, key=lambda e: (levenshtein([SYM[c] for c in e], P), len(e), e))
        E = [SYM[c] for c in best]
        assert E != P
        stats[2] += 1
        edits.append((a - 1 + k, b, E))
    for s, e, E in sorted(edits, reverse=True):  # disjoint: apply from the back
        read[s:e] = E
    return read


def correct_reads(reads, k, min_count, frac_permille, branch_limit, count2):
    """(corrected reads as lists of symbol codes, stats[5]) as msbwt_correct_reads defines them"""
    stats = [0] * 5
    out = [correct_read(r, k, min_count, frac_permille, branch_limit, count2, stats) for r in reads]
    return out, stats
