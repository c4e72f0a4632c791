"""Pins the CPU oracle against every known-answer test the reference holds for the
count_kmer / constrain_range path (SURVEY.md section 4 / 8c).  Citations are
file:line in the reference (rust-msbwt).  CPU only."""
import hashlib
import itertools

import numpy as np
import pytest

from oracle import naive
from oracle import oracle as O

SYMS = "$ACGNT"


def load(strings=None, bwt=None, bin_power=8):
    if bwt is None:
        bwt = naive.naive_bwt(strings)
    b = O.RleBWT(bin_power)
    b.load_vector(O.convert_to_vec(bwt))
    return b, bwt


# ---- string_util.rs:91-120 ----
def test_string_util():
    assert list(O.convert_stoi("ACGTN$")) == [1, 2, 3, 5, 4, 0]
    assert list(O.convert_stoi("acgtnx")) == [1, 2, 3, 5, 4, 4]
    assert O.convert_itos([0, 1, 2, 3, 4, 5]) == "$ACGNT"
    assert list(O.reverse_complement_i([0, 1, 2, 3, 4, 5])) == [1, 4, 2, 3, 5, 0]


# ---- bwt_util.rs:194-236 ----
def test_naive_bwt_kats():
    assert naive.naive_bwt(["CCGT", "N", "ACG"]) == "GTN$$ACCC$G"
    assert naive.naive_bwt(["A", "AA", "AAA"]) == "AAA$AA$A$"
    assert naive.naive_bwt(["ACA", "CA"]) == "AACC$A$"


# ---- bwt_converter.rs:195-256 ----
def test_convert_to_vec_kats():
    assert list(O.convert_to_vec("ACGNT$")) == [9, 10, 11, 12, 13, 8]
    assert list(O.convert_to_vec("\n$$\n$$\nAAA\n")) == [32, 25]
    assert list(O.convert_to_vec("A" * 3104)) == [1, 9, 25]
    assert list(O.convert_to_vec("A" * 31 + "C" * 31)) == [249, 250]
    assert list(O.convert_to_vec("N" * 32767)) == [252, 252, 252]
    assert list(O.convert_to_vec("GTN$$ACCC$G")) == [11, 13, 12, 16, 9, 26, 8, 11]
    assert len(O.convert_to_vec("AAAACCCGGGGNTTTTT$$")) == 6
    with pytest.raises(O.OraclePanic):
        O.convert_to_vec("ACGX")


# ---- bwt_converter.rs:259-321 ----
def test_save_bwt_numpy_bytes(tmp_path):
    head = b"\x93NUMPY\x01\x00\x56\x00{'descr': '|u1', 'fortran_order': False, 'shape': (3, ), }"
    expect = head + b" " * (95 - len(head)) + b"\n" + bytes([1, 9, 25])
    p = str(tmp_path / "a.npy")
    O.save_bwt_numpy(O.convert_to_vec("A" * 3104), p)
    assert open(p, "rb").read() == expect
    # run form (bwt_converter.rs:287-321)
    runs = O.encode_runs([1, 0], [3104, 1])
    assert list(runs) == [1, 9, 25, 8]
    # numpy itself must read what we wrote
    assert list(np.load(p)) == [1, 9, 25]


# ---- rle_bwt.rs:479-503 ----
def test_load_from_npy_totals(tmp_path):
    p = str(tmp_path / "b.npy")
    O.save_bwt_numpy(O.convert_to_vec(naive.naive_bwt(["CCGT", "N", "ACG"])), p)
    b = O.RleBWT()
    b.load_numpy_file(p)
    assert [b.get_symbol_count(i) for i in range(6)] == [3, 1, 3, 2, 1, 1]
    assert b.get_total_size() == 11


# ---- rle_bwt.rs:505-599: literal ref_index / fm_index tables ----
FM_KAT = {
    1: ([0, 2, 3, 5, 5, 7, 8], [[0, 0, 0, 2, 2, 3, 3], [0, 0, 0, 1, 1, 1, 1], [0, 0, 0, 0, 0, 3, 3],
                                [0, 1, 1, 1, 1, 1, 2], [0, 0, 1, 1, 1, 1, 1], [0, 1, 1, 1, 1, 1, 1]]),
    2: ([0, 3, 5, 8], [[0, 0, 2, 3], [0, 0, 1, 1], [0, 0, 0, 3], [0, 1, 1, 2], [0, 1, 1, 1], [0, 1, 1, 1]]),
    3: ([0, 5, 8], [[0, 2, 3], [0, 1, 1], [0, 0, 3], [0, 1, 2], [0, 1, 1], [0, 1, 1]]),
    4: ([0, 8], [[0, 3], [0, 1], [0, 3], [0, 2], [0, 1], [0, 1]]),
}


@pytest.mark.parametrize("bin_power", [1, 2, 3, 4])
def test_fmindex_literals(bin_power):
    b, bwt = load(["CCGT", "N", "ACG"], bin_power=bin_power)
    assert bwt == "GTN$$ACCC$G"
    assert [b.get_symbol_count(i) for i in range(6)] == [3, 1, 3, 2, 1, 1]
    ref, fm = FM_KAT[bin_power]
    assert len(b.ref_index) == -(-len(bwt) // (1 << bin_power)) + 1
    assert b.ref_index == ref
    for s in range(6):
        assert b.fm_index(s) == fm[s]


# ---- rle_bwt.rs:601-675 ----
@pytest.mark.parametrize("bin_power", [1, 2, 3, 4, 8])
def test_constrain_range_every_position(bin_power):
    b, bwt = load(["CCGT", "N", "ACG"], bin_power=bin_power)
    ints = list(O.convert_stoi(bwt))
    n = len(bwt)
    for sym in range(6):
        assert b.constrain_range(sym, 0, n) == (b.start_index(sym), b.end_index(sym))
        cnt = 0
        for ind in range(n + 1):
            assert b.constrain_range(sym, 0, ind) == (b.start_index(sym), b.start_index(sym) + cnt)
            assert b.constrain_range(sym, ind, n) == (b.start_index(sym) + cnt, b.end_index(sym))
            if ind < n and ints[ind] == sym:
                cnt += 1


# ---- rle_bwt.rs:677-710 + dynamic_bwt.rs:702-773 ----
@pytest.mark.parametrize("bin_power", [1, 2, 3, 4, 8])
def test_count_kmer_kats(bin_power):
    data = ["CCGTACGTA", "GGTACAGTA", "ACGACGACG"]
    b, _ = load(data, bin_power=bin_power)
    for c in range(6):
        assert b.count_kmer([c]) == b.get_symbol_count(c)
    for s in data:
        assert b.count_kmer(O.convert_stoi(s)) == 1
    assert b.count_kmer(O.convert_stoi("ACG")) == 4
    assert b.count_kmer(O.convert_stoi("CC")) == 1
    assert b.count_kmer(O.convert_stoi("TAC")) == 2
    data4 = data + ["AAGTCATAT"]  # dynamic_bwt.rs:734-773 (inserted string == naive BWT of 4 strings)
    b4, _ = load(data4, bin_power=bin_power)
    for c in range(6):
        assert b4.count_kmer([c]) == b4.get_symbol_count(c)
    for s in data4:
        assert b4.count_kmer(O.convert_stoi(s)) == 1
    assert b4.count_kmer(O.convert_stoi("ACG")) == 4
    assert b4.count_kmer(O.convert_stoi("CC")) == 1
    assert b4.count_kmer(O.convert_stoi("TAC")) == 2
    assert b4.count_kmer(O.convert_stoi("AA")) == 1
    assert b4.count_kmer(O.convert_stoi("GT")) == 5


# ---- doc-tests msbwt_core.rs:110-122, rle_bwt.rs:165-188 ----
def test_doc_kats():
    b, _ = load(bwt="TG$$CAGCCG")
    assert b.get_total_size() == 10
    assert b.get_symbol_count(0) == 2
    assert b.count_kmer([1, 2, 3, 5]) == 1
    assert b.count_kmer([2, 3]) == 2
    assert b.count_kmer(O.convert_stoi("CG")) == 2
    assert b.count_kmer([]) == 10  # empty k-mer -> total_size (msbwt_core.rs:128-131,160)
    with pytest.raises(O.OraclePanic):
        b.count_kmer([1, 6])  # msbwt_core.rs:127 assert


# ---- test_data/two_string.npy: rle_bwt.rs:76-79, dynamic_bwt.rs:783-793, README.md:62-70 ----
def test_two_string_fixture(two_string_npy):
    raw = open(two_string_npy, "rb").read()
    assert len(raw) == 106 and list(raw[96:]) == [13, 9, 10, 8, 11, 9, 13, 10, 11, 8]
    b = O.RleBWT()
    b.load_numpy_file(two_string_npy)
    assert b.count_kmer(O.convert_stoi("ACGT")) == 1
    assert b.count_kmer(O.convert_stoi("TGCA")) == 1
    assert b.count_kmer(O.convert_stoi("$")) == 2
    # SURVEY.md section 4: non-zero ACGT k-mers for k=1..8 are 4,6,4,2,0,0,0,0
    nonzero = []
    for k in range(1, 9):
        qs = np.array(list(itertools.product([1, 2, 3, 5], repeat=k)), dtype=np.uint8)
        nonzero.append(int((b.count_kmers_fixed(qs, k) > 0).sum()))
    assert nonzero == [4, 6, 4, 2, 0, 0, 0, 0]


def test_reference_fixture_copy_is_reproduced_by_the_oracle(two_string_npy, tmp_path):
    """tests/golden/two_string.npy is a byte-identical copy of the reference's test_data/two_string.npy; its hash pins
    the copy, and the oracle's writer must reproduce it from the fixture's two strings"""
    raw = open(two_string_npy, "rb").read()
    assert hashlib.sha256(raw).hexdigest() == "1849b221e871bcc1a137955db7c1659d4c140d727be18321ce64d917863991de"
    p = str(tmp_path / "two_string.npy")
    O.save_bwt_numpy(O.convert_to_vec(naive.naive_bwt(["ACGT", "TGCA"])), p)
    assert open(p, "rb").read() == raw


# ---- load_numpy_file error classes (rle_bwt.rs:84-147) ----
def test_load_numpy_errors(tmp_path):
    b = O.RleBWT()
    with pytest.raises(O.OracleIoError):
        b.load_numpy_file(str(tmp_path / "missing.npy"))
    p = tmp_path / "short.npy"
    p.write_bytes(b"\x93NUMPY")
    with pytest.raises(O.OraclePanic):
        b.load_numpy_file(str(p))
    good = tmp_path / "good.npy"
    O.save_bwt_numpy([9, 10], str(good))
    raw = good.read_bytes()
    (tmp_path / "trunc_hdr.npy").write_bytes(raw[:50])
    with pytest.raises(O.OracleIoError):
        b.load_numpy_file(str(tmp_path / "trunc_hdr.npy"))
    (tmp_path / "trunc_body.npy").write_bytes(raw[:-1])
    with pytest.raises(O.OracleIoError):
        b.load_numpy_file(str(tmp_path / "trunc_body.npy"))
    (tmp_path / "long_body.npy").write_bytes(raw + b"\x09")
    with pytest.raises(O.OracleIoError):
        b.load_numpy_file(str(tmp_path / "long_body.npy"))
    bad = bytearray(raw)
    bad[10:11] = b"["
    (tmp_path / "bad_json.npy").write_bytes(bytes(bad))
    with pytest.raises(O.OraclePanic):
        b.load_numpy_file(str(tmp_path / "bad_json.npy"))
    # magic/version are not checked (rle_bwt.rs:96): a mangled magic still loads
    ok = bytearray(raw)
    ok[0:6] = b"XXXXXX"
    (tmp_path / "nomagic.npy").write_bytes(bytes(ok))
    b.load_numpy_file(str(tmp_path / "nomagic.npy"))
    assert b.get_total_size() == 2
    # numpy's own writer (different header padding / v1 header) is accepted too
    np.save(str(tmp_path / "np.npy"), np.array([9, 10, 11], dtype=np.uint8))
    b.load_numpy_file(str(tmp_path / "np.npy"))
    assert b.get_total_size() == 3


# ---- beyond the reference's tests: rank identity on awkward streams (SURVEY.md facts table) ----
def _decode(rle):
    out, prev, power = [], 255, 1
    runs = []
    for v in rle:
        v = int(v)
        c, d = v & 7, v >> 3
        if c == prev:
            runs[-1][1] += d * power
            power *= 32
        else:
            runs.append([c, d])
            prev, power = c, 32
    for c, n in runs:
        out.extend([c] * n)
    return out


@pytest.mark.parametrize("bin_power", [1, 3, 5, 8])
def test_constrain_range_is_c_plus_rank_on_long_and_zero_digit_runs(bin_power):
    rng = np.random.default_rng(1234 + bin_power)
    syms, counts = [], []
    prev = -1
    for _ in range(60):
        s = int(rng.integers(0, 6))
        if s == prev:
            continue
        prev = s
        syms.append(s)
        counts.append(int(rng.choice([1, 2, 31, 32, 33, 64, 1024, 1025, 700, 3104])))
    rle = O.encode_runs(syms, counts)
    text = _decode(rle)
    b = O.RleBWT(bin_power)
    b.load_vector(rle)
    n = len(text)
    assert b.get_total_size() == n
    pref = np.zeros((6, n + 1), dtype=np.int64)
    for s in range(6):
        pref[s, 1:] = np.cumsum(np.array(text) == s)
    pos = sorted(set(rng.integers(0, n + 1, size=300).tolist() + [0, n]))
    for s in range(6):
        for l, h in zip(pos[:-1:3], pos[1::3]):
            assert b.constrain_range(s, l, h) == (b.start_index(s) + pref[s, l], b.start_index(s) + pref[s, h])
        for p in pos:
            assert b.constrain_range(s, p, p) == (b.start_index(s) + pref[s, p],) * 2


def test_count_kmer_matches_brute_force_on_random_strings():
    rng = np.random.default_rng(7)
    strings = ["".join(rng.choice(list("ACGT"), size=int(rng.integers(1, 40)))) for _ in range(40)]
    strings[3] = strings[3][:5] + "N" + strings[3][5:]
    b, _ = load(strings, bin_power=4)
    for k in (1, 2, 3, 5, 8):
        for _ in range(60):
            q = "".join(rng.choice(list("ACGT"), size=k))
            assert b.count_kmer(O.convert_stoi(q)) == naive.brute_count(strings, q)
    assert b.count_kmer(O.convert_stoi("N")) == 1
    ends = sum(s.endswith("A") for s in strings)
    assert b.count_kmer(O.convert_stoi("A$")) == ends


def test_threads_split_matches_single():
    rng = np.random.default_rng(11)
    strings = ["".join(rng.choice(list("ACGT"), size=50)) for _ in range(200)]
    b, _ = load(strings)
    qs = rng.choice(np.array([1, 2, 3, 5], dtype=np.uint8), size=(5000, 6))
    a = b.count_kmers_fixed(qs, 6, threads=1)
    c = b.count_kmers_fixed(qs, 6, threads=4)
    assert (a == c).all()
    v = b.count_kmers([q for q in qs[:100]], threads=3)
    assert (v == a[:100]).all()
    steps, two = b.count_kmers_stats(qs, 6, 8)
    assert 0 < steps <= 5000 * 6 and 0 <= two <= steps


def test_golden_fixture_matches_oracle(golden_dir):
    z = np.load(f"{golden_dir}/reads30x_k31.npz")
    b = O.RleBWT()
    b.load_vector(z["rle"])
    assert b.get_total_size() == int(z["total"])
    assert (b.count_kmers_fixed(z["queries"], int(z["k"])) == z["counts"]).all()
    assert (b.count_kmers_fixed(z["queries_k12"], 12) == z["counts_k12"]).all()
