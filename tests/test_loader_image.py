"""CPU checks of the product's host logic: the C ABI library loads and exports every
symbol include/msbwt_gpu.h declares, the loader's block image (layout.h) encodes exact
ranks (checked against the oracle through a numpy reading of the documented layout),
the .npy reader accepts/rejects what the reference does, and without a GPU every
query-capable constructor fails loudly (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

import rust_msbwt_b200 as M
from oracle import naive
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "msbwt_gpu.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(msbwt_[a-z_0-9]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(M.library_path())
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/msbwt_gpu.h but not exported"
    assert declared == set(M.EXPORTED_SYMBOLS)
    assert M.load_library().msbwt_abi_version() == 4


CKPT_SLOT = {1: 0, 2: 1, 3: 2, 5: 3}  # layout.h: A,C in half 0 words 0,1; G,T in half 1 words 0,1; $ / N in aux


def image_rank(blocks, aux, cbase, sb_shift, sym, pos):
    """rank+C read off the block image exactly as layout.h documents it"""
    blk, p = pos >> 7, pos & 127
    w = blocks[blk]
    cnt = 0
    for j in range(4):
        m = 0xFFFFFFFF
        for b in range(3):
            plane = int(w[(j >> 1) * 8 + 2 + 2 * b + (j & 1)])
            m &= plane if (sym >> b) & 1 else (~plane & 0xFFFFFFFF)
        nb = min(max(p - 32 * j, 0), 32)
        cnt += bin(m & ((1 << nb) - 1)).count("1")
    ckpt = int(w[(CKPT_SLOT[sym] >> 1) * 8 + (CKPT_SLOT[sym] & 1)]) if sym in CKPT_SLOT else int(aux[blk][sym >> 2])
    return int(cbase[blk >> sb_shift][sym]) + ckpt + cnt


def random_rle(rng, nruns, big=False):
    syms, counts, prev = [], [], -1
    for _ in range(nruns):
        s = int(rng.choice(6, p=[0.05, 0.27, 0.25, 0.25, 0.03, 0.15]))
        if s == prev:
            continue
        prev = s
        syms.append(s)
        counts.append(int(rng.choice([1, 1, 2, 3, 7, 31, 32, 33, 255, 256, 257, 1025] if big else [1, 1, 1, 2, 3, 5, 9, 40])))
    return O.encode_runs(syms, counts)


@pytest.mark.parametrize("sb_shift", [0, 1, 3])
@pytest.mark.parametrize("big", [False, True])
def test_block_image_ranks_match_oracle(sb_shift, big):
    rng = np.random.default_rng(99 + sb_shift + 10 * big)
    rle = random_rle(rng, 900, big)
    blocks, aux, cbase = M.debug_build_image(rle, sb_shift)
    orc = O.RleBWT()
    orc.load_vector(rle)
    n = orc.get_total_size()
    shift = sb_shift or 25
    assert blocks.shape[0] == aux.shape[0] == (n >> 7) + 1
    assert cbase.shape[0] == ((blocks.shape[0] - 1) >> shift) + 1
    pos = sorted(set(rng.integers(0, n + 1, size=400).tolist() + [0, n, n - 1, 128, 127, 129, 256, 255, 257]))
    for s in range(6):
        for a, b in zip(pos[:-1], pos[1:]):
            want = orc.constrain_range(s, a, b)
            assert (image_rank(blocks, aux, cbase, shift, s, a), image_rank(blocks, aux, cbase, shift, s, b)) == want


def test_block_image_exact_multiple_of_256_and_empty():
    rle = O.encode_runs([1, 2], [256, 256])
    blocks, aux, cbase = M.debug_build_image(rle)
    assert blocks.shape == (5, 16)  # position N itself has a block
    assert image_rank(blocks, aux, cbase, 25, 2, 512) == 256 + 256
    assert image_rank(blocks, aux, cbase, 25, 1, 512) == 256
    assert image_rank(blocks, aux, cbase, 25, 0, 512) == 0 and image_rank(blocks, aux, cbase, 25, 4, 512) == 512
    blocks, aux, cbase = M.debug_build_image(np.zeros(0, np.uint8))
    assert blocks.shape == (1, 16) and image_rank(blocks, aux, cbase, 25, 3, 0) == 0


def test_bad_rle_symbol_is_eformat():
    with pytest.raises(M.MsbwtError) as e:
        M.debug_build_image(np.array([9, 14], dtype=np.uint8))  # 14 = symbol 6
    assert e.value.code == 3


def test_rle_whose_runs_add_up_past_2_pow_62_is_refused_before_any_device_work():
    """the total is accumulated with a check after every byte (validate_rle): five runs of 31 * 32^11 ~ 2^60 symbols
    each must be refused as EFORMAT, not wrap a u64 prefix sum on the device"""
    run_a = np.full(12, 1 | (31 << 3), dtype=np.uint8)   # twelve base-32 digits of symbol A
    run_c = np.full(12, 2 | (31 << 3), dtype=np.uint8)
    rle = np.concatenate([run_a, run_c, run_a, run_c, run_a])
    b = M.RleBWT.new()
    with pytest.raises(M.MsbwtError) as e:
        b.load_vector(rle)
    assert e.value.code == 3 and "2^62" in str(e.value)
    with pytest.raises(M.MsbwtError) as e:                # a thirteenth digit: one run beyond 2^60
        b.load_vector(np.full(13, 1 | (31 << 3), dtype=np.uint8))
    assert e.value.code == 3


def test_host_side_failures_keep_their_messages(tmp_path):
    """msbwt_last_error() of failures found before any device work, verbatim, and "" after a call that succeeds"""
    L = M.load_library()
    b = M.RleBWT.new()
    with pytest.raises(M.MsbwtError) as e:
        b.load_vector(np.array([9, 14], dtype=np.uint8))  # 14 = symbol 6
    assert e.value.code == 3 and L.msbwt_last_error() == b"RLE byte 1 has symbol 6 (>= 6)"
    missing = str(tmp_path / "missing.npy")
    with pytest.raises(OSError):
        b.load_numpy_file(missing)
    assert L.msbwt_last_error() == f"cannot open {missing}: No such file or directory".encode()
    with pytest.raises(M.MsbwtError) as e:
        M.debug_build_image(np.full(13, 1 | (31 << 3), dtype=np.uint8))  # a thirteenth digit: one run beyond 2^60
    assert e.value.code == 3 and L.msbwt_last_error() == b"run longer than 2^60 symbols"
    M.debug_build_image(np.array([9, 10], dtype=np.uint8))
    assert L.msbwt_last_error() == b""


def test_string_util_mirror():
    assert list(M.convert_stoi("ACGTN$acgtnx")) == [1, 2, 3, 5, 4, 0, 1, 2, 3, 5, 4, 4]
    assert M.convert_itos([0, 1, 2, 3, 4, 5]) == "$ACGNT"
    assert list(M.reverse_complement_i([0, 1, 2, 3, 4, 5])) == [1, 4, 2, 3, 5, 0]


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback_without_a_device(two_string_npy):
    b = M.RleBWT()
    with pytest.raises(M.MsbwtError) as e:
        b.load_vector(O.convert_to_vec(naive.naive_bwt(["ACGT", "TGCA"])))
    assert e.value.code == 6  # ENODEV
    with pytest.raises(M.MsbwtError) as e:
        b.load_numpy_file(two_string_npy)
    assert e.value.code == 6
    with pytest.raises(M.MsbwtError):
        b.count_kmer([1, 2])


def test_npy_reader_error_classes_match_oracle(tmp_path, two_string_npy):
    """Same acceptance classes as the reference's load_numpy_file (src/rle_bwt.rs:81-155):
    io::Error -> OSError, panic -> MsbwtError(EFORMAT).  Checked through create_from_npy;
    without a GPU a well-formed file gets as far as ENODEV."""
    good = tmp_path / "good.npy"
    O.save_bwt_numpy([9, 10], str(good))
    raw = good.read_bytes()
    cases = {
        "missing.npy": None,
        "short.npy": b"\x93NUMPY",
        "trunc_hdr.npy": raw[:50],
        "trunc_body.npy": raw[:-1],
        "long_body.npy": raw + b"\x09",
        "bad_json.npy": raw[:10] + b"[" + raw[11:],
        "true.npy": raw.replace(b"False", b"True "),
        "noshape.npy": raw.replace(b"'shape'", b"'shapx'"),
        "nomagic.npy": b"XXXXXX" + raw[6:],
        "badsym.npy": raw[:-1] + b"\x0e",
    }
    np.save(str(tmp_path / "np.npy"), np.array([9, 10, 11], dtype=np.uint8))
    cases["np.npy"] = (tmp_path / "np.npy").read_bytes()
    for name, data in cases.items():
        p = tmp_path / name
        if data is not None:
            p.write_bytes(data)
        orc = O.RleBWT()
        try:
            orc.load_numpy_file(str(p))
            want = "ok"
        except O.OracleIoError:
            want = "io"
        except O.OraclePanic:
            want = "panic"
        b = M.RleBWT()
        try:
            b.load_numpy_file(str(p))
            got = "ok"
        except OSError:
            got = "io"
        except M.MsbwtError as e:
            got = {3: "panic", 6: "ok"}.get(e.code, f"code{e.code}")  # ENODEV == parsed fine, no device here
        assert got == want, name


def test_rust_shim_sources_stay_in_sync_with_the_library():
    """rust/ cannot be compiled here (no cargo): at least its file list and its `extern "C"` block must follow the
    library -- build.rs compiles exactly the translation units build.py does, and gpu_ffi.rs binds only symbols
    include/msbwt_gpu.h declares, every query / construction / codec entry point among them."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import importlib.util
    spec = importlib.util.spec_from_file_location("msbwt_build", os.path.join(root, "rust-msbwt_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    build_rs = open(os.path.join(root, "rust", "build.rs")).read()
    assert set(re.findall(r'"(\w+\.cu)"', build_rs)) == set(b.SOURCES)
    assert set(re.findall(r'"(\w+\.cpp)"', build_rs)) == set(b.HOST_SOURCES)
    header = open(os.path.join(root, "include", "msbwt_gpu.h")).read()
    declared = set(re.findall(r"\b(msbwt_\w+)\s*\(", header))
    bound = set(re.findall(r"pub fn (msbwt_\w+)\(", open(os.path.join(root, "rust", "src", "gpu_ffi.rs")).read()))
    assert bound <= declared, bound - declared
    must = {n for n in declared if not n.startswith("msbwt_debug_") and n not in (
        "msbwt_gather_bench", "msbwt_host_pack_threads", "msbwt_last_transfer_bytes")}
    assert must <= bound, must - bound
