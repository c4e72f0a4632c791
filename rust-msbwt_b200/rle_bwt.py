"""Host-side mirror of the reference's `RleBWT` (src/rle_bwt.rs:14-322) and `BWT` trait
(src/msbwt_core.rs:28-162) over the C ABI in include/msbwt_gpu.h.

Same method names, argument meaning and error behaviour as the reference:

    RleBWT.new() / RleBWT.with_bin_power(p)    src/rle_bwt.rs:297-322
    load_vector(rle_bytes)                     src/rle_bwt.rs:59-66
    load_numpy_file(path)                      src/rle_bwt.rs:81-155  (OSError where the reference
                                               returns io::Error, MsbwtError where it panics)
    get_symbol_count(sym) / get_total_size()   src/rle_bwt.rs:172-193
    constrain_range(sym, BWTRange)             src/rle_bwt.rs:202-287
    count_kmer(kmer)                           src/msbwt_core.rs:125-161 (symbol >= 6 raises, as the
                                               reference's assert panics)
    count_kmers(kmers)                         the batched entry point BASELINE.json adds

Every query goes to the CUDA library; there is no CPU path here.  If the library or a
CUDA device is missing the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MSBWT_LIBRARY_PATH: load another build of the same library (kernel tuning variants, tools/)
_LIB_PATH = os.environ.get("MSBWT_LIBRARY_PATH") or os.path.join(_HERE, "libmsbwt_b200.so")

OK, EINVAL, EIO, EFORMAT, ECUDA, ENOMEM, ENODEV = range(7)
_NAMES = {EINVAL: "EINVAL", EIO: "EIO", EFORMAT: "EFORMAT", ECUDA: "ECUDA", ENOMEM: "ENOMEM", ENODEV: "ENODEV"}

# string_util.rs:3-32 / 6-9 / 12
_STOI = np.full(256, 4, dtype=np.uint8)
for _c, _v in (("$", 0), ("A", 1), ("C", 2), ("G", 3), ("N", 4), ("T", 5), ("a", 1), ("c", 2), ("g", 3), ("n", 4), ("t", 5)):
    _STOI[ord(_c)] = _v
_ITOS = np.frombuffer(b"$ACGNT", dtype=np.uint8)
_COMPLEMENT = np.array([0, 5, 3, 2, 4, 1], dtype=np.uint8)


def convert_stoi(seq: str | bytes) -> np.ndarray:
    """string_util.rs:63-67"""
    raw = seq.encode() if isinstance(seq, str) else bytes(seq)
    return _STOI[np.frombuffer(raw, dtype=np.uint8)]


def convert_itos(iseq) -> str:
    """string_util.rs:80-88"""
    return _ITOS[np.asarray(iseq, dtype=np.uint8)].tobytes().decode()


def reverse_complement_i(seq) -> np.ndarray:
    """string_util.rs:45-50"""
    return _COMPLEMENT[np.asarray(seq, dtype=np.uint8)[::-1]]


class MsbwtError(RuntimeError):
    """A failure the reference would have panicked on (or a CUDA failure)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"{_NAMES.get(code, code)}: {message}")
        self.code = code


@dataclass(frozen=True)
class BWTRange:
    """msbwt_core.rs:18-24: half-open [l, h)."""
    l: int = 0
    h: int = 0


class Options(C.Structure):
    """`msbwt_options` (include/msbwt_gpu.h)."""
    _fields_ = [("struct_size", C.c_uint32), ("superblock_shift", C.c_uint32), ("suffix_table_s", C.c_int32),
                ("pair_index", C.c_int32), ("kernel_lanes", C.c_int32), ("quad_index", C.c_int32), ("oct_index", C.c_int32),
                ("oct_bucket_shift", C.c_int32), ("keep_quad_index", C.c_int32), ("final_index", C.c_int32),
                ("final_bucket_shift", C.c_int32), ("final_lines_log2", C.c_int32)]


_lib = None


def library_path() -> str:
    return _LIB_PATH


def load_library():
    """dlopen libmsbwt_b200.so (built in-tree by build.py).  Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise MsbwtError(ENODEV, f"{_LIB_PATH} is missing: run `python rust-msbwt_b200/build.py` "
                                 "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(_LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    ip = C.POINTER(C.c_int)
    sig = {
        "msbwt_index_create_from_rle": (vp, [vp, u64, ip, i32, ip]),
        "msbwt_index_create_from_npy": (vp, [C.c_char_p, ip, i32, ip]),
        "msbwt_index_create_ex": (vp, [vp, u64, ip, i32, u32, i32, ip]),
        "msbwt_index_create_opts": (vp, [vp, u64, ip, i32, C.POINTER(Options), ip]),
        "msbwt_index_create_from_npy_opts": (vp, [C.c_char_p, ip, i32, C.POINTER(Options), ip]),
        "msbwt_index_destroy": (None, [vp]),
        "msbwt_total_size": (u64, [vp]),
        "msbwt_symbol_count": (u64, [vp, C.c_uint8]),
        "msbwt_start_index": (u64, [vp, C.c_uint8]),
        "msbwt_device_count": (i32, [vp]),
        "msbwt_device_ordinal": (i32, [vp, i32]),
        "msbwt_index_bytes": (u64, [vp]),
        "msbwt_count_kmers": (i32, [vp, vp, vp, u64, vp]),
        "msbwt_count_kmers_fixed": (i32, [vp, vp, u32, u64, vp]),
        "msbwt_constrain_ranges": (i32, [vp, vp, vp, vp, u64, vp, vp]),
        "msbwt_count_kmers_fixed_device": (i32, [vp, i32, vp, u32, u64, vp, vp, vp]),
        "msbwt_constrain_ranges_device": (i32, [vp, i32, vp, vp, vp, u64, vp, vp, vp]),
        "msbwt_packed_bytes": (u64, [vp, u32, u64]),
        "msbwt_suffix_table_s": (i32, [vp]),
        "msbwt_kernel_lanes": (i32, [vp]),
        "msbwt_pair_index": (i32, [vp]),
        "msbwt_quad_index": (i32, [vp]),
        "msbwt_oct_index": (i32, [vp]),
        "msbwt_oct_overflow_lines": (u64, [vp]),
        "msbwt_oct_overflow_occurrences": (u64, [vp]),
        "msbwt_oct_runs": (u64, [vp]),
        "msbwt_oct_bucket_shift": (i32, [vp]),
        "msbwt_oct_symbols": (i32, []),
        "msbwt_table_depth_for_k": (i32, [vp, u32]),
        "msbwt_debug_table_depth": (i32, [u32, u32, u32]),
        "msbwt_debug_plan_layout": (i32, [C.POINTER(Options), u64, i32, u64, u64, u64, u64, vp, i32]),
        "msbwt_count_kmers_u64": (i32, [vp, vp, u32, u64, vp]),
        "msbwt_count_kmers_fixed_u32": (i32, [vp, vp, u32, u64, vp]),
        "msbwt_count_kmers_u64_u32": (i32, [vp, vp, u32, u64, vp]),
        "msbwt_final_index": (i32, [vp]),
        "msbwt_debug_copy_final_image": (i32, [vp, i32, C.POINTER(u64), C.POINTER(u32), C.POINTER(u32), C.POINTER(u64), vp]),
        "msbwt_debug_copy_oct_image": (i32, [vp, i32, C.POINTER(u64), vp]),
        "msbwt_constrain_ranges_fanout": (i32, [vp, vp, vp, u64, vp, vp]),
        "msbwt_constrain_ranges_fanout_device": (i32, [vp, i32, vp, vp, u64, vp, vp, vp]),
        "msbwt_count_read_kmers": (i32, [vp, vp, u32, u64, u32, u32, vp]),
        "msbwt_debug_copy_quad_image": (i32, [vp, i32, C.POINTER(u64), C.POINTER(u32), vp, vp]),
        "msbwt_last_transfer_bytes": (None, [C.POINTER(u64), C.POINTER(u64)]),
        "msbwt_host_pack_threads": (i32, []),
        "msbwt_debug_host_pack": (i32, [vp, u32, u64, i32, vp, vp, u64, C.POINTER(u64)]),
        "msbwt_debug_copy_pair_image": (i32, [vp, i32, C.POINTER(u64), C.POINTER(u32), vp, vp]),
        "msbwt_pack_kmers_device": (i32, [vp, i32, vp, u32, u64, vp, vp, vp, vp]),
        "msbwt_count_kmers_packed_device": (i32, [vp, i32, vp, u32, u64, vp, vp]),
        "msbwt_seed_kmers_u64_device": (i32, [vp, i32, vp, u32, u64, vp, vp, vp]),
        "msbwt_count_kmers_packed_stats_device": (i32, [vp, i32, vp, u32, u64, vp, vp, vp]),
        "msbwt_debug_pack_stats": (i32, [vp, i32, vp, u32, u64, vp]),
        "msbwt_launch_count": (u64, []),
        "msbwt_gather_bench": (i32, [i32, vp, u64, u32, u64, u64, vp, vp]),
        "msbwt_l2_fetch_granularity": (i32, [i32, i32]),
        "msbwt_debug_build_image": (i32, [vp, u64, u32, C.POINTER(u64), C.POINTER(u32), vp, vp, vp]),
        "msbwt_debug_copy_image": (i32, [vp, i32, C.POINTER(u64), C.POINTER(u32), vp, vp, vp]),
        "msbwt_build_rle_bwt": (i32, [vp, u64, u32, i32, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]),
        "msbwt_build_rle_bwt_ragged": (i32, [vp, vp, u64, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]),
        "msbwt_merge_rle_bwts": (i32, [vp, u64, vp, u64, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(u32)]),
        "msbwt_kmer_spectrum": (i32, [vp, u32, u64, vp, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]),
        "msbwt_kmer_spectrum_canonical": (i32, [vp, u32, u64, vp, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]),
        "msbwt_unitigs": (i32, [vp, u32, u64, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]),
        "msbwt_correct_reads": (i32, [vp, vp, vp, u64, u32, u64, u32, u32, C.POINTER(vp), C.POINTER(vp), vp]),
        "msbwt_buffer_free": (None, [vp]),
        "msbwt_convert_to_rle": (i32, [vp, u64, C.POINTER(vp), C.POINTER(u64)]),
        "msbwt_save_rle_npy": (i32, [vp, u64, C.c_char_p]),
        "msbwt_save_runs_npy": (i32, [vp, vp, u64, C.c_char_p]),
        "msbwt_host_alloc": (vp, [C.c_size_t]),
        "msbwt_host_free": (None, [vp]),
        "msbwt_last_error": (C.c_char_p, []),
        "msbwt_abi_version": (i32, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


EXPORTED_SYMBOLS = (
    "msbwt_index_create_from_rle", "msbwt_index_create_from_npy", "msbwt_index_create_ex", "msbwt_index_create_opts",
    "msbwt_index_create_from_npy_opts", "msbwt_count_kmers_packed_stats_device", "msbwt_seed_kmers_u64_device", "msbwt_debug_pack_stats", "msbwt_count_kmers_fixed_u32", "msbwt_count_kmers_u64_u32",
    "msbwt_pair_index", "msbwt_debug_copy_pair_image", "msbwt_quad_index", "msbwt_debug_copy_quad_image", "msbwt_oct_index", "msbwt_oct_overflow_lines",
    "msbwt_oct_overflow_occurrences", "msbwt_oct_runs", "msbwt_oct_bucket_shift", "msbwt_oct_symbols", "msbwt_table_depth_for_k", "msbwt_debug_table_depth", "msbwt_debug_plan_layout", "msbwt_count_kmers_u64", "msbwt_final_index", "msbwt_debug_copy_final_image",
    "msbwt_debug_copy_oct_image", "msbwt_constrain_ranges_fanout", "msbwt_constrain_ranges_fanout_device",
    "msbwt_count_read_kmers", "msbwt_last_transfer_bytes", "msbwt_host_pack_threads",
    "msbwt_debug_host_pack",
    "msbwt_index_destroy", "msbwt_total_size", "msbwt_symbol_count", "msbwt_start_index",
    "msbwt_device_count", "msbwt_device_ordinal", "msbwt_index_bytes", "msbwt_suffix_table_s", "msbwt_kernel_lanes", "msbwt_count_kmers",
    "msbwt_count_kmers_fixed", "msbwt_constrain_ranges", "msbwt_count_kmers_fixed_device",
    "msbwt_constrain_ranges_device", "msbwt_packed_bytes", "msbwt_pack_kmers_device",
    "msbwt_count_kmers_packed_device", "msbwt_launch_count", "msbwt_gather_bench", "msbwt_l2_fetch_granularity", "msbwt_debug_build_image", "msbwt_debug_copy_image",
    "msbwt_host_alloc", "msbwt_build_rle_bwt", "msbwt_build_rle_bwt_ragged", "msbwt_merge_rle_bwts", "msbwt_kmer_spectrum", "msbwt_kmer_spectrum_canonical", "msbwt_unitigs", "msbwt_correct_reads", "msbwt_buffer_free", "msbwt_convert_to_rle", "msbwt_save_rle_npy",
    "msbwt_save_runs_npy",
    "msbwt_host_free", "msbwt_last_error", "msbwt_abi_version",
)


def _check(rc: int, what: str) -> None:
    if rc == OK:
        return
    msg = (load_library().msbwt_last_error() or b"").decode(errors="replace")
    if rc == EIO:
        raise OSError(f"{what}: {msg}")  # the reference returns Err(io::Error) here
    raise MsbwtError(rc, f"{what}: {msg}")


def _u8(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint8))


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


def _p(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def oct_symbols() -> int:
    """m: symbols (constrain_range steps) one oct line answers."""
    return int(load_library().msbwt_oct_symbols())


class RleBWT:
    """GPU-resident `RleBWT`.  `devices`: CUDA ordinals to replicate the index on
    (None = the current device); batches are split across them (no collective)."""

    def __init__(self, bin_power: int = 8, devices: list[int] | None = None, superblock_shift: int = 0,
                 suffix_table_s: int = -1, pair_index: int = -1, kernel_lanes: int = 0, quad_index: int = -1,
                 oct_index: int = -1, oct_bucket_shift: int = 0, keep_quad_index: int = -1, final_index: int = -1,
                 final_bucket_shift: int = 0, final_lines_log2: int = 0):
        # bin_power is accepted for signature parity (src/rle_bwt.rs:309-322); it never
        # changed results in the reference and has no counterpart in the device layout.
        self.bin_power = bin_power
        self._devices = list(devices) if devices else []
        self._sb_shift = superblock_shift
        self._table_s = suffix_table_s  # -1 auto, 0 none, 1..15 explicit (include/msbwt_gpu.h)
        self._pair = pair_index         # -1 auto, 0 never, 1 always: the 128-byte pair image (two steps per line)
        self._lanes = kernel_lanes      # 0 auto, 1, 2
        self._quad = quad_index         # -1 auto, 0 never, 1 always: the 32-byte quad sectors (four steps per sector)
        self._oct = oct_index           # -1 auto, 0 never, 1 always: the 128-byte oct lines (ten steps per line)
        self._oct_shift = oct_bucket_shift  # 0 auto, else log2 of the oct bucket size (8..23)
        self._keep_quad = keep_quad_index   # under an oct image: -1 auto, 0 drop the quad image after the build, 1 keep
        self._final = final_index           # -1 auto (with the oct image), 0 never, 1 always: the final-step lines
        self._final_shift = final_bucket_shift  # 0 = 16
        self._final_lb = final_lines_log2       # 0 auto, else log2 of the lines per bucket (12..20)
        self._h = None

    @classmethod
    def new(cls, **kw) -> "RleBWT":
        return cls(8, **kw)

    @classmethod
    def with_bin_power(cls, bin_power: int, **kw) -> "RleBWT":
        return cls(bin_power, **kw)

    # -- lifetime
    def close(self) -> None:
        h, self._h = self._h, None
        if h and _lib is not None:
            _lib.msbwt_index_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _dev_args(self):
        if not self._devices:
            return None, 0
        arr = (C.c_int * len(self._devices))(*self._devices)
        return arr, len(self._devices)

    @property
    def handle(self):
        if not self._h:
            raise MsbwtError(EINVAL, "no BWT loaded")
        return self._h

    def _options(self) -> Options:
        return Options(C.sizeof(Options), self._sb_shift, self._table_s, self._pair, self._lanes, self._quad, self._oct,
                       self._oct_shift, self._keep_quad, self._final, self._final_shift, self._final_lb)

    # -- BWT trait
    def load_vector(self, bwt) -> None:
        L = load_library()
        self.close()
        a = _u8(bwt)
        err = C.c_int(0)
        devs, nd = self._dev_args()
        opts = self._options()
        h = L.msbwt_index_create_opts(_p(a), a.size, devs, nd, C.byref(opts), C.byref(err))
        if not h:
            _check(err.value or ECUDA, "load_vector")
        self._h = h

    def load_numpy_file(self, filename: str) -> None:
        L = load_library()
        self.close()
        err = C.c_int(0)
        devs, nd = self._dev_args()
        opts = self._options()   # the same layout knobs as load_vector
        h = L.msbwt_index_create_from_npy_opts(os.fsencode(filename), devs, nd, C.byref(opts), C.byref(err))
        if not h:
            _check(err.value or ECUDA, "load_numpy_file")
        self._h = h

    def get_symbol_count(self, symbol: int) -> int:
        return int(load_library().msbwt_symbol_count(self.handle, symbol))

    def get_total_size(self) -> int:
        return int(load_library().msbwt_total_size(self.handle))

    def start_index(self, symbol: int) -> int:
        return int(load_library().msbwt_start_index(self.handle, symbol))

    def constrain_range(self, sym: int, input_range: BWTRange) -> BWTRange:
        lo, hi = self.constrain_ranges([sym], [input_range.l], [input_range.h])
        return BWTRange(int(lo[0]), int(hi[0]))

    def count_kmer(self, kmer) -> int:
        a = _u8(kmer).reshape(-1)
        if a.size == 0:  # empty k-mer counts total_size (msbwt_core.rs:128-131,160)
            return int(self.count_kmers([a])[0])
        return int(self.count_kmers_fixed(a, a.size)[0])

    # -- batched entry points
    def count_kmers(self, kmers) -> np.ndarray:
        """`count_kmers(&[Vec<u8>]) -> Vec<u64>`: variable-length batch."""
        n = len(kmers)
        lens = np.fromiter((len(q) for q in kmers), dtype=np.uint64, count=n)
        offs = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(lens, out=offs[1:])
        flat = _u8(np.concatenate([_u8(q).reshape(-1) for q in kmers])) if n and offs[-1] else np.zeros(1, np.uint8)
        out = np.zeros(n, dtype=np.uint64)
        _check(load_library().msbwt_count_kmers(self.handle, _p(flat), _p(offs), n, _p(out)), "count_kmers")
        return out

    def count_kmers_fixed(self, syms, k: int, counts32: bool = False) -> np.ndarray:
        """Fixed-k batch: `syms` is n*k symbols, row-major.  `counts32`: u32 counts (index below 2^32 symbols)."""
        a = _u8(syms).reshape(-1)
        if k == 0:
            raise MsbwtError(EINVAL, "count_kmers_fixed needs k > 0 (use count_kmers for empty k-mers)")
        if a.size % k:
            raise MsbwtError(EINVAL, "len(syms) is not a multiple of k")
        n = a.size // k
        if counts32:
            out = np.zeros(n, dtype=np.uint32)
            _check(load_library().msbwt_count_kmers_fixed_u32(self.handle, _p(a), k, n, _p(out)), "count_kmers_fixed_u32")
            return out
        out = np.zeros(n, dtype=np.uint64)
        _check(load_library().msbwt_count_kmers_fixed(self.handle, _p(a), k, n, _p(out)), "count_kmers_fixed")
        return out

    @property
    def final_index(self) -> bool:
        """final-step image in use (msbwt_options.final_index)"""
        return bool(load_library().msbwt_final_index(self.handle))

    @property
    def final_bucket_shift(self) -> int:
        """log2 of the final-step image's bucket size, 0 without one"""
        if not self.final_index:
            return 0
        b = C.c_uint32(0)
        _check(load_library().msbwt_debug_copy_final_image(self.handle, 0, None, C.byref(b), None, None, None),
               "debug_copy_final_image")
        return int(b.value)

    def final_image(self, slot: int = 0) -> tuple[np.ndarray, int, int, int]:
        """(lines [nlines, 32] u32, bucket shift, log2 lines per bucket, overflowed lines) of the final-step image"""
        L = load_library()
        n, b, lb, over = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0), C.c_uint64(0)
        _check(L.msbwt_debug_copy_final_image(self.handle, slot, C.byref(n), C.byref(b), C.byref(lb), C.byref(over), None),
               "debug_copy_final_image")
        lines = np.zeros((n.value, 32), dtype=np.uint32)
        _check(L.msbwt_debug_copy_final_image(self.handle, slot, None, None, None, None, _p(lines)), "debug_copy_final_image")
        return lines, int(b.value), int(lb.value), int(over.value)

    def count_kmers_u64(self, kmers, k: int, counts32: bool = False) -> np.ndarray:
        """k-mers held as integers (k <= 32, first symbol in the most significant of the 2k bits, A,C,G,T = 0..3):
        8 bytes per query over the link instead of k.  `counts32`: u32 counts (index below 2^32 symbols)."""
        a = _u64(kmers).reshape(-1)
        if counts32:
            out = np.zeros(a.size, dtype=np.uint32)
            _check(load_library().msbwt_count_kmers_u64_u32(self.handle, _p(a), k, a.size, _p(out)), "count_kmers_u64_u32")
            return out
        out = np.zeros(a.size, dtype=np.uint64)
        _check(load_library().msbwt_count_kmers_u64(self.handle, _p(a), k, a.size, _p(out)), "count_kmers_u64")
        return out

    def constrain_ranges(self, sym, l, h) -> tuple[np.ndarray, np.ndarray]:
        s, lo, hi = _u8(sym).reshape(-1), _u64(l).reshape(-1), _u64(h).reshape(-1)
        if not (s.size == lo.size == hi.size):
            raise MsbwtError(EINVAL, "sym/l/h length mismatch")
        out_l = np.zeros(s.size, dtype=np.uint64)
        out_h = np.zeros(s.size, dtype=np.uint64)
        _check(load_library().msbwt_constrain_ranges(self.handle, _p(s), _p(lo), _p(hi), s.size, _p(out_l), _p(out_h)),
               "constrain_range")
        return out_l, out_h

    def constrain_ranges_fanout(self, l, h) -> tuple[np.ndarray, np.ndarray]:
        """The four `constrain_range` calls (A, C, G, T) of every range at once: (out_l[n,4], out_h[n,4])."""
        lo, hi = _u64(l).reshape(-1), _u64(h).reshape(-1)
        if lo.size != hi.size:
            raise MsbwtError(EINVAL, "l/h length mismatch")
        out_l = np.zeros((lo.size, 4), dtype=np.uint64)
        out_h = np.zeros((lo.size, 4), dtype=np.uint64)
        _check(load_library().msbwt_constrain_ranges_fanout(self.handle, _p(lo), _p(hi), lo.size, _p(out_l), _p(out_h)),
               "constrain_ranges_fanout")
        return out_l, out_h

    def count_read_kmers(self, reads, k: int, both_strands: bool = False) -> np.ndarray:
        """`count_kmer` of every k-mer window of every read (reads[n, read_len] symbol bytes): out[n, read_len-k+1];
        with `both_strands` each entry is count(window) + count(reverse_complement_i(window))."""
        a = _u8(reads)
        if a.ndim != 2:
            raise MsbwtError(EINVAL, "reads must be a 2-D array [n_reads, read_len]")
        n, L = a.shape
        if k < 1 or k > L:
            raise MsbwtError(EINVAL, "k must be in 1..read_len")
        out = np.zeros((n, L - k + 1), dtype=np.uint64)
        _check(load_library().msbwt_count_read_kmers(self.handle, _p(a), L, n, k, 2 if both_strands else 1, _p(out)),
               "count_read_kmers")
        return out

    def _kmer_spectrum(self, k: int, min_count: int, nbins: int, with_list: bool, canonical: bool = False):
        L = load_library()
        if k < 0 or min_count < 0 or nbins < 0:
            raise MsbwtError(EINVAL, "k, min_count and nbins must not be negative")
        hist = np.zeros(nbins, dtype=np.uint64)
        km, cn, n = C.c_void_p(0), C.c_void_p(0), C.c_uint64(0)
        fn = L.msbwt_kmer_spectrum_canonical if canonical else L.msbwt_kmer_spectrum
        _check(fn(self.handle, k, min_count, _p(hist) if nbins else None, nbins,
                  C.byref(km) if with_list else None, C.byref(cn) if with_list else None, C.byref(n)),
               "kmer_spectrum_canonical" if canonical else "kmer_spectrum")
        if not with_list:
            return hist, None, None
        try:
            kmers, counts = (np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(n.value,)).copy() if n.value
                             else np.zeros(0, np.uint64) for p in (km, cn))
        finally:
            L.msbwt_buffer_free(km)
            L.msbwt_buffer_free(cn)
        return hist, kmers, counts

    def kmer_spectrum(self, k: int, min_count: int = 1, nbins: int = 10001, canonical: bool = False) -> np.ndarray:
        """The k-mer spectrum: hist[c] = number of distinct ACGT k-mers (k <= 32) occurring exactly c times (count_kmer),
        the last bin holding those occurring nbins - 1 times or more; bins below min_count are 0.  Computed on the
        device by a pruned backward search; no k-mer crosses the link.  canonical=True counts each k-mer on both
        strands, once per pair {X, rc X}: count_kmer(X) + count_kmer(rc X), or count_kmer(X) for a palindrome
        (msbwt_kmer_spectrum_canonical), the spectrum `jellyfish count -C` gives for the reads."""
        return self._kmer_spectrum(k, min_count, nbins, False, canonical)[0]

    def list_kmers(self, k: int, min_count: int = 2, canonical: bool = False) -> tuple[np.ndarray, np.ndarray]:
        """(kmers u64, counts u64): every ACGT k-mer (k <= 32) with count_kmer >= min_count, as count_kmers_u64 takes
        them (A,C,G,T = 0..3, first symbol most significant), in co-lexicographic order (by the last symbol first).
        canonical=True: the canonical k-mers min(X, rc X) whose canonical count (see kmer_spectrum) is >= min_count,
        with that count, in a deterministic order and no other promised."""
        _, kmers, counts = self._kmer_spectrum(k, min_count, 0, True, canonical)
        return kmers, counts

    def unitigs(self, k: int, min_count: int = 2, canonical: bool = False) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(syms u8, offsets u64[n + 1], count_sums u64[n]): the unitigs of the compacted de Bruijn graph of the k-mers
        with count_kmer >= min_count (k <= 32; node-centric, msbwt_unitigs), ascending by first k-mer.  Unitig i is
        syms[offsets[i]:offsets[i + 1]] in the msbwt alphabet (convert_itos turns it into text); count_sums[i] sums the
        counts of its k-windows.  canonical=True: nodes are both members of every pair whose canonical count (see
        kmer_spectrum) is >= min_count, and each unitig is returned once per reverse-complement pair."""
        if k < 0 or min_count < 0:
            raise MsbwtError(EINVAL, "k and min_count must not be negative")
        L = load_library()
        s, o, c, n = C.c_void_p(0), C.c_void_p(0), C.c_void_p(0), C.c_uint64(0)
        _check(L.msbwt_unitigs(self.handle, k, min_count, 1 if canonical else 0, C.byref(s), C.byref(o), C.byref(c),
                               C.byref(n)), "unitigs")
        try:
            if not n.value:
                return np.zeros(0, np.uint8), np.zeros(1, np.uint64), np.zeros(0, np.uint64)
            offsets = np.ctypeslib.as_array(C.cast(o, C.POINTER(C.c_uint64)), shape=(n.value + 1,)).copy()
            sums = np.ctypeslib.as_array(C.cast(c, C.POINTER(C.c_uint64)), shape=(n.value,)).copy()
            syms = np.ctypeslib.as_array(C.cast(s, C.POINTER(C.c_uint8)), shape=(int(offsets[-1]),)).copy()
            return syms, offsets, sums
        finally:
            for p in (s, o, c):
                L.msbwt_buffer_free(p)

    def correct_reads(self, reads, k: int, min_count: int = 5, frac_permille: int = 100,
                      branch_limit: int = 4) -> tuple[list[np.ndarray], np.ndarray]:
        """Reads corrected against the index in the manner of fmlrc (msbwt_correct_reads; include/msbwt_gpu.h holds
        the definition): every weak run of k-mer windows inside a read is bridged through the k-mers whose
        both-strand count reaches the read's threshold, breadth-first, and replaced by the bridge closest to it in
        edit distance.  `reads`: a sequence of uint8 symbol arrays / strings over ACGNT, as build_rle_bwt_ragged takes.
        Returns (the corrected reads as uint8 arrays, stats u64[5]: weak runs, eligible runs, bridged, abandoned over
        the budget, eligible with no bridge)."""
        if k < 0 or min_count < 0 or frac_permille < 0 or branch_limit < 0:
            raise MsbwtError(EINVAL, "k, min_count, frac_permille and branch_limit must not be negative")
        L = load_library()
        arrs = [convert_stoi(r) if isinstance(r, (str, bytes)) else _u8(r).reshape(-1) for r in reads]
        offs = np.zeros(len(arrs) + 1, dtype=np.uint64)
        if arrs:
            np.cumsum([a.size for a in arrs], out=offs[1:])
        flat = _u8(np.concatenate(arrs)) if arrs and offs[-1] else np.zeros(1, np.uint8)
        s, o, stats = C.c_void_p(0), C.c_void_p(0), np.zeros(5, np.uint64)
        _check(L.msbwt_correct_reads(self.handle, _p(flat), _p(offs), len(arrs), k, min_count, frac_permille,
                                     branch_limit, C.byref(s), C.byref(o), _p(stats)), "correct_reads")
        try:
            o_arr = np.ctypeslib.as_array(C.cast(o, C.POINTER(C.c_uint64)), shape=(len(arrs) + 1,)).copy()
            total = int(o_arr[-1])
            syms = (np.ctypeslib.as_array(C.cast(s, C.POINTER(C.c_uint8)), shape=(total,)).copy() if total
                    else np.zeros(0, np.uint8))
        finally:
            L.msbwt_buffer_free(s)
            L.msbwt_buffer_free(o)
        return [syms[o_arr[r]:o_arr[r + 1]] for r in range(len(arrs))], stats

    # -- device-buffer entry points (raw pointers: torch `.data_ptr()` / stream handles)
    def count_kmers_fixed_device(self, d_syms: int, k: int, n: int, d_out: int, d_status: int = 0,
                                 stream: int = 0, slot: int = 0) -> None:
        _check(load_library().msbwt_count_kmers_fixed_device(self.handle, slot, d_syms, k, n, d_out, d_status or None,
                                                             stream or None), "count_kmers_fixed_device")

    def pack_kmers_device(self, d_syms: int, k: int, n: int, d_packed: int, d_out: int, d_status: int,
                          stream: int = 0, slot: int = 0) -> None:
        _check(load_library().msbwt_pack_kmers_device(self.handle, slot, d_syms, k, n, d_packed, d_out, d_status,
                                                      stream or None), "pack_kmers_device")

    def seed_kmers_u64_device(self, d_kmers: int, k: int, n: int, d_packed: int, d_out: int, stream: int = 0, slot: int = 0) -> None:
        """pack stage for device-resident k-mers held as 2-bit-per-symbol integers (k <= 32)"""
        _check(load_library().msbwt_seed_kmers_u64_device(self.handle, slot, d_kmers, k, n, d_packed, d_out, stream),
               "seed_kmers_u64_device")

    def count_kmers_packed_device(self, d_packed: int, k: int, n: int, d_out: int, stream: int = 0,
                                  slot: int = 0) -> None:
        _check(load_library().msbwt_count_kmers_packed_device(self.handle, slot, d_packed, k, n, d_out,
                                                              stream or None), "count_kmers_packed_device")

    def pack_stats(self, d_packed: int, k: int, n: int, slot: int = 0) -> dict:
        """what the last pack_kmers_device call on this scratch left for the search and what its one-request path did"""
        out = np.zeros(6, dtype=np.uint64)
        _check(load_library().msbwt_debug_pack_stats(self.handle, slot, d_packed, k, n, _p(out)), "debug_pack_stats")
        keys = ("live_a", "live_b", "final_lines", "final_overflowed", "two_buckets", "table_empty")
        return dict(zip(keys, (int(v) for v in out)))

    def count_kmers_packed_stats_device(self, d_packed: int, k: int, n: int, d_out: int, d_stats: int, stream: int = 0,
                                        slot: int = 0) -> None:
        """the search with the counting build of the oct kernel: d_stats = 8 u64 on the device (msbwt_gpu.h)"""
        _check(load_library().msbwt_count_kmers_packed_stats_device(self.handle, slot, d_packed, k, n, d_out, d_stats, stream),
               "count_kmers_packed_stats_device")

    def constrain_ranges_device(self, d_sym: int, d_l: int, d_h: int, n: int, d_out_l: int, d_out_h: int,
                                stream: int = 0, slot: int = 0) -> None:
        _check(load_library().msbwt_constrain_ranges_device(self.handle, slot, d_sym, d_l, d_h, n, d_out_l, d_out_h,
                                                            stream or None), "constrain_ranges_device")

    def packed_bytes(self, k: int, n: int) -> int:
        return int(load_library().msbwt_packed_bytes(self.handle, k, n))

    @property
    def suffix_table_s(self) -> int:
        return int(load_library().msbwt_suffix_table_s(self.handle))

    def device_image(self, slot: int = 0) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(blocks[nblocks,16] u32, aux[nblocks,2] u32, cbase[n_super,8] u64) copied back from the device."""
        L = load_library()
        nb, ns = C.c_uint64(0), C.c_uint32(0)
        _check(L.msbwt_debug_copy_image(self.handle, slot, C.byref(nb), C.byref(ns), None, None, None), "image")
        blocks = np.zeros((nb.value, 16), dtype=np.uint32)
        aux = np.zeros((nb.value, 2), dtype=np.uint32)
        cbase = np.zeros((ns.value, 8), dtype=np.uint64)
        _check(L.msbwt_debug_copy_image(self.handle, slot, C.byref(nb), C.byref(ns), _p(blocks), _p(aux), _p(cbase)),
               "image")
        return blocks, aux, cbase

    def pair_image(self, slot: int = 0) -> tuple[np.ndarray, np.ndarray]:
        """(lines[npair,32] u32, c2base[n_super2,16] u64) of the pair image, copied back from the device."""
        L = load_library()
        nb, ns = C.c_uint64(0), C.c_uint32(0)
        _check(L.msbwt_debug_copy_pair_image(self.handle, slot, C.byref(nb), C.byref(ns), None, None), "pair image")
        lines = np.zeros((nb.value, 32), dtype=np.uint32)
        c2base = np.zeros((ns.value, 16), dtype=np.uint64)
        _check(L.msbwt_debug_copy_pair_image(self.handle, slot, C.byref(nb), C.byref(ns), _p(lines), _p(c2base)),
               "pair image")
        return lines, c2base

    def quad_image(self, slot: int = 0) -> tuple[np.ndarray, np.ndarray]:
        """(sectors[256, nsec4, 8] u32, c4base[n_super4, 256] u64) of the quad image, copied back from the device."""
        L = load_library()
        nb, ns = C.c_uint64(0), C.c_uint32(0)
        _check(L.msbwt_debug_copy_quad_image(self.handle, slot, C.byref(nb), C.byref(ns), None, None), "quad image")
        sectors = np.zeros((256, nb.value, 8), dtype=np.uint32)
        c4base = np.zeros((ns.value, 256), dtype=np.uint64)
        _check(L.msbwt_debug_copy_quad_image(self.handle, slot, C.byref(nb), C.byref(ns), _p(sectors), _p(c4base)),
               "quad image")
        return sectors, c4base

    def oct_image(self, slot: int = 0) -> np.ndarray:
        """lines[4^m, nbuck8, 32] u32 of the oct image (m = oct_symbols()), copied back from the device."""
        L = load_library()
        nb = C.c_uint64(0)
        _check(L.msbwt_debug_copy_oct_image(self.handle, slot, C.byref(nb), None), "oct image")
        lines = np.zeros((4 ** oct_symbols(), nb.value, 32), dtype=np.uint32)
        _check(L.msbwt_debug_copy_oct_image(self.handle, slot, C.byref(nb), _p(lines)), "oct image")
        return lines

    @property
    def oct_index(self) -> bool:
        return bool(load_library().msbwt_oct_index(self.handle))

    @property
    def oct_overflow_lines(self) -> int:
        return int(load_library().msbwt_oct_overflow_lines(self.handle))

    @property
    def oct_overflow_occurrences(self) -> int:
        return int(load_library().msbwt_oct_overflow_occurrences(self.handle))

    @property
    def oct_runs(self) -> int:
        return int(load_library().msbwt_oct_runs(self.handle))

    def table_depth_for_k(self, k: int) -> int:
        """The suffix-table level an all-ACGT k-mer starts from (one of the kept levels, or 0)."""
        return int(load_library().msbwt_table_depth_for_k(self.handle, k))

    @property
    def oct_bucket_shift(self) -> int:
        return int(load_library().msbwt_oct_bucket_shift(self.handle))

    @property
    def quad_index(self) -> bool:
        return bool(load_library().msbwt_quad_index(self.handle))

    @property
    def pair_index(self) -> bool:
        return bool(load_library().msbwt_pair_index(self.handle))

    @property
    def kernel_lanes(self) -> int:
        return int(load_library().msbwt_kernel_lanes(self.handle))

    @property
    def index_bytes(self) -> int:
        return int(load_library().msbwt_index_bytes(self.handle))

    @property
    def device_ordinals(self) -> list[int]:
        L = load_library()
        return [L.msbwt_device_ordinal(self.handle, i) for i in range(L.msbwt_device_count(self.handle))]


def debug_build_image(rle, superblock_shift: int = 0) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Host-side block image (layout.h) of an RLE stream:
    (blocks[nblocks,16] u32, aux[nblocks,2] u32, cbase[n_super,8] u64).  Inspection only; needs no device."""
    L = load_library()
    a = _u8(rle)
    nb, ns = C.c_uint64(0), C.c_uint32(0)
    _check(L.msbwt_debug_build_image(_p(a), a.size, superblock_shift, C.byref(nb), C.byref(ns), None, None, None),
           "image")
    blocks = np.zeros((nb.value, 16), dtype=np.uint32)
    aux = np.zeros((nb.value, 2), dtype=np.uint32)
    cbase = np.zeros((ns.value, 8), dtype=np.uint64)
    _check(L.msbwt_debug_build_image(_p(a), a.size, superblock_shift, C.byref(nb), C.byref(ns), _p(blocks), _p(aux),
                                     _p(cbase)), "image")
    return blocks, aux, cbase


def build_rle_bwt(reads, device: int = 0, n_reads: int | None = None, read_len: int | None = None) -> tuple[np.ndarray, int]:
    """Multi-string BWT of equal-length reads, built on the GPU, as msbwt RLE bytes: what `msbwt2-build`
    writes for the same reads (sorted insertion; src/bin/msbwt2-build.rs, src/bwt_util.rs:154-171).
    `reads`: an [n, L] uint8 array of symbols 1..5, or a raw device pointer (int) with n_reads / read_len.
    Returns (rle bytes, total symbols)."""
    L = load_library()
    if isinstance(reads, int):
        ptr, on_dev, n, ln = C.c_void_p(reads), 1, int(n_reads), int(read_len)
        keep = None
    else:
        keep = _u8(reads)
        if keep.ndim != 2:
            raise MsbwtError(EINVAL, "reads must be an [n, L] array")
        n, ln = keep.shape
        ptr, on_dev = _p(keep), 0
    out, nbytes, total = C.c_void_p(0), C.c_uint64(0), C.c_uint64(0)
    _check(L.msbwt_build_rle_bwt(ptr, n, ln, on_dev, device, C.byref(out), C.byref(nbytes), C.byref(total)), "build_rle_bwt")
    try:
        rle = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(nbytes.value,)).copy() if nbytes.value else np.zeros(0, np.uint8)
    finally:
        L.msbwt_buffer_free(out)
    return rle, int(total.value)


def build_rle_bwt_ragged(reads, device: int = 0) -> tuple[np.ndarray, int]:
    """The same for reads of any lengths (`reads`: a sequence of uint8 symbol arrays / strings over ACGNT), in
    naive_bwt's order (src/bwt_util.rs:154-171).  Returns (rle bytes, total symbols = sum of length + 1)."""
    L = load_library()
    arrs = [convert_stoi(r) if isinstance(r, (str, bytes)) else _u8(r).reshape(-1) for r in reads]
    offs = np.zeros(len(arrs) + 1, dtype=np.uint64)
    if arrs:
        np.cumsum([a.size for a in arrs], out=offs[1:])
    flat = _u8(np.concatenate(arrs)) if arrs and offs[-1] else np.zeros(1, np.uint8)
    out, nbytes, total = C.c_void_p(0), C.c_uint64(0), C.c_uint64(0)
    _check(L.msbwt_build_rle_bwt_ragged(_p(flat), _p(offs), len(arrs), device, C.byref(out), C.byref(nbytes), C.byref(total)),
           "build_rle_bwt_ragged")
    try:
        rle = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(nbytes.value,)).copy() if nbytes.value else np.zeros(0, np.uint8)
    finally:
        L.msbwt_buffer_free(out)
    return rle, int(total.value)


def merge_rle_bwts(rle_a, rle_b, device: int = 0) -> tuple[np.ndarray, int, int]:
    """Merge two multi-string BWTs (msbwt RLE bytes) on the GPU: Holt and McMillan's interleave, as the reference's
    pairwise_bwt_merge (src/bwt_util.rs:108-141).  For BWTs built from reads the result is the BWT of the union of the
    read sets, byte for byte what build_rle_bwt(_ragged) makes from all the reads.  Returns (rle bytes, total symbols,
    interleave passes run -- the last of which changed nothing)."""
    L = load_library()
    a, b = _u8(rle_a).reshape(-1), _u8(rle_b).reshape(-1)
    out, nbytes, total, iters = C.c_void_p(0), C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
    _check(L.msbwt_merge_rle_bwts(_p(a) if a.size else None, a.size, _p(b) if b.size else None, b.size, device, C.byref(out),
                                  C.byref(nbytes), C.byref(total), C.byref(iters)), "merge_rle_bwts")
    try:
        rle = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(nbytes.value,)).copy() if nbytes.value else np.zeros(0, np.uint8)
    finally:
        L.msbwt_buffer_free(out)
    return rle, int(total.value), int(iters.value)


def convert_to_vec(text) -> np.ndarray:
    """bwt_converter.rs:26-80: a text BWT over `$ACGNT` (newlines skipped) -> msbwt RLE bytes"""
    raw = text.encode() if isinstance(text, str) else bytes(text)
    a = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(0, dtype=np.uint8)
    L = load_library()
    out, n = C.c_void_p(0), C.c_uint64(0)
    _check(L.msbwt_convert_to_rle(_p(a) if a.size else None, a.size, C.byref(out), C.byref(n)), "convert_to_vec")
    try:
        return np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(n.value,)).copy() if n.value else np.zeros(0, np.uint8)
    finally:
        L.msbwt_buffer_free(out)


def save_bwt_numpy(rle, filename: str) -> None:
    """bwt_converter.rs:102-130: the 96-byte header msbwt2 writes + the RLE bytes"""
    a = _u8(rle).reshape(-1)
    _check(load_library().msbwt_save_rle_npy(_p(a) if a.size else None, a.size, os.fsencode(filename)), "save_bwt_numpy")


def save_bwt_runs_numpy(runs, filename: str) -> None:
    """bwt_converter.rs:152-184: the same container from an iterable of (symbol, count) runs"""
    runs = list(runs)
    s = np.array([r[0] for r in runs], dtype=np.uint8)
    c = np.array([r[1] for r in runs], dtype=np.uint64)
    _check(load_library().msbwt_save_runs_npy(_p(s) if s.size else None, _p(c) if c.size else None, s.size, os.fsencode(filename)),
           "save_bwt_runs_numpy")


def l2_fetch_granularity(device: int, nbytes: int = 0) -> int:
    return int(load_library().msbwt_l2_fetch_granularity(device, nbytes))


def last_transfer_bytes() -> tuple[int, int]:
    """(host->device, device->host) bytes of the calling thread's last count_kmers_fixed."""
    a, b = C.c_uint64(0), C.c_uint64(0)
    load_library().msbwt_last_transfer_bytes(C.byref(a), C.byref(b))
    return int(a.value), int(b.value)


def debug_host_pack(syms, k: int, threads: int = 1) -> tuple[np.ndarray, np.ndarray]:
    """(words[ceil(k/32), n] u64, sorted exception indices) from the host-side 2-bit packer.  Needs no device."""
    a = _u8(syms).reshape(-1)
    n = a.size // k
    words = np.zeros((-(-k // 32), n), dtype=np.uint64)
    exc = np.zeros(max(n, 1), dtype=np.uint64)
    ne = C.c_uint64(0)
    _check(load_library().msbwt_debug_host_pack(_p(a), k, n, threads, _p(words), _p(exc), exc.size, C.byref(ne)),
           "host_pack")
    return words, np.sort(exc[:ne.value])


def host_pack_threads() -> int:
    return int(load_library().msbwt_host_pack_threads())


def launch_count() -> int:
    return int(load_library().msbwt_launch_count())


def gather_bench(device: int, d_buf: int, buf_bytes: int, granule: int, n_gathers: int, seed: int, d_sink: int,
                 stream: int = 0) -> None:
    _check(load_library().msbwt_gather_bench(device, d_buf, buf_bytes, granule, n_gathers, seed, d_sink,
                                             stream or None), "gather_bench")
