"""msbwt_index_bytes: the device memory an index reports is the sum of the images it holds -- the one-step blocks,
the pair, quad, oct and final-step images and the kept suffix-table levels -- for every layout the options select.
The image sizes come from the debug accessors (called with NULL buffers), the table levels from the depth rule of
capi.cu build_suffix_table: level s, plus the 3 levels below it under a quad or oct image, 1 under a pair image
only, never below level 1; 8 bytes per entry, 16 with 64-bit positions."""
import ctypes as C

import pytest

import rust_msbwt_b200 as M

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def rle():
    from harness import bwt_build, synth
    reads = synth.make_reads(40000, read_len=100, coverage=25.0, error_rate=0.01, device="cuda")
    return bwt_build.build_rle_bwt(reads)[0].cpu().numpy()


def expected_bytes(g) -> int:
    L = M.load_library()
    h = g.handle
    u64, u32 = C.c_uint64(0), C.c_uint32(0)
    assert L.msbwt_debug_copy_image(h, 0, C.byref(u64), C.byref(u32), None, None, None) == 0
    nblocks, n_super = u64.value, u32.value
    total = nblocks * 64 + nblocks * 2 * 4 + n_super * 8 * 8
    if g.pair_index:
        assert L.msbwt_debug_copy_pair_image(h, 0, C.byref(u64), C.byref(u32), None, None) == 0
        total += u64.value * 128 + u32.value * 16 * 8
    if g.quad_index:
        assert L.msbwt_debug_copy_quad_image(h, 0, C.byref(u64), C.byref(u32), None, None) == 0
        total += 256 * u64.value * 32 + u32.value * 256 * 8
    if g.oct_index:
        assert L.msbwt_debug_copy_oct_image(h, 0, C.byref(u64), None) == 0
        total += 4 ** M.oct_symbols() * u64.value * 128
    if g.final_index:
        assert L.msbwt_debug_copy_final_image(h, 0, C.byref(u64), None, None, None, None) == 0
        total += u64.value * 128
    s = g.suffix_table_s
    if s > 0:
        wide = n_super > 1 or g.get_total_size() >= 1 << 32
        lower = 3 if (g.quad_index or g.oct_index) else (1 if g.pair_index else 0)
        total += sum(4 ** j for j in range(max(1, s - lower), s + 1)) * (16 if wide else 8)
    return total


# (options, (pair, quad, oct, final) flags the index ends up with)
LAYOUTS = [
    ({}, (0, 0, 0, 0)),
    ({"pair_index": 1}, (1, 0, 0, 0)),
    ({"quad_index": 1}, (0, 1, 1, 1)),
    ({"oct_index": 1}, (0, 1, 1, 1)),
    ({"oct_index": 1, "keep_quad_index": 0}, (0, 0, 1, 1)),
    ({"oct_index": 1, "final_index": 0}, (0, 1, 1, 0)),
    ({"suffix_table_s": 0}, (0, 0, 0, 0)),
    ({"superblock_shift": 5, "oct_index": 1}, (0, 0, 1, 1)),  # 64-bit positions: the wide oct and final-step images
]


@pytest.mark.parametrize("opts,flags", LAYOUTS, ids=[",".join(f"{k}={v}" for k, v in o.items()) or "default" for o, _ in LAYOUTS])
def test_index_bytes_is_the_sum_of_the_images(rle, opts, flags):
    g = M.RleBWT(**opts)
    g.load_vector(rle)
    assert (g.pair_index, g.quad_index, g.oct_index, g.final_index) == tuple(bool(f) for f in flags)
    if "suffix_table_s" in opts:
        assert g.suffix_table_s == opts["suffix_table_s"]
    else:
        assert g.suffix_table_s > 0
    assert g.index_bytes == expected_bytes(g)
