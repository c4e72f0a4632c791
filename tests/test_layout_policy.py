"""The layout policy of index construction (capi.cu plan_layout) on its own, through msbwt_debug_plan_layout: which
images a replica gets, its suffix-table depth and its kernel lanes, from the options, the layout environment variables,
the index's size and the device's sizes.  The rules are restated below and compared at the sizes where they decide
something (1.5 to 4.6 Gsymbols on 8 to 180 GiB devices), which a GPU run reaches only with a very large index.
Needs no GPU."""
import ctypes as C

import pytest

import rust_msbwt_b200 as M

EINVAL = 1  # MSBWT_EINVAL, include/msbwt_gpu.h
GiB = 1 << 30
L2 = 126 << 20
FIELDS = ("table_s", "explicit_s", "hbm", "wide_oct", "quad", "oct", "fin", "pair", "keep_quad", "oct_required",
          "fin_required", "fin_lb", "lanes", "oct_shift", "fin_shift")
ENV = {"MSBWT_SUFFIX_TABLE_S": "suffix_table_s", "MSBWT_PAIR_INDEX": "pair_index", "MSBWT_QUAD_INDEX": "quad_index",
       "MSBWT_OCT_INDEX": "oct_index", "MSBWT_OCT_BUCKET_SHIFT": "oct_bucket_shift", "MSBWT_KEEP_QUAD": "keep_quad_index",
       "MSBWT_FINAL_INDEX": "final_index", "MSBWT_FINAL_BUCKET_SHIFT": "final_bucket_shift",
       "MSBWT_FINAL_LINES_LOG2": "final_lines_log2", "MSBWT_LANES": "kernel_lanes"}

CFG2, CFG4, WIDE_N = 1_510_000_000, 3_020_000_000, 4_600_000_000
# (N, wide): 64-bit positions for any N (several superblocks), and always from 2^32 symbols on
SIZES = [(n, w) for n in (10**6, 151_000_000, CFG2, CFG4) for w in (False, True)] + [(WIDE_N, True)]
DEVICES = {"8GiB": (8 * GiB, 7 * GiB + (600 << 20)), "80GiB": (80 * GiB, 79 * GiB), "180GiB": (180 * GiB, 178 * GiB)}
B200 = DEVICES["180GiB"]


@pytest.fixture(autouse=True)
def _no_layout_environment(monkeypatch):
    for var in ENV:
        monkeypatch.delenv(var, raising=False)


def options(**fields) -> M.Options:
    o = M.Options(C.sizeof(M.Options), 0, -1, -1, 0, -1, -1, 0, -1, -1, 0, 0)
    for name, value in fields.items():
        setattr(o, name, value)
    return o


def block_bytes(n: int, wide: bool) -> int:
    """the bare replica: 64-byte blocks + 8 bytes of aux per block + 8 u64 counts per superblock"""
    nblocks = n // 128 + 1
    return nblocks * 72 + (max(2, -(-n // 2**32)) if wide else 1) * 64


def plan(opts: M.Options, n: int, wide: bool, device) -> dict:
    total, free = device
    out = (C.c_int32 * len(FIELDS))()
    rc = M.load_library().msbwt_debug_plan_layout(C.byref(opts), n, int(wide), block_bytes(n, wide), L2, free, total,
                                                  out, len(FIELDS))
    assert rc == 0
    return dict(zip(FIELDS, out))


def quad_bytes(n):
    return 256 * (n // 224 + 2) * 32


def oct_bytes(n, b):
    return 4**10 * ((n >> b) + 1) * 128


def fin_bytes(n, b, lb):
    return (((n >> b) + 1) << lb) * 128


def reference(o: M.Options, n: int, wide: bool, device) -> dict:
    """The policy restated; `o` already holds what the environment sets.  "pinned" = 0 or 1."""
    total, free = device
    pinned = lambda v: v in (0, 1)  # noqa: E731
    explicit = o.suffix_table_s >= 0
    s = min(o.suffix_table_s, 15) if explicit else 0
    while not explicit and s < 13 and 4**s < n // 32:
        s += 1
    one_step = block_bytes(n, wide) + (4**s * (16 if wide else 8) if s else 0)
    hbm = one_step > 2 * L2
    wide_oct = wide and (o.oct_index == 1 or (
        o.oct_index != 0 and o.pair_index == -1 and o.quad_index == -1 and hbm and n < 2**40 and
        oct_bytes(n, 24) + fin_bytes(n, 16, 12) + 12 * n + 8 * GiB <= free))
    q = quad_bytes(n)
    narrow_oct = not wide and o.oct_index != 0
    if o.oct_index == 1 or o.quad_index == 1:
        quad = True
    elif o.quad_index == 0 or pinned(o.pair_index):
        quad = False
    else:
        quad = one_step > L2 and (q <= free // 100 * 65 if narrow_oct else q <= 64 * GiB and q <= free // 2)
    octi = quad and narrow_oct
    fin_shift = o.final_bucket_shift or 16
    return dict(
        table_s=s, explicit_s=explicit, hbm=hbm, wide_oct=wide_oct, quad=quad, oct=octi,
        fin=(octi or wide_oct) and o.final_index != 0,
        pair=not quad and (o.pair_index == 1 if pinned(o.pair_index) else hbm),
        keep_quad=o.keep_quad_index != 0 if o.keep_quad_index != -1 else q + 40 * n <= total // 10 * 7,
        oct_required=o.oct_index == 1, fin_required=o.final_index == 1,
        fin_lb=o.final_lines_log2 or (13 if fin_bytes(n, fin_shift, 13) <= total // 10 * 3 else 12),
        lanes=o.kernel_lanes if o.kernel_lanes in (1, 2) else (2 if hbm else 1),
        oct_shift=o.oct_bucket_shift, fin_shift=fin_shift)


SINGLE = [dict()] + [{f: v} for f in ("pair_index", "quad_index", "oct_index", "keep_quad_index", "final_index")
                     for v in (0, 1)]
SINGLE += [{"suffix_table_s": v} for v in (0, 1, 9, 16)] + [{"kernel_lanes": v} for v in (1, 2)]
SINGLE += [{"oct_bucket_shift": 18}, {"final_bucket_shift": 12}, {"final_lines_log2": 14}]
PAIRS = [{a: x, b: y} for a, b in (("pair_index", "quad_index"), ("oct_index", "pair_index"), ("oct_index", "quad_index"))
         for x in (0, 1) for y in (0, 1)]


@pytest.mark.parametrize("fields", SINGLE + PAIRS, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()) or "auto")
def test_plan_matches_the_stated_rules(fields):
    o = options(**fields)
    for n, wide in SIZES:
        for name, device in DEVICES.items():
            assert plan(o, n, wide, device) == reference(o, n, wide, device), (n, wide, name)


def test_configs2_index_on_a_b200_gets_quad_oct_and_final_and_keeps_quad():
    p = plan(options(), CFG2, False, B200)
    assert p["quad"] and p["oct"] and p["fin"] and p["keep_quad"] and not p["wide_oct"] and not p["pair"]
    assert p["lanes"] == 2 and p["table_s"] == 13 and not p["explicit_s"] and p["fin_lb"] == 13


def test_configs4_index_drops_the_quad_image():
    p = plan(options(), CFG4, False, B200)
    assert p["quad"] and p["oct"] and p["fin"] and not p["keep_quad"]


def test_wide_index_takes_the_wide_oct_route():
    p = plan(options(), WIDE_N, True, B200)
    assert p["wide_oct"] and p["fin"] and not p["oct_required"]
    # the images and the builders' scratch do not fit 8 GiB: the automatic route is not taken there
    assert not plan(options(), WIDE_N, True, DEVICES["8GiB"])["wide_oct"]


def test_index_that_fits_l2_gets_no_multi_step_image_and_one_lane():
    for wide in (False, True):
        p = plan(options(), 10**6, wide, B200)
        assert not (p["hbm"] or p["wide_oct"] or p["quad"] or p["oct"] or p["fin"] or p["pair"])
        assert p["lanes"] == 1


ENV_CASES = [("MSBWT_SUFFIX_TABLE_S", "9", 9), ("MSBWT_SUFFIX_TABLE_S", "-3", 0), ("MSBWT_SUFFIX_TABLE_S", "99", 15),
             ("MSBWT_LANES", "1", 1), ("MSBWT_LANES", "2", 2), ("MSBWT_LANES", "3", 1),
             ("MSBWT_PAIR_INDEX", "0", 0), ("MSBWT_PAIR_INDEX", "1", 1), ("MSBWT_PAIR_INDEX", "5", 1),
             ("MSBWT_QUAD_INDEX", "0", 0), ("MSBWT_QUAD_INDEX", "1", 1),
             ("MSBWT_OCT_INDEX", "0", 0), ("MSBWT_OCT_INDEX", "1", 1),
             ("MSBWT_OCT_BUCKET_SHIFT", "18", 18), ("MSBWT_KEEP_QUAD", "0", 0), ("MSBWT_KEEP_QUAD", "1", 1),
             ("MSBWT_FINAL_INDEX", "0", 0), ("MSBWT_FINAL_INDEX", "1", 1), ("MSBWT_FINAL_BUCKET_SHIFT", "12", 12),
             ("MSBWT_FINAL_LINES_LOG2", "14", 14)]


@pytest.mark.parametrize("var,value,field_value", ENV_CASES, ids=lambda x: str(x))
def test_each_variable_means_what_its_field_means(monkeypatch, var, value, field_value):
    want = {(n, w, d): plan(options(**{ENV[var]: field_value}), n, w, DEVICES[d]) for n, w in SIZES for d in DEVICES}
    monkeypatch.setenv(var, value)
    for (n, w, d), p in want.items():
        assert plan(options(), n, w, DEVICES[d]) == p, (n, w, d)


def test_a_field_the_caller_set_wins_over_its_variable(monkeypatch):
    set_by_caller = options(pair_index=1, kernel_lanes=1, suffix_table_s=7, oct_index=0)
    want = plan(set_by_caller, CFG2, False, B200)
    for var, value in (("MSBWT_PAIR_INDEX", "0"), ("MSBWT_LANES", "2"), ("MSBWT_SUFFIX_TABLE_S", "12"),
                       ("MSBWT_OCT_INDEX", "1")):
        monkeypatch.setenv(var, value)
    assert plan(set_by_caller, CFG2, False, B200) == want


def test_oct_index_variable_forces_the_oct_images(monkeypatch):
    """MSBWT_OCT_INDEX=1 builds the quad + oct images of an index that would get none, and requires the wide ones"""
    monkeypatch.setenv("MSBWT_OCT_INDEX", "1")
    p = plan(options(), 10**6, False, B200)
    assert p["quad"] and p["oct"] and p["fin"] and p["oct_required"]
    p = plan(options(), WIDE_N, True, DEVICES["8GiB"])
    assert p["wide_oct"] and p["oct_required"]


def test_pair_index_variable_pins_the_layout(monkeypatch):
    """MSBWT_PAIR_INDEX=0|1 keeps a configs[2]-size index off the quad route, as pair_index = 0|1 does"""
    for value in (0, 1):
        monkeypatch.setenv("MSBWT_PAIR_INDEX", str(value))
        p = plan(options(), CFG2, False, B200)
        assert not p["quad"] and not p["oct"] and p["pair"] == value


def test_quad_index_variable_goes_before_a_pinned_pair_index(monkeypatch):
    """quad_index is read before the "pair_index pinned" rule; MSBWT_QUAD_INDEX now is too"""
    monkeypatch.setenv("MSBWT_QUAD_INDEX", "1")
    p = plan(options(pair_index=0), CFG2, False, B200)
    assert p["quad"] and p["oct"] and not p["pair"]


def test_bad_arguments():
    L = M.load_library()
    out = (C.c_int32 * len(FIELDS))()
    args = (CFG2, 0, block_bytes(CFG2, False), L2, *B200[::-1])
    assert L.msbwt_debug_plan_layout(C.byref(options()), *args, out, len(FIELDS) - 1) == EINVAL
    assert L.msbwt_debug_plan_layout(C.byref(options()), *args, None, len(FIELDS)) == EINVAL
    short = options()
    short.struct_size = 8
    assert L.msbwt_debug_plan_layout(C.byref(short), *args, out, len(FIELDS)) == EINVAL
    assert L.msbwt_debug_plan_layout(None, *args, out, len(FIELDS)) == 0
    assert dict(zip(FIELDS, out)) == plan(options(), CFG2, False, B200)
