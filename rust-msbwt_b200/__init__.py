"""rust-msbwt_b200 -- B200-native batched FM-index queries for msbwt2's RLE multi-string BWT.

The package holds only the hot path named in BASELINE.json: `csrc/` (sm_100a kernels +
the C ABI of include/msbwt_gpu.h, built in-tree into libmsbwt_b200.so) and `rle_bwt.py`,
the host-side mirror of the reference's `RleBWT` / `BWT` trait
(src/rle_bwt.rs:14-322, src/msbwt_core.rs:28-162) over that C ABI.

The directory name carries a hyphen, so import it as `rust_msbwt_b200` (the shim module
of that name at the repo root loads this package).
"""
from .rle_bwt import (  # noqa: F401
    BWTRange,
    build_rle_bwt,
    build_rle_bwt_ragged,
    merge_rle_bwts,
    MsbwtError,
    RleBWT,
    convert_itos,
    convert_stoi,
    convert_to_vec,
    save_bwt_numpy,
    save_bwt_runs_numpy,
    debug_build_image,
    debug_host_pack,
    gather_bench,
    host_pack_threads,
    last_transfer_bytes,
    Options,
    launch_count,
    l2_fetch_granularity,
    EXPORTED_SYMBOLS,
    library_path,
    load_library,
    oct_symbols,
    reverse_complement_i,
)
from . import build as _build  # noqa: F401


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a with nvcc (in-tree)."""
    return _build.build(force=force, verbose=verbose)
