//! `extern "C"` bindings for include/msbwt_gpu.h -- UNVERIFIED (no Rust toolchain in the build image).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct msbwt_index {
    _private: [u8; 0],
}

/// `msbwt_options` (include/msbwt_gpu.h): which device images serve the path.  Results never depend on it.
#[repr(C)]
pub struct msbwt_options {
    pub struct_size: u32,
    pub superblock_shift: u32,
    pub suffix_table_s: i32,
    pub pair_index: i32,
    pub kernel_lanes: i32,
    pub quad_index: i32,
    pub oct_index: i32,
    pub oct_bucket_shift: i32,
    pub keep_quad_index: i32,     // ABI 4: -1 automatic
    pub final_index: i32,         // ABI 4: -1 automatic
    pub final_bucket_shift: i32,  // ABI 4: 0 default
    pub final_lines_log2: i32,    // ABI 4: 0 automatic
}

pub const MSBWT_OK: c_int = 0;
pub const MSBWT_EINVAL: c_int = 1;
pub const MSBWT_EIO: c_int = 2;
pub const MSBWT_EFORMAT: c_int = 3;
pub const MSBWT_ECUDA: c_int = 4;
pub const MSBWT_ENOMEM: c_int = 5;
pub const MSBWT_ENODEV: c_int = 6;

extern "C" {
    pub fn msbwt_index_create_from_rle(rle: *const u8, len: u64, devices: *const c_int, ndev: c_int, err: *mut c_int) -> *mut msbwt_index;
    pub fn msbwt_index_create_from_npy(path: *const c_char, devices: *const c_int, ndev: c_int, err: *mut c_int) -> *mut msbwt_index;
    pub fn msbwt_index_create_ex(rle: *const u8, len: u64, devices: *const c_int, ndev: c_int, superblock_shift: u32, suffix_table_s: c_int, err: *mut c_int) -> *mut msbwt_index;
    pub fn msbwt_index_create_opts(rle: *const u8, len: u64, devices: *const c_int, ndev: c_int, opts: *const msbwt_options, err: *mut c_int) -> *mut msbwt_index;
    pub fn msbwt_index_create_from_npy_opts(path: *const c_char, devices: *const c_int, ndev: c_int, opts: *const msbwt_options, err: *mut c_int) -> *mut msbwt_index;
    pub fn msbwt_index_destroy(idx: *mut msbwt_index);
    pub fn msbwt_total_size(idx: *const msbwt_index) -> u64;
    pub fn msbwt_symbol_count(idx: *const msbwt_index, sym: u8) -> u64;
    pub fn msbwt_start_index(idx: *const msbwt_index, sym: u8) -> u64;
    pub fn msbwt_device_count(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_device_ordinal(idx: *const msbwt_index, slot: c_int) -> c_int;
    pub fn msbwt_index_bytes(idx: *const msbwt_index) -> u64;
    pub fn msbwt_count_kmers(idx: *const msbwt_index, syms: *const u8, offsets: *const u64, n: u64, out: *mut u64) -> c_int;
    pub fn msbwt_count_kmers_fixed(idx: *const msbwt_index, syms: *const u8, k: u32, n: u64, out: *mut u64) -> c_int;
    pub fn msbwt_constrain_ranges(idx: *const msbwt_index, sym: *const u8, l: *const u64, h: *const u64, n: u64, out_l: *mut u64, out_h: *mut u64) -> c_int;
    pub fn msbwt_count_kmers_fixed_device(idx: *const msbwt_index, slot: c_int, d_syms: *const u8, k: u32, n: u64, d_out: *mut u64, d_status: *mut u32, stream: *mut c_void) -> c_int;
    pub fn msbwt_packed_bytes(idx: *const msbwt_index, k: u32, n: u64) -> u64;
    pub fn msbwt_suffix_table_s(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_kernel_lanes(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_pair_index(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_quad_index(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_oct_index(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_oct_bucket_shift(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_oct_symbols() -> c_int;
    pub fn msbwt_table_depth_for_k(idx: *const msbwt_index, k: u32) -> c_int;
    pub fn msbwt_debug_table_depth(k: u32, table_s: u32, steps: u32) -> c_int;
    pub fn msbwt_debug_plan_layout(opts: *const msbwt_options, total: u64, wide: c_int, block_bytes: u64, l2_bytes: u64, free_bytes: u64, device_bytes: u64, plan: *mut i32, nplan: c_int) -> c_int;
    pub fn msbwt_final_index(idx: *const msbwt_index) -> c_int;
    pub fn msbwt_debug_copy_final_image(idx: *const msbwt_index, slot: c_int, nlines: *mut u64, bucket_shift: *mut u32, lines_log2: *mut u32, overflow_lines: *mut u64, lines: *mut u32) -> c_int;
    pub fn msbwt_count_kmers_u64(idx: *const msbwt_index, kmers: *const u64, k: u32, n: u64, out: *mut u64) -> c_int;
    pub fn msbwt_count_kmers_fixed_u32(idx: *const msbwt_index, syms: *const u8, k: u32, n: u64, out: *mut u32) -> c_int;
    pub fn msbwt_count_kmers_u64_u32(idx: *const msbwt_index, kmers: *const u64, k: u32, n: u64, out: *mut u32) -> c_int;
    pub fn msbwt_seed_kmers_u64_device(idx: *const msbwt_index, slot: c_int, d_kmers: *const u64, k: u32, n: u64, d_packed: *mut u64, d_out: *mut u64, stream: *mut c_void) -> c_int;
    pub fn msbwt_debug_pack_stats(idx: *const msbwt_index, slot: c_int, d_packed: *const u64, k: u32, n: u64, out6: *mut u64) -> c_int;
    pub fn msbwt_count_kmers_packed_stats_device(idx: *const msbwt_index, slot: c_int, d_packed: *const u64, k: u32, n: u64, d_out: *mut u64, d_stats: *mut u64, stream: *mut c_void) -> c_int;
    pub fn msbwt_build_rle_bwt(reads: *const u8, n_reads: u64, read_len: u32, reads_on_device: c_int, device: c_int, rle: *mut *mut u8, rle_len: *mut u64, total: *mut u64) -> c_int;
    pub fn msbwt_build_rle_bwt_ragged(syms: *const u8, offsets: *const u64, n_reads: u64, device: c_int, rle: *mut *mut u8, rle_len: *mut u64, total: *mut u64) -> c_int;
    pub fn msbwt_merge_rle_bwts(rle_a: *const u8, len_a: u64, rle_b: *const u8, len_b: u64, device: c_int, rle: *mut *mut u8, rle_len: *mut u64, total: *mut u64, iterations: *mut u32) -> c_int;
    pub fn msbwt_kmer_spectrum(idx: *const msbwt_index, k: u32, min_count: u64, hist: *mut u64, nbins: u32, kmers: *mut *mut u64, counts: *mut *mut u64, n_kmers: *mut u64) -> c_int;
    pub fn msbwt_unitigs(idx: *const msbwt_index, k: u32, min_count: u64, canonical: c_int, syms: *mut *mut u8, offsets: *mut *mut u64, count_sums: *mut *mut u64, n_unitigs: *mut u64) -> c_int;
    pub fn msbwt_kmer_spectrum_canonical(idx: *const msbwt_index, k: u32, min_count: u64, hist: *mut u64, nbins: u32, kmers: *mut *mut u64, counts: *mut *mut u64, n_kmers: *mut u64) -> c_int;
    pub fn msbwt_correct_reads(idx: *const msbwt_index, syms: *const u8, offsets: *const u64, n_reads: u64, k: u32, min_count: u64, frac_permille: u32, branch_limit: u32, out_syms: *mut *mut u8, out_offsets: *mut *mut u64, stats: *mut u64) -> c_int;
    pub fn msbwt_buffer_free(p: *mut u8);
    pub fn msbwt_convert_to_rle(text: *const u8, n: u64, rle: *mut *mut u8, rle_len: *mut u64) -> c_int;
    pub fn msbwt_save_rle_npy(rle: *const u8, len: u64, path: *const c_char) -> c_int;
    pub fn msbwt_save_runs_npy(syms: *const u8, counts: *const u64, nruns: u64, path: *const c_char) -> c_int;
    pub fn msbwt_oct_runs(idx: *const msbwt_index) -> u64;
    pub fn msbwt_oct_overflow_lines(idx: *const msbwt_index) -> u64;
    pub fn msbwt_oct_overflow_occurrences(idx: *const msbwt_index) -> u64;
    pub fn msbwt_pack_kmers_device(idx: *const msbwt_index, slot: c_int, d_syms: *const u8, k: u32, n: u64, d_packed: *mut u64, d_out: *mut u64, d_status: *mut u32, stream: *mut c_void) -> c_int;
    pub fn msbwt_count_kmers_packed_device(idx: *const msbwt_index, slot: c_int, d_packed: *const u64, k: u32, n: u64, d_out: *mut u64, stream: *mut c_void) -> c_int;
    pub fn msbwt_constrain_ranges_device(idx: *const msbwt_index, slot: c_int, d_sym: *const u8, d_l: *const u64, d_h: *const u64, n: u64, d_out_l: *mut u64, d_out_h: *mut u64, stream: *mut c_void) -> c_int;
    pub fn msbwt_constrain_ranges_fanout(idx: *const msbwt_index, l: *const u64, h: *const u64, n: u64, out_l: *mut u64, out_h: *mut u64) -> c_int;
    pub fn msbwt_constrain_ranges_fanout_device(idx: *const msbwt_index, slot: c_int, d_l: *const u64, d_h: *const u64, n: u64, d_out_l: *mut u64, d_out_h: *mut u64, stream: *mut c_void) -> c_int;
    pub fn msbwt_count_read_kmers(idx: *const msbwt_index, reads: *const u8, read_len: u32, n_reads: u64, k: u32, strands: u32, out: *mut u64) -> c_int;
    pub fn msbwt_launch_count() -> u64;
    pub fn msbwt_l2_fetch_granularity(device: c_int, bytes: c_int) -> c_int;
    pub fn msbwt_host_alloc(bytes: usize) -> *mut c_void;
    pub fn msbwt_host_free(p: *mut c_void);
    pub fn msbwt_last_error() -> *const c_char;
    pub fn msbwt_abi_version() -> c_int;
}
