//! `GpuRleBWT`: the reference's `BWT` trait (src/msbwt_core.rs:28-162) over the CUDA engine,
//! plus the batched `count_kmers`.  UNVERIFIED (no Rust toolchain in the build image).
use std::ffi::{CStr, CString};
use std::io;
use std::ptr;

use crate::gpu_ffi as ffi;
use crate::msbwt_core::{BWTRange, BWT, VC_LEN};

pub struct GpuRleBWT {
    handle: *mut ffi::msbwt_index,
    devices: Vec<i32>,
}

// The handle is immutable after creation and the C ABI allows concurrent queries.
unsafe impl Send for GpuRleBWT {}
unsafe impl Sync for GpuRleBWT {}

fn last_error() -> String {
    unsafe { CStr::from_ptr(ffi::msbwt_last_error()).to_string_lossy().into_owned() }
}

impl GpuRleBWT {
    /// Mirrors `RleBWT::new()` (src/rle_bwt.rs:297-299); index lives on the current CUDA device.
    pub fn new() -> Self {
        Self { handle: ptr::null_mut(), devices: vec![] }
    }
    /// Replicate the index on these CUDA ordinals; batches are split across them.
    pub fn with_devices(devices: &[i32]) -> Self {
        Self { handle: ptr::null_mut(), devices: devices.to_vec() }
    }
    /// `bin_power` never changed results (src/rle_bwt.rs:309-322); accepted and ignored.
    pub fn with_bin_power(_bin_power: u8) -> Self {
        Self::new()
    }
    fn replace(&mut self, h: *mut ffi::msbwt_index) {
        if !self.handle.is_null() {
            unsafe { ffi::msbwt_index_destroy(self.handle) };
        }
        self.handle = h;
    }
    /// The batched entry point: one count per k-mer, same values as calling `count_kmer` on each.
    pub fn count_kmers(&self, kmers: &[Vec<u8>]) -> Vec<u64> {
        let mut offsets = Vec::with_capacity(kmers.len() + 1);
        let mut flat = Vec::with_capacity(kmers.iter().map(|k| k.len()).sum());
        offsets.push(0u64);
        for k in kmers {
            flat.extend_from_slice(k);
            offsets.push(flat.len() as u64);
        }
        let mut out = vec![0u64; kmers.len()];
        let rc = unsafe {
            ffi::msbwt_count_kmers(self.handle, flat.as_ptr(), offsets.as_ptr(), kmers.len() as u64, out.as_mut_ptr())
        };
        // the reference asserts on symbols >= VC_LEN (src/msbwt_core.rs:127)
        assert!(rc == ffi::MSBWT_OK, "count_kmers failed: {}", last_error());
        out
    }
    /// Flat fixed-k form (avoids 10^9 heap `Vec`s): `syms.len() == n * k`.
    pub fn count_kmers_fixed(&self, syms: &[u8], k: usize) -> Vec<u64> {
        assert!(k > 0 && syms.len() % k == 0);
        let n = syms.len() / k;
        let mut out = vec![0u64; n];
        let rc = unsafe { ffi::msbwt_count_kmers_fixed(self.handle, syms.as_ptr(), k as u32, n as u64, out.as_mut_ptr()) };
        assert!(rc == ffi::MSBWT_OK, "count_kmers_fixed failed: {}", last_error());
        out
    }
    /// K-mers the caller holds as 2-bit-per-symbol integers (k <= 32, first symbol most significant, A,C,G,T = 0..3):
    /// 8 bytes per query over the link instead of k.
    pub fn count_kmers_u64(&self, kmers: &[u64], k: usize) -> Vec<u64> {
        let mut out = vec![0u64; kmers.len()];
        let rc = unsafe { ffi::msbwt_count_kmers_u64(self.handle, kmers.as_ptr(), k as u32, kmers.len() as u64, out.as_mut_ptr()) };
        assert!(rc == ffi::MSBWT_OK, "count_kmers_u64 failed: {}", last_error());
        out
    }
    /// The same with 32-bit counts (index below 2^32 symbols): 4 bytes per query on the way back.
    pub fn count_kmers_u64_u32(&self, kmers: &[u64], k: usize) -> Vec<u32> {
        let mut out = vec![0u32; kmers.len()];
        let rc = unsafe { ffi::msbwt_count_kmers_u64_u32(self.handle, kmers.as_ptr(), k as u32, kmers.len() as u64, out.as_mut_ptr()) };
        assert!(rc == ffi::MSBWT_OK, "count_kmers_u64_u32 failed: {}", last_error());
        out
    }

    /// Reads corrected against the index in the manner of fmlrc (msbwt_correct_reads, include/msbwt_gpu.h): weak
    /// interior runs of k-mer windows bridged through the solid k-mers, and the five counters of the call.
    pub fn correct_reads(&self, reads: &[Vec<u8>], k: u32, min_count: u64, frac_permille: u32, branch_limit: u32) -> (Vec<Vec<u8>>, [u64; 5]) {
        let mut offsets = Vec::with_capacity(reads.len() + 1);
        offsets.push(0u64);
        let mut flat = Vec::new();
        for r in reads {
            flat.extend_from_slice(r);
            offsets.push(flat.len() as u64);
        }
        let (mut s, mut o, mut stats) = (ptr::null_mut(), ptr::null_mut(), [0u64; 5]);
        let rc = unsafe {
            ffi::msbwt_correct_reads(self.handle, flat.as_ptr(), offsets.as_ptr(), reads.len() as u64, k, min_count, frac_permille, branch_limit, &mut s, &mut o, stats.as_mut_ptr())
        };
        assert!(rc == ffi::MSBWT_OK, "correct_reads failed: {}", last_error());
        let out = unsafe {
            let o = std::slice::from_raw_parts(o, reads.len() + 1);
            let v = (0..reads.len()).map(|r| std::slice::from_raw_parts(s.add(o[r] as usize), (o[r + 1] - o[r]) as usize).to_vec()).collect();
            v
        };
        unsafe {
            ffi::msbwt_buffer_free(s);
            ffi::msbwt_buffer_free(o as *mut u8);
        }
        (out, stats)
    }
}

impl Default for GpuRleBWT {
    fn default() -> Self {
        Self::new()
    }
}

impl Drop for GpuRleBWT {
    fn drop(&mut self) {
        self.replace(ptr::null_mut());
    }
}

impl BWT for GpuRleBWT {
    fn load_vector(&mut self, bwt: Vec<u8>) {
        let mut err = 0;
        let h = unsafe {
            ffi::msbwt_index_create_from_rle(bwt.as_ptr(), bwt.len() as u64, self.devices.as_ptr(), self.devices.len() as i32, &mut err)
        };
        assert!(!h.is_null(), "load_vector failed ({}): {}", err, last_error());
        self.replace(h);
    }

    fn load_numpy_file(&mut self, filename: &str) -> io::Result<()> {
        let path = CString::new(filename).map_err(|e| io::Error::new(io::ErrorKind::InvalidInput, e))?;
        let mut err = 0;
        let h = unsafe { ffi::msbwt_index_create_from_npy(path.as_ptr(), self.devices.as_ptr(), self.devices.len() as i32, &mut err) };
        if h.is_null() {
            return match err {
                // where the reference returns Err(io::Error) (src/rle_bwt.rs:84,101-112,128-147)
                ffi::MSBWT_EIO => Err(io::Error::new(io::ErrorKind::UnexpectedEof, last_error())),
                // where the reference panics (src/rle_bwt.rs:91-93,115-125)
                ffi::MSBWT_EFORMAT => panic!("{}", last_error()),
                _ => Err(io::Error::new(io::ErrorKind::Other, last_error())),
            };
        }
        self.replace(h);
        Ok(())
    }

    fn get_symbol_count(&self, symbol: u8) -> u64 {
        assert!((symbol as usize) < VC_LEN);
        unsafe { ffi::msbwt_symbol_count(self.handle, symbol) }
    }

    fn get_total_size(&self) -> u64 {
        unsafe { ffi::msbwt_total_size(self.handle) }
    }

    unsafe fn constrain_range(&self, sym: u8, input_range: &BWTRange) -> BWTRange {
        let (mut l, mut h) = (0u64, 0u64);
        let rc = ffi::msbwt_constrain_ranges(self.handle, &sym, &input_range.l, &input_range.h, 1, &mut l, &mut h);
        assert!(rc == ffi::MSBWT_OK, "constrain_range failed: {}", last_error());
        BWTRange { l, h }
    }

    // override of the default loop (src/msbwt_core.rs:125-161): one launch instead of k round trips
    fn count_kmer(&self, kmer: &[u8]) -> u64 {
        let offsets = [0u64, kmer.len() as u64];
        let mut out = 0u64;
        let rc = unsafe { ffi::msbwt_count_kmers(self.handle, kmer.as_ptr(), offsets.as_ptr(), 1, &mut out) };
        assert!(rc == ffi::MSBWT_OK, "count_kmer failed: {}", last_error());
        out
    }
}
