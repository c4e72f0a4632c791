/*
 * msbwt_gpu.h -- C ABI of the B200-native FM-index query engine for msbwt2's
 * run-length-encoded multi-string BWT.
 *
 * This is the drop-in boundary for ONE path of HudsonAlpha/rust-msbwt: the
 * `BWT` trait surface that `RleBWT` implements (src/msbwt_core.rs:28-162,
 * src/rle_bwt.rs:44-322) plus the batched `count_kmers` entry point.  A Rust
 * `extern "C"` module binds exactly these symbols (see INTEGRATION.md and
 * rust/src/gpu_ffi.rs).  Plain pointers and sizes only; the caller owns every
 * buffer it passes; the opaque handle owns the device-resident index replicas.
 *
 * There is no CPU fallback: if no CUDA device is usable, create fails with
 * MSBWT_ENODEV.
 *
 * Symbol alphabet (src/msbwt_core.rs:4-14): $=0 A=1 C=2 G=3 N=4 T=5, one symbol
 * per byte in every `syms` argument, exactly the `&[u8]` the reference takes.
 *
 * Thread-safety: a handle is immutable after create.  Concurrent query calls on
 * one handle are allowed; calls that target the same device serialise on an
 * internal per-device mutex (they share that device's staging workspace).
 * create/destroy must not race with queries on the same handle.
 */
#ifndef MSBWT_GPU_H
#define MSBWT_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSBWT_ABI_VERSION 4

/* Return codes.  The reference panics where we return EINVAL / EFORMAT; the
 * Rust shim turns those back into panics to keep trait behaviour
 * (src/msbwt_core.rs:127, src/rle_bwt.rs:91-93,115-125). */
enum msbwt_status {
    MSBWT_OK = 0,
    MSBWT_EINVAL = 1,  /* symbol >= 6, l > h, h > total_size, NULL where data is required */
    MSBWT_EIO = 2,     /* open / short read / size mismatch: where the reference returns io::Error
                          (src/rle_bwt.rs:84,101-112,128-147) */
    MSBWT_EFORMAT = 3, /* malformed .npy header or RLE symbol >= 6: where the reference panics */
    MSBWT_ECUDA = 4,   /* a CUDA call failed; msbwt_last_error() has the CUDA string */
    MSBWT_ENOMEM = 5,
    MSBWT_ENODEV = 6   /* no usable CUDA device (there is no CPU fallback) */
};

typedef struct msbwt_index msbwt_index;

/* ---- construction: RleBWT::new + BWT::load_vector / load_numpy_file ---- */

/* Replaces `RleBWT::new()` + `load_vector(Vec<u8>)` (src/rle_bwt.rs:59-66,297-299).
 * `rle` is the msbwt RLE byte stream (byte = sym | digit<<3, consecutive equal-sym
 * bytes are little-endian base-32 digits of one run).  The bytes are consumed
 * during the call (re-laid-out into the device block image) and not retained.
 * `devices`/`ndev`: CUDA ordinals to replicate the index on; ndev == 0 means the
 * calling thread's current device.  Returns NULL and sets *err on failure. */
msbwt_index *msbwt_index_create_from_rle(const uint8_t *rle, uint64_t len,
                                         const int *devices, int ndev, int *err);

/* Replaces `load_numpy_file` (src/rle_bwt.rs:81-155).  Same acceptance rules:
 * npy magic/version are not checked, header length is bytes 8..9 little-endian,
 * the data offset is rounded up to 16, dtype/fortran_order are ignored,
 * `shape[0]` must equal the remaining file size. */
msbwt_index *msbwt_index_create_from_npy(const char *path, const int *devices, int ndev, int *err);

/* Same as create_from_rle with explicit layout knobs (testing / tuning):
 * `superblock_shift` = log2(blocks per superblock), 0 selects the default (25:
 * 2^32 symbols per superblock).  The reference's only tuning knob, `bin_power`
 * (RleBWT::with_bin_power, src/rle_bwt.rs:309-322), has no effect on results
 * and no equivalent here: the device block covers a fixed 128 symbols.
 * `suffix_table_s`: depth of the suffix table -- the range after the first s backward-search
 * steps, precomputed for all 4^s ACGT suffixes (the `kmer_cache` the reference author planned
 * but never implemented, src/msbwt_core.rs:133-146); k-mers whose last s symbols are ACGT
 * start from it, bit-exactly.  -1 = automatic (ceil(log4(N/32)), at most 13 -- deepened up to 15 for
 * an index that lives in HBM, while the tables stay below 4x the block images and a quarter of the
 * free device memory), 0 = none, 1..15 explicit. */
msbwt_index *msbwt_index_create_ex(const uint8_t *rle, uint64_t len, const int *devices, int ndev,
                                   uint32_t superblock_shift, int suffix_table_s, int *err);

/* The same with every knob in one growable struct (set struct_size = sizeof(msbwt_options)).
 * `pair_index`: the PAIR image -- one 128-byte line per 96 BWT positions that answers TWO
 * constrain_range steps with one line fill (layout.h) -- is built next to the one-step blocks when
 * the index lives in HBM (-1 = automatic: one-step blocks + suffix table > 2 x L2), 0 = never,
 * 1 = always.  Results are identical either way.  `kernel_lanes`: 0 = automatic, 1 or 2 (see msbwt_kernel_lanes).
 * `quad_index`: the QUAD image -- one occurrence bit-vector per 4-symbol code in self-contained
 * 32-byte sectors (layout.h), FOUR constrain_range steps per line fill, 256*N/7 bytes -- replaces the
 * pair image (-1 = automatic: the index lives in HBM and the image is <= 64 GB and <= half the free
 * device memory), 0 = never, 1 = always.  Results are identical.
 * `oct_index`: the OCT image -- one 128-byte line of explicit occurrence RUNS per (m-symbol code, 2^b-position
 * bucket), m = msbwt_oct_symbols() = 10 constrain_range steps per line fill, 128 * 4^m * (N / 2^b + 1) bytes --
 * is built next to the quad image (-1 = automatic: whenever the quad image is built and the oct image fits a quarter
 * of the device memory left), 0 = never, 1 = always (implies quad_index).  An index
 * whose positions need 64 bits (2^32 symbols and more -- the reference is u64 throughout, src/msbwt_core.rs:18-24 --
 * or several superblocks) gets the same lines with 40-bit checkpoints, built by walking LF through the one-step
 * blocks, and no quad image (36.6 bytes per position have no room): automatic when it lives in HBM and the images
 * fit.  Lines that cannot hold their bucket's runs are answered through the quad image or one-symbol ranks, so
 * results are identical on any input.  `oct_bucket_shift`: b, 8..24 (0 = automatic: the largest b
 * that keeps the mean number of runs per line <= 6).  Under an oct image the automatic suffix-table depth is
 * 14 with levels 11..13 kept: a 31-mer is one L2-resident table entry (depth 11) + two oct lines.
 * `keep_quad_index` (under an oct image): the quad image is what the builders walk LF^4 with; afterwards it only
 * serves remainders of 4..9 symbols and the oct kernel's rare fallbacks, which one-symbol ranks answer as well.
 * -1 = automatic (kept when quad + 40 bytes per symbol for the other images fit 70 % of the device: 55 GB at
 * 1.51 Gsymbols; dropped at 3.02 Gsymbols, where it would be 110 GB), 0 = drop it once the images are built,
 * 1 = keep.  Results are identical either way.
 * `final_index`: the FINAL-STEP image on top of the oct image -- the LAST 20 symbols a count_kmer consumes need no
 * rank, only the number of positions of [l, h) preceded by those 20 symbols, so one hashed 128-byte line of explicit
 * runs per (20-symbol code, 2^16-position bucket) answers them: a 31-mer is one L2-resident depth-11 table entry +
 * ONE line fill.  -1 = automatic (built whenever the oct image is), 0 = never,
 * 1 = always (create fails if it cannot be built).  A line whose groups do not fit, or a range over two buckets,
 * takes the two oct steps instead, so results are identical on any input.  `final_bucket_shift` (8..16, 0 = 16) and
 * `final_lines_log2` (12..20 lines per bucket; 0 = automatic: 13 = 16 bytes per symbol when that fits 30 % of
 * the device memory, else 12 = 8 bytes per symbol).
 * Environment: ten variables set the same knobs for every create call, the ones without an msbwt_options
 * argument included -- MSBWT_SUFFIX_TABLE_S (suffix_table_s), MSBWT_PAIR_INDEX (pair_index), MSBWT_QUAD_INDEX
 * (quad_index), MSBWT_OCT_INDEX (oct_index), MSBWT_OCT_BUCKET_SHIFT (oct_bucket_shift), MSBWT_KEEP_QUAD
 * (keep_quad_index), MSBWT_FINAL_INDEX (final_index), MSBWT_FINAL_BUCKET_SHIFT (final_bucket_shift),
 * MSBWT_FINAL_LINES_LOG2 (final_lines_log2) and MSBWT_LANES (kernel_lanes).  One rule for all ten: a variable
 * applies only when its field is automatic (suffix_table_s < 0; pair_index, quad_index, oct_index,
 * keep_quad_index, final_index = -1; the shifts and final_lines_log2 = 0; kernel_lanes neither 1 nor 2), and then
 * means exactly what setting the field would.  Values are read as integers: the suffix table depth is clamped to
 * 0..15, any value of MSBWT_PAIR_INDEX / MSBWT_QUAD_INDEX / MSBWT_OCT_INDEX other than 0 means 1, and any value
 * of MSBWT_LANES other than 2 means 1. */
typedef struct msbwt_options {
    uint32_t struct_size;
    uint32_t superblock_shift; /* 0 = default */
    int32_t suffix_table_s;    /* -1 = automatic */
    int32_t pair_index;        /* -1 = automatic */
    int32_t kernel_lanes;      /* 0 = automatic */
    int32_t quad_index;        /* -1 = automatic (ABI 3; a caller's shorter ABI-2 struct means -1) */
    int32_t oct_index;         /* -1 = automatic (ABI 3) */
    int32_t oct_bucket_shift;  /* 0 = automatic (ABI 3) */
    int32_t keep_quad_index;   /* -1 = automatic (ABI 4; a caller's shorter struct means automatic for all four) */
    int32_t final_index;       /* -1 = automatic (ABI 4) */
    int32_t final_bucket_shift; /* 0 = default (ABI 4) */
    int32_t final_lines_log2;  /* 0 = automatic (ABI 4) */
} msbwt_options;
msbwt_index *msbwt_index_create_opts(const uint8_t *rle, uint64_t len, const int *devices, int ndev,
                                     const msbwt_options *opts, int *err);
/* load_numpy_file (src/rle_bwt.rs:81-155) with the same knobs; opts == NULL is msbwt_index_create_from_npy */
msbwt_index *msbwt_index_create_from_npy_opts(const char *path, const int *devices, int ndev,
                                              const msbwt_options *opts, int *err);

void msbwt_index_destroy(msbwt_index *idx);

/* ---- accessors: get_total_size / get_symbol_count (src/rle_bwt.rs:172-193) ---- */
uint64_t msbwt_total_size(const msbwt_index *idx);
uint64_t msbwt_symbol_count(const msbwt_index *idx, uint8_t sym); /* 0 for sym >= 6 */
/* start_index[sym] (the C array, src/rle_bwt.rs:374-381); total_size for sym >= 6 */
uint64_t msbwt_start_index(const msbwt_index *idx, uint8_t sym);
int msbwt_device_count(const msbwt_index *idx);
int msbwt_device_ordinal(const msbwt_index *idx, int slot);
uint64_t msbwt_index_bytes(const msbwt_index *idx); /* device bytes per replica, suffix table included */
int msbwt_suffix_table_s(const msbwt_index *idx);     /* suffix table depth in use (0 = none) */
/* lanes per query of the search kernel chosen for this index: 1 = one thread per query (index
 * L2-resident), 2 = a lane pair per query (index in HBM); msbwt_options.kernel_lanes sets it */
int msbwt_kernel_lanes(const msbwt_index *idx);
int msbwt_pair_index(const msbwt_index *idx); /* 1 when the pair image is in use */
int msbwt_quad_index(const msbwt_index *idx); /* 1 when the quad image is in use (it replaces the pair image) */
int msbwt_oct_index(const msbwt_index *idx);  /* 1 when the oct image is in use (with or without the quad image beside it) */
uint64_t msbwt_oct_overflow_lines(const msbwt_index *idx); /* oct lines answered through the quad image */
uint64_t msbwt_oct_overflow_occurrences(const msbwt_index *idx); /* BWT positions those lines cover */
uint64_t msbwt_oct_runs(const msbwt_index *idx);           /* runs of equal m-symbol codes in the BWT (chose b) */
int msbwt_oct_bucket_shift(const msbwt_index *idx);        /* b of the oct image in use, 0 without one */
int msbwt_oct_symbols(void);                               /* m: symbols (constrain_range steps) per oct line */
int msbwt_table_depth_for_k(const msbwt_index *idx, uint32_t k); /* suffix-table level an all-ACGT k-mer starts from */
/* final-step image (msbwt_options.final_index; specification: oracle/final_step.py): 1 when in use; the debug copy
 * returns its geometry and, when `lines` is not NULL, the lines themselves */
int msbwt_final_index(const msbwt_index *idx);
int msbwt_debug_copy_final_image(const msbwt_index *idx, int slot, uint64_t *nlines, uint32_t *bucket_shift,
                                 uint32_t *lines_log2, uint64_t *overflow_lines, uint32_t *lines /* nlines * 32, or NULL */);
/* the same policy without an index: `steps` = symbols per step of the image (1, 2, 4 or msbwt_oct_symbols()); -1 otherwise */
int msbwt_debug_table_depth(uint32_t k, uint32_t table_s, uint32_t steps);
/* The layout policy without a device: what create plans for one replica from `opts` (NULL = all automatic) and the
 * environment, for an index of `total` symbols (`wide` != 0: 64-bit positions) whose bare replica -- block image,
 * aux and superblock counts -- takes `block_bytes`, on a device with `l2_bytes` of L2, `free_bytes` free and
 * `device_bytes` in all.  plan[0..14] = suffix-table depth before the deepening for HBM, depth fixed by the caller or
 * the environment (not deepened), index in HBM, wide oct route, quad route, oct image on the quad route, final-step
 * image, pair image alone, keep the quad image under the oct image, oct image required, final-step image required,
 * log2 of final-step lines per bucket, kernel lanes, oct bucket shift (0 = automatic), final-step bucket shift.  The quad,
 * oct-on-quad and pair fields say what is built when the wide oct route is not taken or runs out of memory.
 * EINVAL when nplan < 15 or opts is invalid. */
int msbwt_debug_plan_layout(const msbwt_options *opts, uint64_t total, int wide, uint64_t block_bytes,
                            uint64_t l2_bytes, uint64_t free_bytes, uint64_t device_bytes, int32_t *plan, int nplan);

/* ---- queries from HOST buffers (the drop-in calls) ---- */

/* Batched BWT::count_kmer (src/msbwt_core.rs:125-161): query i is
 * syms[offsets[i] .. offsets[i+1]); out[i] = count.  An empty query counts
 * total_size.  Any symbol >= 6 anywhere in the batch -> MSBWT_EINVAL (the reference
 * asserts, src/msbwt_core.rs:127) and the contents of `out` are unspecified: symbols
 * are checked on the device while the batch streams through, never silently accepted.
 * The batch is split across the handle's devices. */
int msbwt_count_kmers(const msbwt_index *idx, const uint8_t *syms, const uint64_t *offsets,
                      uint64_t n, uint64_t *out);

/* Fixed-length form: query i is syms[i*k .. (i+1)*k).  This is the fast path.
 * How the batch reaches the device: with enough host threads (>= 8 usable by this process;
 * MSBWT_HOST_PACK=0|1 overrides, MSBWT_HOST_THREADS=n sets the pool size) a worker pool packs all-ACGT
 * k-mers 2 bits per symbol into pinned staging while earlier chunks are copied and searched, so the
 * link carries 8*ceil(k/32) bytes per query instead of k; k-mers holding any other symbol, and every
 * batch when the pool is off, are copied as bytes and packed / validated on the device.  Counts
 * are identical either way.  `syms` and `out` may be pageable or pinned (msbwt_host_alloc): pinned buffers are read
 * and written by the copy engines directly; pageable ones are staged chunk by chunk through pinned buffers of the
 * library by its worker threads (about half the throughput of pinned memory, host-memory-bound). */
int msbwt_count_kmers_fixed(const msbwt_index *idx, const uint8_t *syms, uint32_t k, uint64_t n,
                            uint64_t *out);
/* The same counts for k-mers the caller already holds as integers, 2 bits per symbol -- what k-mer counting
 * pipelines keep: k <= 32, kmers[i] = sum over j of code(s_j) << 2*(k-1-j) with A,C,G,T = 0,1,2,3 and s_0 the FIRST
 * symbol (bits above 2k are ignored); out[i] = BWT::count_kmer of that k-mer (src/msbwt_core.rs:125-161).  Nothing is
 * packed or validated anywhere (such a k-mer cannot hold `$` or `N`): the link carries 8 bytes per query each way
 * instead of k bytes in.  EINVAL when k == 0 or k > 32. */
int msbwt_count_kmers_u64(const msbwt_index *idx, const uint64_t *kmers, uint32_t k, uint64_t n, uint64_t *out);
/* 32-bit counts: the same two calls for an index below 2^32 symbols (a count can reach total_size; EINVAL
 * otherwise) -- the copy back to the host carries 4 bytes per query instead of 8. */
int msbwt_count_kmers_fixed_u32(const msbwt_index *idx, const uint8_t *syms, uint32_t k, uint64_t n, uint32_t *out);
int msbwt_count_kmers_u64_u32(const msbwt_index *idx, const uint64_t *kmers, uint32_t k, uint64_t n, uint32_t *out);
/* host->device and device->host bytes moved by the calling thread's last msbwt_count_kmers_fixed */
void msbwt_last_transfer_bytes(uint64_t *h2d, uint64_t *d2h);
int msbwt_host_pack_threads(void); /* size the packing pool would have in this process */

/* Batched BWT::constrain_range (src/rle_bwt.rs:202-287): for each i,
 * [out_l, out_h) = [C[sym]+rank(sym,l), C[sym]+rank(sym,h)).  The reference's
 * version is `unsafe` and unchecked; here sym >= 6, l > h or h > total_size
 * -> MSBWT_EINVAL with outputs untouched. */
int msbwt_constrain_ranges(const msbwt_index *idx, const uint8_t *sym, const uint64_t *l,
                           const uint64_t *h, uint64_t n, uint64_t *out_l, uint64_t *out_h);

/* ---- queries on DEVICE buffers (zero-copy callers, kernel-only timing) ----
 * `slot` indexes the handle's device list; all pointers must be device memory on
 * that device; `stream` is a cudaStream_t (NULL = legacy default stream).  The
 * call is asynchronous; `d_status` (device uint32, may be NULL) receives 0 or
 * MSBWT_EINVAL when a symbol >= 6 was seen (in which case d_out is unspecified). */
int msbwt_count_kmers_fixed_device(const msbwt_index *idx, int slot, const uint8_t *d_syms,
                                   uint32_t k, uint64_t n, uint64_t *d_out, uint32_t *d_status,
                                   void *stream);
int msbwt_constrain_ranges_device(const msbwt_index *idx, int slot, const uint8_t *d_sym,
                                  const uint64_t *d_l, const uint64_t *d_h, uint64_t n,
                                  uint64_t *d_out_l, uint64_t *d_out_h, void *stream);

/* The two stages of msbwt_count_kmers_fixed_device as separate calls, for callers that want to
 * time or overlap them (n <= 2^30 per pair; d_packed = msbwt_packed_bytes(idx,k,n) bytes of device
 * scratch, opaque):
 *   pack : validates the n*k symbol bytes, looks each k-mer's last symbols up in the suffix table -- and, when the
 *          index has a final-step image and the k-mer is a table entry + exactly 20 symbols (k = 31, 32), answers
 *          it right there from ONE 128-byte line (pack_seed_final_kernel) --,
 *          packs the remaining symbols 3 bits each (the k-mer's LAST symbol first, because backward
 *          search consumes it first), writes d_out[q] directly for k-mers that need no further
 *          search step (e.g. the table says "absent") and appends the rest to a compacted list;
 *   count: the backward search over that list; afterwards every d_out[q] is final. */
uint64_t msbwt_packed_bytes(const msbwt_index *idx, uint32_t k, uint64_t n);
int msbwt_pack_kmers_device(const msbwt_index *idx, int slot, const uint8_t *d_syms, uint32_t k,
                            uint64_t n, uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status,
                            void *stream);
/* the pack stage for k-mers already on the device as 2-bit-per-symbol integers (msbwt_count_kmers_u64's format, k <= 32):
 * nothing to validate; followed by msbwt_count_kmers_packed_device like msbwt_pack_kmers_device */
int msbwt_seed_kmers_u64_device(const msbwt_index *idx, int slot, const uint64_t *d_kmers, uint32_t k, uint64_t n,
                                uint64_t *d_packed, uint64_t *d_out, void *stream);
int msbwt_count_kmers_packed_device(const msbwt_index *idx, int slot, const uint64_t *d_packed,
                                    uint32_t k, uint64_t n, uint64_t *d_out, void *stream);
/* Measurement aid: what the last msbwt_pack_kmers_device on this scratch left for the search (out6[0] live list A,
 * [1] live list B) and what its one-request path did ([2] final-step lines fetched, [3] of which had overflowed,
 * [4] ranges over two buckets, [5] k-mers the suffix table answered with an empty range).  Synchronises the device. */
int msbwt_debug_pack_stats(const msbwt_index *idx, int slot, const uint64_t *d_packed, uint32_t k, uint64_t n,
                           uint64_t *out6);
/* Measurement aid (bench.py's roofline accounting): the search over the oct image with a counting build of the
 * kernel.  d_stats = 8 u64 on the device: oct lines fetched, final-step lines fetched, of which had overflowed,
 * quad steps, distinct 128-byte lines those read, one-symbol steps, distinct 64-byte blocks those read, queries
 * walked.  Counts land in d_out as usual.  EINVAL when the index has no oct image. */
int msbwt_count_kmers_packed_stats_device(const msbwt_index *idx, int slot, const uint64_t *d_packed, uint32_t k,
                                          uint64_t n, uint64_t *d_out, uint64_t *d_stats, void *stream);

/* Number of kernel launches the library has issued so far (all devices). */
uint64_t msbwt_launch_count(void);

/* ---- measurement aid: random-gather roofline microbenchmark (SURVEY.md 8d, K4) ----
 * Issues n_gathers (< 2^31) independent, uniformly random, `granule`-byte-aligned reads of
 * `granule` bytes (32, 64 or 128) over the largest power-of-two number of granules that
 * fits in `d_buf` (buf_bytes, device memory) on `stream`. */
int msbwt_gather_bench(int device, const void *d_buf, uint64_t buf_bytes, uint32_t granule,
                       uint64_t n_gathers, uint64_t seed, uint64_t *d_sink, void *stream);

/* cudaLimitMaxL2FetchGranularity of `device` (bytes, 0 = query only).  Returns the value in
 * effect afterwards, or a negative msbwt_status.  Measurement aid: on B200 an L2 miss of a
 * 32/64-byte request fills a whole 128-byte line by default. */
int msbwt_l2_fetch_granularity(int device, int bytes);

/* ---- inspection: the host-side block image (no device needed) ----
 * Builds the layout.h block image of `rle` exactly as create does and copies it out so
 * tests can check the loader without a GPU.  Call with the array pointers NULL to size:
 * *nblocks blocks of 16 u32 words, *nblocks pairs of u32 in aux, *n_super rows of 8 u64
 * in cbase. */
int msbwt_debug_build_image(const uint8_t *rle, uint64_t len, uint32_t superblock_shift,
                            uint64_t *nblocks, uint32_t *n_super, uint32_t *blocks, uint32_t *aux,
                            uint64_t *cbase);

/* Copies a replica's device-resident image out in the same form (NULL arrays: sizes only).  The image
 * is built on the device (builder.cu); tests compare it with the host builder's word for word. */
int msbwt_debug_copy_image(const msbwt_index *idx, int slot, uint64_t *nblocks, uint32_t *n_super,
                           uint32_t *blocks, uint32_t *aux, uint64_t *cbase);

/* The pair image of a replica: *npair lines of 32 u32 words; *n_super2 rows of 16 u64 in c2base
 * (0 rows when positions are 32-bit: the checkpoints are then absolute).  NULL arrays: sizes only. */
int msbwt_debug_copy_pair_image(const msbwt_index *idx, int slot, uint64_t *npair, uint32_t *n_super2,
                                uint32_t *lines, uint64_t *c2base);

/* The quad image of a replica: 256 * *nsec4 sectors of 8 u32 words, code-major; *n_super4 rows of 256 u64
 * in c4base (0 rows when positions are 32-bit).  NULL arrays: sizes only. */
int msbwt_debug_copy_quad_image(const msbwt_index *idx, int slot, uint64_t *nsec4, uint32_t *n_super4,
                                uint32_t *sectors, uint64_t *c4base);

/* ---- batched callers of the path (what a correction / assembly loop around msbwt2 does with it) ---- */

/* Fan-out: the four constrain_range calls of a backward-search extension at once.  For every input range i
 * and j = 0..3: (out_l[4*i+j], out_h[4*i+j]) = RleBWT::constrain_range(ACGT[j], [l[i], h[i]))
 * (src/rle_bwt.rs:202-287 called with sym = 1, 2, 3, 5); the index blocks holding l and h are fetched once
 * for the four symbols.  EINVAL (nothing written) when some l > h or h > total_size. */
int msbwt_constrain_ranges_fanout(const msbwt_index *idx, const uint64_t *l, const uint64_t *h, uint64_t n,
                                  uint64_t *out_l /* 4n */, uint64_t *out_h /* 4n */);
int msbwt_constrain_ranges_fanout_device(const msbwt_index *idx, int slot, const uint64_t *d_l, const uint64_t *d_h,
                                         uint64_t n, uint64_t *d_out_l, uint64_t *d_out_h, void *stream);

/* Pileup: BWT::count_kmer (src/msbwt_core.rs:125-161) of every k-mer window of every read.  `reads` =
 * n_reads * read_len symbol bytes (0..5); out[r * (read_len-k+1) + w] = count_kmer(reads[r][w .. w+k)) when
 * strands == 1, and count_kmer(window) + count_kmer(reverse_complement_i(window)) (src/string_util.rs:45-50)
 * when strands == 2.  Only the reads cross PCIe (read_len bytes per read instead of k per window); the
 * windows are laid out on the device and go through the same pack / search kernels as msbwt_count_kmers_fixed.
 * A read is never split across launches, so one read's (read_len-k+1) * strands * k window bytes must fit the
 * device; they may pass 2^32.
 * EINVAL when k == 0, k > read_len, strands not in {1,2}, (read_len-k+1) * strands >= 2^32 (nothing written) or a
 * symbol is >= 6 (found by the pack kernel, as for msbwt_count_kmers_fixed: `out` is then unspecified). */
int msbwt_count_read_kmers(const msbwt_index *idx, const uint8_t *reads, uint32_t read_len, uint64_t n_reads,
                           uint32_t k, uint32_t strands, uint64_t *out /* n_reads * (read_len-k+1) */);

/* The oct image of a replica: 4^m * *nbuck8 lines of 32 u32 words, code-major (nbuck8 = (N >> b) + 1).
 * NULL array: size only. */
int msbwt_debug_copy_oct_image(const msbwt_index *idx, int slot, uint64_t *nbuck8, uint32_t *lines);

/* The host-side 2-bit packer of the end-to-end path, on its own (no device needed): packs n k-mers of k
 * symbol bytes with `threads` workers into words[w * n + q], w < ceil(k/32) (the k-mer's last symbol in
 * the top bits of word 0, A,C,G,T = 0..3) and lists the queries holding any symbol outside ACGT
 * (*n_exceptions of them, the first max_exceptions written to `exceptions`, in no particular order). */
int msbwt_debug_host_pack(const uint8_t *syms, uint32_t k, uint64_t n, int threads, uint64_t *words,
                          uint64_t *exceptions, uint64_t max_exceptions, uint64_t *n_exceptions);

/* ---- building the BWT itself (the step before the query path; SURVEY.md 8f N2) ----
 * Multi-string BWT of `n_reads` reads of `read_len` symbols each (one symbol per byte, 1..5 = A,C,G,N,T;
 * 0 or >= 6 -> MSBWT_EINVAL), built on `device` and returned in the msbwt RLE byte format
 * (src/bwt_converter.rs:52-56) -- what `msbwt2-build` produces for the same reads with its default sorted
 * insertion (src/bin/msbwt2-build.rs:19-114, src/dynamic_bwt.rs:305-381), i.e. naive_bwt's order
 * (src/bwt_util.rs:154-171).  `reads` is host memory, or device memory on `device` when reads_on_device != 0.
 * *rle is a buffer of *rle_len bytes owned by the caller: release it with msbwt_buffer_free.
 * *total = n_reads * (read_len + 1). */
int msbwt_build_rle_bwt(const uint8_t *reads, uint64_t n_reads, uint32_t read_len, int reads_on_device,
                        int device, uint8_t **rle, uint64_t *rle_len, uint64_t *total);
/* The same for reads of ANY lengths (create_from_fastx takes them as they come, src/dynamic_bwt.rs:453-473): read r is
 * syms[offsets[r] .. offsets[r+1]) (host memory, n_reads + 1 offsets; an empty read contributes its `$` alone).
 * Order = naive_bwt's (src/bwt_util.rs:154-171): a suffix that ends sooner sorts first (`$` is the smallest symbol),
 * equal suffixes by the lexicographic rank of their whole reads.  *total = sum of (length + 1). */
int msbwt_build_rle_bwt_ragged(const uint8_t *syms, const uint64_t *offsets, uint64_t n_reads, int device,
                               uint8_t **rle, uint64_t *rle_len, uint64_t *total);
/* Merge two multi-string BWTs (pairwise_bwt_merge, src/bwt_util.rs:108-141): Holt and McMillan's interleave, run on
 * `device`.  `rle_a` / `rle_b` are host RLE byte streams, as msbwt_index_create_from_rle takes them (either may be
 * empty).  The result is the stable interleave of both inputs' rows by their infinite forward symbol sequences (rows
 * that tie keep A's before B's), in the canonical RLE encoding msbwt_build_rle_bwt emits.  For BWTs built from reads
 * it is the BWT of the union of the two read sets, byte for byte what msbwt_build_rle_bwt(_ragged) makes from all the
 * reads at once, and merge(A, B) == merge(B, A).  *rle is a buffer of *rle_len bytes owned by the caller (release it
 * with msbwt_buffer_free); *total = N_A + N_B; *iterations (may be NULL) = interleave passes run, the last of which
 * changed nothing (at most 2 L + 2 for reads of at most L symbols; 0 when both inputs are empty).
 * Device memory: about 0.82 byte per merged symbol while iterating (the two inputs' one-step block images, 0.56; two
 * interleave bit-vectors, 0.25), then 1 byte per merged symbol for the merged symbols plus the encoder's run table
 * (17 bytes per run) and the RLE bytes.  While an input is loaded, the loader's scan buffers come on top for a moment
 * (up to 26 bytes per RLE byte of that input, plus 0.56 byte per symbol).
 * EINVAL: a NULL output pointer, or a NULL input with a length above 0.  EFORMAT: an input holds a symbol >= 6 or a
 * run of 2^60 symbols or more, or N_A + N_B >= 2^62.  ENOMEM / ECUDA: nothing is leaked and *rle is NULL. */
int msbwt_merge_rle_bwts(const uint8_t *rle_a, uint64_t len_a, const uint8_t *rle_b, uint64_t len_b, int device,
                         uint8_t **rle, uint64_t *rle_len, uint64_t *total, uint32_t *iterations /* may be NULL */);
void msbwt_buffer_free(uint8_t *p);
/* The k-mer spectrum of the index, and optionally its k-mers.  S = every string X of k symbols over {A,C,G,T}
 * (1 <= k <= 32) with count_kmer(X) >= min_count (>= 1), count_kmer being BWT::count_kmer (src/msbwt_core.rs:125-161),
 * i.e. what msbwt_count_kmers_u64 returns for X; for a BWT built from reads, the occurrences of X inside the reads (X
 * never spans a read boundary or an N).  *n_kmers = |S|.  hist: nbins u64 (may be NULL when nbins == 0);
 * hist[c] = #{X in S : count = c} for c < nbins - 1 and hist[nbins - 1] = #{X in S : count >= nbins - 1}, so entries
 * below min_count and hist[0] are 0.  kmers / counts: both NULL (histogram only) or both non-NULL, in which case *kmers
 * and *counts become buffers of *n_kmers u64 owned by the caller (release each with msbwt_buffer_free; NULL when
 * *n_kmers == 0): S in msbwt_count_kmers_u64's encoding (A,C,G,T = 0..3, first symbol in the most significant of the
 * 2k bits, upper bits zero) in co-lexicographic order -- ascending by the last symbol, then the one before it, and so
 * on -- with their counts.  Two calls return identical arrays.
 * The walk is a depth-first backward search from [0, N) that extends every surviving range by A, C, G and T and drops
 * ranges narrower than min_count, over slices of at most B = 2^20 ranges per depth.  It reads only the one-step
 * blocks, so it works the same whatever images the index carries, and runs on the handle's first replica on a stream
 * and scratch of its own (it may run concurrently with queries on the same handle).
 * Device memory: at most (k - 1) * 4B stored ranges of 8 bytes (16 with 64-bit positions), plus 8 bytes each for the
 * packed k-mer when the list is requested, one slice's 4B children before compaction, 4B flag bytes, 2^22 staged
 * (k-mer, count) pairs of 16 bytes when the list is requested, nbins * 8 bytes and CUB's scratch: independent of N and
 * of |S| (and no buffer is larger than N / min_count entries).  At k = 31 with 32-bit positions: 1.0 GB for the
 * histogram, 2.1 GB with the list.  Host memory for the list grows with |S| (16 bytes per k-mer, and up to twice that
 * while a buffer grows).
 * EINVAL (nothing written): k == 0 or k > 32, min_count == 0, n_kmers NULL, hist NULL with nbins > 0, nbins == 1 or
 * nbins > 2^20, exactly one of kmers / counts NULL.  An index with no ACGT k-mer of length k (or min_count > N) gives
 * *n_kmers = 0 and an all-zero hist.  ENOMEM / ECUDA: nothing is leaked, nothing is left running on the device and
 * *kmers / *counts are NULL. */
int msbwt_kmer_spectrum(const msbwt_index *idx, uint32_t k, uint64_t min_count, uint64_t *hist, uint32_t nbins,
                        uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers);
/* The canonical k-mer spectrum: msbwt_kmer_spectrum with each k-mer counted on both strands, as `jellyfish count -C`
 * and KMC count the reads.  For a k-mer X in msbwt_count_kmers_u64's encoding, rc(X) reverses its k 2-bit groups and
 * maps each code c to 3 - c; canon(X) = min(X, rc(X)) as integers; the canonical count is
 * C(X) = count_kmer(X) + count_kmer(rc(X)) when X != rc(X), and count_kmer(X) when X is its own reverse complement (a
 * palindrome, possible for even k only).  S_c = { canon(X) : C(X) >= min_count }, each pair {X, rc(X)} once as its
 * canonical member; *n_kmers = |S_c|, hist counts C over S_c with msbwt_kmer_spectrum's bin rules (the last bin holds
 * C >= nbins - 1, bins below min_count and hist[0] are 0), and *kmers / *counts are S_c and its canonical counts.
 * Every N-free k-window of every read adds exactly 1 to exactly one canonical k-mer, so for an index built from reads
 * sum of c * hist[c] is the number of N-free k-windows, and reverse-complementing any subset of the reads before the
 * index is built changes neither S_c, nor the counts, nor hist.  This differs from msbwt_count_read_kmers with
 * strands == 2 on palindromes, which that call counts twice.  An index that already holds the reads' reverse
 * complements gets every count doubled here: for such an index msbwt_kmer_spectrum already is the two-strand spectrum.
 * Arguments, EINVAL cases (nothing written), ownership of the list (release each buffer with msbwt_buffer_free) and
 * concurrency are msbwt_kmer_spectrum's.  The list is in a deterministic order (two calls return identical arrays);
 * no other order is promised.
 * The walk is msbwt_kmer_spectrum's with the k-mer values, pruned at ceil(min_count / 2) (a pair reaching min_count has
 * a member counting at least that).  Its k-mers are staged on the device, 2^22 at a time, and each staged batch is
 * resolved there: the count of every rc(X) comes from the query path, so the call reads whatever images
 * msbwt_count_kmers_u64 reads (suffix table, oct and final-step images, one-step blocks), not only the one-step blocks.
 * Device memory: the list mode of msbwt_kmer_spectrum at min_count ceil(min_count / 2) (also for the histogram alone),
 * plus, per staged k-mer, 8 + 8 bytes for its reverse complement and that one's count, 1 flag byte and the query
 * path's scratch of 20 bytes (28 with 64-bit positions): 155 MB (189 MB) for 2^22 staged k-mers, fewer when the index
 * holds fewer than 2^22 * ceil(min_count / 2) symbols. */
int msbwt_kmer_spectrum_canonical(const msbwt_index *idx, uint32_t k, uint64_t min_count, uint64_t *hist,
                                  uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers);
/* The unitigs of the compacted de Bruijn graph of the solid k-mers (1 <= k <= 32), node-centric as in BCALM2 and
 * cuttlefish.  Nodes V: canonical == 0, the k-mers msbwt_kmer_spectrum lists (count_kmer(X) >= min_count);
 * canonical == 1, every X with C(X) >= min_count, C as in msbwt_kmer_spectrum_canonical, so both members of each pair
 * are nodes and V is closed under rc.  X -> Y is an edge iff X[1..k) = Y[0..k-1) and both are in V (the (k+1)-mer need
 * not occur; self-loops count toward the degrees), and it is compacted iff outdeg(X) = 1, indeg(Y) = 1 and X != Y.
 * Plain mode: every node lies on exactly one maximal path of compacted edges, its unitig.  A linear path starts at its
 * node with no compacted in-edge; a cycle of compacted edges is cut before its smallest node (by the integer value of
 * msbwt_count_kmers_u64's encoding), starts there and has |C| + k - 1 symbols.  Canonical mode: the plain unitigs of
 * that V, each unitig U kept iff first(U) <= first(U'), U' being the unitig holding rc(first(U)): one unitig per
 * reverse-complement pair and a self-reverse-complementary unitig once (for a linear U: first(U) <= rc(last(U)); for
 * a pair of cycles {C, rc C}: min(C) <= min(rc C)).  On an index that already holds both strands of its reads, plain
 * mode returns every unitig together with its reverse complement; on an index of the reads as they are, canonical
 * mode is what an assembler wants.
 * Outputs: *n_unitigs unitigs, strictly ascending by the value of their first k-mer.  *syms: their sequences one after
 * the other in the msbwt alphabet (A,C,G,T = 1,2,3,5, the bytes msbwt_count_kmers_fixed takes); *offsets: n + 1 u64,
 * unitig i = (*syms)[offsets[i], offsets[i + 1]); *count_sums[i] = the sum of count_kmer (C in canonical mode) over
 * its k-windows, so its mean abundance is count_sums[i] / (length - k + 1).  All three are owned by the caller
 * (release each with msbwt_buffer_free) and NULL when n == 0.  Two calls return identical arrays.
 * Runs on the handle's first replica with a stream and scratch of its own and takes no lock (it may run beside queries
 * on the same handle).  It lists V with the spectrum walk twice (a histogram-only pass sizes the device arrays the
 * second pass fills, so no k-mer crosses the link), radix-sorts it, links every node by one binary search, ranks the
 * unitigs by pointer jumping and writes them out on the device.  Device memory: the spectrum's walk (see
 * msbwt_kmer_spectrum) on top of V's 32 bytes per node while V is listed, then 53 bytes per node (53.1-53.3 measured
 * at 58-727 M nodes on configs[2] on a B200, tools/unitig_bench.py) (keys, counts and the sort's alternates 32, links 8,
 * offsets and numbers 12, a flag 1), 16 more while cycles of compacted edges are cut, then the outputs (16 bytes per
 * unitig and its symbols) in place of the counts (8 per node).  Canonical mode doubles the node count against the
 * canonical spectrum's list.
 * EINVAL (nothing written): bad handle, k == 0 or k > 32, min_count == 0, canonical not 0 or 1, any output pointer
 * NULL.  ENOMEM / ECUDA: nothing is leaked, nothing is left running, the outputs are NULL / 0; a V of 2^32 nodes or
 * more (node ids are 32-bit) is ENOMEM. */
int msbwt_unitigs(const msbwt_index *idx, uint32_t k, uint64_t min_count, int canonical, uint8_t **syms,
                  uint64_t **offsets, uint64_t **count_sums, uint64_t *n_unitigs);
/* Read correction against the index in the manner of fmlrc (not bit-compatible with fmlrc2): weak runs of a read's
 * k-mer windows are bridged through the de Bruijn graph of the solid k-mers, breadth-first.  Read r is
 * syms[offsets[r] .. offsets[r+1]) over A,C,G,N,T = 1,2,3,4,5, reads of any lengths.  Parameters: k in 1..32,
 * min_count >= 1, frac_permille in 0..1000 (fmlrc's frac 0.1 is 100), branch_limit >= 1 (fmlrc's branch-limit factor,
 * 4 there).  Each read is corrected on its own, from the counts of the read as given:
 *  1. Window counts.  Windows w = 0 .. nwin-1, nwin = len - k + 1, window w = read[w .. w+k).  A window holding N has
 *     count2 = 0; otherwise count2(X) = count_kmer(X) + count_kmer(rc X), what msbwt_count_read_kmers(strands = 2)
 *     gives (a palindrome counts twice).  Reads shorter than k + 2 are returned unchanged.
 *  2. Threshold.  v = the ascending list of the read's non-zero count2 values, m its length.  m = 0: the read is
 *     unchanged.  Otherwise T = max(min_count, floor(v[floor(m/2)] * frac_permille / 1000)), in integers.
 *  3. Weak runs.  A window is weak when count2 < T; a weak run is a maximal run [a, b) of weak windows.  It is
 *     eligible when 1 <= a, b <= nwin - 1 and b - a >= k - 1: then X = window a-1 is its solid seed, Y = window b its
 *     solid target, and P = read[a-1+k .. b) the bases between them, of length L0 = b - a + 1 - k >= 0 (a substitution
 *     gives L0 = 1, a deletion 0, an insertion 1).  Runs that touch either end of the read, or are shorter than k - 1
 *     windows, are left as they are.
 *  4. Bridges.  Emax = floor(13 L0 / 10) + 2.  A walk is a string over ACGT that starts with X and whose every
 *     k-window Z has count2(Z) >= T; walks grow breadth-first, one symbol per round, for rounds t = 1 .. k + Emax.  At
 *     round t >= k a walk whose newest window is Y is a bridge S = X E Y with |E| = t - k and is not extended; every
 *     other walk is extended at the next round (also one that meets Y before round k).  The gap's work is the number
 *     of walks created over all rounds (bridges included, X not); when it exceeds branch_limit * (k + Emax) the gap is
 *     abandoned and left unchanged, even if bridges were found.
 *  5. Choice.  Among the bridges, the E with the smallest Levenshtein distance to P (unit costs over symbol codes; an
 *     N in P matches nothing); ties go to the shorter E, then to the lexicographically smaller (A < C < G < T).  No
 *     bridge: unchanged.  Otherwise P is replaced by E (E != P, since X P Y holds a weak window).  All gaps of a read
 *     are decided from the read as given and applied together (their P's are disjoint).
 * Outputs: *out_syms and *out_offsets (n_reads + 1 u64, from 0) hold the corrected reads in input order in the same
 * ragged form; release both with msbwt_buffer_free.  stats (u64[5], may be NULL), summed over the call: [0] weak runs,
 * [1] eligible runs, [2] bridged (replaced), [3] abandoned over the budget, [4] eligible runs with no bridge.
 * The result depends only on the index's counts and the reads: not on chunking, the number of replicas or which
 * images the index carries.
 * Not covered: runs at either end of a read (they need an open-ended extension rule), k > 32 (fmlrc's second pass at
 * K = 59), fmlrc2's depth-first order and choice rules.  fmlrc's two passes are two calls.
 * The reads are split into one contiguous slice per replica; each replica corrects its slice on its own stream and
 * scratch in chunks of whole reads of about 2^22 symbols, and takes no lock (the call may run beside queries on the
 * same handle).  Per chunk everything runs on the device: window counts through the query path, per-read medians by a
 * segmented sort, weak runs, one breadth-first search over every gap of the chunk (each round's 4 children x 2 strands
 * counted in one batch, one small read-back per round), Levenshtein scoring per bridge and the assembly of the new
 * reads.  Device memory per replica follows the chunk, not the batch: the buffers hold about 130 bytes per chunk
 * symbol (the query path's scratch for two queries per symbol included) and about 500 per walk of the widest round,
 * and grow by half again when a chunk needs more.  Measured peaks (tools/correct_bench.py, configs[2]'s index on a
 * B200): 0.27-0.36 GB for one chunk of 2 M symbols of 10 kbp reads, 0.94-1.10 GB for chunks of 2^22 symbols of
 * 150 bp reads.  A read longer than 2^22 symbols is a chunk of its own.
 * EINVAL (nothing written): bad handle, k outside 1..32, min_count == 0, frac_permille > 1000, branch_limit == 0,
 * a NULL output pointer, NULL syms / offsets with n_reads > 0, decreasing offsets, a read of 2^31 symbols or more, or
 * a symbol 0 ($) or >= 6.  ENOMEM / ECUDA: nothing is leaked and nothing is left running; one chunk whose walks need
 * 2^32 node ids or more is ENOMEM. */
int msbwt_correct_reads(const msbwt_index *idx, const uint8_t *syms, const uint64_t *offsets, uint64_t n_reads,
                        uint32_t k, uint64_t min_count, uint32_t frac_permille, uint32_t branch_limit,
                        uint8_t **out_syms, uint64_t **out_offsets, uint64_t *stats);

/* ---- the data format either side of the path: src/bwt_converter.rs ----
 * convert_to_vec (:26-80): a text BWT over `$ACGNT` (newlines are skipped and do not end a run) -> msbwt RLE bytes
 * (malloc'd: release with msbwt_buffer_free).  Any other byte -> MSBWT_EFORMAT (the reference panics, :43-46). */
int msbwt_convert_to_rle(const uint8_t *text, uint64_t n, uint8_t **rle, uint64_t *rle_len);
/* save_bwt_numpy (:102-130): the 96-byte npy-v1 header msbwt2 writes -- `{'descr': '|u1', 'fortran_order': False,
 * 'shape': (<len>, ), }` padded with spaces, newline-terminated -- followed by the RLE bytes, byte for byte what the
 * reference writes and what msbwt_index_create_from_npy / load_numpy_file read.  MSBWT_EIO on any file error. */
int msbwt_save_rle_npy(const uint8_t *rle, uint64_t len, const char *path);
/* save_bwt_runs_numpy (:152-184): the same container from (symbol, count) runs; a zero count writes nothing */
int msbwt_save_runs_npy(const uint8_t *syms, const uint64_t *counts, uint64_t nruns, const char *path);

/* ---- pinned host buffers for callers that want full copy/compute overlap ---- */
void *msbwt_host_alloc(size_t bytes);
void msbwt_host_free(void *p);

/* Thread-local description of the last failure in the calling thread ("" if none). */
const char *msbwt_last_error(void);
int msbwt_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MSBWT_GPU_H */
