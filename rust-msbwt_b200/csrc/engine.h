// engine.h -- internal interface between the C ABI (capi.cu), the host-side layout
// builder (loader.cu) and the kernels (kernels.cu).
//
// Errors and launch counts are reported where they happen.  A failing function returns an msbwt_status and leaves
// its message in g_last_error (msbwt_last_error) through fail() or CU_TRY.  Every launch wrapper, image builder and the
// spectrum add the kernels they launch to g_launches (msbwt_launch_count); the block image of create (builder.cu) is
// the one build step that is not counted.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/msbwt_gpu.h"
#include "layout.h"

namespace msbwt {

extern thread_local std::string g_last_error;
extern std::atomic<uint64_t> g_launches;

inline int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

// return MSBWT_ENOMEM (out of device memory) or MSBWT_ECUDA, with "<prefix><expr>: <CUDA error>" as the message
#define CU_TRY_IN(prefix, expr)                                                                   \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(e_ == cudaErrorMemoryAllocation ? MSBWT_ENOMEM : MSBWT_ECUDA,             \
                        std::string(prefix) + #expr + ": " + cudaGetErrorString(e_));            \
    } while (0)
#define CU_TRY(expr) CU_TRY_IN("", expr)

// one cudaMalloc'd buffer, freed when it goes out of scope unless release()d
struct CudaFree {
    void operator()(void *p) const { cudaFree(p); }
};
template <class T> using DevicePtr = std::unique_ptr<T, CudaFree>;

// cudaMalloc'd scratch buffers of one build step: whatever is still listed is freed when it goes out of scope
struct DeviceScratch {
    std::vector<void *> ptrs;
    DeviceScratch() = default;
    DeviceScratch(const DeviceScratch &) = delete;
    DeviceScratch &operator=(const DeviceScratch &) = delete;
    ~DeviceScratch() { release_all(); }
    template <class T> cudaError_t alloc(T **p, size_t count) {
        cudaError_t e = cudaMalloc((void **)p, (count ? count : 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    void release(void *p) {
        auto it = std::find(ptrs.begin(), ptrs.end(), p);
        if (it != ptrs.end()) { cudaFree(p); ptrs.erase(it); }
    }
    // unlists p without freeing it: whoever it is handed to owns it from here on
    template <class T> T *take(T *p) {
        auto it = std::find(ptrs.begin(), ptrs.end(), (void *)p);
        if (it != ptrs.end()) ptrs.erase(it);
        return p;
    }
    void release_all() {
        for (void *p : ptrs) cudaFree(p);
        ptrs.clear();
    }
};

// a call's own stream: drained and destroyed on every way out, before the scratch it used is freed (declare it after
// that scratch)
struct OwnStream {
    cudaStream_t s = nullptr;
    ~OwnStream() {
        if (s) {
            cudaStreamSynchronize(s);
            cudaStreamDestroy(s);
        }
    }
};

constexpr int kCountThreads = 256;
constexpr uint64_t kMaxPerLaunch = 1ull << 30;  // queries per pack/count launch (u32 indices inside the kernels)
// resident CTAs per SM the kernels are compiled for (register budget = 65536 / (256 * min_ctas)):
// one thread per query keeps two 64-byte blocks (32 registers) in flight, a lane pair half of that
constexpr int min_ctas(bool wide, int lanes) { return lanes == 2 ? (wide ? 4 : 5) : (wide ? 3 : 4); }

inline uint32_t words_for_k(uint32_t k) { return k ? (k + kSymsPerWord - 1) / kSymsPerWord : 1; }

// ---- loader.cu: RLE byte stream / .npy -> host block image ----
struct HostImage {
    std::vector<uint32_t> blocks;  // nblocks * 16 words
    std::vector<uint32_t> aux;     // nblocks * 2 ($, N checkpoints)
    std::vector<uint64_t> cbase;   // n_super * 8
    uint64_t counts[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t start[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t total = 0;
    uint64_t nblocks = 0;
    uint32_t n_super = 0;
    uint32_t sb_shift = kDefaultSuperShift;
};

// ---- builder.cu: RLE byte stream -> block image built ON the current device ----
struct DeviceImage {
    uint4 *blocks = nullptr;
    uint32_t *aux = nullptr;
    uint64_t *cbase = nullptr;
    uint64_t counts[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t start[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t total = 0;
    uint64_t nblocks = 0;
    uint32_t n_super = 0;
    uint32_t sb_shift = kDefaultSuperShift;
};
int build_image_on_device(const uint8_t *h_rle, uint64_t len, uint32_t sb_shift, DeviceImage &img);
void free_device_image(DeviceImage &img);

// ---- pair_builder.cu: one-step image (resident on the current device) -> pair image ----
struct PairImage {
    uint4 *lines = nullptr;      // npair * 128 B
    uint64_t *c2base = nullptr;  // n_super2 * 16, WIDE only
    uint64_t npair = 0;
    uint32_t n_super2 = 0;
};
// `keep_codes` (optional): receives the per-position pair-code bytes (16 | code, or 0 when invalid;
// npair * 96 of them, device memory the caller must cudaFree) -- the quad builder's input.
int build_pair_image_on_device(int device, const IndexView &ix, const uint64_t start[kAlphabet], PairImage &img,
                               uint8_t **keep_codes = nullptr);
void free_pair_image(PairImage &img);

// ---- quad_builder.cu: pair image + pair codes (resident on the current device) -> quad image ----
struct QuadImage {
    uint4 *sectors = nullptr;    // 256 * nsec4 * 32 B
    uint64_t *c4base = nullptr;  // n_super4 * 256, WIDE only
    uint64_t nsec4 = 0;
    uint32_t n_super4 = 0;
    uint32_t sb_shift4 = 0;
};
uint64_t quad_image_bytes(uint64_t total);
// `ix` must carry the one-step blocks and the pair image; `d_codes2` = build_pair_image_on_device's keep_codes
// `keep_codes` (optional): receives the per-position quad codes (0x100 | code, or 0 when invalid; device
// memory the caller must cudaFree) -- the oct builder's input.
int build_quad_image_on_device(int device, const IndexView &ix, const uint8_t *d_codes2, QuadImage &img,
                               uint16_t **keep_codes = nullptr);
void free_quad_image(QuadImage &img);

// ---- oct_builder.cu: quad image + quad codes (resident on the current device) -> oct image ----
struct OctImage {
    uint4 *lines = nullptr;  // 4^m * nbuck8 * 128 B
    uint64_t nbuck8 = 0;
    int shift = 0;                      // b: log2 of the bucket size
    uint64_t runs = 0;                  // code8 runs of the BWT (what chose b)
    uint64_t overflow_lines = 0;        // (code, bucket) lines with more than kOctCapacity runs
    uint64_t overflow_occurrences = 0;  // positions whose line overflowed (answered through the quad image)
};
uint64_t oct_image_bytes(uint64_t total, int shift);
// stage 1 (needs the quad image): the kOctSyms-symbol code of every position, `1 << kOctCodeBits | code` or 0 when one of
// the symbols is not ACGT (4 bytes per position, device memory the caller frees).  `d_codes4` = the quad builder's
// keep_codes, OWNED by this call; `d_codes2` = the pair builder's keep_codes (borrowed).  N < 2^32 only.
int build_oct_codes_on_device(int device, const IndexView &ix, uint16_t *d_codes4, const uint8_t *d_codes2,
                              uint32_t **d_codes10);
// stage 1 without a quad image: the same codes by walking LF through the one-step blocks (any index; the only way when
// N >= 2^32, whose quad image has no room)
int build_oct_codes_by_walk(int device, const IndexView &ix, uint32_t **d_codes10);
// stage 2 (needs only the one-step blocks and the codes): the lines.  `requested_shift` 0 = automatic (layout.h).
// When even the coarsest buckets exceed `max_bytes` nothing is built (img.lines stays null) and MSBWT_OK is returned.
int build_oct_lines_on_device(int device, const IndexView &ix, const uint32_t *d_codes10, int requested_shift,
                              uint64_t max_bytes, OctImage &img);
void free_oct_image(OctImage &img);

// ---- fin_builder.cu: the oct builder's 10-symbol codes -> final-step lines (layout.h) ----
struct FinImage {
    uint4 *lines = nullptr;  // nlines * 128 B
    uint64_t nlines = 0;     // ((N >> shift) + 1) << lb
    int shift = 0, lb = 0;
    uint64_t runs = 0;            // run records stored
    uint64_t overflow_lines = 0;  // lines whose groups did not fit
};
uint64_t fin_image_bytes(uint64_t total, int shift, int lb);
// stage 1 (needs the quad image and the one-step blocks): the kFinSyms-symbol code of every position,
// `1 << kFinCodeBits | code` or 0 (8 bytes per position, device memory OWNED by stage 2)
int build_fin_codes_on_device(int device, const IndexView &ix, const uint32_t *d_codes10, uint64_t **d_codes20);
int build_fin_codes_by_walk(int device, const IndexView &ix, const uint32_t *d_codes10, uint64_t **d_codes20);
// stage 2 (needs only the codes, which it frees as soon as the run records exist): the lines
int build_fin_lines_on_device(int device, uint64_t total, uint64_t *d_codes20, int shift, int lb, FinImage &img);
void free_fin_image(FinImage &img);

// ---- bwt_build.cu: reads (device) -> RLE bytes of their multi-string BWT (device).  d_offsets == nullptr: n_reads reads
// of read_len symbols each; otherwise read r = d_reads[d_offsets[r] .. d_offsets[r + 1]) and read_len = the longest ----
int build_rle_bwt_on_device(const uint8_t *d_reads, const uint64_t *d_offsets, uint64_t n_reads, uint32_t read_len,
                            uint8_t **d_rle_out, uint64_t *rle_len, uint64_t *total);
// n symbol bytes (device) -> their msbwt RLE bytes (a cudaMalloc'd device buffer the caller frees); step 4b of the builder
int encode_rle_on_device(const uint8_t *d_bwt, uint64_t n, uint8_t **d_rle_out, uint64_t *rle_len);

// ---- bwt_merge.cu: two RLE byte streams (host) -> RLE bytes of their Holt-McMillan merge (device buffer the caller
// frees); *iterations = interleave passes run, the last of which changed nothing ----
int merge_rle_bwts_on_device(const uint8_t *h_rle_a, uint64_t len_a, const uint8_t *h_rle_b, uint64_t len_b,
                             uint8_t **d_rle_out, uint64_t *rle_len, uint64_t *total, uint32_t *iterations);

// ---- spectrum.cu: the k-mer spectrum of an index (one replica, on the current device): hist[nbins] (nbins may be 0)
// and *n_kmers; when `kmers` is not null, also the k-mers with count >= min_count and their counts in co-lexicographic
// order (*kmers, *counts: malloc'd host arrays the caller frees, null when there are none).  1 <= k <= 32, min_count >= 1.
// `canonical`: the same over canonical pairs {X, rc X} (msbwt_kmer_spectrum_canonical), whose reverse-complement
// lookups run on the query path with `lanes` (the replica's kernel mapping) on the call's own stream and scratch.
int kmer_spectrum_on_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                            uint64_t *hist, uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers);

// the same list (LIST mode, `canonical` as above) written to device arrays of `sink.cap` entries, which a first,
// histogram-only call sized: *n_kmers entries of sink.kmers / sink.counts, in the order the host list would have
struct DeviceKmerList {
    uint64_t *kmers = nullptr, *counts = nullptr;
    uint64_t cap = 0;
};
int kmer_spectrum_to_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                            const DeviceKmerList &sink, uint64_t *n_kmers);

// ---- unitigs.cu: the unitigs of the compacted de Bruijn graph of the solid k-mers (msbwt_unitigs; one replica, on the
// current device).  *syms, *offsets, *count_sums: malloc'd host arrays the caller frees, null when *n_unitigs == 0 ----
int unitigs_on_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                      uint8_t **syms, uint64_t **offsets, uint64_t **count_sums, uint64_t *n_unitigs);

// ---- correct.cu: msbwt_correct_reads for reads [0, n_reads) of `offsets` (one replica, on the current device, with
// its own stream and scratch).  Appends the corrected reads' symbols and lengths; stats[5] as in msbwt_gpu.h ----
struct CorrectParams {
    uint32_t k;
    uint64_t min_count;
    uint32_t frac_permille, branch_limit;
};
int correct_reads_on_device(int device, const IndexView &ix, int lanes, const uint8_t *syms, const uint64_t *offsets,
                            uint64_t n_reads, const CorrectParams &prm, std::vector<uint8_t> &out_syms,
                            std::vector<uint64_t> &out_lens, uint64_t stats[5]);

// ---- loader.cu: RLE stream checks, the host builder (msbwt_debug_build_image) and the .npy reader ----
int validate_rle(const uint8_t *rle, uint64_t len);
int build_image_from_rle(const uint8_t *rle, uint64_t len, uint32_t sb_shift, HostImage &img);
int read_npy_payload(const char *path, std::vector<uint8_t> &payload);

// ---- kernels.cu ----
cudaError_t launch_pack_seed(const IndexView &ix, const uint8_t *d_syms, uint32_t k, uint64_t n, uint64_t *d_packed,
                             uint64_t *d_out, uint32_t *d_status, cudaStream_t st);
cudaError_t launch_table_extend(int device, const IndexView &ix, const void *d_parent, void *d_child,
                                uint32_t n_child, cudaStream_t st);
bool index_is_wide(const IndexView &ix);
// Device scratch produced by pack_seed_kernel and consumed by the search kernels (all u64 units,
// n = queries in the batch, `words` = words_for_k(k)).  Two compacted live lists share the arrays:
// list A (pair path: every remaining symbol is ACGT and their number is even) grows from index 0
// upwards, list B (one-step path) from index n-1 downwards.
//   [0, n)                      W0    first symbol word of a live query: A = 32 x 2-bit symbols,
//                                     B = 21 x 3-bit symbols, first-consumed symbol in the top bits
//   [n, n + seedw*n)            SEED  starting range: l | h<<32, or l then h (WIDE)
//   [.., + (n+1)/2)             QIDX  u32: original query index | table depth used << 30
//                                     (0 = none, 1 = table_s, 2 = table_s - 1)
//   [.., + (words-1)*n)         WX    symbol words 1.. of query q, word-major, by ORIGINAL index
//   [.., + 2)                   LIVE  number of live queries in list A, list B (u64 counters)
//   [.., + 2)                   WORK  the oct kernel's chunk dispenser over list A (u32 counter; + padding)
//   [.., + 4)                   FSTAT counters of pack_seed_final_kernel (final_kernels.cu): final-step lines fetched,
//                                     of which had overflowed, ranges over two buckets, k-mers the suffix table
//                                     already answered (empty range)
// Queries that need no search step (empty seed range, or the suffix table answered every symbol)
// are finished by the pack kernel itself and never reach the search kernels.
constexpr uint32_t kQidxMask = (1u << 30) - 1u;
struct PackedLayout {
    uint64_t n;
    uint32_t words, seedw;
    __host__ __device__ uint64_t w0() const { return 0; }
    __host__ __device__ uint64_t seed() const { return n; }
    __host__ __device__ uint64_t qidx() const { return n + (uint64_t)seedw * n; }
    __host__ __device__ uint64_t wx() const { return qidx() + (n + 1) / 2; }
    __host__ __device__ uint64_t live() const { return wx() + (uint64_t)(words - 1) * n; }
    __host__ __device__ uint64_t work() const { return live() + 2; }
    __host__ __device__ uint64_t fstat() const { return live() + 4; }
    __host__ __device__ uint64_t total() const { return live() + 8; }
};
inline PackedLayout packed_layout(const IndexView &ix, uint32_t k, uint64_t n) {
    return PackedLayout{n, words_for_k(k), index_is_wide(ix) ? 2u : 1u};
}
// Runs the pair kernel over list A (when the index has a pair image) and the one-step kernel over list B.
cudaError_t launch_count_packed(int device, const IndexView &ix, int lanes, const uint64_t *d_packed, uint32_t k,
                                uint64_t n, uint64_t *d_out, cudaStream_t st, bool with_b = true);
// host-packed batches (hostpack.cpp): words[w * n + q], 2-bit ACGT symbols, the k-mer's last symbol in the
// top bits of word 0 -> live list A (same scratch layout as launch_pack_seed produces)
cudaError_t launch_seed_packed(const IndexView &ix, const uint64_t *d_words, uint32_t k, uint64_t n,
                               uint64_t *d_packed, uint64_t *d_out, cudaStream_t st);
// caller-packed batches, k <= 32: kmers[q] = the k-mer as a 2k-bit integer, first symbol most significant -> live list A
cudaError_t launch_seed_u64(const IndexView &ix, const uint64_t *d_kmers, uint32_t k, uint64_t n,
                            uint64_t *d_packed, uint64_t *d_out, cudaStream_t st);
// final_kernels.cu: the one-request path of k-mers that are a suffix-table entry + exactly kFinSyms symbols
// (k = 31 / 32 with table levels 11 / 12): pack (or take the packed word), seed and answer from ONE final-step line
// in one regular kernel; what it cannot answer (range over two buckets, overflowed line, `$` / `N`) goes to the live
// lists for launch_count_packed.  `src_kind`: 0 = symbol bytes (n * k, 16-byte aligned), 1 = caller-packed integers
// (msbwt_count_kmers_u64's format), 2 = host-packed words (word 0 of hostpack.cpp's format).
bool final_fast_path_applies(const IndexView &ix, uint32_t k, const void *d_src, int src_kind);
cudaError_t launch_pack_seed_final(int device, const IndexView &ix, const void *d_src, int src_kind, uint32_t k, uint64_t n,
                                   uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status, cudaStream_t st);
// quad_kernels.cu: live list A over the quad (and oct) image
cudaError_t launch_count_quad(int device, const IndexView &ix, const uint64_t *d_packed, const PackedLayout &lay,
                              uint32_t k, uint64_t *d_out, cudaStream_t st);
// wide_kernels.cu: live list A over the oct (and final-step) image of an index with 64-bit positions
cudaError_t launch_count_oct_wide(int device, const IndexView &ix, const uint64_t *d_packed, const PackedLayout &lay,
                                  uint32_t k, uint64_t *d_out, cudaStream_t st);
// stats_kernels.cu: live list A over the oct image with the counting instantiation -- d_stats[8] (oct_kernel.cuh)
cudaError_t launch_count_oct_stats(int device, const IndexView &ix, const uint64_t *d_packed, uint32_t k, uint64_t n,
                                   uint64_t *d_out, unsigned long long *d_stats, cudaStream_t st);
bool packed_batch_needs_list_b(const IndexView &ix, uint32_t k);
uint32_t max_host_packed_k();  // seed_packed_kernel handles k-mers of at most this many symbols
cudaError_t launch_count_bytes(int device, const IndexView &ix, const uint8_t *d_syms,
                               const uint64_t *d_offsets, uint64_t n, uint64_t *d_out, uint32_t *d_status,
                               cudaStream_t st);
cudaError_t launch_constrain_ranges(int device, const IndexView &ix, const uint8_t *d_sym, const uint64_t *d_l,
                                    const uint64_t *d_h, uint64_t n, uint64_t *d_out_l, uint64_t *d_out_h,
                                    cudaStream_t st);
// ext_kernels.cu: the four constrain_range calls (A,C,G,T) of every range from one fetch of its blocks
// (out[4 * i + j]); the k-mers of every window of every read (and their reverse complements) as symbol bytes;
// per-window sums of the two strands' counts
cudaError_t launch_constrain_fanout(int device, const IndexView &ix, const uint64_t *d_l, const uint64_t *d_h,
                                    uint64_t n, uint64_t *d_out_l, uint64_t *d_out_h, cudaStream_t st);
cudaError_t launch_expand_read_kmers(int device, const uint8_t *d_reads, uint32_t read_len, uint64_t n_reads, uint32_t k,
                                     uint32_t strands, uint8_t *d_syms, cudaStream_t st);
cudaError_t launch_sum_strands(int device, const uint64_t *d_per_query, uint64_t n_windows, uint64_t *d_out, cudaStream_t st);
cudaError_t launch_narrow_counts(int device, const uint64_t *d_in, uint64_t n, uint32_t *d_out, cudaStream_t st);
cudaError_t launch_gather(int device, const void *d_buf, uint64_t buf_bytes, uint32_t granule,
                          uint64_t n_gathers, uint64_t seed, uint64_t *d_sink, cudaStream_t st);

}  // namespace msbwt
