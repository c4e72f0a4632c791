// bwt_merge.cu -- merge two multi-string BWTs on the device: the Holt-McMillan interleave.
//
// Replaces the reference's pairwise_bwt_merge (src/bwt_util.rs:108-141), a single-threaded pass per iteration over
// the two inputs.  Within one input the rows are sorted by their infinite forward symbol sequences; the merge is the
// stable interleave of both inputs' rows by those sequences (ties keep A before B).  It is the fixed point of
//
//     I_0     = N_A zeros (A's rows) followed by N_B ones (B's rows)
//     I_{t+1} = walk I_t in order, take each row's symbol c from its own input (the next unread one of that input),
//               and append the row's source bit to bucket c; bucket c starts at C_A[c] + C_B[c].
//
// For BWTs built from reads the result is the BWT of the union of the read sets, byte for byte what the builder
// (bwt_build.cu) makes from all the reads at once; oracle/merge.py restates the iteration in numpy.
//
// Device layout:
//   inputs : the one-step block images of both inputs (builder.cu: the loader's validation and decoding), 0.56 B per
//            symbol.  A row's symbol is read from the bit-planes (symbol_at); ranks at tile starts from
//            device_rank.cuh.
//   I_t    : a bit-vector (bit r of word r / 32 = row r's source), two of them, 0.25 B per symbol.
//   pass   : one warp per tile of kTileRows merged rows.  z = A-rows before the tile (exclusive scan of the previous
//            pass's per-tile zero counts); symbol c's bits from the tile go to C_A[c] + rank_c(A, z) + C_B[c] +
//            rank_c(B, start - z), so no scan over symbols across tiles is needed.  The warp walks the tile 32 rows at
//            a time; lane c (< 6) keeps symbol c's output stream, stores its interior words and ORs (atomicOr into
//            the zeroed vector) the at most two words it shares with neighbouring segments.
//   count  : per-tile zero counts of I_{t+1} for the next pass, and whether I_{t+1} differs from I_t.
//   output : after the fixed point, one pass writes the merged symbols (one byte each); encode_rle_on_device
//            (bwt_build.cu) turns them into RLE bytes exactly as the builder does.
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <string>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "kernel_common.cuh"

namespace msbwt {

namespace {

// one warp per tile of 32 * kTileWords merged rows.  Measured on B200 (profiles/merge_tile_sweep.jsonl, 1.51 Gsymbols):
// the pass takes 8.96-9.05 ms for 128..1024 words and the count pass 0.24 -> 0.07 ms; pass + count is flat within
// 0.7 % from 256 words up, so 256 stays.  The pass is bound by instruction issue (DESIGN.md section 4), not by the tile.
#ifndef MSBWT_MERGE_TILE_WORDS
#define MSBWT_MERGE_TILE_WORDS 256
#endif
constexpr uint32_t kTileWords = MSBWT_MERGE_TILE_WORDS;
static_assert(kTileWords % 128 == 0, "tile_zeros_kernel reads a tile as whole uint4 rounds of a warp");
constexpr uint64_t kTileRows = 32ull * kTileWords;
constexpr int kMergeThreads = 256;
constexpr uint32_t kFull = 0xffffffffu;

__device__ __forceinline__ uint32_t low_bits(uint32_t k) { return k >= 32 ? kFull : ((1u << k) - 1u); }

// symbol_at over a bare block array: the merge picks the input per lane without diverging
__device__ __forceinline__ uint32_t symbol_in(const uint4 *blocks, uint64_t p) {
    const uint32_t *w = reinterpret_cast<const uint32_t *>(blocks) + (p >> kBlockShift) * (uint64_t)kWordsPerBlock +
                        (((uint32_t)p >> 6) & 1u) * 8u + (((uint32_t)p >> 5) & 1u);
    const uint32_t b = (uint32_t)p & 31u;
    return ((__ldg(w + 2) >> b) & 1u) | (((__ldg(w + 4) >> b) & 1u) << 1) | (((__ldg(w + 6) >> b) & 1u) << 2);
}

// the lanes whose symbol is `c`, from the warp's three symbol bit-planes
__device__ __forceinline__ uint32_t lanes_with(uint32_t c, uint32_t p0, uint32_t p1, uint32_t p2) {
    return (p0 ^ ((c & 1u) - 1u)) & (p1 ^ (((c >> 1) & 1u) - 1u)) & (p2 ^ (((c >> 2) & 1u) - 1u));
}

// I_0: rows [n_a, n) come from B
__global__ void init_interleave_kernel(uint32_t *__restrict__ v, uint64_t n_a, uint64_t n, uint64_t words) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += step) {
        const uint64_t lo = w * 32;
        uint32_t m = 0;
        if (lo + 32 > n_a && lo < n) {
            const uint32_t from = n_a > lo ? (uint32_t)(n_a - lo) : 0u;
            const uint32_t to = n < lo + 32 ? (uint32_t)(n - lo) : 32u;
            m = low_bits(to) & ~low_bits(from);
        }
        v[w] = m;
    }
}

// one warp per tile: A-rows (zero bits) of `v` in the tile, and whether the tile differs from `prev` (may be null)
__global__ void __launch_bounds__(kMergeThreads) tile_zeros_kernel(const uint4 *__restrict__ v, const uint4 *__restrict__ prev,
                                                                   uint64_t n, uint64_t n_tiles, uint64_t *__restrict__ zeros,
                                                                   uint32_t *__restrict__ changed) {
    const uint64_t tile = ((uint64_t)blockIdx.x * kMergeThreads + threadIdx.x) >> 5;
    if (tile >= n_tiles) return;  // whole warps
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t ones = 0, diff = 0;
#pragma unroll
    for (uint32_t i = 0; i < kTileWords / 4 / 32; i++) {
        const uint64_t at = tile * (kTileWords / 4) + i * 32 + lane;
        const uint4 x = v[at];
        ones += __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
        if (prev) {
            const uint4 y = prev[at];
            diff |= (x.x ^ y.x) | (x.y ^ y.y) | (x.z ^ y.z) | (x.w ^ y.w);
        }
    }
    ones = __reduce_add_sync(kFull, ones);
    const bool any = __any_sync(kFull, diff != 0);
    if (lane == 0) {
        const uint64_t rows = n - tile * kTileRows < kTileRows ? n - tile * kTileRows : kTileRows;  // padding bits are zero
        zeros[tile] = rows - ones;
        if (any) atomicOr(changed, 1u);
    }
}

// One interleave pass (EMIT = false: I_t -> I_{t+1} into the zeroed `next`) or the output pass (EMIT = true: the
// merged symbols, one byte per row).  `zbefore[t]` = A-rows of I_t before tile t.
template <bool EMIT>
__global__ void __launch_bounds__(kMergeThreads) merge_pass_kernel(const IndexView a, const IndexView b,
                                                                   const uint32_t *__restrict__ cur,
                                                                   const uint64_t *__restrict__ zbefore, uint64_t n,
                                                                   uint64_t n_tiles, uint32_t *__restrict__ next,
                                                                   uint8_t *__restrict__ out) {
    // the ballots and reductions below follow a divergent symbol fetch and lane-dependent rank (n_tiles < 2^49: never
    // prints)
    warp_sync_guard(PackedLayout{n_tiles, 0, 0});
    const uint64_t tile = ((uint64_t)blockIdx.x * kMergeThreads + threadIdx.x) >> 5;
    if (tile >= n_tiles) return;  // whole warps
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt = (1u << lane) - 1u;
    const uint64_t row0 = tile * kTileRows, row_end = row0 + kTileRows < n ? row0 + kTileRows : n;
    uint64_t pa = zbefore[tile], pb = row0 - pa;

    // lane c < 6: the output stream of symbol c -- `acc` holds the bits of word `wi` from bit 0 up to `fill`; `shared`:
    // the word's low bits belong to the segment before (it is ORed in, not stored)
    uint64_t acc = 0, wi = 0;
    uint32_t fill = 0;
    bool shared = false;
    if (!EMIT && lane < (uint32_t)kAlphabet) {
        const uint64_t pos = lf_step<true>(a, CBase<true>{a.cbase, a.sb_shift}, lane, pa) +
                             lf_step<true>(b, CBase<true>{b.cbase, b.sb_shift}, lane, pb);
        wi = pos >> 5;
        fill = (uint32_t)pos & 31u;
        shared = fill != 0;
    }

    for (uint64_t r0 = row0; r0 < row_end; r0 += 32) {
        const uint32_t nr = row_end - r0 < 32 ? (uint32_t)(row_end - r0) : 32u;
        const uint32_t w = __ldg(cur + (r0 >> 5));
        const uint32_t s = (w >> lane) & 1u;
        const uint32_t ones_before = __popc(w & lt);
        uint32_t c = 7;  // matches no symbol
        if (lane < nr) c = symbol_in(s ? b.blocks : a.blocks, s ? pb + ones_before : pa + (lane - ones_before));
        const uint32_t ones = __popc(w & low_bits(nr));
        pa += nr - ones;
        pb += ones;
        if constexpr (EMIT) {
            if (lane < nr) out[r0 + lane] = (uint8_t)c;
        } else {
            const uint32_t p0 = __ballot_sync(kFull, c & 1u), p1 = __ballot_sync(kFull, c & 2u), p2 = __ballot_sync(kFull, c & 4u);
            const uint32_t bit = s << __popc(lanes_with(c, p0, p1, p2) & lt);  // at the row's rank among its symbol's
            const uint32_t cnt = lane < (uint32_t)kAlphabet ? __popc(lanes_with(lane, p0, p1, p2) & low_bits(nr)) : 0u;
            uint32_t v = 0;
#pragma unroll
            for (uint32_t j = 0; j < (uint32_t)kAlphabet; j++) {
                const uint32_t vj = __reduce_or_sync(kFull, c == j ? bit : 0u);
                if (lane == j) v = vj;
            }
            if (cnt) {  // lanes 0..5 only
                acc |= (uint64_t)v << fill;
                fill += cnt;
                if (fill >= 32) {
                    const uint32_t word = (uint32_t)acc;
                    if (word) {
                        if (shared) atomicOr(next + wi, word);
                        else next[wi] = word;
                    }
                    acc >>= 32;
                    fill -= 32;
                    wi++;
                    shared = false;
                }
            }
        }
    }
    if (!EMIT && fill && (uint32_t)acc) atomicOr(next + wi, (uint32_t)acc);  // shared with the segment after
}

IndexView view_of(const DeviceImage &img) {
    IndexView v{};
    v.blocks = img.blocks;
    v.aux = img.aux;
    v.cbase = img.cbase;
    v.total = img.total;
    v.nblocks = img.nblocks;
    v.n_super = img.n_super;
    v.sb_shift = img.sb_shift;
    return v;
}

struct ImageOwner {
    DeviceImage img;
    ~ImageOwner() { free_device_image(img); }
};

#define M_TRY(e) CU_TRY_IN("bwt merge: ", e)

}  // namespace

int merge_rle_bwts_on_device(const uint8_t *h_rle_a, uint64_t len_a, const uint8_t *h_rle_b, uint64_t len_b,
                             uint8_t **d_rle_out, uint64_t *rle_len, uint64_t *total, uint32_t *iterations) {
    *d_rle_out = nullptr;
    *rle_len = 0;
    *total = 0;
    *iterations = 0;
    ImageOwner A, B;
    if (int rc = build_image_on_device(h_rle_a, len_a, 0, A.img); rc != MSBWT_OK) return fail(rc, "input A: " + g_last_error);
    if (int rc = build_image_on_device(h_rle_b, len_b, 0, B.img); rc != MSBWT_OK) return fail(rc, "input B: " + g_last_error);
    const uint64_t n_a = A.img.total, n = A.img.total + B.img.total;
    if (n >> 62) return fail(MSBWT_EFORMAT, "bwt merge: the merged BWT would hold 2^62 symbols or more");
    if (!n) return MSBWT_OK;
    const IndexView va = view_of(A.img), vb = view_of(B.img);

    const uint64_t n_tiles = (n + kTileRows - 1) / kTileRows, words = n_tiles * kTileWords;
    const unsigned grid = (unsigned)((n_tiles * 32 + kMergeThreads - 1) / kMergeThreads);
    DeviceScratch bufs;
    uint32_t *cur = nullptr, *next = nullptr, *d_changed = nullptr;
    uint64_t *d_zeros = nullptr, *d_zbefore = nullptr;
    void *d_temp = nullptr;
    size_t temp_bytes = 0;
    M_TRY(bufs.alloc(&cur, words));
    M_TRY(bufs.alloc(&next, words));
    M_TRY(bufs.alloc(&d_zeros, n_tiles));
    M_TRY(bufs.alloc(&d_zbefore, n_tiles));
    M_TRY(bufs.alloc(&d_changed, 1));
    M_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, d_zeros, d_zbefore, (int64_t)n_tiles));
    M_TRY(bufs.alloc((uint8_t **)&d_temp, temp_bytes));

    init_interleave_kernel<<<(unsigned)std::min<uint64_t>((words + 255) / 256, 148 * 64), 256>>>(cur, n_a, n, words);
    M_TRY(cudaGetLastError());
    tile_zeros_kernel<<<grid, kMergeThreads>>>(reinterpret_cast<const uint4 *>(cur), nullptr, n, n_tiles, d_zeros, d_changed);
    M_TRY(cudaGetLastError());
    g_launches += 2;
    // the iteration ends after at most N_A + N_B passes; more means a broken invariant, not a slow input
    for (uint64_t it = 1;; it++) {
        M_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_zeros, d_zbefore, (int64_t)n_tiles));
        M_TRY(cudaMemsetAsync(next, 0, words * sizeof(uint32_t)));
        merge_pass_kernel<false><<<grid, kMergeThreads>>>(va, vb, cur, d_zbefore, n, n_tiles, next, nullptr);
        M_TRY(cudaGetLastError());
        M_TRY(cudaMemsetAsync(d_changed, 0, sizeof(uint32_t)));
        tile_zeros_kernel<<<grid, kMergeThreads>>>(reinterpret_cast<const uint4 *>(next), reinterpret_cast<const uint4 *>(cur),
                                                   n, n_tiles, d_zeros, d_changed);
        M_TRY(cudaGetLastError());
        g_launches += 3;
        uint32_t changed = 0;
        M_TRY(cudaMemcpy(&changed, d_changed, sizeof(changed), cudaMemcpyDeviceToHost));
        std::swap(cur, next);
        if (!changed) {
            *iterations = (uint32_t)std::min<uint64_t>(it, 0xFFFFFFFFull);
            break;
        }
        if (it > n) return fail(MSBWT_ECUDA, "bwt merge: internal error: the interleave did not reach its fixed point");
    }

    // the merged symbols, then the images and bit-vectors are no longer needed
    uint8_t *d_bwt = nullptr;
    M_TRY(cudaMalloc((void **)&d_bwt, n));
    struct BwtOwner { uint8_t *p; ~BwtOwner() { cudaFree(p); } } bwt_owner{d_bwt};
    M_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_zeros, d_zbefore, (int64_t)n_tiles));
    merge_pass_kernel<true><<<grid, kMergeThreads>>>(va, vb, cur, d_zbefore, n, n_tiles, nullptr, d_bwt);
    M_TRY(cudaGetLastError());
    M_TRY(cudaDeviceSynchronize());
    g_launches += 2;
    bufs.release_all();
    free_device_image(A.img);
    free_device_image(B.img);
    if (int rc = encode_rle_on_device(d_bwt, n, d_rle_out, rle_len); rc != MSBWT_OK) return rc;
    *total = n;
    return MSBWT_OK;
}

}  // namespace msbwt
