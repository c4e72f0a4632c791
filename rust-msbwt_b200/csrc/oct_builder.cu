// oct_builder.cu -- device-side construction of the OCT image (layout.h) from the quad image and the
// per-position quad codes that are already resident on the device.
//
// The reference has no counterpart (its index is the sampled table of construct_fmindex,
// src/rle_bwt.rs:387-467); what the oct image must reproduce is the composition of several
// RleBWT::constrain_range calls (src/rle_bwt.rs:202-287) -- kOctSyms of them since the image holds ten
// symbols per line; layout.h states the identity.
//
// Two stages, so that the caller can drop the (large) quad image between them:
//   1. codes  : one thread per BWT position j with a valid quad code a: j4 = LF^4(j) = rank4(a, j) through the
//               quad image (one sector), b = code4(j4) (one random read), j8 = rank4(b, j4), c = the pair code
//               (two symbols) at j8; code(j) = a * 4^6 + b * 4^2 + c when all three are valid.
//   2. count  : run heads (code8 changes) are counted; the bucket shift b is the largest one that keeps the
//               mean number of runs per line <= kOctTargetRuns (and the image within the caller's budget).
//   3. emit   : every run head (also forced at multiples of 2^cs, layout.h) walks to the end of its run and
//               appends `(len << b) | offset` to line (code8, j >> b): the slot comes from an atomicAdd on
//               the line's run counter, which keeps counting past the line's capacity; word 0 gathers the
//               line's occurrences.
//   4. stamp  : one warp per code: exclusive prefix sum of the occurrence counts over the code's buckets,
//               plus C8[code]; lines holding more than kOctCapacity runs are counted (the kernel answers
//               those through the quad image).
//   Cm[c] = kOctSyms constrain_range calls of our own kernel applied to position 0.
#include <algorithm>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "engine.h"

namespace msbwt {

namespace {

static_assert(kOctSyms == 8 || kOctSyms == 10, "the code kernel composes quad codes (+ one pair code)");
constexpr uint32_t kValid8 = 1u << kOctCodeBits;
constexpr uint32_t kCodeMask = kValid8 - 1u;

__global__ void __launch_bounds__(256) oct_code8_kernel(IndexView ix, const uint16_t *__restrict__ codes4,
                                                        const uint8_t *__restrict__ codes2,
                                                        uint32_t *__restrict__ codes8) {
    const C4Base<false> c4{};
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < ix.total; j += step) {
        const uint32_t a = codes4[j];
        uint32_t v = 0;
        if (a & 0x100u) {
            uint32_t l = (uint32_t)j, h = (uint32_t)j;
            quad_step<false>(ix, c4, a & 255u, l, h);  // l = LF^4(j)
            const uint32_t b = codes4[l];
            if (b & 0x100u) {
                if constexpr (kOctSyms == 8) {
                    v = kValid8 | ((a & 255u) << 8) | (b & 255u);
                } else {
                    h = l;
                    quad_step<false>(ix, c4, b & 255u, l, h);  // l = LF^8(j)
                    const uint32_t c = codes2[l];                // 16 | pair code (B[l], B[LF l]) when both are ACGT
                    if (c & 16u) v = kValid8 | ((a & 255u) << 12) | ((b & 255u) << 4) | (c & 15u);
                }
            }
        }
        codes8[j] = v;
    }
}

// The same codes without a quad image: every position walks LF through the one-step blocks, kOctSyms symbols, one
// 64-byte block per step (indexes of 2^32 positions and more, whose quad image -- 36.6 B per position -- has no room).
template <bool WIDE>
__global__ void __launch_bounds__(256) oct_code_walk_kernel(IndexView ix, uint32_t *__restrict__ codes) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < ix.total; j += step) {
        P p = (P)j;
        uint32_t code = 0;
        bool ok = true;
        for (int r = 0; r < kOctSyms; r++) {
            const uint32_t s = symbol_at(ix, p);
            if (!((0x2Eu >> s) & 1u)) { ok = false; break; }  // not one of A,C,G,T = 1,2,3,5
            code = (code << 2) | ((s - 1u - (s >> 2)) & 3u);
            if (r + 1 < kOctSyms) p = lf_step<WIDE>(ix, cb, s, p);
        }
        codes[j] = ok ? (kValid8 | code) : 0u;
    }
}

__global__ void __launch_bounds__(256) oct_count_runs_kernel(const uint32_t *__restrict__ codes8, uint64_t total,
                                                             unsigned long long *__restrict__ runs) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    uint32_t mine = 0;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += step) {
        const uint32_t v = codes8[j];
        mine += (v & kValid8) && (j == 0 || codes8[j - 1] != v);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
    if ((threadIdx.x & 31u) == 0 && mine) atomicAdd(runs, (unsigned long long)mine);
}

__global__ void __launch_bounds__(256) oct_emit_kernel(const uint32_t *__restrict__ codes8, uint64_t total,
                                                       uint32_t shift, uint64_t nbuck8, uint32_t *__restrict__ lines) {
    const uint64_t chunk_mask = (1ull << oct_chunk_shift((int)shift)) - 1ull;
    const uint32_t off_mask = (1u << shift) - 1u;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += step) {
        const uint32_t v = codes8[j];
        if (!(v & kValid8)) continue;
        if (!((j & chunk_mask) == 0 || codes8[j - 1] != v)) continue;
        uint32_t len = 1;
        while (j + len < total && ((j + len) & chunk_mask) != 0 && codes8[j + len] == v) len++;
        uint32_t *line = lines + ((uint64_t)(v & kCodeMask) * nbuck8 + (j >> shift)) * kOctLineWords;
        atomicAdd(line, len);
        const uint32_t slot = atomicAdd(line + 1, 1u);
        if (slot < (uint32_t)kOctCapacity) line[2 + slot] = (len << shift) | ((uint32_t)j & off_mask);
    }
}

// one warp per code: occurrence counts of its buckets (word 0) -> checkpoints.  WIDE (positions of 2^32 and more):
// word 0 = the low 32 bits of the checkpoint, word 1 = min(runs, 31) | (the bits above them) << 8 (layout.h).
template <bool WIDE>
__global__ void __launch_bounds__(256) oct_stamp_kernel(const uint64_t *__restrict__ c8, uint64_t nbuck8,
                                                        uint32_t *__restrict__ lines, unsigned long long *__restrict__ overflow) {
    using P = typename Pos<WIDE>::type;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t code = blockIdx.x * 8u + (threadIdx.x >> 5);
    if (code >= (uint32_t)kOctCodes) return;
    uint32_t *base = lines + (uint64_t)code * nbuck8 * kOctLineWords;
    P run = (P)c8[code];
    uint32_t over = 0;
    unsigned long long over_occ = 0;
    for (uint64_t b0 = 0; b0 < nbuck8; b0 += 32) {
        const uint64_t b = b0 + lane;
        const uint32_t cnt = b < nbuck8 ? base[b * kOctLineWords] : 0u;
        const uint32_t nruns = b < nbuck8 ? base[b * kOctLineWords + 1] : 0u;
        if (nruns > (uint32_t)kOctCapacity) { over++; over_occ += cnt; }
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += t;
        }
        if (b < nbuck8) {
            const P ck = run + (P)(incl - cnt);
            base[b * kOctLineWords] = (uint32_t)ck;
            if constexpr (WIDE) base[b * kOctLineWords + 1] = min(nruns, (uint32_t)kOctCapacity + 1u) | ((uint32_t)(ck >> 32) << 8);
        }
        run += (P)__shfl_sync(0xffffffffu, incl, 31);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        over += __shfl_xor_sync(0xffffffffu, over, d);
        over_occ += __shfl_xor_sync(0xffffffffu, over_occ, d);
    }
    if (lane == 0 && over) {
        atomicAdd(overflow, (unsigned long long)over);
        atomicAdd(overflow + 1, over_occ);
    }
}

#define O_TRY(e) CU_TRY_IN("oct image: ", e)

}  // namespace

uint64_t oct_image_bytes(uint64_t total, int shift) {
    return (uint64_t)kOctCodes * ((total >> shift) + 1) * kOctLineBytes;
}

// Stage 1: the kOctSyms-symbol code of every position (4 bytes each; the caller frees them).  `ix` must carry the
// one-step blocks and the quad image; `d_codes4` (the quad builder's keep_codes) is OWNED by this call and freed as
// soon as the codes exist; `d_codes2` (the pair builder's keep_codes) is borrowed.
int build_oct_codes_on_device(int device, const IndexView &ix, uint16_t *d_codes4, const uint8_t *d_codes2,
                              uint32_t **d_codes10) {
    DevicePtr<uint16_t> codes4(d_codes4);
    *d_codes10 = nullptr;
    if (!ix.quad || !d_codes4 || !d_codes2) return fail(MSBWT_EINVAL, "oct image: needs the quad image, its codes and the pair codes");
    if (index_is_wide(ix)) return fail(MSBWT_EINVAL, "oct image: only for indexes with 32-bit positions (N < 2^32, one superblock)");
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((ix.total + 255) / 256, (uint64_t)sms * 32));
    uint32_t *d_codes8 = nullptr;
    O_TRY(cudaMalloc((void **)&d_codes8, std::max<uint64_t>(1, ix.total) * sizeof(uint32_t)));
    oct_code8_kernel<<<grid, 256>>>(ix, d_codes4, d_codes2, d_codes8);
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(d_codes8);
        return fail(MSBWT_ECUDA, std::string("oct image: code kernel: ") + cudaGetErrorString(e));
    }
    *d_codes10 = d_codes8;
    return MSBWT_OK;
}

// Stage 1 without a quad image (any index; the only way for one of 2^32 positions and more): the codes by walking LF
// through the one-step blocks -- `ix` needs nothing else.
int build_oct_codes_by_walk(int device, const IndexView &ix, uint32_t **d_codes10) {
    *d_codes10 = nullptr;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((ix.total + 255) / 256, (uint64_t)sms * 32));
    uint32_t *d_codes = nullptr;
    O_TRY(cudaMalloc((void **)&d_codes, std::max<uint64_t>(1, ix.total) * sizeof(uint32_t)));
    if (index_is_wide(ix)) oct_code_walk_kernel<true><<<grid, 256>>>(ix, d_codes);
    else oct_code_walk_kernel<false><<<grid, 256>>>(ix, d_codes);
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(d_codes);
        return fail(MSBWT_ECUDA, std::string("oct image: code walk kernel: ") + cudaGetErrorString(e));
    }
    *d_codes10 = d_codes;
    return MSBWT_OK;
}

// Stage 2: the lines, from the codes alone (plus the one-step blocks for Cm[c]): the quad image is not read, so
// the caller may already have dropped it.  `requested_shift` 0 = automatic (layout.h).  When even the coarsest
// buckets exceed `max_bytes` nothing is built (img.lines stays null) and MSBWT_OK is returned.
int build_oct_lines_on_device(int device, const IndexView &ix, const uint32_t *d_codes8, int requested_shift,
                              uint64_t max_bytes, OctImage &img) {
    if (!d_codes8) return fail(MSBWT_EINVAL, "oct image: needs the position codes");
    if ((ix.total >> 40) != 0) return fail(MSBWT_EINVAL, "oct image: a line's checkpoint holds 40 bits (N < 2^40)");
    const bool wide = index_is_wide(ix);
    if (requested_shift && (requested_shift < kOctMinShift || requested_shift > kOctMaxShift))
        return fail(MSBWT_EINVAL, "oct image: bucket shift out of range");
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((ix.total + 255) / 256, (uint64_t)sms * 32));

    DeviceScratch tmp;
    uint8_t *d_sym = nullptr;
    uint64_t *d_pos = nullptr;
    unsigned long long *d_stat = nullptr;  // [0] runs, [1] overflowed lines, [2] their occurrences
    O_TRY(tmp.alloc(&d_stat, 3));
    O_TRY(cudaMemsetAsync(d_stat, 0, 3 * sizeof(unsigned long long)));
    oct_count_runs_kernel<<<grid, 256>>>(d_codes8, ix.total, d_stat);
    O_TRY(cudaGetLastError());
    g_launches++;
    unsigned long long runs = 0;
    O_TRY(cudaMemcpy(&runs, d_stat, sizeof(runs), cudaMemcpyDeviceToHost));
    img.runs = runs;

    int shift = requested_shift;
    if (!shift) {  // mean runs per line = runs * 2^shift / (4^m * N)
        shift = kOctMaxShift;
        while (shift > kOctAutoMinShift &&
               (long double)runs * (long double)(1ull << shift) >
                   (long double)kOctTargetRuns * (long double)kOctCodes * (long double)std::max<uint64_t>(ix.total, 1))
            shift--;
        while (shift < kOctMaxShift && oct_image_bytes(ix.total, shift) > max_bytes) shift++;
    }
    if (oct_image_bytes(ix.total, shift) > max_bytes) return MSBWT_OK;  // no room: img.lines stays null
    const uint64_t nbuck8 = (ix.total >> shift) + 1;
    const uint64_t nlines = (uint64_t)kOctCodes * nbuck8;
    img.nbuck8 = nbuck8;
    img.shift = shift;

    O_TRY(cudaMalloc((void **)&img.lines, nlines * kOctLineBytes));
    O_TRY(cudaMemsetAsync(img.lines, 0, nlines * kOctLineBytes));
    O_TRY(tmp.alloc(&d_sym, kOctCodes));
    O_TRY(tmp.alloc(&d_pos, 3 * (size_t)kOctCodes));

    // Cm[c]: the kOctSyms steps applied to position 0
    static const uint8_t acgt[4] = {1, 2, 3, 5};
    O_TRY(cudaMemsetAsync(d_pos, 0, 3 * (size_t)kOctCodes * sizeof(uint64_t)));
    uint64_t *cur = d_pos, *nxt = d_pos + kOctCodes, *spare = d_pos + 2 * (size_t)kOctCodes;
    std::vector<uint8_t> h_sym(kOctCodes);
    for (int r = 0; r < kOctSyms; r++) {
        for (int c = 0; c < kOctCodes; c++) h_sym[(size_t)c] = acgt[(c >> (2 * (kOctSyms - 1 - r))) & 3];
        O_TRY(cudaMemcpy(d_sym, h_sym.data(), h_sym.size(), cudaMemcpyHostToDevice));
        O_TRY(launch_constrain_ranges(device, ix, d_sym, cur, cur, kOctCodes, nxt, spare, nullptr));
        std::swap(cur, nxt);
    }

    // emit
    if (ix.total) {
        oct_emit_kernel<<<grid, 256>>>(d_codes8, ix.total, (uint32_t)shift, nbuck8, reinterpret_cast<uint32_t *>(img.lines));
        O_TRY(cudaGetLastError());
        g_launches++;
    }
    // stamp
    if (wide) oct_stamp_kernel<true><<<kOctCodes / 8, 256>>>(cur, nbuck8, reinterpret_cast<uint32_t *>(img.lines), d_stat + 1);
    else oct_stamp_kernel<false><<<kOctCodes / 8, 256>>>(cur, nbuck8, reinterpret_cast<uint32_t *>(img.lines), d_stat + 1);
    O_TRY(cudaGetLastError());
    g_launches++;
    unsigned long long over[2] = {0, 0};
    O_TRY(cudaMemcpy(over, d_stat + 1, sizeof(over), cudaMemcpyDeviceToHost));
    img.overflow_lines = over[0];
    img.overflow_occurrences = over[1];
    O_TRY(cudaDeviceSynchronize());
    return MSBWT_OK;
}

void free_oct_image(OctImage &img) {
    if (img.lines) cudaFree(img.lines);
    img = {};
}

}  // namespace msbwt
