// pair_builder.cu -- device-side construction of the PAIR image (layout.h) from the one-step
// image that is already resident on the device.
//
// The reference has no counterpart: its index is the sampled table of construct_fmindex
// (src/rle_bwt.rs:387-467).  What the pair image must reproduce is the composition of two
// RleBWT::constrain_range calls (src/rle_bwt.rs:202-287); layout.h states the identity.
//
//   1. codes : one thread per BWT position j: b = B[j]; LF(j) = C[b] + rank(b, j) through the
//              one-step blocks; a = B[LF(j)] (one random read); code byte = 16 | 4*idx(b) | idx(a)
//              when both are ACGT, else 0.
//   2. fill  : one thread per 96-position line paints the five bit-planes of its four quarters and
//              counts the 16 codes.
//   3. scan  : per code, an exclusive prefix sum of the per-line counts (CUB, plumbing).
//   4. stamp : checkpoints -- absolute (C2 included) when N < 2^32, otherwise relative to the pair
//              superblock with the base in c2base.
//   C2[b,a] = C[a] + rank(a, C[b]) comes from 16 constrain_range calls of our own kernel.
#include <algorithm>

#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "engine.h"

namespace msbwt {

namespace {

__device__ __forceinline__ bool is_acgt(uint32_t sy) { return ((0x2Eu >> sy) & 1u) != 0; }  // sy < 8
__device__ __forceinline__ uint32_t acgt_idx(uint32_t sy) { return (sy - 1u - (sy >> 2)) & 3u; }

// (symbol_at: B[pos] from the one-step block planes, device_rank.cuh)

template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads) pair_codes_kernel(IndexView ix, uint8_t *__restrict__ codes) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t threads = (uint64_t)gridDim.x * kCountThreads;
    for (uint64_t j = (uint64_t)blockIdx.x * kCountThreads + threadIdx.x; j < ix.total; j += threads) {
        const uint32_t b = symbol_at(ix, j);
        uint8_t code = 0;
        if (is_acgt(b)) {
            P l = (P)j, h = (P)j;
            rank_step<WIDE, 1>(ix, cb, b, l, h);  // l = LF(j)
            const uint32_t a = symbol_at(ix, l);
            if (is_acgt(a)) code = (uint8_t)(16u | (acgt_idx(b) << 2) | acgt_idx(a));
        }
        codes[j] = code;
    }
}

// one thread per line: planes of the four quarters + per-line code counts (SoA: counts[code * npair + line])
__global__ void __launch_bounds__(128) pair_fill_kernel(const uint8_t *__restrict__ codes, uint64_t npair,
                                                        uint32_t *__restrict__ lines, uint8_t *__restrict__ counts) {
    const uint64_t line = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= npair) return;
    const uint4 *src = reinterpret_cast<const uint4 *>(codes + line * kPairSyms);  // 96 = 6 x 16 bytes
    uint32_t cnt[16];
#pragma unroll
    for (int c = 0; c < 16; c++) cnt[c] = 0;
    uint32_t *dst = lines + line * kPairWords;
    uint32_t raw[kPairSyms / 4];
#pragma unroll
    for (int i = 0; i < kPairSyms / 16; i++) {
        const uint4 v = src[i];
        raw[4 * i] = v.x; raw[4 * i + 1] = v.y; raw[4 * i + 2] = v.z; raw[4 * i + 3] = v.w;
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
        uint32_t pl[4] = {0, 0, 0, 0}, valid = 0;
#pragma unroll
        for (int sidx = 0; sidx < kPairQuarterSyms; sidx++) {
            const int at = t * kPairQuarterSyms + sidx;
            const uint32_t c = (raw[at >> 2] >> (8 * (at & 3))) & 0xffu;
            if (c & 16u) {
                valid |= 1u << sidx;
#pragma unroll
                for (int p = 0; p < 4; p++) pl[p] |= ((c >> p) & 1u) << sidx;
                cnt[c & 15u]++;
            }
        }
        const uint4 zero = make_uint4(0, 0, 0, 0);
        reinterpret_cast<uint4 *>(dst + t * 8)[0] = zero;  // checkpoints: stamped after the scans
        reinterpret_cast<uint4 *>(dst + t * 8)[1] =
            make_uint4(pl[0] | ((valid & 0xffu) << 24), pl[1] | (((valid >> 8) & 0xffu) << 24),
                       pl[2] | (((valid >> 16) & 0xffu) << 24), pl[3]);
    }
#pragma unroll
    for (int c = 0; c < 16; c++) counts[(uint64_t)c * npair + line] = (uint8_t)cnt[c];
}

struct WidenU8 {
    __host__ __device__ uint64_t operator()(uint8_t v) const { return v; }
};

template <bool WIDE>
__global__ void pair_stamp_kernel(const uint64_t *__restrict__ before, uint64_t npair, uint32_t sb_shift, uint32_t code,
                                  uint64_t c2, uint32_t *__restrict__ lines, uint64_t *__restrict__ c2base) {
    const uint64_t line = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= npair) return;
    uint32_t v;
    if constexpr (WIDE) {
        const uint64_t first = (line >> sb_shift) << sb_shift;
        const uint64_t base = before[first];
        v = (uint32_t)(before[line] - base);
        if (line == first) c2base[(line >> sb_shift) * 16 + code] = c2 + base;
    } else {
        v = (uint32_t)(c2 + before[line]);
    }
    lines[line * kPairWords + (code >> 2) * 8 + (code & 3u)] = v;
}

#define P_TRY(e) CU_TRY_IN("pair image: ", e)

}  // namespace

int build_pair_image_on_device(int device, const IndexView &ix, const uint64_t start[kAlphabet], PairImage &img,
                               uint8_t **keep_codes) {
    const bool wide = index_is_wide(ix);
    const uint64_t npair = ix.total / kPairSyms + 1;
    const uint32_t sb_shift = ix.sb_shift;
    img.npair = npair;
    img.n_super2 = (uint32_t)(((npair - 1) >> sb_shift) + 1);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);

    DeviceScratch tmp;
    uint8_t *d_codes = nullptr, *d_counts = nullptr, *d_sym = nullptr;
    uint64_t *d_before = nullptr, *d_q = nullptr;
    P_TRY(cudaMalloc((void **)&img.lines, npair * kPairBytes));
    if (wide) P_TRY(cudaMalloc((void **)&img.c2base, (size_t)img.n_super2 * 16 * sizeof(uint64_t)));
    P_TRY(tmp.alloc(&d_codes, npair * kPairSyms));
    P_TRY(tmp.alloc(&d_counts, npair * 16));
    P_TRY(tmp.alloc(&d_before, npair));
    P_TRY(tmp.alloc(&d_sym, 16));
    P_TRY(tmp.alloc(&d_q, 16 * 4));
    P_TRY(cudaMemset(d_codes + ix.total, 0, npair * kPairSyms - ix.total));  // positions >= N are invalid

    // C2[b,a] = C[a] + rank(a, C[b]): constrain_range(a, [C[b], C[b])) for the 16 ACGT pairs
    static const uint8_t acgt[4] = {1, 2, 3, 5};
    uint8_t h_sym[16];
    uint64_t h_pos[16], h_c2[16];
    for (int c = 0; c < 16; c++) {
        h_sym[c] = acgt[c & 3];
        h_pos[c] = start[acgt[c >> 2]];
    }
    P_TRY(cudaMemcpy(d_sym, h_sym, sizeof(h_sym), cudaMemcpyHostToDevice));
    P_TRY(cudaMemcpy(d_q, h_pos, sizeof(h_pos), cudaMemcpyHostToDevice));
    P_TRY(launch_constrain_ranges(device, ix, d_sym, d_q, d_q, 16, d_q + 16, d_q + 32, nullptr));
    P_TRY(cudaMemcpy(h_c2, d_q + 16, sizeof(h_c2), cudaMemcpyDeviceToHost));

    // 1. codes
    if (ix.total) {
        const uint64_t want = (ix.total + kCountThreads - 1) / kCountThreads;
        const unsigned grid = (unsigned)std::min<uint64_t>(want, (uint64_t)sms * 32);
        if (wide) pair_codes_kernel<true><<<grid, kCountThreads>>>(ix, d_codes);
        else pair_codes_kernel<false><<<grid, kCountThreads>>>(ix, d_codes);
        P_TRY(cudaGetLastError());
        g_launches++;
    }
    // 2. planes + per-line counts
    pair_fill_kernel<<<(unsigned)((npair + 127) / 128), 128>>>(d_codes, npair, reinterpret_cast<uint32_t *>(img.lines), d_counts);
    P_TRY(cudaGetLastError());
    g_launches++;
    // 3 + 4. per-code prefix sums over lines, stamped as they are produced
    {
        cub::TransformInputIterator<uint64_t, WidenU8, const uint8_t *> in(d_counts, WidenU8{});
        void *d_temp = nullptr;
        size_t temp_bytes = 0;
        P_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, in, d_before, npair));
        P_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        const unsigned sgrid = (unsigned)((npair + 255) / 256);
        for (uint32_t c = 0; c < 16; c++) {
            cub::TransformInputIterator<uint64_t, WidenU8, const uint8_t *> in_c(d_counts + (uint64_t)c * npair, WidenU8{});
            P_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, in_c, d_before, npair));
            if (wide) pair_stamp_kernel<true><<<sgrid, 256>>>(d_before, npair, sb_shift, c, h_c2[c],
                                                               reinterpret_cast<uint32_t *>(img.lines), img.c2base);
            else pair_stamp_kernel<false><<<sgrid, 256>>>(d_before, npair, sb_shift, c, h_c2[c],
                                                          reinterpret_cast<uint32_t *>(img.lines), img.c2base);
            P_TRY(cudaGetLastError());
            g_launches++;
        }
    }
    P_TRY(cudaDeviceSynchronize());
    if (keep_codes) *keep_codes = tmp.take(d_codes);  // handed to the caller instead of freed with the scratch
    return MSBWT_OK;
}

void free_pair_image(PairImage &img) {
    if (img.lines) cudaFree(img.lines);
    if (img.c2base) cudaFree(img.c2base);
    img = {};
}

}  // namespace msbwt
