// quad_builder.cu -- device-side construction of the QUAD image (layout.h) from the pair image and
// the per-position pair codes that are already resident on the device.
//
// The reference has no counterpart: its index is the sampled table of construct_fmindex
// (src/rle_bwt.rs:387-467).  What the quad image must reproduce is the composition of four
// RleBWT::constrain_range calls (src/rle_bwt.rs:202-287); layout.h states the identity.
//
//   1. codes : one thread per 96-position pair line.  LF^2 restricted to one pair code is order
//              preserving, so LF^2(j) = (the line's checkpoint for code2(j)) + (occurrences of that
//              code earlier in the line): a running counter per code, no rank query.  The quad code is
//              code2(j) * 16 + code2(LF^2(j)) (one random byte read), valid when both halves are.
//   2. fill  : one warp per 224-position sector span; __match_any_sync groups the lanes of each
//              32-position word by code and the first lane of a group stores the group's lane mask as
//              that code's occurrence word (the image starts zeroed).
//   3. scan  : per code, an exclusive prefix sum over its sectors' popcounts (CUB, plumbing; the
//              popcounts are computed on the fly by the input iterator).
//   4. stamp : checkpoints -- absolute (C4 included) when N < 2^32, otherwise relative to the quad
//              superblock with the base in c4base.
//   C4[c] = four constrain_range calls of our own kernel applied to position 0.
#include <algorithm>

#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "engine.h"

namespace msbwt {

namespace {

constexpr int kCodeThreads = 128;

template <bool WIDE>
__global__ void __launch_bounds__(kCodeThreads) quad_codes_kernel(IndexView ix, const uint8_t *__restrict__ codes2,
                                                                  uint16_t *__restrict__ codes4) {
    using P = typename Pos<WIDE>::type;
    __shared__ P next_at[16][kCodeThreads];  // per thread (column): where the next occurrence of each pair code maps
    const uint64_t line = (uint64_t)blockIdx.x * kCodeThreads + threadIdx.x;
    if (line >= ix.npair) return;
    const uint32_t *lw = reinterpret_cast<const uint32_t *>(ix.pair) + line * kPairWords;
#pragma unroll
    for (int c = 0; c < 16; c++) {
        P v = (P)__ldg(lw + (c >> 2) * 8 + (c & 3));
        if constexpr (WIDE) v += ix.c2base[((line >> ix.sb_shift) << 4) + c];
        next_at[c][threadIdx.x] = v;
    }
    const uint4 *src = reinterpret_cast<const uint4 *>(codes2 + line * kPairSyms);  // 96 = 6 x 16 bytes
    uint4 *dst = reinterpret_cast<uint4 *>(codes4 + line * kPairSyms);              // 8 codes per store
#pragma unroll 1
    for (int v16 = 0; v16 < kPairSyms / 16; v16++) {
        const uint4 rv = src[v16];
        const uint32_t raw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
        for (int g = 0; g < 2; g++) {
            uint32_t first[8], second[8];
            P at[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int b = g * 8 + u;
                first[u] = (raw[b >> 2] >> (8 * (b & 3))) & 0xffu;
                at[u] = 0;
                if (first[u] & 16u) at[u] = next_at[first[u] & 15u][threadIdx.x]++;
            }
#pragma unroll
            for (int u = 0; u < 8; u++) second[u] = (first[u] & 16u) ? (uint32_t)__ldg(codes2 + at[u]) : 0u;
            uint32_t o[4];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const uint32_t c4 = (first[u] & second[u] & 16u) ? (0x100u | ((first[u] & 15u) << 4) | (second[u] & 15u)) : 0u;
                if (u & 1) o[u >> 1] |= c4 << 16; else o[u >> 1] = c4;
            }
            dst[v16 * 2 + g] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

__global__ void __launch_bounds__(256) quad_fill_kernel(const uint16_t *__restrict__ codes4, uint64_t nsec_real,
                                                        uint64_t nsec4, uint32_t *__restrict__ sectors) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = (uint64_t)gridDim.x * 8u;
    for (uint64_t s = (uint64_t)blockIdx.x * 8u + (threadIdx.x >> 5); s < nsec_real; s += warps) {
        const uint16_t *src = codes4 + s * kQuadSyms + lane;
#pragma unroll
        for (int w = 0; w < 7; w++) {
            const uint32_t v = src[w * 32];
            const bool valid = (v & 0x100u) != 0;
            const uint32_t key = valid ? (v & 255u) : 256u + lane;  // invalid positions group with nobody
            const uint32_t m = __match_any_sync(0xffffffffu, key);
            if (valid && (m & ((1u << lane) - 1u)) == 0)
                sectors[((uint64_t)(v & 255u) * nsec4 + s) * kQuadWords + 1 + w] = m;
        }
    }
}

// occurrences in one sector (words 1..7; word 0 is the checkpoint slot)
struct SectorCount {
    const uint4 *base;
    __host__ __device__ uint64_t operator()(uint64_t s) const {
#ifdef __CUDA_ARCH__
        const uint4 a = base[2 * s], b = base[2 * s + 1];
        return (uint64_t)(__popc(a.y) + __popc(a.z) + __popc(a.w) + __popc(b.x) + __popc(b.y) + __popc(b.z) + __popc(b.w));
#else
        (void)s;
        return 0;
#endif
    }
};

template <bool WIDE>
__global__ void quad_stamp_kernel(const uint64_t *__restrict__ before, uint64_t nsec4, uint32_t sb_shift4, uint32_t code,
                                  uint64_t c4, uint32_t *__restrict__ code_sectors, uint64_t *__restrict__ c4base) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsec4) return;
    uint32_t v;
    if constexpr (WIDE) {
        const uint64_t first = (s >> sb_shift4) << sb_shift4;
        const uint64_t base = before[first];
        v = (uint32_t)(before[s] - base);
        if (s == first) c4base[((s >> sb_shift4) << 8) + code] = c4 + base;
    } else {
        v = (uint32_t)(c4 + before[s]);
    }
    code_sectors[s * kQuadWords] = v;
}

#define Q_TRY(e) CU_TRY_IN("quad image: ", e)

}  // namespace

uint64_t quad_image_bytes(uint64_t total) {
    return (uint64_t)kQuadCodes * (total / kQuadSyms + 2) * kQuadSectorBytes;
}

int build_quad_image_on_device(int device, const IndexView &ix, const uint8_t *d_codes2, QuadImage &img,
                               uint16_t **keep_codes) {
    if (!ix.pair || !d_codes2) return fail(MSBWT_EINVAL, "quad image: needs the pair image and its code bytes");
    const bool wide = index_is_wide(ix);
    const uint64_t nsec_real = ix.total / kQuadSyms + 1;  // the last one holds position N
    const uint64_t nsec4 = nsec_real + 1;                 // + one all-zero sector per code: its checkpoint = the code's total
    img.nsec4 = nsec4;
    img.sb_shift4 = std::min<uint32_t>(ix.sb_shift, (uint32_t)kQuadMaxSuperShift);
    img.n_super4 = (uint32_t)(((nsec4 - 1) >> img.sb_shift4) + 1);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);

    DeviceScratch tmp;
    uint16_t *d_codes4 = nullptr;
    uint8_t *d_sym = nullptr;
    uint64_t *d_before = nullptr, *d_pos = nullptr;
    const uint64_t image_bytes = (uint64_t)kQuadCodes * nsec4 * kQuadSectorBytes;
    Q_TRY(cudaMalloc((void **)&img.sectors, image_bytes));
    if (wide) Q_TRY(cudaMalloc((void **)&img.c4base, (size_t)img.n_super4 * kQuadCodes * sizeof(uint64_t)));
    Q_TRY(cudaMemsetAsync(img.sectors, 0, image_bytes));
    const uint64_t ncodes = std::max<uint64_t>(ix.npair * kPairSyms, nsec_real * kQuadSyms);
    Q_TRY(tmp.alloc(&d_codes4, ncodes));
    Q_TRY(tmp.alloc(&d_before, nsec4));
    Q_TRY(tmp.alloc(&d_sym, kQuadCodes));
    Q_TRY(tmp.alloc(&d_pos, 3 * kQuadCodes));
    if (ncodes > ix.npair * kPairSyms)
        Q_TRY(cudaMemsetAsync(d_codes4 + ix.npair * kPairSyms, 0, (ncodes - ix.npair * kPairSyms) * sizeof(uint16_t)));

    // C4[c]: the four steps applied to position 0 (l == h == 0 all the way)
    static const uint8_t acgt[4] = {1, 2, 3, 5};
    uint64_t h_c4[kQuadCodes];
    Q_TRY(cudaMemsetAsync(d_pos, 0, 3 * kQuadCodes * sizeof(uint64_t)));
    uint64_t *cur = d_pos, *nxt = d_pos + kQuadCodes, *spare = d_pos + 2 * kQuadCodes;
    for (int r = 0; r < 4; r++) {
        uint8_t h_sym[kQuadCodes];
        for (int c = 0; c < kQuadCodes; c++) h_sym[c] = acgt[(c >> (2 * (3 - r))) & 3];
        Q_TRY(cudaMemcpy(d_sym, h_sym, sizeof(h_sym), cudaMemcpyHostToDevice));
        Q_TRY(launch_constrain_ranges(device, ix, d_sym, cur, cur, kQuadCodes, nxt, spare, nullptr));
        std::swap(cur, nxt);
    }
    Q_TRY(cudaMemcpy(h_c4, cur, sizeof(h_c4), cudaMemcpyDeviceToHost));

    // 1. codes
    {
        const unsigned grid = (unsigned)((ix.npair + kCodeThreads - 1) / kCodeThreads);
        if (wide) quad_codes_kernel<true><<<grid, kCodeThreads>>>(ix, d_codes2, d_codes4);
        else quad_codes_kernel<false><<<grid, kCodeThreads>>>(ix, d_codes2, d_codes4);
        Q_TRY(cudaGetLastError());
        g_launches++;
    }
    // 2. occurrence bits
    {
        const unsigned grid = (unsigned)std::min<uint64_t>((nsec_real + 7) / 8, (uint64_t)sms * 64);
        quad_fill_kernel<<<grid, 256>>>(d_codes4, nsec_real, nsec4, reinterpret_cast<uint32_t *>(img.sectors));
        Q_TRY(cudaGetLastError());
        g_launches++;
    }
    // 3 + 4. per-code prefix sums over sectors, stamped as they are produced
    {
        using CountIt = cub::TransformInputIterator<uint64_t, SectorCount, cub::CountingInputIterator<uint64_t>>;
        void *d_temp = nullptr;
        size_t temp_bytes = 0;
        CountIt probe(cub::CountingInputIterator<uint64_t>(0), SectorCount{img.sectors});
        Q_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, probe, d_before, nsec4));
        Q_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        const unsigned sgrid = (unsigned)((nsec4 + 255) / 256);
        for (uint32_t c = 0; c < (uint32_t)kQuadCodes; c++) {
            const uint4 *code_base = img.sectors + (uint64_t)c * nsec4 * 2;
            CountIt in(cub::CountingInputIterator<uint64_t>(0), SectorCount{code_base});
            Q_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, in, d_before, nsec4));
            uint32_t *cs = reinterpret_cast<uint32_t *>(img.sectors) + (uint64_t)c * nsec4 * kQuadWords;
            if (wide) quad_stamp_kernel<true><<<sgrid, 256>>>(d_before, nsec4, img.sb_shift4, c, h_c4[c], cs, img.c4base);
            else quad_stamp_kernel<false><<<sgrid, 256>>>(d_before, nsec4, img.sb_shift4, c, h_c4[c], cs, img.c4base);
            Q_TRY(cudaGetLastError());
            g_launches++;
        }
    }
    Q_TRY(cudaDeviceSynchronize());
    if (keep_codes) *keep_codes = tmp.take(d_codes4);  // handed to the caller instead of freed with the scratch
    return MSBWT_OK;
}

void free_quad_image(QuadImage &img) {
    if (img.sectors) cudaFree(img.sectors);
    if (img.c4base) cudaFree(img.c4base);
    img = {};
}

}  // namespace msbwt
