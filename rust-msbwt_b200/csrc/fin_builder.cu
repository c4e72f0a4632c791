// fin_builder.cu -- device-side construction of the FINAL-STEP image (layout.h; specification and CPU checker in
// oracle/final_step.py, DESIGN.md section 7 item 4).  Built by default on top of the oct image; final_index = 0 (or
// MSBWT_FINAL_INDEX=0) turns it off.
//
// The last kFinSyms (20) symbols a BWT::count_kmer (src/msbwt_core.rs:125-161) consumes need no rank, only the number
// of positions of [l, h) whose 20-symbol code matches, so the image holds no checkpoints and nothing for absent codes:
//
//   1. codes : one thread per position j with a valid 10-symbol code a (the oct builder's): ten steps of our own
//              kernels' arithmetic (two quad steps + two one-symbol ranks) give p = LF^10(j); code20(j) =
//              a << 20 | code10(p) when that one is valid too.
//   2. runs  : heads (code changes, bucket boundaries) are counted, then every head walks to the end of its run
//              (cut at 65535 positions) and emits one record: key = line << 28 | tag, value = len << 16 | offset.
//   3. sort  : records by key (CUB radix sort, 56 bits): the runs of a line, and inside it of a code, are contiguous.
//   4. lines : the first record of every line writes the line: groups `(tag << 4) | nruns` + run words, word 0 =
//              words in use, or kFinOverflow when they do not fit (the kernel then takes the oct steps).
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "engine.h"

namespace msbwt {

namespace {

constexpr uint32_t kValid10 = 1u << kOctCodeBits;
constexpr uint32_t kMask10 = kValid10 - 1u;
constexpr uint64_t kValid20 = 1ull << kFinCodeBits;
constexpr uint32_t kMaxRun = 65535u;

__global__ void __launch_bounds__(256) fin_code20_kernel(IndexView ix, const uint32_t *__restrict__ codes10,
                                                         uint64_t *__restrict__ codes20) {
    __shared__ uint64_t cb_smem[4];
    const CBase<false> cb = stage_cbase<false>(ix, cb_smem);
    const C4Base<false> c4{};
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < ix.total; j += step) {
        const uint32_t a = codes10[j];
        uint64_t v = 0;
        if (a & kValid10) {
            uint32_t l = (uint32_t)j, h = (uint32_t)j;
            quad_step<false>(ix, c4, (a >> 12) & 255u, l, h);  // LF^4(j)
            h = l;
            quad_step<false>(ix, c4, (a >> 4) & 255u, l, h);   // LF^8(j)
            h = l;
            rank_step<false, 1>(ix, cb, (0x5321u >> (4u * ((a >> 2) & 3u))) & 7u, l, h);  // A,C,G,T = 1,2,3,5
            h = l;
            rank_step<false, 1>(ix, cb, (0x5321u >> (4u * (a & 3u))) & 7u, l, h);          // l = LF^10(j)
            const uint32_t b = codes10[l];
            if (b & kValid10) v = kValid20 | ((uint64_t)(a & kMask10) << kOctCodeBits) | (uint64_t)(b & kMask10);
        }
        codes20[j] = v;
    }
}

// The same codes without a quad image (indexes of 2^32 positions and more): ten one-symbol steps through the one-step
// blocks -- the symbols are the digits of the position's own 10-symbol code -- then the code found there.
template <bool WIDE>
__global__ void __launch_bounds__(256) fin_code_walk_kernel(IndexView ix, const uint32_t *__restrict__ codes10,
                                                            uint64_t *__restrict__ codes20) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < ix.total; j += step) {
        const uint32_t a = codes10[j];
        uint64_t v = 0;
        if (a & kValid10) {
            P p = (P)j;
#pragma unroll 1
            for (int r = kOctSyms - 1; r >= 0; r--) p = lf_step<WIDE>(ix, cb, (0x5321u >> (4u * ((a >> (2 * r)) & 3u))) & 7u, p);  // A,C,G,T = 1,2,3,5
            const uint32_t b = codes10[p];
            if (b & kValid10) v = kValid20 | ((uint64_t)(a & kMask10) << kOctCodeBits) | (uint64_t)(b & kMask10);
        }
        codes20[j] = v;
    }
}

__device__ __forceinline__ bool fin_is_head(const uint64_t *codes20, uint64_t j, uint64_t bmask) {
    const uint64_t v = codes20[j];
    return (v & kValid20) && (j == 0 || (j & bmask) == 0 || codes20[j - 1] != v);
}

__global__ void __launch_bounds__(256) fin_count_runs_kernel(const uint64_t *__restrict__ codes20, uint64_t total, uint32_t shift,
                                                             unsigned long long *__restrict__ runs) {
    const uint64_t bmask = (1ull << shift) - 1ull, step = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long mine = 0;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += step) {
        if (!fin_is_head(codes20, j, bmask)) continue;
        // a run longer than kMaxRun positions is stored as several records
        uint64_t len = 1;
        const uint64_t v = codes20[j];
        while (j + len < total && ((j + len) & bmask) != 0 && codes20[j + len] == v) len++;
        mine += (len + kMaxRun - 1) / kMaxRun;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
    if ((threadIdx.x & 31u) == 0 && mine) atomicAdd(runs, mine);
}

__global__ void __launch_bounds__(256) fin_emit_kernel(const uint64_t *__restrict__ codes20, uint64_t total, uint32_t shift, uint32_t lb,
                                                       uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                       unsigned long long *__restrict__ cursor) {
    const uint64_t bmask = (1ull << shift) - 1ull, step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += step) {
        if (!fin_is_head(codes20, j, bmask)) continue;
        const uint64_t v = codes20[j];
        uint64_t len = 1;
        while (j + len < total && ((j + len) & bmask) != 0 && codes20[j + len] == v) len++;
        const uint64_t mixed = fin_mix40(v & (kValid20 - 1ull));
        const uint64_t line = ((j >> shift) << lb) | (mixed & ((1ull << lb) - 1ull));
        const uint64_t key = (line << kFinTagBits) | (mixed >> lb);
        const uint64_t pieces = (len + kMaxRun - 1) / kMaxRun;
        unsigned long long slot = atomicAdd(cursor, (unsigned long long)pieces);
        uint64_t at = j;
        while (len) {
            const uint32_t piece = len < (uint64_t)kMaxRun ? (uint32_t)len : kMaxRun;
            keys[slot] = key;
            vals[slot] = (piece << 16) | (uint32_t)(at & bmask);
            slot++;
            at += piece;
            len -= piece;
        }
    }
}

// records sorted by key: the first record of a line writes the whole line
__global__ void __launch_bounds__(256) fin_lines_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals, uint64_t n_runs,
                                                        uint32_t *__restrict__ lines, unsigned long long *__restrict__ overflow) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_runs; i += step) {
        const uint64_t line = keys[i] >> kFinTagBits;
        if (i && (keys[i - 1] >> kFinTagBits) == line) continue;
        uint32_t *w = lines + line * kFinLineWords;
        uint32_t used = 0, header = 0, in_group = 0;
        uint64_t cur_key = ~0ull;
        bool over = false;
        for (uint64_t r = i; r < n_runs && (keys[r] >> kFinTagBits) == line; r++) {
            if (keys[r] != cur_key || in_group == 15u) {  // a new code, or a 16th run of the same one: a new group
                if (used + 2u > (uint32_t)kFinLineWords - 1u) { over = true; break; }
                cur_key = keys[r];
                header = ++used;
                in_group = 0;
                w[header] = (uint32_t)(cur_key & ((1ull << kFinTagBits) - 1ull)) << 4;
            } else if (used + 1u > (uint32_t)kFinLineWords - 1u) {
                over = true;
                break;
            }
            w[++used] = vals[r];
            w[header] = (w[header] & ~15u) | ++in_group;
        }
        w[0] = over ? kFinOverflow : used;
        if (over) atomicAdd(overflow, 1ull);
    }
}

#define F_TRY(e) CU_TRY_IN("final-step image: ", e)

}  // namespace

uint64_t fin_image_bytes(uint64_t total, int shift, int lb) { return (((total >> shift) + 1) << lb) * (uint64_t)kFinLineBytes; }

static void fin_trace(const char *what) {
    static const bool on = getenv("MSBWT_TRACE") != nullptr;
    if (on) {
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        fprintf(stderr, "[msbwt] final-step image: %s (%.1f GB of device memory free)\n", what, (double)free_b / 1e9);
    }
}

// Stage 1 (needs the quad image and the one-step blocks): code20 of every position, 8 bytes each
int build_fin_codes_on_device(int device, const IndexView &ix, const uint32_t *d_codes10, uint64_t **d_codes20_out) {
    *d_codes20_out = nullptr;
    if (!ix.quad || !d_codes10 || index_is_wide(ix)) return fail(MSBWT_EINVAL, "final-step image: needs the quad image, the 10-symbol codes and 32-bit positions");
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((ix.total + 255) / 256, (uint64_t)sms * 32));
    uint64_t *d_codes20 = nullptr;
    F_TRY(cudaMalloc((void **)&d_codes20, std::max<uint64_t>(1, ix.total) * sizeof(uint64_t)));
    fin_trace("codes");
    fin_code20_kernel<<<grid, 256>>>(ix, d_codes10, d_codes20);
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(d_codes20);
        return fail(MSBWT_ECUDA, std::string("final-step image: code kernel: ") + cudaGetErrorString(e));
    }
    *d_codes20_out = d_codes20;
    return MSBWT_OK;
}

// Stage 1 without a quad image (any index; the only way for one of 2^32 positions and more): `ix` needs only the one-step
// blocks
int build_fin_codes_by_walk(int device, const IndexView &ix, const uint32_t *d_codes10, uint64_t **d_codes20_out) {
    *d_codes20_out = nullptr;
    if (!d_codes10) return fail(MSBWT_EINVAL, "final-step image: needs the 10-symbol codes");
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((ix.total + 255) / 256, (uint64_t)sms * 32));
    uint64_t *d_codes20 = nullptr;
    F_TRY(cudaMalloc((void **)&d_codes20, std::max<uint64_t>(1, ix.total) * sizeof(uint64_t)));
    fin_trace("codes (walk)");
    if (index_is_wide(ix)) fin_code_walk_kernel<true><<<grid, 256>>>(ix, d_codes10, d_codes20);
    else fin_code_walk_kernel<false><<<grid, 256>>>(ix, d_codes10, d_codes20);
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(d_codes20);
        return fail(MSBWT_ECUDA, std::string("final-step image: code walk kernel: ") + cudaGetErrorString(e));
    }
    *d_codes20_out = d_codes20;
    return MSBWT_OK;
}

// Stage 2 (needs nothing but the codes, which it OWNS and frees as soon as the run records exist): the lines
int build_fin_lines_on_device(int device, uint64_t total, uint64_t *d_codes20_in, int shift, int lb, FinImage &img) {
    DevicePtr<uint64_t> codes20(d_codes20_in);
    if (!d_codes20_in) return fail(MSBWT_EINVAL, "final-step image: no position codes");
    if (shift < 8 || shift > 16 || lb < kFinCodeBits - kFinTagBits || lb > 20) return fail(MSBWT_EINVAL, "final-step image: bucket shift 8..16, lines per bucket 2^12..2^20");
    if (((((total >> shift) + 1) << lb) >> (64 - kFinTagBits)) != 0) return fail(MSBWT_EINVAL, "final-step image: line index and tag do not fit one 64-bit sort key");
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((total + 255) / 256, (uint64_t)sms * 32));
    const uint64_t *d_codes20 = codes20.get();

    DeviceScratch tmp;
    unsigned long long *d_stat = nullptr;  // [0] records, [1] emit cursor, [2] overflowed lines
    F_TRY(tmp.alloc(&d_stat, 3));
    F_TRY(cudaMemsetAsync(d_stat, 0, 3 * sizeof(unsigned long long)));
    fin_count_runs_kernel<<<grid, 256>>>(d_codes20, total, (uint32_t)shift, d_stat);
    F_TRY(cudaGetLastError());
    g_launches++;
    unsigned long long n_runs = 0;
    F_TRY(cudaMemcpy(&n_runs, d_stat, sizeof(n_runs), cudaMemcpyDeviceToHost));

    const uint64_t nlines = ((total >> shift) + 1) << lb;
    img.shift = shift;
    img.lb = lb;
    img.nlines = nlines;
    img.runs = n_runs;
    uint64_t *k0 = nullptr, *k1 = nullptr;
    uint32_t *v0 = nullptr, *v1 = nullptr;
    if (n_runs) {
        fin_trace("run records");
        F_TRY(tmp.alloc(&k0, n_runs));
        F_TRY(tmp.alloc(&v0, n_runs));
        fin_emit_kernel<<<grid, 256>>>(d_codes20, total, (uint32_t)shift, (uint32_t)lb, k0, v0, d_stat + 1);
        F_TRY(cudaGetLastError());
        F_TRY(cudaDeviceSynchronize());
        g_launches++;
    }
    codes20.reset();  // the records carry everything from here on
    F_TRY(cudaMalloc((void **)&img.lines, nlines * kFinLineBytes));
    F_TRY(cudaMemsetAsync(img.lines, 0, nlines * kFinLineBytes));
    if (n_runs) {
        fin_trace("sort");
        F_TRY(tmp.alloc(&k1, n_runs));
        F_TRY(tmp.alloc(&v1, n_runs));
        cub::DoubleBuffer<uint64_t> keys(k0, k1);
        cub::DoubleBuffer<uint32_t> vals(v0, v1);
        size_t temp_bytes = 0;
        int line_bits = 1;  // bits of a line index
        while (line_bits < 64 && (nlines >> line_bits) != 0) line_bits++;
        const int end_bit = std::min(64, kFinTagBits + line_bits);
        F_TRY(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, vals, (int64_t)n_runs, 0, end_bit));
        void *d_temp = nullptr;
        F_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        F_TRY(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, keys, vals, (int64_t)n_runs, 0, end_bit));
        fin_trace("lines");
        fin_lines_kernel<<<grid, 256>>>(keys.Current(), vals.Current(), n_runs, reinterpret_cast<uint32_t *>(img.lines), d_stat + 2);
        F_TRY(cudaGetLastError());
        g_launches += 2;
    }
    unsigned long long over = 0;
    F_TRY(cudaMemcpy(&over, d_stat + 2, sizeof(over), cudaMemcpyDeviceToHost));
    img.overflow_lines = over;
    F_TRY(cudaDeviceSynchronize());
    fin_trace("done");
    return MSBWT_OK;
}

void free_fin_image(FinImage &img) {
    if (img.lines) cudaFree(img.lines);
    img = {};
}

}  // namespace msbwt
