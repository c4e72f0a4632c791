// builder.cu -- device-side construction of the block image (layout.h) from the msbwt RLE byte
// stream: the GPU counterpart of the reference's load path, standard_init -> calculate_totals +
// construct_fmindex (src/rle_bwt.rs:324-467), which is a serial host pass over every byte.
//
//   1. scan   : every RLE byte contributes digit * 32^j symbols (j = its index inside the run of
//               equal-symbol bytes, src/msbwt_core.rs:4-14); an exclusive prefix sum of the
//               contributions gives the BWT position at which each byte's run begins.
//   2. select : the bytes that start a run -> run table (start position, symbol).
//   3. fill   : one thread per 128-symbol block binary-searches the run table and paints the three
//               bit-planes of its block, counting the six symbols as it goes.
//   4. scan   : per-symbol exclusive prefix sums of the block counts -> checkpoints.
//   5. stamp  : checkpoints (relative to the superblock), aux ($,N) and cbase rows.
//
// The scans / select are CUB device primitives (plumbing, like the radix sort a loader would
// use); fill/stamp are ours.  The host builder in loader.cu stays as the inspection path
// (msbwt_debug_build_image) and tests compare the two images word for word.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "../../include/msbwt_gpu.h"
#include "engine.h"

namespace msbwt {

namespace {

struct Contribution {  // symbols contributed by RLE byte i
    const uint8_t *rle;
    __host__ __device__ uint64_t operator()(uint64_t i) const {
        const uint8_t v = rle[i], c = v & 7u;
        int j = 0;
        while (j < 12 && (uint64_t)j < i && (rle[i - 1 - j] & 7u) == c) j++;
        return (uint64_t)(v >> 3) << (5 * j);
    }
};

struct StartsRun {
    const uint8_t *rle;
    __host__ __device__ bool operator()(uint64_t i) const { return i == 0 || ((rle[i] ^ rle[i - 1]) & 7u) != 0; }
};

struct Widen {
    __host__ __device__ uint64_t operator()(uint32_t v) const { return v; }
};

// symbol >= 6 or a run of 13+ bytes (>= 2^60 symbols) -> flag, as the host builder refuses them
__global__ void validate_rle_kernel(const uint8_t *__restrict__ rle, uint64_t len, uint32_t *__restrict__ flag) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    const uint8_t c = rle[i] & 7u;
    bool bad = c >= kAlphabet;
    if (i >= 12) {
        bool same = true;
        for (int j = 1; j <= 12; j++) same &= (rle[i - j] & 7u) == c;
        bad |= same;
    }
    if (bad) atomicOr(flag, 1u);
}

__global__ void run_table_kernel(const uint8_t *__restrict__ rle, const uint64_t *__restrict__ before,
                                 const uint64_t *__restrict__ run_byte, uint64_t n_runs,
                                 uint64_t *__restrict__ run_pos, uint8_t *__restrict__ run_sym) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint64_t i = run_byte[r];
    run_pos[r] = before[i];
    run_sym[r] = rle[i] & 7u;
}

__device__ __forceinline__ void paint(uint32_t *w, uint32_t off, uint32_t end, uint32_t sym) {
    // symbol `sym` at block offsets [off, end); half-major layout of layout.h
    for (uint32_t j = off >> 5; j <= (end - 1) >> 5; j++) {
        const uint32_t lo = off > (j << 5) ? off - (j << 5) : 0;
        const uint32_t hi = end < ((j + 1) << 5) ? end - (j << 5) : 32;
        const uint32_t m = (hi == 32 ? ~0u : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
        uint32_t *hw = w + (j >> 1) * 8 + (j & 1);
        if (sym & 1u) hw[2] |= m;
        if (sym & 2u) hw[4] |= m;
        if (sym & 4u) hw[6] |= m;
    }
}

// one thread per block: planes + per-block symbol counts (SoA: counts[s * nblocks + b])
__global__ void fill_blocks_kernel(const uint64_t *__restrict__ run_pos, const uint8_t *__restrict__ run_sym,
                                   uint64_t n_runs, uint64_t total, uint64_t nblocks, uint32_t *__restrict__ blocks,
                                   uint32_t *__restrict__ counts) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const uint64_t lo = b << kBlockShift;
    uint32_t w[kWordsPerBlock];
#pragma unroll
    for (int i = 0; i < kWordsPerBlock; i++) w[i] = 0;
    uint32_t cnt[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t pos = lo;
    const uint64_t stop = (lo + kBlockSyms < total) ? lo + kBlockSyms : total;
    if (pos < stop) {
        // last run whose start is <= lo
        uint64_t a = 0, z = n_runs;
        while (z - a > 1) {
            const uint64_t mid = (a + z) >> 1;
            if (run_pos[mid] <= lo) a = mid; else z = mid;
        }
        uint64_t r = a;
        while (pos < stop) {
            const uint64_t run_end = (r + 1 < n_runs) ? run_pos[r + 1] : total;
            if (run_end <= pos) { r++; continue; }  // empty runs (all-zero digits) and the run before lo
            const uint64_t e = run_end < stop ? run_end : stop;
            const uint32_t s = run_sym[r];
            paint(w, (uint32_t)(pos - lo), (uint32_t)(e - lo), s);
            cnt[s] += (uint32_t)(e - pos);
            pos = e;
        }
    }
    if (pos < lo + kBlockSyms) paint(w, (uint32_t)(pos - lo), kBlockSyms, 7u);  // padding matches no symbol
    uint4 *dst = reinterpret_cast<uint4 *>(blocks + b * kWordsPerBlock);
#pragma unroll
    for (int i = 0; i < 4; i++) dst[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
#pragma unroll
    for (int s = 0; s < kAlphabet; s++) counts[(uint64_t)s * nblocks + b] = cnt[s];
}

struct Starts { uint64_t c[kAlphabet]; };

// checkpoints relative to the superblock, aux, cbase
__global__ void stamp_checkpoints_kernel(const uint64_t *__restrict__ before, uint64_t nblocks, uint32_t sb_shift,
                                         Starts start, uint32_t *__restrict__ blocks, uint32_t *__restrict__ aux,
                                         uint64_t *__restrict__ cbase) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const uint64_t first = (b >> sb_shift) << sb_shift;
    uint32_t rel[kAlphabet];
#pragma unroll
    for (int s = 0; s < kAlphabet; s++) {
        const uint64_t here = before[(uint64_t)s * nblocks + b], base = before[(uint64_t)s * nblocks + first];
        rel[s] = (uint32_t)(here - base);
        if (b == first) cbase[(b >> sb_shift) * 8 + s] = start.c[s] + base;
    }
    if (b == first) { cbase[(b >> sb_shift) * 8 + 6] = 0; cbase[(b >> sb_shift) * 8 + 7] = 0; }
    uint32_t *w = blocks + b * kWordsPerBlock;
    w[0] = rel[1]; w[1] = rel[2];  // A, C in half 0
    w[8] = rel[3]; w[9] = rel[5];  // G, T in half 1
    aux[b * 2] = rel[0];
    aux[b * 2 + 1] = rel[4];
}

#define B_TRY(e) CU_TRY(e)

}  // namespace

int build_image_on_device(const uint8_t *h_rle, uint64_t len, uint32_t sb_shift, DeviceImage &img) {
    if (len && !h_rle) return fail(MSBWT_EINVAL, "rle is NULL");
    if (sb_shift == 0) sb_shift = kDefaultSuperShift;
    if (sb_shift > (uint32_t)kDefaultSuperShift) return fail(MSBWT_EINVAL, "superblock_shift > 25 would overflow the u32 block counters");
    DeviceScratch tmp;
    uint8_t *d_rle = nullptr;
    uint64_t *d_before = nullptr, *d_run_byte = nullptr, *d_nruns = nullptr, *d_run_pos = nullptr;
    uint8_t *d_run_sym = nullptr;
    uint32_t *d_flag = nullptr;
    uint64_t total = 0, n_runs = 0;

    B_TRY(tmp.alloc(&d_rle, len));
    B_TRY(tmp.alloc(&d_before, len + 1));
    B_TRY(tmp.alloc(&d_flag, 1));
    B_TRY(tmp.alloc(&d_nruns, 1));
    B_TRY(cudaMemset(d_flag, 0, sizeof(uint32_t)));
    if (len) {
        B_TRY(cudaMemcpy(d_rle, h_rle, len, cudaMemcpyHostToDevice));
        validate_rle_kernel<<<(unsigned)((len + 255) / 256), 256>>>(d_rle, len, d_flag);
        B_TRY(cudaGetLastError());
        uint32_t flag = 0;
        B_TRY(cudaMemcpy(&flag, d_flag, sizeof(flag), cudaMemcpyDeviceToHost));
        if (flag) return fail(MSBWT_EFORMAT, "RLE stream has a symbol >= 6 or a run longer than 2^60 symbols");

        // 1. positions: exclusive sum over len + 1 items (the extra item yields the total)
        cub::CountingInputIterator<uint64_t> idx(0);
        cub::TransformInputIterator<uint64_t, Contribution, cub::CountingInputIterator<uint64_t>> contrib(idx, Contribution{d_rle});
        void *d_temp = nullptr;
        size_t temp_bytes = 0;
        B_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, contrib, d_before, len));
        B_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        B_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, contrib, d_before, len));
        uint64_t last_before = 0;
        B_TRY(cudaMemcpy(&last_before, d_before + (len - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost));
        total = last_before + Contribution{h_rle}(len - 1);
        if (total >> 62) return fail(MSBWT_EFORMAT, "BWT longer than 2^62 symbols");

        // 2. run table
        B_TRY(tmp.alloc(&d_run_byte, len));
        cub::TransformInputIterator<bool, StartsRun, cub::CountingInputIterator<uint64_t>> flags(idx, StartsRun{d_rle});
        void *d_temp2 = nullptr;
        size_t temp2_bytes = 0;
        B_TRY(cub::DeviceSelect::Flagged(nullptr, temp2_bytes, idx, flags, d_run_byte, d_nruns, (int64_t)len));
        B_TRY(tmp.alloc((uint8_t **)&d_temp2, temp2_bytes));
        B_TRY(cub::DeviceSelect::Flagged(d_temp2, temp2_bytes, idx, flags, d_run_byte, d_nruns, (int64_t)len));
        B_TRY(cudaMemcpy(&n_runs, d_nruns, sizeof(uint64_t), cudaMemcpyDeviceToHost));
        B_TRY(tmp.alloc(&d_run_pos, n_runs));
        B_TRY(tmp.alloc(&d_run_sym, n_runs));
        run_table_kernel<<<(unsigned)((n_runs + 255) / 256), 256>>>(d_rle, d_before, d_run_byte, n_runs, d_run_pos, d_run_sym);
        B_TRY(cudaGetLastError());
    }

    img.total = total;
    img.sb_shift = sb_shift;
    img.nblocks = (total >> kBlockShift) + 1;
    img.n_super = (uint32_t)(((img.nblocks - 1) >> sb_shift) + 1);
    B_TRY(cudaMalloc((void **)&img.blocks, img.nblocks * kBlockBytes));
    B_TRY(cudaMalloc((void **)&img.aux, img.nblocks * 2 * sizeof(uint32_t)));
    B_TRY(cudaMalloc((void **)&img.cbase, (size_t)img.n_super * 8 * sizeof(uint64_t)));

    // 3. planes + block counts
    uint32_t *d_counts = nullptr;
    uint64_t *d_before_blk = nullptr;
    B_TRY(tmp.alloc(&d_counts, img.nblocks * kAlphabet));
    B_TRY(tmp.alloc(&d_before_blk, img.nblocks * kAlphabet));
    const unsigned blk_grid = (unsigned)((img.nblocks + 127) / 128);
    fill_blocks_kernel<<<blk_grid, 128>>>(d_run_pos, d_run_sym, n_runs, total, img.nblocks,
                                          reinterpret_cast<uint32_t *>(img.blocks), d_counts);
    B_TRY(cudaGetLastError());

    // 4. per-symbol prefix sums over blocks
    {
        cub::TransformInputIterator<uint64_t, Widen, const uint32_t *> in(d_counts, Widen{});
        void *d_temp = nullptr;
        size_t temp_bytes = 0;
        B_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, in, d_before_blk, img.nblocks));
        B_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        for (int s = 0; s < kAlphabet; s++) {
            cub::TransformInputIterator<uint64_t, Widen, const uint32_t *> in_s(d_counts + (uint64_t)s * img.nblocks, Widen{});
            B_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, in_s, d_before_blk + (uint64_t)s * img.nblocks, img.nblocks));
        }
    }
    // totals = prefix before the last block + the last block's own counts
    Starts start{};
    uint64_t sum = 0;
    for (int s = 0; s < kAlphabet; s++) {
        uint64_t bef = 0;
        uint32_t last = 0;
        B_TRY(cudaMemcpy(&bef, d_before_blk + (uint64_t)s * img.nblocks + (img.nblocks - 1), sizeof(bef), cudaMemcpyDeviceToHost));
        B_TRY(cudaMemcpy(&last, d_counts + (uint64_t)s * img.nblocks + (img.nblocks - 1), sizeof(last), cudaMemcpyDeviceToHost));
        img.counts[s] = bef + last;
        img.start[s] = sum;
        start.c[s] = sum;
        sum += img.counts[s];
    }
    if (sum != total) return fail(MSBWT_ECUDA, "internal error: block counts do not add up to the stream total");

    // 5. checkpoints
    stamp_checkpoints_kernel<<<(unsigned)((img.nblocks + 255) / 256), 256>>>(
        d_before_blk, img.nblocks, sb_shift, start, reinterpret_cast<uint32_t *>(img.blocks), img.aux, img.cbase);
    B_TRY(cudaGetLastError());
    B_TRY(cudaDeviceSynchronize());
    return MSBWT_OK;
}

void free_device_image(DeviceImage &img) {
    if (img.blocks) cudaFree(img.blocks);
    if (img.aux) cudaFree(img.aux);
    if (img.cbase) cudaFree(img.cbase);
    img.blocks = nullptr; img.aux = nullptr; img.cbase = nullptr;
}

}  // namespace msbwt
