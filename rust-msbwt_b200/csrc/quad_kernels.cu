// quad_kernels.cu -- the search kernel over live list A for an index with a quad (and oct) image.
// Same structure as the pair / one-step kernels of kernels.cu (persistent grid, every thread walks its
// own query stream and refills itself); kept in its own translation unit because ptxas 12.9 crashes on
// the module that holds every search kernel together.
//
// Replaces the reference's hot loop: BWT::count_kmer (src/msbwt_core.rs:125-161) calling
// RleBWT::constrain_range (src/rle_bwt.rs:202-287) once per symbol -- here four symbols per index access,
// ten with the oct image (oct_kernel.cuh; layout.h states the identities).
#include "device_rank.cuh"
#include "engine.h"
#include "kernel_common.cuh"
#include "oct_kernel.cuh"

namespace msbwt {

// Persistent kernel over live list A with a QUAD image: one thread per query, four symbols per step
// (one 32-byte sector per boundary).  The depth the suffix table answered is a function of k alone for
// an all-ACGT k-mer (acgt_table_depth), so the remaining count is uniform across the list; a remainder
// that is not a multiple of four (k below the kept table levels) ends with one-step ranks.
constexpr int quad_min_ctas(bool wide) { return wide ? 4 : 6; }

// the rare remainder step of the quad kernel, kept out of line so that its 32 load registers do not
// set the register budget of the quad loop
// (one copy per kernel instantiation: ptxas 12.9 crashes when two entries with different register budgets
// share one out-of-line function)
template <bool WIDE>
__device__ __noinline__ void remainder_step(const IndexView &ix, const CBase<WIDE> &cb, uint32_t sym,
                                            typename Pos<WIDE>::type &l, typename Pos<WIDE>::type &h) {
    rank_step<WIDE, 1>(ix, cb, sym, l, h);
}

template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, quad_min_ctas(WIDE))
count_kmers_quad_kernel(IndexView ix, const uint64_t *__restrict__ packed, PackedLayout lay, uint32_t k,
                        uint64_t *__restrict__ out) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t c4_smem[WIDE ? kQuadMaxSuperInSmem * kQuadCodes : 1];
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const C4Base<WIDE> c4 = stage_c4base<WIDE>(ix, c4_smem);
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t stream = policy_evict_first();

    const uint32_t n = (uint32_t)packed[lay.live()];  // live queries of list A
    const uint32_t owners = gridDim.x * kCountThreads;
    uint32_t i = blockIdx.x * kCountThreads + threadIdx.x;
    if (i >= n) return;
    const uint64_t *w0 = packed + lay.w0(), *seeds = packed + lay.seed(), *wx = packed + lay.wx();
    const uint32_t *qidx = reinterpret_cast<const uint32_t *>(packed + lay.qidx());
    const uint32_t rem0 = k - acgt_table_depth(k, ix.table_s, 4u);

    P l = 0, h = 0;
    uint64_t word = 0, pend = 0, next_word = 0, next_lo = 0;
    [[maybe_unused]] uint64_t next_hi = 0;
    uint32_t q = 0, next_q = 0;
    uint32_t rem = 0;   // symbols still to consume
    int shift = 62;     // bit offset of the next symbol (2 bits) in `word`
    uint32_t widx = 0;

    auto prefetch = [&](uint32_t ii) {
        next_word = ldg_stream(w0 + ii, stream);
        next_lo = ldg_stream(seeds + ii, stream);
        if constexpr (WIDE) next_hi = ldg_stream(seeds + lay.n + ii, stream);
        next_q = __ldg(qidx + ii);
    };
    auto begin = [&]() {
        word = next_word;
        q = next_q & kQidxMask;
        if constexpr (WIDE) { l = next_lo; h = next_hi; } else { l = (uint32_t)next_lo; h = (uint32_t)(next_lo >> 32); }
        rem = rem0;
        shift = 62;
        widx = 0;
        if (rem > (uint32_t)kPairSymsPerWord) pend = ldg_stream(wx + q, stream);  // needed 8 quad steps from now
    };

    prefetch(i);
    begin();
    if (i + owners < n) prefetch(i + owners);

    for (;;) {
        while (rem == 0 || l == h) {
            stg_stream(out + q, (uint64_t)(h - l), stream);
            i += owners;
            if (i >= n) return;
            begin();
            if (i + owners < n) prefetch(i + owners);
        }
        if (shift < 0) {  // 32 symbols per word: a quad never straddles two words
            word = pend;
            widx++;
            shift = 62;
            if (rem > (uint32_t)kPairSymsPerWord) pend = ldg_stream(wx + (uint64_t)widx * lay.n + q, stream);
        }
        if (rem >= 4u) {
            const uint32_t code = (uint32_t)(word >> (shift - 6)) & 255u;
            quad_step<WIDE>(ix, c4, code, l, h);
            rem -= 4;
            shift -= 8;
        } else {
            const uint32_t sym = (0x5321u >> (4u * ((uint32_t)(word >> shift) & 3u))) & 7u;  // A,C,G,T = 1,2,3,5
            remainder_step<WIDE>(ix, cb, sym, l, h);
            rem--;
            shift -= 2;
        }
    }
}

template <bool WIDE>
static cudaError_t launch_count_quad_t(int device, const IndexView &ix, const uint64_t *d_packed,
                                       const PackedLayout &lay, uint32_t k, uint64_t *d_out, cudaStream_t st) {
    const unsigned grid = persistent_grid(device, (const void *)count_kmers_quad_kernel<WIDE>, kCountThreads, lay.n,
                                          kCountThreads);
    count_kmers_quad_kernel<WIDE><<<grid, kCountThreads, 0, st>>>(ix, d_packed, lay, k, d_out);
    return cudaGetLastError();
}

cudaError_t launch_count_quad(int device, const IndexView &ix, const uint64_t *d_packed, const PackedLayout &lay,
                              uint32_t k, uint64_t *d_out, cudaStream_t st) {
    if (index_is_wide(ix))
        return ix.oct ? launch_count_oct_wide(device, ix, d_packed, lay, k, d_out, st)
                      : launch_count_quad_t<true>(device, ix, d_packed, lay, k, d_out, st);
    if (ix.oct) {
        static bool prepared[64] = {};  // per device: 4 CTAs x 47 KB of staging per SM need the large shared-memory configuration
        if (device < 0 || device >= 64 || !prepared[device]) {
            cudaFuncSetAttribute((const void *)count_kmers_oct_kernel<>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOctSmemPacked);
            cudaFuncSetAttribute((const void *)count_kmers_oct_kernel<>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (device >= 0 && device < 64) prepared[device] = true;
        }
        // the chunk dispenser lives in the scratch buffer next to the live counters (engine bookkeeping: the
        // buffer is the engine's own scratch, `const` only towards the caller's data in it)
        uint32_t *work = reinterpret_cast<uint32_t *>(const_cast<uint64_t *>(d_packed) + lay.work());
        if (cudaError_t e = cudaMemsetAsync(work, 0, sizeof(uint32_t), st); e != cudaSuccess) return e;
        const unsigned grid = oct_grid(device, (const void *)count_kmers_oct_kernel<>, kOctSmemPacked, lay.n);
        count_kmers_oct_kernel<><<<grid, kCountThreads, kOctSmemPacked, st>>>(ix, d_packed, lay, k, d_out, work);
        return cudaGetLastError();
    }
    return launch_count_quad_t<false>(device, ix, d_packed, lay, k, d_out, st);
}

}  // namespace msbwt
