// kernel_common.cuh -- helpers shared by the translation units that hold the search kernels
// (kernels.cu, quad_kernels.cu; split because ptxas 12.9 crashes on the module that holds them all).
#pragma once
#include <cuda_runtime.h>

#include <cstdio>

#include "engine.h"

namespace msbwt {

// Symbols per step of the kernel that walks live list A: 4 with a quad image, 2 with a pair image, else 1.
__host__ __device__ __forceinline__ uint32_t list_a_stride(const IndexView &ix) {
    return ix.quad ? 4u : (ix.pair ? 2u : 1u);
}

// Suffix-table depth for an all-ACGT k-mer.  With a multi-step image (stride 2 or 4) the depth is
// picked from the `stride` deepest levels {ts, ts-1, ..} so that the number of symbols left is a
// multiple of the stride (k below those levels: no table).
__host__ __device__ __forceinline__ uint32_t acgt_table_depth(uint32_t k, uint32_t ts, uint32_t stride) {
    if (!ts) return 0;
    if (k >= ts) {
        const uint32_t back = (stride - (k - ts) % stride) % stride;
        return back < ts ? ts - back : 0;
    }
    return k + stride > ts ? k : 0;  // level k itself is one of the kept ones: the table answers everything
}

// With an oct image (kOctSyms symbols per line, quad steps of four for what is left, one-symbol steps for the
// rest) the depth is the one of the four kept levels {ts, .., ts-3} that leaves the cheapest walk: one index
// access per oct and per quad step, two per one-symbol step (a one-step block per boundary); ties go to the
// deeper level.
__host__ __device__ __forceinline__ uint32_t oct_walk_cost(uint32_t rest) {
    const uint32_t r = rest % (uint32_t)kOctSyms;
    return rest / (uint32_t)kOctSyms + r / 4u + 2u * (r % 4u);
}
__host__ __device__ __forceinline__ uint32_t oct_table_depth(uint32_t k, uint32_t ts) {
    if (!ts) return 0;
    if (k < ts) return k + 4u > ts ? k : 0;  // level k itself is one of the kept ones: the table answers everything
    uint32_t best = 0, best_cost = oct_walk_cost(k);
    for (uint32_t back = 0; back < 4u && back < ts; back++) {
        const uint32_t c = oct_walk_cost(k - (ts - back));
        if (c < best_cost) { best_cost = c; best = ts - back; }
    }
    return best;
}

// The depth the pack / seed kernels look an all-ACGT k-mer up at, and the search kernels resume from.
__host__ __device__ __forceinline__ uint32_t list_a_table_depth(const IndexView &ix, uint32_t k) {
    return ix.oct ? oct_table_depth(k, ix.table_s) : acgt_table_depth(k, ix.table_s, list_a_stride(ix));
}

// ---- four symbols per 32-bit word (SWAR)
// Checking four symbol bytes for a symbol outside ACGT and packing them, in one pass through an 8-entry byte table
// (PRMT): the four symbol bytes become four selector nibbles, the table answers A,C,G,T = 1,2,3,5 with their 2-bit
// codes and every other symbol < 8 with 0x80.  `acc` collects x | table bytes: the k-mer holds a symbol outside ACGT
// iff (acc & kSwarBadMask) != 0 at the end (a byte >= 8 shows in x itself, whatever the table then answers).
// Returns the four codes packed into the TOP byte (byte i of x at bits 24 + 2i; one multiply: the partial products
// do not overlap), meaningful only when the word is clean; swar_gather4 collects the top bytes of four such words.
// 7 instructions per word against 17 for a check and a pack in plain SWAR arithmetic and the shift into place.
constexpr uint32_t kSwarBadMask = 0xF8F8F8F8u;
__device__ __forceinline__ uint32_t prmt_b32(uint32_t a, uint32_t b, uint32_t sel) {  // no & 0x7777 as in __byte_perm
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ uint32_t swar_lut_pack4_top(uint32_t x, uint32_t &acc) {
    const uint32_t t = x + (x >> 4);                                // byte 0 = b0 | b1 << 4, byte 2 = b2 | b3 << 4
    const uint32_t sel = prmt_b32(t, 0u, 0x4420u);                  // selector nibbles b0, b1, b2, b3 (all < 8 if clean)
    const uint32_t y = prmt_b32(0x02010080u, 0x80800380u, sel);     // table[0..7] = 80 00 01 02 80 03 80 80
    acc |= x | y;
    return y * 0x01041040u;
}
// top bytes of four words -> one word, word i at byte i
__device__ __forceinline__ uint32_t swar_gather4(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    return prmt_b32(prmt_b32(m0, m1, 0x0073u), prmt_b32(m2, m3, 0x0073u), 0x5410u);
}

// CONVERGENCE GUARD for kernels whose lanes exchange data (shuffles, ballots, shared memory + __syncwarp) after
// divergent code.  ptxas 12.9 may "prove" such a warp converged, drop every __syncwarp() and issue the collectives
// without a WARPSYNC; on B200 that assumption failed under load in the oct search kernel (oct_kernel.cuh has the
// story, profiles/r2t_convergence.md the evidence).  A call ptxas cannot see through -- a printf that never runs: the
// bits of a launch's query count above 2^40 are never set -- makes it compile the kernel conservatively, with
// WARPSYNC.COLLECTIVE before every collective.  tests/test_sass_contract.py checks the SASS for it.
__device__ __forceinline__ void warp_sync_guard(const PackedLayout &lay) {
    if ((uint32_t)(lay.n >> 40) == 0x5EEDu) printf("%u", (uint32_t)lay.n);
}

inline int sm_count(int device) {
    static int cached[64];
    if (device < 0 || device >= 64) return 148;
    if (!cached[device]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
        cached[device] = v;
    }
    return cached[device];
}

// rc(v) of a k-mer in msbwt_count_kmers_u64's encoding: every code c becomes 3 - c (= c ^ 3) and the k 2-bit groups
// are reversed.  The bit reversal also swaps the two bits inside each group, so they are swapped back.
__device__ __forceinline__ uint64_t revcomp_kmer(uint64_t v, uint32_t k) {
    uint64_t r = __brevll(~v);
    r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
    return r >> (64 - 2 * k);  // the complemented zero bits above the k-mer end up below it
}

// one full wave of CTAs (a multiple of the SM count), fewer if there is less work
inline unsigned persistent_grid(int device, const void *kernel, int threads, uint64_t work_groups,
                                int groups_per_cta) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    uint64_t full = (uint64_t)sm_count(device) * (uint64_t)per_sm;
    uint64_t need = (work_groups + groups_per_cta - 1) / groups_per_cta;
    if (need < 1) need = 1;
    return (unsigned)(need < full ? need : full);
}

}  // namespace msbwt
