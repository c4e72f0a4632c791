// oct_kernel.cuh -- the search kernel over the oct image (layout.h), shared by the three translation units that
// instantiate it: quad_kernels.cu (the search), stats_kernels.cu (the counting instantiation) and wide_kernels.cu
// (64-bit positions).  One instantiation per module because ptxas 12.9 crashes on a module that holds two.
#pragma once
#include "device_rank.cuh"
#include "engine.h"
#include "kernel_common.cuh"

namespace msbwt {

// ---------------------------------------------------------------- oct image (with or without the quad image beside it)
//
// While kOctSyms (ten) or more symbols are left a step reads one 128-byte line of the oct image (layout.h); when
// exactly kFinSyms (twenty) are left, one final-step line answers the count; the quad image (if it was kept) and
// one-symbol ranks serve remainders, ranges that straddle two buckets and the lines that overflowed.  32-bit
// positions, or 64-bit ones in the WIDE instantiation (wide_kernels.cu), which has no quad image.
//
// What HBM random access is bound by is the number of L2 requests that miss -- about 40 G/s whatever their
// size (profiles/r1_gather_*.json) -- and what reaches that bound is the number of them in flight.  So:
//
//  * one thread per query (1024 queries in flight per SM), but the index lines are fetched by the WARP:
//    every lane publishes the address of the line (or the two quad sectors) its query needs next (in the 16
//    spare bytes of its shared-memory row), and in eight rounds the warp copies the 32 lines into shared memory
//    with cp.async, eight lanes x 16 bytes per line, i.e. ONE 128-byte request per line and no load registers.  (A thread that read its own line with
//    four 256-bit loads paid four requests per line and ran at a quarter of the line rate; a quad of lanes
//    per query kept only 384 queries per SM in flight: profiles/r1_o2_*, r1_o6_* summaries.)
//  * every iteration is ISSUE (branch-free, whatever kind of step each lane needs), one wait, CONSUME (each
//    lane ranks in its own staged line; divergent, but without memory accesses): one memory round trip per
//    iteration even when the lanes of a warp need different kinds of step -- one lane in fourteen lands on
//    an overflowed line on 30x reads with 1 % errors.
//  * every warp takes chunks of 512 consecutive queries of the live list from an atomic counter and stages
//    them through shared memory 32 queries at a time, double-buffered (coalesced cp.async one pool ahead);
//    lanes that finished take the next queries of the pool in lane order, so the warp stays full whatever the
//    mix of early exits and no warp is left with a slow slice of a skewed batch.
#ifndef MSBWT_OCT_CTAS
#define MSBWT_OCT_CTAS 4
#endif
constexpr int kOctRowBytes = 144;    // a 128-byte line + 16: rows of consecutive lanes start 4 banks apart (conflict-free LDS.128)
constexpr int kOctPoolBytes = 640;   // 32 x (u64 symbol word, u64 seed range, u32 original index)
constexpr int kOctWidePoolBytes = 896;  // WIDE: 32 x (u64 symbol word, u64 l, u64 h, u32 original index)
constexpr int kOctChunk = 512;       // queries a warp takes from the live list at a time (fewer when the list is short)

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem, bool on) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem), "r"(on ? 16u : 0u) : "memory");
}
// the same with an L2 eviction policy (createpolicy): index lines and query bytes are read once -- evict first
__device__ __forceinline__ void cp_async16_hint(void *smem, const void *gmem, bool on, uint64_t policy) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;" ::"r"(dst), "l"(gmem), "r"(on ? 16u : 0u), "l"(policy)
                 : "memory");
}
// 16 bytes when `bytes` is 16, sixteen zero bytes (and no read) when it is 0
__device__ __forceinline__ void cp_async16_bytes(void *smem, const void *gmem, uint32_t bytes) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem), "r"(bytes) : "memory");
}
// `bytes` (0..16) from gmem, the rest of the 16 zero-filled
__device__ __forceinline__ void cp_async16_partial(void *smem, const void *gmem, uint32_t bytes) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem, bool on) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(gmem), "r"(on ? 8u : 0u) : "memory");
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem, bool on) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(gmem), "r"(on ? 4u : 0u) : "memory");
}

// the rare one-symbol remainder step, out of line and by value so that neither its 32 load registers nor a
// stack slot for l / h burden the main loop
static __device__ __noinline__ uint2 oct_remainder_step(const IndexView &ix, const uint32_t *cbase, uint32_t sym, uint32_t l, uint32_t h) {
    const CBase<false> cb{cbase};
    rank_step<false, 1>(ix, cb, sym, l, h);
    return make_uint2(l, h);
}
static __device__ __noinline__ ulonglong2 oct_remainder_step_wide(const IndexView &ix, const uint64_t *cbase, uint32_t sb_shift, uint32_t sym,
                                                                  uint64_t l, uint64_t h) {
    const CBase<true> cb{cbase, sb_shift};
    rank_step<true, 1>(ix, cb, sym, l, h);
    return make_ulonglong2(l, h);
}

// occurrences below bucket offsets pl / ph contributed by one stored run `(len << b) | off` (0 = empty slot)
__device__ __forceinline__ void oct_add_run(uint32_t e, uint32_t b, uint32_t mask, int pl, int ph, int &sl, int &sh) {
    const int off = (int)(e & mask), len = (int)(e >> b);
    sl += min(max(pl - off, 0), len);
    sh += min(max(ph - off, 0), len);
}
__device__ __forceinline__ void oct_add_runs(const uint4 &v, uint32_t b, uint32_t mask, int pl, int ph, int &sl, int &sh) {
    oct_add_run(v.x, b, mask, pl, ph, sl, sh);
    oct_add_run(v.y, b, mask, pl, ph, sl, sh);
    oct_add_run(v.z, b, mask, pl, ph, sl, sh);
    oct_add_run(v.w, b, mask, pl, ph, sl, sh);
}
// a staged quad sector {checkpoint, 224 occurrence bits}: checkpoint + set bits at offsets < p
__device__ __forceinline__ uint32_t staged_sector_rank(const uint4 &a, const uint4 &b, int p) {
    return a.x + __popc(a.y & below_mask(p)) + __popc(a.z & below_mask(p - 32)) + __popc(a.w & below_mask(p - 64)) +
           __popc(b.x & below_mask(p - 96)) + __popc(b.y & below_mask(p - 128)) + __popc(b.z & below_mask(p - 160)) +
           __popc(b.w & below_mask(p - 192));
}

// The queries come packed and seeded from the pack / seed kernels (live list A of `packed`).
// STATS = true (stats_kernels.cu, never on a timed path): the same walk also counts what it fetches -- stats[0] oct
// lines, [1] final-step lines, [2] final-step lines that had overflowed (their query then takes the oct steps),
// [3] quad steps, [4] distinct 128-byte lines those read, [5] one-symbol steps, [6] distinct 64-byte blocks those
// read, [7] queries walked: the exact index traffic of the implemented algorithm on a batch, for the roofline
// accounting of bench.py.
// WIDE = true (wide_kernels.cu): positions of 64 bits -- an index of 2^32 symbols and more, or one cut into several
// superblocks.  The seeds come as two words per query, a line's checkpoint is word 0 | (word 1 >> 8) << 32 and its run
// count the low byte of word 1 (layout.h); such an index has no quad image beside the oct image (36.6 B per position
// have no room), so remainders, overflowed lines and ranges over two buckets take one-symbol steps.
constexpr int kOctStatWords = 8;
template <bool STATS = false, bool WIDE = false>
__global__ void __launch_bounds__(kCountThreads, WIDE ? 3 : MSBWT_OCT_CTAS)
count_kmers_oct_kernel(IndexView ix, const uint64_t *__restrict__ packed, PackedLayout lay, uint32_t k,
                       uint64_t *__restrict__ out, uint32_t *__restrict__ work, unsigned long long *__restrict__ stats = nullptr) {
    using P = typename Pos<WIDE>::type;
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t stream = policy_evict_first();
    constexpr uint32_t kFull = 0xffffffffu;
    constexpr uint32_t kPool = WIDE ? kOctWidePoolBytes : kOctPoolBytes;
    constexpr uint32_t kWarpSmem = 32 * kOctRowBytes + 2 * kPool;

    const uint32_t n = (uint32_t)packed[lay.live()];  // queries to walk (live list A)
    // CONVERGENCE.  The warp protocol below (a ballot, requests and lines other lanes read from shared memory, four
    // __syncwarp(), a warp-wide scan -- and, when the trouble was found, 24 shuffles per iteration) needs the 32
    // lanes together at every one of those points.  Left alone, ptxas 12.9 "proves" that they are (the divergent
    // regions all close with BSYNC.RECONVERGENT), drops every __syncwarp() and issues the shuffles / votes without a
    // WARPSYNC -- and on B200 that assumption does not hold under load: on batches of 50-100 M k-mers that take oct
    // steps AND a final-step line (k = 43, 53, 63) about every other launch left a few hundred queries unanswered and
    // some warps never finished, while every build whose SASS carries WARPSYNC.COLLECTIVE ran clean (profiles/
    // r2t_convergence.md).  warp_sync_guard (kernel_common.cuh) makes ptxas compile the kernel conservatively:
    // a path with WARPSYNC.COLLECTIVE before every collective for a warp that is not all there, which is what the
    // source asks for.  tests/test_sass_contract.py
    // checks the SASS of every instantiation for it, so that a toolchain that changes its mind cannot silently take
    // it away again.
    warp_sync_guard(lay);
    const uint32_t lane = threadIdx.x & 31u;
    if ((blockIdx.x * (kCountThreads / 32) + (threadIdx.x >> 5)) * 32u >= n) return;  // more warps than pools of work
    const uint64_t *w0 = packed + lay.w0(), *seeds = packed + lay.seed(), *wx = packed + lay.wx();
    const uint32_t *qidx = reinterpret_cast<const uint32_t *>(packed + lay.qidx());
    const uint32_t depth0 = list_a_table_depth(ix, k);
    const uint32_t rem0 = k - depth0;
    const uint32_t bshift = ix.oct_shift, bmask = (1u << bshift) - 1u;
    const char *const oct_base = reinterpret_cast<const char *>(ix.oct);
    const char *const quad_base = reinterpret_cast<const char *>(ix.quad);
    uint8_t *const rows = smem + (threadIdx.x >> 5) * kWarpSmem;  // 32 rows of kOctRowBytes
    uint8_t *const pools = rows + 32 * kOctRowBytes;               // 2 pools of 32 queries
    const uint4 *const my_row = reinterpret_cast<const uint4 *>(rows + lane * kOctRowBytes);
    // this lane copies bytes [16 j, 16 j + 16) of the lines of rows 4 c + (lane >> 3): of every oct / final-step line
    // (kind 1) and of a quad request (kind 2) when j < 4 -- bit `kind` of piece_on
    const uint32_t piece_off = 16u * (lane & 7u);
    const uint32_t piece_on = 2u | ((lane & 7u) < 4u ? 4u : 0u);
    const uint32_t piece_hmask = (lane & 7u) >= 2u ? ~0u : 0u;  // pieces 2, 3 of a quad request: the sector of h

    // A list that is not long against the grid (the leftovers of the one-request kernel: a percent of the batch; a
    // 10 M-query batch of long k-mers) is cut into smaller chunks, about sixteen per resident warp: a warp walks its
    // chunk 32 queries at a time, each a chain of dependent line fetches, and with 512-query chunks the last round
    // of chunks would keep a fraction of the grid busy for a fifth of the run (10 M queries = 4.1 chunks per warp).
    const uint32_t warps_in_grid = gridDim.x * (kCountThreads / 32);
    const uint32_t chunk_size = min((uint32_t)kOctChunk, max(32u, ((n / (warps_in_grid * 16u)) + 31u) & ~31u));
    // The queries are handed out in chunks of `chunk_size` (an atomic counter: a warp whose queries die early
    // simply comes back sooner, whatever the order of the batch) and staged pool by pool: pool A (sequence
    // number `seq`, buffer seq & 1) is being handed to the lanes, pool B (the other buffer) is already staged
    // or on its way.
    uint32_t chunk_next = 0, chunk_end = 0;  // the rest of this warp's current chunk (warp-uniform)
    auto next_pool = [&](uint32_t &base, uint32_t &cnt) {
        if (chunk_next >= chunk_end) {
            uint32_t c = 0;
            if (lane == 0) c = atomicAdd(work, chunk_size);
            c = __shfl_sync(kFull, c, 0);
            chunk_next = min(c, n);
            chunk_end = min(c + chunk_size, n);
        }
        base = chunk_next;
        cnt = min(32u, chunk_end - chunk_next);
        chunk_next += cnt;
    };
    auto load_pool = [&](uint32_t buf, uint32_t base, uint32_t cnt) {
        uint8_t *p = pools + buf * kPool;
        const uint32_t idx = base + lane;
        const bool on = lane < cnt;
        cp_async8(p + 8u * lane, w0 + idx, on);
        cp_async8(p + 256u + 8u * lane, seeds + idx, on);
        if constexpr (WIDE) {
            cp_async8(p + 512u + 8u * lane, seeds + lay.n + idx, on);
            cp_async4(p + 768u + 4u * lane, qidx + idx, on);
        } else {
            cp_async4(p + 512u + 4u * lane, qidx + idx, on);
        }
    };
    uint32_t seq = 0, a_pos = 0, a_cnt, b_cnt, a_base, b_base;
    next_pool(a_base, a_cnt);
    load_pool(0u, a_base, a_cnt);
    next_pool(b_base, b_cnt);
    load_pool(1u, b_base, b_cnt);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();

    uint32_t st_cnt[kOctStatWords] = {0, 0, 0, 0, 0, 0, 0, 0};  // STATS only (dead code otherwise)
    auto flush_stats = [&]() {
        if constexpr (STATS) {
#pragma unroll
            for (int i = 0; i < kOctStatWords; i++) {
                uint32_t v = st_cnt[i];
#pragma unroll
                for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
                if (lane == 0 && v) atomicAdd(stats + i, (unsigned long long)v);
            }
        }
    };
    bool active = false;
    P l = 0, h = 0;
    uint64_t word = 0, pend = 0;
    uint32_t q = 0;
    uint32_t rem = 0;     // symbols still to consume
    int shift = 62;       // bit offset of the next symbol (2 bits) in `word`; negative: already inside `pend`
    uint32_t widx = 0;
    uint32_t forced = 0;  // symbols to take without the oct image (overflowed line / two buckets)
    bool no_fin = false;  // this query's final-step line overflowed: its last kFinSyms symbols go through the oct steps
#ifdef MSBWT_OCT_WATCHDOG
    uint32_t wd_age = 0;  // debug build: iterations this lane has spent on its current query
#endif
    const char *const fin_base = reinterpret_cast<const char *>(ix.fin);
    const uint32_t fshift = ix.fin_shift, fmask = (1u << fshift) - 1u, flb = ix.fin_lb;

    // the next `nsym` symbols as one code (first consumed most significant); a step may straddle two words
    auto peek = [&](uint32_t nsym) -> uint32_t {
        const int bits = 2 * (int)nsym, avail = shift + 2;  // avail >= 2 here
        if (avail >= bits) return (uint32_t)(word >> (avail - bits)) & ((1u << bits) - 1u);
        const int need = bits - avail;
        return (uint32_t)(((word & ((1ull << avail) - 1ull)) << need) | (pend >> (64 - need)));
    };

    // the next kFinSyms symbols as one 40-bit code (first consumed most significant)
    auto peek_fin = [&]() -> uint64_t {
        const int bits = kFinCodeBits, avail = shift + 2;
        if (avail >= bits) return (word >> (avail - bits)) & ((1ull << bits) - 1ull);
        const int need = bits - avail;
        return ((word & ((1ull << avail) - 1ull)) << need) | (pend >> (64 - need));
    };

    for (;;) {
        // ---- RETIRE + REFILL (warp-uniform control)
        if (active && (rem == 0 || l == h)) {
            stg_stream(out + q, (uint64_t)(h - l), stream);
            active = false;
        }
        const uint32_t want = __ballot_sync(kFull, !active);
        if (want) {
            const uint32_t avail_a = a_cnt - a_pos, avail = avail_a + b_cnt;
            if (avail) {
                const uint32_t r = __popc(want & ((1u << lane) - 1u));  // idle lanes take queries in lane order
                if (!active && r < avail) {
                    const bool from_a = r < avail_a;
                    const uint8_t *p = pools + ((from_a ? seq : seq + 1u) & 1u) * kPool;
                    const uint32_t slot = from_a ? a_pos + r : r - avail_a;
                    shift = 62;
                    widx = 0;
                    forced = 0;
                    no_fin = false;
                    active = true;
#ifdef MSBWT_OCT_WATCHDOG
                    wd_age = 0;
#endif
                    if constexpr (STATS) st_cnt[7]++;
                    word = *reinterpret_cast<const volatile uint64_t *>(p + 8u * slot);
                    const uint64_t lo = *reinterpret_cast<const volatile uint64_t *>(p + 256u + 8u * slot);
                    const uint32_t qraw = *reinterpret_cast<const volatile uint32_t *>(p + (WIDE ? 768u : 512u) + 4u * slot);
                    q = qraw & kQidxMask;
                    no_fin = ((qraw >> 30) & 1u) != 0u;  // pack_seed_final_kernel already found this query's line overflowed
                    if constexpr (WIDE) {
                        l = lo;
                        h = *reinterpret_cast<const volatile uint64_t *>(p + 512u + 8u * slot);
                    } else {
                        l = (uint32_t)lo;
                        h = (uint32_t)(lo >> 32);
                    }
                    rem = rem0;
                    if (rem > (uint32_t)kPairSymsPerWord) pend = ldg_stream(wx + q, stream);
                }
                const uint32_t taken = min((uint32_t)__popc(want), avail);
                if (taken >= avail_a) {  // pool A is used up: B becomes A, the next pool is staged into A's buffer
                    a_cnt = b_cnt;
                    a_base = b_base;
                    a_pos = taken - avail_a;
                    seq++;
                    next_pool(b_base, b_cnt);
                    __syncwarp();
                    load_pool((seq + 1u) & 1u, b_base, b_cnt);  // (committed with this iteration's lines)
                } else {
                    a_pos += taken;
                }
            } else if (want == kFull) {
                flush_stats();
                return;  // nothing left to hand out and every lane is done
            }
        }
        if (active && shift < 0) {  // 32 symbols per word: on to the next one (a step may have ended inside it)
            word = pend;
            widx++;
            shift += 64;
            if (2u * rem > (uint32_t)(shift + 2)) pend = ldg_stream(wx + (uint64_t)widx * lay.n + q, stream);
        }

#ifdef MSBWT_OCT_WATCHDOG
        if (active && ++wd_age > 4096u) {  // no k-mer needs more than k iterations: say what this one is doing and drop it
            printf("[oct watchdog] q %u rem %u l %llu h %llu shift %d widx %u forced %u no_fin %d word %016llx pend %016llx k %u n %u\n", q, rem,
                   (unsigned long long)l, (unsigned long long)h, shift, widx, forced, (int)no_fin, (unsigned long long)word,
                   (unsigned long long)pend, k, n);
            rem = 0;
        }
#endif
        // ---- ISSUE (branch-free): every lane publishes what its query needs, the warp fetches it
        // (a range over two buckets, like an overflowed line, takes its kOctSyms symbols as quad steps and, for
        // the last two of ten, one-symbol steps)
        const bool live = active && rem != 0 && l != h;
        const P bl = l >> bshift, bh = h >> bshift;
        // exactly kFinSyms symbols left: ONE final-step line answers the count (no rank needed for the last step)
        const bool is_fin = live && fin_base != nullptr && rem == (uint32_t)kFinSyms && forced == 0u && !no_fin &&
                            (l >> fshift) == (h >> fshift);
        const uint64_t fin_mixed = is_fin ? fin_mix40(peek_fin()) : 0ull;  // (a dozen instructions: only where they are used)
        const bool want_oct = live && !is_fin && rem >= (uint32_t)kOctSyms && forced == 0u;
        const bool is_oct = want_oct && bl == bh;
        if (want_oct && !is_oct) forced = (uint32_t)kOctSyms;  // symbols to take without the oct image
        const bool is_quad = !WIDE && live && quad_base != nullptr && !is_oct && !is_fin && rem >= 4u && (forced == 0u || forced >= 4u);
        const uint32_t codem = peek((uint32_t)kOctSyms);
        const uint32_t code8 = peek(4u);
        const uint32_t sl = WIDE ? 0u : (uint32_t)l / (uint32_t)kQuadSyms, sh = WIDE ? 0u : (uint32_t)h / (uint32_t)kQuadSyms;
        const char *p0 = is_oct ? oct_base + ((size_t)codem * ix.nbuck8 + bl) * kOctLineBytes
                                : quad_base + ((size_t)code8 * ix.nsec4 + sl) * kQuadSectorBytes;
        if (is_fin) p0 = fin_base + ((((size_t)(l >> fshift)) << flb) | (size_t)(fin_mixed & ((1ull << flb) - 1ull))) * kFinLineBytes;
        // kind: 1 oct line or final-step line (all eight 16-byte pieces), 2 quad (the sector of l into bytes 0..31 of the
        // row, the sector of h into 32..63), 0 nothing.  h_adj (quad): what pieces 2 and 3 add to `p0 + 16 j` to land in
        // the sector of h -- its byte distance from the sector of l, less the 32 bytes the two pieces already skipped
        // (mod 2^32: 16 j >= 32 there, the sum is never negative)
        const uint32_t kind = (is_oct || is_fin) ? 1u : (is_quad ? 2u : 0u);
        const uint32_t h_adj = is_quad ? (sh - sl) * (uint32_t)kQuadSectorBytes - 32u : 0u;
        if constexpr (STATS) {
            st_cnt[0] += is_oct;
            st_cnt[1] += is_fin;
            st_cnt[3] += is_quad;
            if (is_quad) st_cnt[4] += (((size_t)code8 * ix.nsec4 + sl) >> 2) == (((size_t)code8 * ix.nsec4 + sh) >> 2) ? 1u : 2u;
        }
#ifdef MSBWT_OCT_WATCHDOG
        {   // debug build: every address a live lane is about to ask for must lie inside its image
            const uint64_t fin_lines = ((ix.total >> fshift) + 1ull) << flb;
            const uint64_t fin_line = (((uint64_t)(l >> fshift)) << flb) | (fin_mixed & ((1ull << flb) - 1ull));
            const bool bad = (live && ((uint64_t)l > (uint64_t)h || (uint64_t)h > ix.total)) || (active && q >= (uint32_t)lay.n) ||
                             (is_fin && fin_line >= fin_lines) || (is_oct && ((uint64_t)bl >= ix.nbuck8 || codem >= (uint32_t)kOctCodes)) ||
                             (is_quad && ((uint64_t)sl >= ix.nsec4 || (uint64_t)sh >= ix.nsec4 || code8 >= 256u));
            if (bad) {
                printf("[oct watchdog] BAD STATE q %u rem %u l %llu h %llu shift %d widx %u forced %u no_fin %d word %016llx pend %016llx fin %d oct %d quad %d "
                       "codem %u code8 %u age %u total %llu\n", q, rem, (unsigned long long)l, (unsigned long long)h, shift, widx, forced, (int)no_fin,
                       (unsigned long long)word, (unsigned long long)pend, (int)is_fin, (int)is_oct, (int)is_quad, codem, code8, wd_age,
                       (unsigned long long)ix.total);
            }
        }
#endif
        // every lane leaves {address, kind, h_adj} in the 16 spare bytes at the end of its own row (a row is 128 + 16 bytes
        // and the copies only write the first 128): one 16-byte store and eight 16-byte reads per lane instead of the 24
        // shuffles that used to carry the same words; what depends only on the lane (which pieces of which kind it copies)
        // is in piece_on / piece_hmask, computed once
        *reinterpret_cast<uint4 *>(rows + lane * kOctRowBytes + kOctLineBytes) =
            make_uint4((uint32_t)(uintptr_t)p0, (uint32_t)((uintptr_t)p0 >> 32), kind, h_adj);
        __syncwarp();
#pragma unroll
        for (uint32_t c = 0; c < 8u; c++) {
            const uint32_t o = 4u * c + (lane >> 3);  // the lane whose line this is
            const uint4 want_o = *reinterpret_cast<const uint4 *>(rows + o * kOctRowBytes + kOctLineBytes);
            const uint64_t a = ((uint64_t)want_o.y << 32) | want_o.x;
            const uint64_t src = a + (uint64_t)(piece_off + (want_o.w & piece_hmask));
            cp_async16_bytes(rows + o * kOctRowBytes + piece_off, reinterpret_cast<const void *>(src), ((piece_on >> want_o.z) & 1u) << 4);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();

        // ---- CONSUME (each lane ranks in its own staged line)
        bool fin_scan = false;                 // this lane's final-step line is good: its runs are summed in phase 2
        uint32_t fin_at = 0, fin_left = 0;     // header word of the first group of its code, groups of that code
        if (is_fin) {
            const uint4 first = my_row[0];
            const uint32_t used = first.x;  // <= 31 in any line the builder wrote
            if (used == kFinOverflow) {
                no_fin = true;  // the same symbols through two oct steps
                if constexpr (STATS) st_cnt[2]++;
            } else {
                // Phase 1, per lane: hop from group header to group header (layout.h) to the FIRST group of this query's
                // code and count its groups (they are adjacent: the builder writes a line's groups in key order) -- a
                // handful of 4-byte reads with nothing nested inside, so the lanes differ only in their trip counts.
                // The runs are summed by the warp in step, below the branches (phase 2).
                const uint32_t tag = (uint32_t)(fin_mixed >> flb);
                const uint32_t *roww = reinterpret_cast<const uint32_t *>(my_row);
                const uint32_t lim = min(used, (uint32_t)kFinLineWords - 1u);  // (bounded whatever the row holds)
                uint32_t hw = first.y;
#ifdef MSBWT_OCT_WATCHDOG
                if (used > 31u) printf("[oct watchdog] final-step line of q %u says %u words in use (l %llu h %llu)\n", q, used, (unsigned long long)l, (unsigned long long)h);
#endif
                fin_scan = true;
                for (uint32_t idx = 1u; idx <= lim;) {
                    const bool eq = (hw >> 4) == tag;
                    if (eq && fin_left == 0u) fin_at = idx;
                    fin_left += eq ? 1u : 0u;
                    idx += 1u + (hw & 15u);
                    if (idx <= lim) hw = roww[idx];
                }
            }
        } else if (is_oct) {
            const uint4 a = my_row[0], b = my_row[1];
            const uint32_t nruns = WIDE ? (a.y & 255u) : a.y;
            if (nruns > (uint32_t)kOctCapacity) {
                forced = (uint32_t)kOctSyms;  // this line cannot hold its runs: the same symbols without the oct image
            } else {
                const int pl = (int)((uint32_t)l & bmask), ph = (int)((uint32_t)h & bmask);
                int cl = 0, ch = 0;
                oct_add_run(a.z, bshift, bmask, pl, ph, cl, ch);
                oct_add_run(a.w, bshift, bmask, pl, ph, cl, ch);
                oct_add_runs(b, bshift, bmask, pl, ph, cl, ch);
                if (nruns > 6u) {
                    oct_add_runs(my_row[2], bshift, bmask, pl, ph, cl, ch);
                    oct_add_runs(my_row[3], bshift, bmask, pl, ph, cl, ch);
                    if (nruns > 14u) {
                        oct_add_runs(my_row[4], bshift, bmask, pl, ph, cl, ch);
                        oct_add_runs(my_row[5], bshift, bmask, pl, ph, cl, ch);
                        if (nruns > 22u) {
                            oct_add_runs(my_row[6], bshift, bmask, pl, ph, cl, ch);
                            oct_add_runs(my_row[7], bshift, bmask, pl, ph, cl, ch);
                        }
                    }
                }
                const P ck = WIDE ? (P)(((uint64_t)(a.y >> 8) << 32) | a.x) : (P)a.x;
                l = ck + (uint32_t)cl;
                h = ck + (uint32_t)ch;
                rem -= (uint32_t)kOctSyms;
                shift -= 2 * kOctSyms;
            }
        } else if (is_quad) {
            const uint32_t nl = staged_sector_rank(my_row[0], my_row[1], (int)((uint32_t)l - sl * (uint32_t)kQuadSyms));
            const uint32_t nh = staged_sector_rank(my_row[2], my_row[3], (int)((uint32_t)h - sh * (uint32_t)kQuadSyms));
            l = nl;
            h = nh;
            rem -= 4;
            shift -= 8;
            forced = forced >= 4u ? forced - 4u : 0u;
        } else if (live) {  // one symbol: the tail of a k-mer, or the last two of ten symbols taken without the oct image
            const uint32_t sym = (0x5321u >> (4u * peek(1u))) & 7u;  // A,C,G,T = 1,2,3,5
            if constexpr (STATS) {
                st_cnt[5]++;
                st_cnt[6] += (l >> kBlockShift) == (h >> kBlockShift) ? 1u : 2u;
            }
            if constexpr (WIDE) {
                const ulonglong2 r = oct_remainder_step_wide(ix, cb.c, cb.sb_shift, sym, l, h);
                l = r.x;
                h = r.y;
            } else {
                const uint2 r = oct_remainder_step(ix, cb.c, sym, l, h);
                l = r.x;
                h = r.y;
            }
            rem--;
            shift -= 2;
            forced = forced ? forced - 1u : 0u;
        }
        // Phase 2 of the final-step lines, the warp in step: every lane adds up the runs of its group, four words per
        // trip, as many trips as the longest group among the lanes needs; a code with more than 15 runs in the bucket
        // continues in the group right behind.  (One lane after the other, inside the branch above, this scan was a
        // quarter of all the warp instructions of a 63-mer batch: profiles/r2w_oct_k63_ncu_summary.txt.)
        if (__any_sync(kFull, fin_scan)) {
            const uint32_t *roww = reinterpret_cast<const uint32_t *>(my_row);
            const int pl = (int)((uint32_t)l & fmask), ph = (int)((uint32_t)h & fmask);
            int acc = 0;
            do {
                const uint32_t n1 = fin_left ? (roww[fin_at] & 15u) : 0u;
                const uint32_t trips = __reduce_max_sync(kFull, n1);
                for (uint32_t r = 0; r < trips; r += 4u) {
#pragma unroll
                    for (uint32_t u = 0; u < 4u; u++) {
                        if (r + u < n1) {
                            const uint32_t w = roww[fin_at + 1u + r + u];
                            const int off = (int)(w & 0xFFFFu), len = (int)(w >> 16);
                            acc += min(max(ph - off, 0), len) - min(max(pl - off, 0), len);
                        }
                    }
                }
                if (fin_left) {
                    fin_at += 1u + n1;
                    fin_left--;
                }
            } while (__any_sync(kFull, fin_left != 0u));
            if (fin_scan) {
                l = 0;
                h = (uint32_t)acc;  // only h - l is read from here on
                rem = 0;
            }
        }
        __syncwarp();  // the rows are rewritten by the next ISSUE
    }
}

// dynamic shared memory per CTA
constexpr int kOctSmemPacked = (kCountThreads / 32) * (32 * kOctRowBytes + 2 * kOctPoolBytes);
constexpr int kOctSmemWide = (kCountThreads / 32) * (32 * kOctRowBytes + 2 * kOctWidePoolBytes);

// one full wave of CTAs for a kernel with `smem` bytes of dynamic shared memory, fewer if there is less work
inline unsigned oct_grid(int device, const void *kernel, int smem, uint64_t n) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kCountThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const uint64_t full = (uint64_t)sm_count(device) * (uint64_t)per_sm, need = (n + kCountThreads - 1) / kCountThreads;
    return (unsigned)(need < 1 ? 1 : (need < full ? need : full));
}

}  // namespace msbwt
