// kernels.cu -- sm_100a kernels for the batched backward search.
//
// Replaces the reference's hot loop: BWT::count_kmer (src/msbwt_core.rs:125-161)
// calling RleBWT::constrain_range (src/rle_bwt.rs:202-287) once per symbol.
// Integer-only, random-gather (HBM access rate / L2) bound; no tensor cores (nothing
// here is a dense contraction).  See layout.h for the block format.
//
// Two work mappings over the same block image (template parameter LANES):
//   LANES = 1  one thread per query: the thread reads both 32-byte halves of a block with
//              two 256-bit ld.global.nc, matches 4 x 32 symbols (3 LOP3 each), masks and
//              popcounts.  No shuffles.  ~4 warp instructions per query-step: the mapping
//              for an L2-resident index, where issue slots are the limit.
//   LANES = 2  a lane pair per query: each lane reads ONE half (one coalesced 64-byte
//              request per block -- HBM serves ~39 G random requests/s whatever their
//              size, so one request per rank matters more than instruction count), counts
//              its 64 symbols, and three shuffles combine the pair.
// A third kernel walks the PAIR image (layout.h): a quad of lanes per query, one coalesced
// 128-byte line per TWO backward-search steps -- the mapping for an index that lives in HBM,
// where every L2 miss costs a whole 128-byte line fill whatever the request size.
// In all of them a lane (group) whose k-mer ends refills itself from its own query stream, so
// every lane of a warp stays busy.  (v1-v3 used 8- then 4-lane groups per query; ncu
// showed them issue-bound at ~12 warp instructions per query-step -- profiles/.)
#include <cstdlib>
#include <string>
#include <type_traits>

#include "device_rank.cuh"
#include "engine.h"
#include "kernel_common.cuh"
#include "pack_common.cuh"

namespace msbwt {

// One thread per query.  The CTA first stages its 256 * k query bytes in shared memory with
// coalesced 16-byte loads (the caller's layout is k-byte rows: read straight from global memory a
// thread would touch one sector per byte load), then every thread
//   1. packs its k-mer four symbols at a time (SWAR on 32-bit shared-memory words) into 2-bit words,
//      the last symbol in the top bits, noting whether every symbol is ACGT;
//   2. all-ACGT k-mers (list A): suffix-table lookup -- if the index has a pair image the depth is
//      chosen from {table_s, table_s - 1} so that an EVEN number of symbols is left for the pair
//      kernel -- and the remaining symbols shifted to the top (seed_acgt);
//      any other k-mer (list B, rare): validated symbol by symbol (symbol >= 6 sets *status), table
//      depth table_s when its last table_s symbols are ACGT, 3 bits per symbol (seed_general);
//   3. finishes the query right here when nothing is left to search (empty range -> count 0,
//      msbwt_core.rs:151-153; or no symbols left -> h-l), or appends it to its live list.
// K = the k-mer length when it is one the library is compiled for (31: the headline query; every shift, mask
// and word count of steps 1-2 is then a constant), 0 = any length (`k_rt`).
template <bool WIDE, uint32_t K>
__global__ void __launch_bounds__(256, K ? MSBWT_PACK_CTAS_FIXED_K : 6)
pack_seed_kernel(IndexView ix, const uint8_t *__restrict__ syms, uint32_t k_rt, SeedPlan plan, PackedLayout lay,
                 uint64_t *__restrict__ packed, uint64_t *__restrict__ out, uint32_t *__restrict__ status) {
    const uint32_t k = K ? K : k_rt;
    extern __shared__ uint4 pack_smem_v[];
    uint8_t *smem = reinterpret_cast<uint8_t *>(pack_smem_v);
    const uint64_t q0 = (uint64_t)blockIdx.x * kPackThreads;
    const uint64_t q = q0 + threadIdx.x;
    const bool valid = q < lay.n;
    const bool staged = k <= kPackSmemMaxK;
    const uint8_t *src = syms + (valid ? q : 0) * k;
    uint32_t row = 0;  // byte offset of this thread's k-mer in shared memory
    if (staged) {
        const uint8_t *g = syms + q0 * k;
        const uint32_t rows = (uint32_t)min((uint64_t)kPackThreads, lay.n - q0);
        const uint32_t bytes = rows * k;
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(g) & 15u);  // smem mirrors the global alignment
        const uint32_t head = min(bytes, (16u - mis) & 15u);                    // < 16 <= kPackThreads: one pass
        if (threadIdx.x < head) smem[mis + threadIdx.x] = g[threadIdx.x];
        const uint32_t vecs = (bytes - head) >> 4;
        const uint4 *gv = reinterpret_cast<const uint4 *>(g + head);
        uint4 *sv = reinterpret_cast<uint4 *>(smem + mis + head);
        // no registers held: every round in flight
        if constexpr (K != 0) {
            constexpr uint32_t kRounds = (K + 15u) / 16u;  // vecs <= 256 * K / 16: two rounds for K = 31
#pragma unroll
            for (uint32_t r = 0; r < kRounds; r++) {
                const uint32_t i = threadIdx.x + r * kPackThreads;
                if (i < vecs) stage_cp_async16(sv + i, gv + i);
            }
        } else {
            for (uint32_t i = threadIdx.x; i < vecs; i += kPackThreads) stage_cp_async16(sv + i, gv + i);
        }
        const uint32_t at = head + (vecs << 4) + threadIdx.x;                    // < 16 bytes are left
        if (at < bytes) smem[mis + at] = g[at];
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
        row = mis + threadIdx.x * k;
        src = smem + row;
    }

    uint64_t lo = 0, hi = 0, word0 = 0;
    uint32_t flag = 0;
    bool list_a = false, finished = false, bad = false;
    bool general = valid && !staged;
    if (valid && staged) {
        // 1. 2-bit words: chunk w = the 32 symbols consumed at steps 32w .. 32w+31 (the last chunk is short)
        const uint32_t nw = (k + kPairSymsPerWord - 1) / kPairSymsPerWord, tail = k - kPairSymsPerWord * (nw - 1);
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(smem);
        uint64_t w2[kPackMaxWords];
        uint32_t other = 0;
#pragma unroll
        for (uint32_t w = 0; w < kPackMaxWords; w++) {
            w2[w] = 0;
            if (w < nw) {
                const bool last = w + 1 == nw;
                const uint32_t c = last ? tail : kPairSymsPerWord;
                const uint32_t o = row + (last ? 0u : k - kPairSymsPerWord * (w + 1));
                const uint32_t *p = sw + (o >> 2);
                const uint32_t sh = (o & 3u) * 8u;
                uint32_t prev = p[0];
                uint32_t m[8];
#pragma unroll
                for (uint32_t i = 0; i < 8; i++) {
                    const uint32_t nxt = p[i + 1];
                    uint32_t x = __funnelshift_r(prev, nxt, sh);
                    prev = nxt;
                    if (c < 4u * (i + 1)) {  // bytes past the chunk count as 'A' (code 0, never an exception)
                        const uint32_t keep = c > 4u * i ? (1u << (8u * (c - 4u * i))) - 1u : 0u;
                        x = (x & keep) | (0x01010101u & ~keep);
                    }
                    m[i] = swar_lut_pack4_top(x, other);
                }
                const uint64_t le = (uint64_t)swar_gather4(m[0], m[1], m[2], m[3]) |
                                    ((uint64_t)swar_gather4(m[4], m[5], m[6], m[7]) << 32);
                w2[w] = le << (64u - 2u * c);
            }
        }
        if (other & kSwarBadMask) {
            general = true;
        } else {
            auto get = [&](uint32_t w) {
                uint64_t v = w2[0];
#pragma unroll
                for (uint32_t j = 1; j < kPackMaxWords; j++) if (j == w) v = w2[j];
                return v;
            };
            seed_acgt<WIDE>(ix, k, plan, nw, get, lay, q, packed, lo, hi, flag, list_a, finished, word0);
        }
    }
    if (general) seed_general<WIDE>(ix, src, k, lay, q, packed, lo, hi, flag, finished, word0, bad);
    if (valid && finished) out[q] = hi - lo;
    const bool live = valid && !finished;
    const uint64_t pos = append_live(live, list_a, reinterpret_cast<unsigned long long *>(packed + lay.live()), lay.n);
    if (live) {
        packed[lay.w0() + pos] = word0;
        if constexpr (WIDE) {
            packed[lay.seed() + pos] = lo;
            packed[lay.seed() + lay.n + pos] = hi;
        } else {
            packed[lay.seed() + pos] = lo | (hi << 32);
        }
        reinterpret_cast<uint32_t *>(packed + lay.qidx())[pos] = (uint32_t)q | (flag << 30);
    }
    if (bad) atomicOr(status, 1u);
}

// K0b: the same job for a batch the HOST has already packed (capi.cu, hostpack.cpp): all-ACGT
// k-mers as ceil(k/32) words of 2-bit symbols, word-major (`words[w * n + q]`), the k-mer's last
// symbol in the top bits of word 0.  Takes the table index off the top, shifts the rest up and
// appends to list A (or finishes the query).  No symbol bytes ever reach the device on this path.
template <bool WIDE>
__global__ void __launch_bounds__(256)
seed_packed_kernel(IndexView ix, const uint64_t *__restrict__ words, uint32_t k, SeedPlan plan, PackedLayout lay,
                   uint64_t *__restrict__ packed, uint64_t *__restrict__ out) {
    warp_sync_guard(lay);  // append_live's ballots follow a divergent table lookup
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = q < lay.n;
    const uint32_t nw = (k + kPairSymsPerWord - 1) / kPairSymsPerWord;  // <= kPackMaxWords (the host checks)
    uint64_t lo = 0, hi = 0, word0 = 0;
    uint32_t flag = 0;
    bool list_a = false, finished = false;
    if (valid) {
        auto get = [&](uint32_t w) { return __ldg(words + (uint64_t)w * lay.n + q); };
        seed_acgt<WIDE>(ix, k, plan, nw, get, lay, q, packed, lo, hi, flag, list_a, finished, word0);
        if (finished) out[q] = hi - lo;
    }
    const bool live = valid && !finished;
    const uint64_t pos = append_live(live, list_a, reinterpret_cast<unsigned long long *>(packed + lay.live()), lay.n);
    if (live) {
        packed[lay.w0() + pos] = word0;
        if constexpr (WIDE) {
            packed[lay.seed() + pos] = lo;
            packed[lay.seed() + lay.n + pos] = hi;
        } else {
            packed[lay.seed() + pos] = lo | (hi << 32);
        }
        reinterpret_cast<uint32_t *>(packed + lay.qidx())[pos] = (uint32_t)q | (flag << 30);
    }
}

// K0c: the same job for k-mers the CALLER holds as integers -- k <= 32, kmers[q] = sum code(s_i) << 2 (k-1-i), A,C,G,T =
// 0..3, the first symbol in the most significant of the 2k bits: what k-mer counters keep.  Reversing the 2-bit groups of
// the word puts the k-mer's LAST symbol in the top bits, which is the word format of live list A; bits above 2k are ignored.
// Every such k-mer is all-ACGT by construction: nothing to validate, no list B unless the pair image leaves an odd remainder.
template <bool WIDE>
__global__ void __launch_bounds__(256)
seed_u64_kernel(IndexView ix, const uint64_t *__restrict__ kmers, uint32_t k, SeedPlan plan, PackedLayout lay,
                uint64_t *__restrict__ packed, uint64_t *__restrict__ out) {
    warp_sync_guard(lay);  // append_live's ballots follow a divergent table lookup
    const uint64_t q = (uint64_t)blockIdx.x * kPackThreads + threadIdx.x;
    const bool valid = q < lay.n;
    uint64_t lo = 0, hi = 0, word0 = 0;
    uint32_t flag = 0;
    bool list_a = false, finished = false;
    if (valid) {
        const uint64_t x = __ldg(kmers + q) & (k >= 32u ? ~0ull : ((1ull << (2u * k)) - 1ull));
        const uint64_t w = reverse_symbol_pairs(x);
        auto get = [&](uint32_t) { return w; };
        seed_acgt<WIDE>(ix, k, plan, 1u, get, lay, q, packed, lo, hi, flag, list_a, finished, word0);
        if (finished) out[q] = hi - lo;
    }
    const bool live = valid && !finished;
    const uint64_t pos = append_live(live, list_a, reinterpret_cast<unsigned long long *>(packed + lay.live()), lay.n);
    if (live) {
        packed[lay.w0() + pos] = word0;
        if constexpr (WIDE) {
            packed[lay.seed() + pos] = lo;
            packed[lay.seed() + lay.n + pos] = hi;
        } else {
            packed[lay.seed() + pos] = lo | (hi << 32);
        }
        reinterpret_cast<uint32_t *>(packed + lay.qidx())[pos] = (uint32_t)q | (flag << 30);
    }
}

// ---------------------------------------------------------------- K1: count_kmers

__device__ __forceinline__ uint32_t table_depth(uint32_t flag, uint32_t ts) { return flag == 0 ? 0u : (flag == 1 ? ts : ts - 1u); }

// Persistent one-step kernel over a live list -- BITS = 2: list A (all-ACGT k-mers, 32 symbols per word,
// stored front to back; used when the index has no pair image), BITS = 3: list B (21 symbols per word,
// stored back to front).  Every owner -- a thread (LANES = 1) or a lane pair (LANES = 2) -- walks its own
// stream of live queries (i, i+T, i+2T, ... of the compacted list) and refills itself as soon as its
// current k-mer is finished.  The next query's first word, seed and index are loaded one query ahead
// and the next symbol word a whole word of steps ahead, so neither exposes memory latency.
template <bool WIDE, int LANES, int BITS>
__global__ void __launch_bounds__(kCountThreads, min_ctas(WIDE, LANES))
count_kmers_packed_kernel(IndexView ix, const uint64_t *__restrict__ packed, PackedLayout lay, uint32_t k,
                          uint64_t *__restrict__ out) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint64_t stream = policy_evict_first();
    if constexpr (LANES == 2) warp_sync_guard(lay);  // the lanes of a pair exchange their halves through shuffles

    constexpr uint32_t kPerWord = BITS == 3 ? kSymsPerWord : kPairSymsPerWord;
    constexpr int kTop = 64 - BITS - (BITS == 3 ? 1 : 0);  // bit offset of a word's first symbol: 60 / 62
    const uint32_t n = (uint32_t)packed[lay.live() + (BITS == 3 ? 1 : 0)];  // live queries of this list
    const uint32_t tid = blockIdx.x * kCountThreads + threadIdx.x;
    const uint32_t owners = gridDim.x * kCountThreads / LANES;  // concurrent query streams
    const uint32_t half = tid & (LANES - 1);
    uint32_t i = tid / LANES;
    if (i >= n) return;
    const uint32_t last = (uint32_t)lay.n - 1u;  // list B is stored back to front
    auto slot = [&](uint32_t ii) { return BITS == 3 ? last - ii : ii; };
    const uint64_t *w0 = packed + lay.w0(), *seeds = packed + lay.seed(), *wx = packed + lay.wx();
    const uint32_t *qidx = reinterpret_cast<const uint32_t *>(packed + lay.qidx());
    const uint32_t ts = ix.table_s;

    P l = 0, h = 0;
    uint64_t word = 0, pend = 0, next_word = 0, next_lo = 0;
    [[maybe_unused]] uint64_t next_hi = 0;
    uint32_t q = 0, next_q = 0;
    uint32_t rem = 0;   // symbols still to consume
    int shift = kTop;   // bit offset of the next symbol in `word`
    uint32_t widx = 0;  // index of `word` within the query's remaining symbols

    auto prefetch = [&](uint32_t ii) {
        const uint32_t at = slot(ii);
        next_word = ldg_stream(w0 + at, stream);
        next_lo = ldg_stream(seeds + at, stream);
        if constexpr (WIDE) next_hi = ldg_stream(seeds + lay.n + at, stream);
        next_q = __ldg(qidx + at);
    };
    auto begin = [&]() {  // start the prefetched query
        word = next_word;
        q = next_q & kQidxMask;
        if constexpr (WIDE) { l = next_lo; h = next_hi; } else { l = (uint32_t)next_lo; h = (uint32_t)(next_lo >> 32); }
        rem = k - table_depth(next_q >> 30, ts);  // the suffix table already answered that many steps
        shift = kTop;
        widx = 0;
        if (rem > kPerWord) pend = ldg_stream(wx + q, stream);  // symbol word 1, needed a word of steps from now
    };

    prefetch(i);
    begin();
    if (i + owners < n) prefetch(i + owners);

    for (;;) {
        // retire + refill (msbwt_core.rs:151-153,160: empty range or all symbols consumed)
        while (rem == 0 || l == h) {
            if (half == 0) stg_stream(out + q, (uint64_t)(h - l), stream);
            i += owners;
            if (i >= n) return;
            begin();
            if (i + owners < n) prefetch(i + owners);
        }
        if (shift < 0) {  // next word of symbols: already in flight since the previous word began
            word = pend;
            widx++;
            shift = kTop;
            if (rem > kPerWord) pend = ldg_stream(wx + (uint64_t)widx * lay.n + q, stream);
        }
        uint32_t sym;
        if constexpr (BITS == 3) sym = (uint32_t)(word >> shift) & 7u;
        else sym = (0x5321u >> (4u * ((uint32_t)(word >> shift) & 3u))) & 7u;  // A,C,G,T = 1,2,3,5
        rank_step<WIDE, LANES>(ix, cb, sym, l, h, half);
        rem--;
        shift -= BITS;
    }
}

// Persistent kernel over live list A: a quad of lanes per query walks the PAIR image, two symbols per
// step (one 128-byte line per boundary); same refill / prefetch structure as above.
#ifndef MSBWT_PAIR_CTAS
#define MSBWT_PAIR_CTAS 6
#endif
constexpr int pair_min_ctas(bool wide) { return wide ? 4 : MSBWT_PAIR_CTAS; }

template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, pair_min_ctas(WIDE))
count_kmers_pair_kernel(IndexView ix, const uint64_t *__restrict__ packed, PackedLayout lay, uint32_t k,
                        uint64_t *__restrict__ out) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t c2_smem[WIDE ? kMaxSuperInSmem * 16 : 1];
    const C2Base<WIDE> c2 = stage_c2base<WIDE>(ix, c2_smem);
    const uint64_t stream = policy_evict_first();
    warp_sync_guard(lay);  // the lanes of a quad exchange their quarters through shuffles

    const uint32_t n = (uint32_t)packed[lay.live()];  // live queries of list A
    const uint32_t tid = blockIdx.x * kCountThreads + threadIdx.x;
    const uint32_t owners = gridDim.x * kCountThreads / 4;
    const uint32_t quarter = tid & 3u;
    uint32_t i = tid >> 2;
    if (i >= n) return;
    const uint64_t *w0 = packed + lay.w0(), *seeds = packed + lay.seed(), *wx = packed + lay.wx();
    const uint32_t *qidx = reinterpret_cast<const uint32_t *>(packed + lay.qidx());
    const uint32_t ts = ix.table_s;

    P l = 0, h = 0;
    uint64_t word = 0, pend = 0, next_word = 0, next_lo = 0;
    [[maybe_unused]] uint64_t next_hi = 0;
    uint32_t q = 0, next_q = 0;
    uint32_t rem = 0;   // symbols still to consume (even)
    int shift = 60;     // bit offset of the next pair (4 bits) in `word`
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
        rem = k - table_depth(next_q >> 30, ts);
        shift = 60;
        widx = 0;
        if (rem > (uint32_t)kPairSymsPerWord) pend = ldg_stream(wx + q, stream);  // needed 16 pair steps from now
    };

    prefetch(i);
    begin();
    if (i + owners < n) prefetch(i + owners);

    for (;;) {
        while (rem == 0 || l == h) {
            if (quarter == 0) stg_stream(out + q, (uint64_t)(h - l), stream);
            i += owners;
            if (i >= n) return;
            begin();
            if (i + owners < n) prefetch(i + owners);
        }
        if (shift < 0) {
            word = pend;
            widx++;
            shift = 60;
            if (rem > (uint32_t)kPairSymsPerWord) pend = ldg_stream(wx + (uint64_t)widx * lay.n + q, stream);
        }
        const uint32_t code = (uint32_t)(word >> shift) & 15u;
        pair_step<WIDE>(ix, c2, code, l, h, quarter);
        rem -= 2;
        shift -= 4;
    }
}

// Variable-length form, symbols read straight from the caller's byte layout.
template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, min_ctas(WIDE, 1))
count_kmers_bytes_kernel(IndexView ix, const uint8_t *__restrict__ syms, const uint64_t *__restrict__ offsets,
                         uint32_t n, uint64_t *__restrict__ out, uint32_t *__restrict__ status) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    uint32_t q = blockIdx.x * kCountThreads + threadIdx.x;
    if (q >= n) return;
    P l = 0, h = (P)ix.total;
    uint64_t beg = offsets[q], cur = offsets[q + 1];  // cur: one past the next symbol to consume
    for (;;) {
        while (cur == beg || l == h) {
            out[q] = (uint64_t)(h - l);
            q += threads;
            if (q >= n) return;
            l = 0; h = (P)ix.total; beg = offsets[q]; cur = offsets[q + 1];
        }
        uint32_t sym = syms[cur - 1];
        if (sym >= (uint32_t)kAlphabet) { atomicOr(status, 1u); sym = 0; }
        rank_step<WIDE, 1>(ix, cb, sym, l, h);
        cur--;
    }
}

// ---------------------------------------------------------------- K2: constrain_ranges

template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, min_ctas(WIDE, 1))
constrain_ranges_kernel(IndexView ix, const uint8_t *__restrict__ sym, const uint64_t *__restrict__ l,
                        const uint64_t *__restrict__ h, uint32_t n, uint64_t *__restrict__ out_l,
                        uint64_t *__restrict__ out_h) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    for (uint64_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += threads) {
        P a = (P)l[i], b = (P)h[i];
        rank_step<WIDE, 1>(ix, cb, sym[i], a, b);
        out_l[i] = a;
        out_h[i] = b;
    }
}

// ---------------------------------------------------------------- K3: suffix table levels

// child[idx] = constrain_range(ACGT[idx & 3], parent[idx >> 2]); an empty parent stays empty
// (count_kmer returns 0 as soon as the range is empty, msbwt_core.rs:151-153).
template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, min_ctas(WIDE, 1))
table_extend_kernel(IndexView ix, const void *__restrict__ parent_v, void *__restrict__ child_v, uint32_t n_child) {
    using P = typename Pos<WIDE>::type;
    using E = typename std::conditional<WIDE, ulonglong2, uint2>::type;
    const E *parent = reinterpret_cast<const E *>(parent_v);
    E *child = reinterpret_cast<E *>(child_v);
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    for (uint64_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n_child; i += threads) {
        const E e = parent[i >> 2];
        P a = (P)e.x, b = (P)e.y;
        E o;
        o.x = 0; o.y = 0;
        if (a != b) {
            const uint32_t sym = (0x5321u >> ((i & 3u) * 4u)) & 7u;  // A,C,G,T = 1,2,3,5
            rank_step<WIDE, 1>(ix, cb, sym, a, b);
            o.x = a; o.y = b;
        }
        child[i] = o;
    }
}

// ---------------------------------------------------------------- K4: gather roofline

__device__ __forceinline__ uint32_t mix32(uint32_t x) {  // murmur3 finaliser
    x ^= x >> 16; x *= 0x85EBCA6Bu;
    x ^= x >> 13; x *= 0xC2B2AE35u;
    return x ^ (x >> 16);
}

// LANES lanes x 16 B = one granule.  Every group issues independent random granule
// reads, 8 in flight per lane, and xors what it read into a sink so nothing is elided.
// The index stream is a 32-bit hash masked to a power-of-two granule count so that the
// kernel stays far from issue-bound (a 64-bit modulo here would dominate).
template <int LANES>
__global__ void __launch_bounds__(256) gather_kernel(const uint4 *__restrict__ buf, uint32_t granule_mask,
                                                     uint32_t n_gathers, uint32_t seed,
                                                     uint64_t *__restrict__ sink) {
    constexpr int kInFlight = 8;
    const uint32_t sub = threadIdx.x % LANES;
    const uint32_t groups = gridDim.x * (256 / LANES);
    const uint32_t g = blockIdx.x * (256 / LANES) + threadIdx.x / LANES;
    uint32_t acc = 0;
    for (uint32_t i = g; i < n_gathers; i += kInFlight * groups) {
        uint4 v[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; u++) {
            const uint32_t j = i + (uint32_t)u * groups;
            const uint32_t gi = mix32(j ^ seed) & granule_mask;
            v[u] = make_uint4(0, 0, 0, 0);
            if (j < n_gathers) v[u] = ldg_plain(buf + (size_t)gi * LANES + sub);
        }
#pragma unroll
        for (int u = 0; u < kInFlight; u++) acc ^= v[u].x ^ v[u].y ^ v[u].z ^ v[u].w;
    }
    if (acc == 0x9E3779B9u) atomicAdd((unsigned long long *)sink, 1ull);  // practically never; defeats DCE
}

// The same measurement with the Hopper / Blackwell bulk copy: every LANE asks for its own 128-byte line with ONE
// cp.async.bulk into its shared-memory row (completion counted in bytes by an mbarrier per warp and stage), two
// stages per warp in flight -- against eight lanes x cp.async 16 B per line in the search kernels.  `granule` 129.
__global__ void __launch_bounds__(256) gather_bulk_kernel(const uint4 *__restrict__ buf, uint32_t line_mask, uint32_t n_gathers,
                                                          uint32_t seed, uint64_t *__restrict__ sink) {
    extern __shared__ __align__(128) uint8_t gather_smem[];  // rows[8 warps][2 stages][32 x 128 B], then bars[8][2]
    uint8_t(*rows)[2][32 * 128] = reinterpret_cast<uint8_t(*)[2][32 * 128]>(gather_smem);
    uint64_t(*bars)[2] = reinterpret_cast<uint64_t(*)[2]>(gather_smem + 8 * 2 * 32 * 128);
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t warps = gridDim.x * 8u, wg = blockIdx.x * 8u + warp;
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&bars[warp][0]), bar1 = (uint32_t)__cvta_generic_to_shared(&bars[warp][1]);
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar1));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    const uint32_t batches = (n_gathers + 31u) / 32u;
    uint32_t acc = 0;
    auto issue = [&](uint32_t b, uint32_t stage) {
        const uint32_t bar = stage ? bar1 : bar0;
        if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(32u * 128u) : "memory");
        __syncwarp();
        const uint32_t gi = mix32((b * 32u + lane) ^ seed) & line_mask;
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&rows[warp][stage][lane * 128u]);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 128, [%2];" ::"r"(dst),
                     "l"(buf + (size_t)gi * 8u), "r"(bar)
                     : "memory");
    };
    auto wait = [&](uint32_t stage, uint32_t parity) {
        const uint32_t bar = stage ? bar1 : bar0;
        uint32_t done = 0;
        while (!done) {
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        }
    };
    uint32_t it = 0;
    uint32_t b = wg;
    if (b < batches) issue(b, 0);
    for (; b < batches; b += warps, it++) {
        const uint32_t stage = it & 1u;
        if (b + warps < batches) issue(b + warps, stage ^ 1u);
        wait(stage, (it >> 1) & 1u);
        acc ^= *reinterpret_cast<const uint32_t *>(&rows[warp][stage][lane * 128u + 4u * (lane & 31u)]);
        __syncwarp();
    }
    if (acc == 0x9E3779B9u) atomicAdd((unsigned long long *)sink, 1ull);
}

// ---------------------------------------------------------------- launch wrappers

static bool is_wide(const IndexView &ix) { return ix.n_super > 1 || (ix.total >> 32) != 0; }


static int current_device() {
    int d = 0;
    cudaGetDevice(&d);
    return d;
}

cudaError_t launch_pack_seed(const IndexView &ix, const uint8_t *d_syms, uint32_t k, uint64_t n, uint64_t *d_packed,
                             uint64_t *d_out, uint32_t *d_status, cudaStream_t st) {
    if (!n) return cudaSuccess;
    g_launches++;  // one kernel, whichever route
    // a suffix-table entry + exactly kFinSyms symbols (k = 31, 32): pack, seed and answer in one regular kernel
    if (final_fast_path_applies(ix, k, d_syms, 0))
        return launch_pack_seed_final(current_device(), ix, d_syms, 0, k, n, d_packed, d_out, d_status, st);
    const PackedLayout lay = packed_layout(ix, k, n);
    cudaError_t e = cudaMemsetAsync(d_packed + lay.live(), 0, 8 * sizeof(uint64_t), st);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const size_t smem = k <= kPackSmemMaxK ? 256u * (size_t)k + 64u : 0u;
    const SeedPlan plan = make_seed_plan(ix, k);
    // fixed-k instantiations (every shift, mask and word count a constant): measured on B200 against the runtime-k
    // build on 10 M queries each (profiles/r2a_pack_fixed_k.json, equal checksums): k = 31 0.250 -> 0.150 ms,
    // k = 15 0.188 -> 0.131 ms; k = 63 no difference and k = 101 slower (0.336 -> 0.406 ms: three fully unrolled
    // words cost more registers than the loop), so those two stay on the runtime-k build
    if (is_wide(ix)) pack_seed_kernel<true, 0><<<blocks, 256, smem, st>>>(ix, d_syms, k, plan, lay, d_packed, d_out, d_status);
    else if (k == 31) pack_seed_kernel<false, 31><<<blocks, 256, smem, st>>>(ix, d_syms, k, plan, lay, d_packed, d_out, d_status);
    else if (k == 15) pack_seed_kernel<false, 15><<<blocks, 256, smem, st>>>(ix, d_syms, k, plan, lay, d_packed, d_out, d_status);
    else pack_seed_kernel<false, 0><<<blocks, 256, smem, st>>>(ix, d_syms, k, plan, lay, d_packed, d_out, d_status);
    return cudaGetLastError();
}

template <bool WIDE, int LANES, int BITS>
static cudaError_t launch_count_packed_t(int device, const IndexView &ix, const uint64_t *d_packed,
                                         const PackedLayout &lay, uint32_t k, uint64_t *d_out, cudaStream_t st) {
    const unsigned grid = persistent_grid(device, (const void *)count_kmers_packed_kernel<WIDE, LANES, BITS>, kCountThreads,
                                          lay.n, kCountThreads / LANES);
    count_kmers_packed_kernel<WIDE, LANES, BITS><<<grid, kCountThreads, 0, st>>>(ix, d_packed, lay, k, d_out);
    return cudaGetLastError();
}

template <int BITS>
static cudaError_t launch_one_step(int device, const IndexView &ix, int lanes, const uint64_t *d_packed,
                                   const PackedLayout &lay, uint32_t k, uint64_t *d_out, cudaStream_t st) {
    if (is_wide(ix))
        return lanes == 2 ? launch_count_packed_t<true, 2, BITS>(device, ix, d_packed, lay, k, d_out, st)
                          : launch_count_packed_t<true, 1, BITS>(device, ix, d_packed, lay, k, d_out, st);
    return lanes == 2 ? launch_count_packed_t<false, 2, BITS>(device, ix, d_packed, lay, k, d_out, st)
                      : launch_count_packed_t<false, 1, BITS>(device, ix, d_packed, lay, k, d_out, st);
}

template <bool WIDE>
static cudaError_t launch_count_pair_t(int device, const IndexView &ix, const uint64_t *d_packed,
                                       const PackedLayout &lay, uint32_t k, uint64_t *d_out, cudaStream_t st) {
    const unsigned grid = persistent_grid(device, (const void *)count_kmers_pair_kernel<WIDE>, kCountThreads, lay.n,
                                          kCountThreads / 4);
    count_kmers_pair_kernel<WIDE><<<grid, kCountThreads, 0, st>>>(ix, d_packed, lay, k, d_out);
    return cudaGetLastError();
}

// n <= kMaxPerLaunch (the callers chunk): query indices are u32 inside the kernels.
// list A: quad kernel when the index has a quad image, pair kernel when it has a pair image, else the
// one-step kernel on 2-bit words;
// list B: the one-step kernel on 3-bit words (`with_b` false: the caller knows list B is empty).
cudaError_t launch_count_packed(int device, const IndexView &ix, int lanes, const uint64_t *d_packed, uint32_t k,
                                uint64_t n, uint64_t *d_out, cudaStream_t st, bool with_b) {
    if (!n) return cudaSuccess;
    if (n > kMaxPerLaunch) return cudaErrorInvalidValue;
    const PackedLayout lay = packed_layout(ix, k, n);
    cudaError_t e;
    if (ix.quad || ix.oct)  // (the oct kernel works with or without the quad image beside it)
        e = launch_count_quad(device, ix, d_packed, lay, k, d_out, st);
    else if (ix.pair)
        e = is_wide(ix) ? launch_count_pair_t<true>(device, ix, d_packed, lay, k, d_out, st)
                        : launch_count_pair_t<false>(device, ix, d_packed, lay, k, d_out, st);
    else
        e = launch_one_step<2>(device, ix, lanes, d_packed, lay, k, d_out, st);
    g_launches++;
    if (e != cudaSuccess || !with_b) return e;
    e = launch_one_step<3>(device, ix, lanes, d_packed, lay, k, d_out, st);
    g_launches++;
    return e;
}

cudaError_t launch_seed_packed(const IndexView &ix, const uint64_t *d_words, uint32_t k, uint64_t n,
                               uint64_t *d_packed, uint64_t *d_out, cudaStream_t st) {
    if (!n) return cudaSuccess;
    g_launches++;  // one kernel, whichever route
    if (k <= 32u && final_fast_path_applies(ix, k, d_words, 2))  // one word per k-mer: word 0 is the whole k-mer
        return launch_pack_seed_final(current_device(), ix, d_words, 2, k, n, d_packed, d_out, nullptr, st);
    const PackedLayout lay = packed_layout(ix, k, n);
    cudaError_t e = cudaMemsetAsync(d_packed + lay.live(), 0, 8 * sizeof(uint64_t), st);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const SeedPlan plan = make_seed_plan(ix, k);
    if (is_wide(ix)) seed_packed_kernel<true><<<blocks, 256, 0, st>>>(ix, d_words, k, plan, lay, d_packed, d_out);
    else seed_packed_kernel<false><<<blocks, 256, 0, st>>>(ix, d_words, k, plan, lay, d_packed, d_out);
    return cudaGetLastError();
}

cudaError_t launch_seed_u64(const IndexView &ix, const uint64_t *d_kmers, uint32_t k, uint64_t n,
                            uint64_t *d_packed, uint64_t *d_out, cudaStream_t st) {
    if (!n) return cudaSuccess;
    if (!k || k > 32u) return cudaErrorInvalidValue;
    g_launches++;  // one kernel, whichever route
    if (final_fast_path_applies(ix, k, d_kmers, 1))
        return launch_pack_seed_final(current_device(), ix, d_kmers, 1, k, n, d_packed, d_out, nullptr, st);
    const PackedLayout lay = packed_layout(ix, k, n);
    cudaError_t e = cudaMemsetAsync(d_packed + lay.live(), 0, 8 * sizeof(uint64_t), st);
    if (e != cudaSuccess) return e;
    const unsigned blocks = (unsigned)((n + kPackThreads - 1) / kPackThreads);
    const SeedPlan plan = make_seed_plan(ix, k);
    if (is_wide(ix)) seed_u64_kernel<true><<<blocks, kPackThreads, 0, st>>>(ix, d_kmers, k, plan, lay, d_packed, d_out);
    else seed_u64_kernel<false><<<blocks, kPackThreads, 0, st>>>(ix, d_kmers, k, plan, lay, d_packed, d_out);
    return cudaGetLastError();
}

// does a host-packed all-ACGT batch of this k ever reach list B? (odd remainder with no usable table depth)
uint32_t max_host_packed_k() { return kPackSmemMaxK; }

bool packed_batch_needs_list_b(const IndexView &ix, uint32_t k) {
    return list_a_stride(ix) == 2u && ((k - acgt_table_depth(k, ix.table_s, 2u)) & 1u) != 0;
}

cudaError_t launch_table_extend(int device, const IndexView &ix, const void *d_parent, void *d_child,
                                uint32_t n_child, cudaStream_t st) {
    g_launches++;
    if (is_wide(ix)) {
        const unsigned grid = persistent_grid(device, (const void *)table_extend_kernel<true>, kCountThreads, n_child, kCountThreads);
        table_extend_kernel<true><<<grid, kCountThreads, 0, st>>>(ix, d_parent, d_child, n_child);
    } else {
        const unsigned grid = persistent_grid(device, (const void *)table_extend_kernel<false>, kCountThreads, n_child, kCountThreads);
        table_extend_kernel<false><<<grid, kCountThreads, 0, st>>>(ix, d_parent, d_child, n_child);
    }
    return cudaGetLastError();
}

bool index_is_wide(const IndexView &ix) { return is_wide(ix); }

cudaError_t launch_count_bytes(int device, const IndexView &ix, const uint8_t *d_syms,
                               const uint64_t *d_offsets, uint64_t n, uint64_t *d_out, uint32_t *d_status,
                               cudaStream_t st) {
    for (uint64_t q0 = 0; q0 < n; q0 += kMaxPerLaunch) {
        const uint32_t m = (uint32_t)((n - q0) < kMaxPerLaunch ? (n - q0) : kMaxPerLaunch);
        if (is_wide(ix)) {
            const unsigned grid = persistent_grid(device, (const void *)count_kmers_bytes_kernel<true>, kCountThreads, m, kCountThreads);
            count_kmers_bytes_kernel<true><<<grid, kCountThreads, 0, st>>>(ix, d_syms, d_offsets + q0, m, d_out + q0, d_status);
        } else {
            const unsigned grid = persistent_grid(device, (const void *)count_kmers_bytes_kernel<false>, kCountThreads, m, kCountThreads);
            count_kmers_bytes_kernel<false><<<grid, kCountThreads, 0, st>>>(ix, d_syms, d_offsets + q0, m, d_out + q0, d_status);
        }
        g_launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_constrain_ranges(int device, const IndexView &ix, const uint8_t *d_sym, const uint64_t *d_l,
                                    const uint64_t *d_h, uint64_t n, uint64_t *d_out_l, uint64_t *d_out_h,
                                    cudaStream_t st) {
    for (uint64_t q0 = 0; q0 < n; q0 += kMaxPerLaunch) {
        const uint32_t m = (uint32_t)((n - q0) < kMaxPerLaunch ? (n - q0) : kMaxPerLaunch);
        if (is_wide(ix)) {
            const unsigned grid = persistent_grid(device, (const void *)constrain_ranges_kernel<true>, kCountThreads, m, kCountThreads);
            constrain_ranges_kernel<true><<<grid, kCountThreads, 0, st>>>(ix, d_sym + q0, d_l + q0, d_h + q0, m, d_out_l + q0, d_out_h + q0);
        } else {
            const unsigned grid = persistent_grid(device, (const void *)constrain_ranges_kernel<false>, kCountThreads, m, kCountThreads);
            constrain_ranges_kernel<false><<<grid, kCountThreads, 0, st>>>(ix, d_sym + q0, d_l + q0, d_h + q0, m, d_out_l + q0, d_out_h + q0);
        }
        g_launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_gather(int device, const void *d_buf, uint64_t buf_bytes, uint32_t granule,
                          uint64_t n_gathers, uint64_t seed, uint64_t *d_sink, cudaStream_t st) {
    uint64_t n_granules = buf_bytes / (granule == 129 ? 128 : granule);
    if (!n_granules || !n_gathers || n_gathers >= (1ull << 31)) return cudaErrorInvalidValue;
    while (n_granules & (n_granules - 1)) n_granules &= n_granules - 1;  // round down to a power of two
    if (n_granules > (1ull << 31)) n_granules = 1ull << 31;
    const uint32_t mask = (uint32_t)(n_granules - 1);
    const unsigned grid = (unsigned)sm_count(device) * 8u;
    const uint4 *buf = (const uint4 *)d_buf;
    g_launches++;
    switch (granule) {
        case 32: gather_kernel<2><<<grid, 256, 0, st>>>(buf, mask, (uint32_t)n_gathers, (uint32_t)seed, d_sink); break;
        case 64: gather_kernel<4><<<grid, 256, 0, st>>>(buf, mask, (uint32_t)n_gathers, (uint32_t)seed, d_sink); break;
        case 128: gather_kernel<8><<<grid, 256, 0, st>>>(buf, mask, (uint32_t)n_gathers, (uint32_t)seed, d_sink); break;
        case 129:  // 128-byte lines, one cp.async.bulk per lane (64 KB of shared memory per CTA: 3 CTAs per SM)
        {
            constexpr int kBulkSmem = 8 * 2 * 32 * 128 + 8 * 2 * 8;
            if (cudaError_t e = cudaFuncSetAttribute((const void *)gather_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBulkSmem); e != cudaSuccess) return e;
            gather_bulk_kernel<<<(unsigned)sm_count(device) * 3u, 256, kBulkSmem, st>>>(buf, mask, (uint32_t)n_gathers, (uint32_t)seed, d_sink);
            break;
        }
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace msbwt
