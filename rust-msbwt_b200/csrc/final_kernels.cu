// final_kernels.cu -- the ONE-REQUEST path of BWT::count_kmer (src/msbwt_core.rs:125-161) for k-mers that are a
// suffix-table entry plus exactly kFinSyms = 20 symbols: k = 31 (table level 11) and k = 32 (level 12).
//
// Such a k-mer needs, per query: its symbols (k bytes, or 8 bytes when the caller holds it packed), one L2-resident
// table entry (the range after its last 11 / 12 symbols), ONE 128-byte final-step line (layout.h: the number of
// positions of that range preceded by its first 20 symbols) and 8 bytes for the count.  The general search kernel
// (oct_kernel.cuh) walks every query as a little state machine and pays for that generality in instructions
// (measured on B200, profiles/r2b_*: 4.6 ms per 100 M 31-mers with one line per query, against 2.6 ms for 100 M
// independent random line reads).  Here the work is REGULAR -- every query does the same three things -- so a warp
// simply streams through consecutive batches of 32 queries as a software pipeline, nothing diverges, nothing is
// compacted, and the counts are written back coalesced:
//
//   iteration i of a warp (its batches are i = 0, 1, ..):
//     -- cp.async.wait_all: what iteration i-1 issued has landed = the lines of batch i and the bytes of batch i+2
//     D  batch i   : every lane scans its own line (groups `tag | nruns` + runs, layout.h), writes its count to
//                    out[32 * batch + lane] (one coalesced 256-byte store per warp), or queues the query for the
//                    general kernel: overflowed line, range over two buckets
//     B  batch i+2 : every lane packs its k-mer from the byte buffer (SWAR, four symbols per step), and requests
//                    its table entry (ld.global.nc: an L2 hit, consumed by C in the next iteration)
//     C  batch i+1 : range [l, h) from the table entry requested one iteration ago; 40-bit code -> fin_mix40 -> line
//                    index + tag; the WARP copies the 32 lines into the row buffer (8 lanes x 16 bytes per line: one
//                    128-byte request per line)
//     A  batch i+3 : the batch's 32 k symbol bytes -> the byte buffer (coalesced 16-byte cp.async)
//
// What the pipeline cannot answer goes where pack_seed_kernel would have put it, in the same scratch layout
// (engine.h PackedLayout), for launch_count_packed to finish: live list A (all-ACGT: the remaining 20 symbols + the
// range; bit 30 of the index word tells the oct kernel that the final-step line is known to have overflowed) and
// live list B (k-mers holding `$` / `N`: seed_general, one symbol at a time -- rare).  Appends to list A are staged
// per warp in shared memory and flushed 32+ at a time: one atomic per flush, not per query.
#include <cstdlib>
#include <type_traits>

#include "oct_kernel.cuh"
#include "pack_common.cuh"

namespace msbwt {

namespace {

constexpr int kFinWarps = 8;                 // warps per CTA
constexpr int kFinThreads = 32 * kFinWarps;
constexpr int kFinRowBytes = 144;            // a 128-byte line + 16: the rows of consecutive lanes start 4 banks apart
constexpr int kFinByteBuf = 32 * 32 + 16;    // 32 k-mers of k <= 32 symbol bytes, + the slack an unaligned 4-byte read needs
// One row buffer and one byte buffer per warp: a warp waits for its own lines and the OTHER warps of the SM hide
// that.  The loop is bound by the latency of its own dependent instructions (ncu, profiles/r2g_*: 640 instructions
// per batch issue in 5600 cycles per warp at 4 warps per scheduler), which only more resident warps can hide -- so
// the shape that keeps the most warps resident: 6.3 KB of shared memory per warp and 64 registers per thread, 4 CTAs
// of 8 warps per SM (32 warps).
// WIDE (64-bit positions: an index of 2^32 symbols and more, or one cut into several superblocks): 16-byte table
// entries, two seed words per queued query, 3 CTAs per SM for the registers the wider ranges take.
template <bool WIDE = false> struct FinShape {
    static constexpr int kQueue = 32;  // list-A entries a warp stages before it flushes
    static constexpr int kWarpSmem = 32 * kFinRowBytes + kFinByteBuf + kQueue * (WIDE ? 28 : 20);
    static constexpr int kSmem = kFinWarps * kWarpSmem;
    static constexpr int kCtasPerSm = WIDE ? 3 : 4;
};

enum : uint32_t { kKindNone = 0, kKindZero = 1, kKindLine = 2, kKindTwoBuckets = 3 };

// SRC 0: symbol bytes; 1: caller-packed integers (first symbol most significant); 2: host-packed words (last symbol
// in the top bits).  K = 31: every shift, mask and copy count a constant; K = 0: k_rt (k <= 32).
template <int SRC, uint32_t K, bool WIDE = false>
__global__ void __launch_bounds__(kFinThreads, FinShape<WIDE>::kCtasPerSm)
pack_seed_final_kernel(IndexView ix, const void *__restrict__ src_v, uint32_t k_rt, SeedPlan plan, PackedLayout lay,
                       uint64_t *__restrict__ packed, uint64_t *__restrict__ out, uint32_t *__restrict__ status) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr uint32_t kFull = 0xffffffffu;
    const uint32_t k = K ? K : k_rt;
    const uint32_t depth = plan.depth;  // k - depth == kFinSyms (the host checked)
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t n = (uint32_t)lay.n;  // <= 2^30 per launch (kMaxPerLaunch): query and batch numbers are 32-bit
    const uint32_t n_batches = (n + 31u) / 32u;
    const uint32_t warps_total = gridDim.x * kFinWarps;
    const uint32_t warp_gid = blockIdx.x * kFinWarps + warp;
    if (warp_gid >= n_batches) return;
    const uint32_t my_batches = (n_batches - warp_gid + warps_total - 1u) / warps_total;  // batches warp_gid + s * warps_total

    using Shape = FinShape<WIDE>;
    using P = typename Pos<WIDE>::type;                                       // a BWT position
    using E = typename std::conditional<WIDE, ulonglong2, uint2>::type;       // a suffix-table entry {l, h}
    constexpr int kFinQueue = Shape::kQueue;
    uint8_t *const wsm = smem + warp * Shape::kWarpSmem;
    uint8_t *const rows = wsm;                                              // 32 rows
    uint8_t *const bytes = wsm + 32 * kFinRowBytes;                         // the byte buffer (SRC 0)
    uint8_t *const queue = bytes + kFinByteBuf;                             // kQueue x {u64 word, u64 seed, u32 index}
    uint64_t *const q_word = reinterpret_cast<uint64_t *>(queue);
    uint64_t *const q_seed = q_word + kFinQueue;                             // l | h << 32; WIDE: l, and h in q_seed_hi
    [[maybe_unused]] uint64_t *const q_seed_hi = q_seed + kFinQueue;
    uint32_t *const q_idx = reinterpret_cast<uint32_t *>(q_seed + (WIDE ? 2 : 1) * kFinQueue);
    uint32_t q_fill = 0;  // warp-uniform

    const E *const table = reinterpret_cast<const E *>(plan.tab);
    const char *const fin_base = reinterpret_cast<const char *>(ix.fin);
    const uint32_t fshift = ix.fin_shift, fmask = (1u << fshift) - 1u, flb = ix.fin_lb;
    const uint64_t stream_pol = policy_evict_first();  // query bytes, final-step lines, results: read or written once
    const uint64_t table_pol = policy_evict_last();    // the suffix-table level: 33 MB read a hundred million times
    unsigned long long *const live = reinterpret_cast<unsigned long long *>(packed + lay.live());
    uint32_t *const qidx_arr = reinterpret_cast<uint32_t *>(packed + lay.qidx());
    uint32_t st_lines = 0, st_over = 0, st_two = 0, st_zero = 0;

    auto first_query = [&](uint32_t s) { return (warp_gid + s * warps_total) * 32u; };

    // ---- A: symbol bytes of batch sequence number s -> the byte buffer (SRC 0), or this lane's word (SRC 1, 2)
    auto stage_a = [&](uint32_t s, uint64_t &word_reg) {
        if (s >= my_batches) return;
        const uint32_t q0 = first_query(s);
        if constexpr (SRC == 0) {
            const uint8_t *g = reinterpret_cast<const uint8_t *>(src_v) + (size_t)q0 * k;  // 16-byte aligned: 32 k bytes per batch
            uint8_t *dst = bytes;
            if (q0 + 32u <= n) {  // a whole batch: 2 k pieces of 16 bytes, every one of them full
                cp_async16_hint(dst + 16u * lane, g + 16u * lane, true, stream_pol);
                if (lane + 32u < 2u * k) cp_async16_hint(dst + 16u * (lane + 32u), g + 16u * (lane + 32u), true, stream_pol);
            } else {              // the batch's tail: the pieces past the last query are zero-filled, not read
                const uint32_t nbytes = (n - q0) * k;
#pragma unroll
                for (uint32_t c = lane; c < 64u; c += 32u) {
                    const uint32_t at = 16u * c;
                    if (at < 32u * k) cp_async16_partial(dst + at, g + at, at < nbytes ? min(16u, nbytes - at) : 0u);
                }
            }
        } else {
            const uint32_t q = q0 + lane;
            word_reg = q < n ? ldg_stream(reinterpret_cast<const uint64_t *>(src_v) + q, stream_pol) : 0ull;
        }
    };

    // ---- B: pack (SRC 0) / normalise (SRC 1, 2) the k-mer of batch s: `word` = its symbols 2 bits each, the LAST
    //         symbol in the top bits; request the table entry.  A k-mer holding `$` / `N` is seeded one symbol at a
    //         time (seed_general) and goes to live list B here and now; kind = what stage C has to do with the query.
    auto stage_b = [&](uint32_t s, uint64_t word_reg, uint64_t &word, E &entry, uint32_t &kind) {
        kind = kKindNone;
        word = 0;
        entry.x = 0;
        entry.y = 0;
        if (s >= my_batches) return;
        const uint32_t q = first_query(s) + lane;
        if (q >= n) return;
        if constexpr (SRC == 0) {
            const uint8_t *buf = bytes;
            const uint32_t o = lane * k;
            const volatile uint32_t *p = reinterpret_cast<const volatile uint32_t *>(buf + (o & ~3u));
            const uint32_t sh = (o & 3u) * 8u;
            uint32_t prev = p[0], other = 0;
            uint32_t m[8];
#pragma unroll
            for (uint32_t i = 0; i < 8; i++) {
                const uint32_t nxt = p[i + 1];
                uint32_t x = __funnelshift_r(prev, nxt, sh);
                prev = nxt;
                if (k < 4u * (i + 1)) {  // bytes past the k-mer count as 'A' (code 0, never an exception)
                    const uint32_t keep = k > 4u * i ? (1u << (8u * (k - 4u * i))) - 1u : 0u;
                    x = (x & keep) | (0x01010101u & ~keep);
                }
                m[i] = swar_lut_pack4_top(x, other);
            }
            if (other & kSwarBadMask) {  // `$`, `N` or an invalid byte: the general path, list B
                uint64_t lo = 0, hi = 0, word0 = 0;
                uint32_t flag = 0;
                bool finished = false, bad = false;
                seed_general<WIDE>(ix, const_cast<const uint8_t *>(buf) + o, k, lay, q, packed, lo, hi, flag, finished, word0, bad);
                if (bad) atomicOr(status, 1u);
                if (finished) {
                    out[q] = hi - lo;
                } else {
                    const uint64_t pos = (uint64_t)n - 1 - atomicAdd(live + 1, 1ull);
                    packed[lay.w0() + pos] = word0;
                    if constexpr (WIDE) {
                        packed[lay.seed() + pos] = lo;
                        packed[lay.seed() + lay.n + pos] = hi;
                    } else {
                        packed[lay.seed() + pos] = lo | (hi << 32);
                    }
                    qidx_arr[pos] = q | (flag << 30);
                }
                return;
            }
            const uint64_t le = (uint64_t)swar_gather4(m[0], m[1], m[2], m[3]) | ((uint64_t)swar_gather4(m[4], m[5], m[6], m[7]) << 32);
            word = le << (64u - 2u * k);
        } else if constexpr (SRC == 1) {
            word = reverse_symbol_pairs(word_reg & (k >= 32u ? ~0ull : ((1ull << (2u * k)) - 1ull)));
        } else {
            word = word_reg;
        }
        entry = ldg_table_entry(table + (word >> (64u - 2u * depth)), table_pol);
        kind = kKindLine;  // refined in stage C, once the entry has arrived
    };

    // ---- C: batch s: the range, the line, and the warp's copy of the 32 lines into the row buffer
    auto stage_c = [&](uint32_t s, uint64_t word, E entry, uint32_t &kind, P &l, P &h, uint32_t &tag) {
        l = entry.x;
        h = entry.y;
        uint32_t line = 0;
        tag = 0;
        if (kind == kKindLine) {
            if (l == h) {
                kind = kKindZero;  // the table already says the k-mer's suffix does not occur
            } else if ((l >> fshift) != (h >> fshift)) {
                kind = kKindTwoBuckets;
            } else {
                const uint64_t mixed = fin_mix40((word << (2u * depth)) >> (64 - kFinCodeBits));
                line = ((uint32_t)(l >> fshift) << flb) | (uint32_t)(mixed & ((1ull << flb) - 1ull));
                tag = (uint32_t)(mixed >> flb);
            }
        }
        if (s >= my_batches) return;  // (warp-uniform)
        const uint32_t pub = line | (kind == kKindLine ? 0x80000000u : 0u);  // a line index is below 2^31 (checked by the host)
        const uint32_t j = lane & 7u;
#pragma unroll
        for (uint32_t c = 0; c < 8u; c++) {
            const uint32_t o = 4u * c + (lane >> 3);  // the lane whose line this is
            const uint32_t v = __shfl_sync(kFull, pub, o);
            cp_async16_hint(rows + o * kFinRowBytes + 16u * j, fin_base + (size_t)(v & 0x7fffffffu) * kFinLineBytes + 16u * j,
                            (v >> 31) != 0u, stream_pol);
        }
    };

    // list A: the warp's queue -> global memory (one atomic for all of it)
    auto flush_queue = [&]() {
        if (!q_fill) return;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(live, (unsigned long long)q_fill);
        base = __shfl_sync(kFull, base, 0);
        for (uint32_t i = lane; i < q_fill; i += 32u) {
            packed[lay.w0() + base + i] = q_word[i];
            packed[lay.seed() + base + i] = q_seed[i];
            if constexpr (WIDE) packed[lay.seed() + lay.n + base + i] = q_seed_hi[i];
            qidx_arr[base + i] = q_idx[i];
        }
        __syncwarp();
        q_fill = 0;
    };

    // occurrences inside [pl, ph) of the runs `(len << 16) | offset` at words first .. first + nruns - 1 of a row: the
    // same loop for every lane of the warp (trip count = the longest list among them), four runs per trip
    auto add_runs = [&](const uint32_t *roww, uint32_t first, uint32_t nruns, int pl, int ph, int &acc) {
        const uint32_t trips = __reduce_max_sync(kFull, nruns);
        for (uint32_t r = 0; r < trips; r += 4u) {
#pragma unroll
            for (uint32_t u = 0; u < 4u; u++) {
                if (r + u < nruns) {
                    const uint32_t w = roww[first + r + u];
                    const int off = (int)(w & 0xFFFFu), len = (int)(w >> 16);
                    acc += min(max(ph - off, 0), len) - min(max(pl - off, 0), len);
                }
            }
        }
    };

    // ---- D: batch s: scan the line, write the count, or queue the query for the general kernel
    auto stage_d = [&](uint32_t s, uint64_t word, uint32_t kind, P l, P h, uint32_t tag) {
        if (s >= my_batches) return;  // (warp-uniform)
        const uint32_t q = first_query(s) + lane;
        bool to_queue = kind == kKindTwoBuckets;
        uint32_t nofin = 0;
        // Phase 1, per lane: hop from group header to group header (`tag << 4 | nruns`, then nruns run words) to the
        // FIRST group of this query's code -- a line holds a few groups, so this is a handful of 4-byte shared-memory
        // reads.  A code with more than 15 runs in the bucket (a 31-mer seen 30 times is ~13 runs of consecutive
        // positions) continues in the groups right behind (layout.h: the groups of one code are adjacent).
        const uint32_t *roww = reinterpret_cast<const uint32_t *>(rows + lane * kFinRowBytes);
        uint32_t i1 = 0, matches = 0, used = 0;
        if (kind == kKindLine) {
            const uint2 first = *reinterpret_cast<const uint2 *>(roww);
            used = first.x;
            st_lines++;
            if (used == kFinOverflow) {
                to_queue = true;
                nofin = 1u;
                st_over++;
                used = 0;
            } else {
                uint32_t hw = first.y;  // word 1: the first header (meaningless when used == 0)
                for (uint32_t idx = 1u; idx <= used;) {
                    const bool eq = (hw >> 4) == tag;
                    if (eq && matches == 0u) i1 = idx;
                    matches += eq ? 1u : 0u;
                    idx += 1u + (hw & 15u);
                    if (idx <= used) hw = roww[idx];
                }
            }
        }
        // Phase 2, the warp in step: every lane adds up the runs of its group (and, when some lane's code has one, of
        // the group behind it); a third group of one code is rare enough to leave to the general kernel
        int acc = 0;
        {
            const int pl = (int)((uint32_t)l & fmask), ph = (int)((uint32_t)h & fmask);
            const uint32_t n1 = matches ? (roww[i1] & 15u) : 0u;
            add_runs(roww, i1 + 1u, n1, pl, ph, acc);
            if (__any_sync(kFull, matches > 1u)) {
                const uint32_t i2 = i1 + 1u + n1;
                const uint32_t n2 = matches > 1u ? (roww[i2] & 15u) : 0u;
                add_runs(roww, i2 + 1u, n2, pl, ph, acc);
                if (matches > 2u) to_queue = true;
            }
        }
        st_two += kind == kKindTwoBuckets;
        st_zero += kind == kKindZero;
        if ((kind == kKindLine && !to_queue) || kind == kKindZero) stg_stream(out + q, (uint64_t)(uint32_t)acc, stream_pol);
        const uint32_t qm = __ballot_sync(kFull, to_queue);
        if (qm) {
            if (q_fill + (uint32_t)__popc(qm) > (uint32_t)kFinQueue) flush_queue();
            if (to_queue) {
                const uint32_t at = q_fill + __popc(qm & ((1u << lane) - 1u));
                q_word[at] = word << (2u * depth);  // the kFinSyms symbols still to consume, first in the top bits
                if constexpr (WIDE) {
                    q_seed[at] = l;
                    q_seed_hi[at] = h;
                } else {
                    q_seed[at] = (uint64_t)l | ((uint64_t)h << 32);
                }
                q_idx[at] = q | (nofin << 30);
            }
            q_fill += (uint32_t)__popc(qm);
            __syncwarp();
        }
    };

    // ---- the pipeline (one row buffer, one byte buffer).  Iteration s: everything issued so far has landed
    //      (lines of batch s, bytes of batch s+2) -> D(s) -> B(s+2) -> C(s+1) (its table entry was requested an
    //      iteration ago) -> A(s+3) -> commit.  Register state: batch s in D (d_*), s+1 in C (c_*).
    uint64_t a_word = 0, b_wordreg = 0, w1 = 0;
    uint64_t c_word = 0, d_word = 0;
    E c_entry{};
    uint32_t c_kind = kKindNone, d_kind = kKindNone, d_tag = 0;
    P d_l = 0, d_h = 0;
    auto land = [&]() {
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
    };
    stage_a(0, b_wordreg);
    land();
    E e0;
    uint32_t k0;
    stage_b(0, b_wordreg, d_word, e0, k0);                  // B(0)
    __syncwarp();
    stage_a(1, w1);
    land();
    stage_b(1, w1, c_word, c_entry, c_kind);                // B(1)
    __syncwarp();
    stage_c(0, d_word, e0, k0, d_l, d_h, d_tag);            // C(0)
    d_kind = k0;
    stage_a(2, b_wordreg);                                  // A(2)
    for (uint32_t s = 0; s < my_batches; s++) {
        land();                                             // lines(s), bytes(s+2)
        stage_d(s, d_word, d_kind, d_l, d_h, d_tag);
        uint64_t b_word;
        E b_entry;
        uint32_t b_kind;
        stage_b(s + 2, b_wordreg, b_word, b_entry, b_kind); // requests the table entry C(s+2) reads next iteration
        __syncwarp();                                       // rows were read by D(s), the byte buffer by B(s+2)
        P n_l, n_h;
        uint32_t n_tag;
        stage_c(s + 1, c_word, c_entry, c_kind, n_l, n_h, n_tag);
        stage_a(s + 3, a_word);
        b_wordreg = a_word;
        d_word = c_word; d_kind = c_kind; d_l = n_l; d_h = n_h; d_tag = n_tag;
        c_word = b_word; c_entry = b_entry; c_kind = b_kind;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    flush_queue();
    // counters (one atomic per warp and counter)
    uint32_t st[4] = {st_lines, st_over, st_two, st_zero};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t v = st[i];
#pragma unroll
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
        if (lane == 0 && v) atomicAdd(reinterpret_cast<unsigned long long *>(packed + lay.fstat()) + i, (unsigned long long)v);
    }
}

template <int SRC, uint32_t K, bool WIDE = false>
cudaError_t launch_shape(int device, const IndexView &ix, const void *d_src, uint32_t k, const SeedPlan &plan, const PackedLayout &lay,
                     uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status, cudaStream_t st) {
    static bool prepared[64] = {};
    constexpr int kFinSmem = FinShape<WIDE>::kSmem;
    const void *fn = (const void *)pack_seed_final_kernel<SRC, K, WIDE>;
    if (device < 0 || device >= 64 || !prepared[device]) {
        if (cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kFinSmem); e != cudaSuccess) return e;
        cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (device >= 0 && device < 64) prepared[device] = true;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kFinThreads, kFinSmem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const uint64_t full = (uint64_t)sm_count(device) * (uint64_t)per_sm;
    const uint64_t need = ((lay.n + 31) / 32 + kFinWarps - 1) / kFinWarps;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min(need, full));
    pack_seed_final_kernel<SRC, K, WIDE><<<grid, kFinThreads, kFinSmem, st>>>(ix, d_src, k, plan, lay, d_packed, d_out, d_status);
    return cudaGetLastError();
}

template <int SRC, uint32_t K>
cudaError_t launch_t(int device, const IndexView &ix, const void *d_src, uint32_t k, const SeedPlan &plan, const PackedLayout &lay,
                     uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status, cudaStream_t st) {
    if (index_is_wide(ix)) return launch_shape<SRC, 0, true>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);  // 64-bit positions: runtime k
    return launch_shape<SRC, K>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);
}

}  // namespace

bool final_fast_path_applies(const IndexView &ix, uint32_t k, const void *d_src, int src_kind) {
    const char *env = getenv("MSBWT_FINAL_FAST");  // =0: the general kernels only (A/B measurements, tests)
    if ((env && atoi(env) == 0) || !ix.fin || !ix.oct || k > 32u || k <= (uint32_t)kFinSyms) return false;
    const uint32_t depth = list_a_table_depth(ix, k);
    if (depth == 0 || k - depth != (uint32_t)kFinSyms) return false;
    if ((((ix.total >> ix.fin_shift) + 1) << ix.fin_lb) >= (1ull << 31)) return false;  // line indices travel as 31 bits
    return (reinterpret_cast<uintptr_t>(d_src) & (src_kind == 0 ? 15u : 7u)) == 0;
}

cudaError_t launch_pack_seed_final(int device, const IndexView &ix, const void *d_src, int src_kind, uint32_t k, uint64_t n,
                                   uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status, cudaStream_t st) {
    if (!n) return cudaSuccess;
    if (n > kMaxPerLaunch) return cudaErrorInvalidValue;
    const PackedLayout lay = packed_layout(ix, k, n);
    if (cudaError_t e = cudaMemsetAsync(d_packed + lay.live(), 0, 8 * sizeof(uint64_t), st); e != cudaSuccess) return e;  // LIVE, WORK, FSTAT
    const SeedPlan plan = make_seed_plan(ix, k);
    if (src_kind == 0) {
        if (k == 31) return launch_t<0, 31>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);
        return launch_t<0, 0>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);
    }
    if (src_kind == 1) return launch_t<1, 0>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);
    return launch_t<2, 0>(device, ix, d_src, k, plan, lay, d_packed, d_out, d_status, st);
}

}  // namespace msbwt
