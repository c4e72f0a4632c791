// unitigs.cu -- the unitigs of the compacted de Bruijn graph of an index's solid k-mers (msbwt_unitigs).
//
// Nodes: V = the k-mers the spectrum walk lists (spectrum.cu), copied device-to-device into arrays a histogram-only
// pass sized; in canonical mode the canonical members plus rc of every non-palindromic one, so V is closed under rc.
// (value, count) pairs are radix-sorted over the low 2k bits, so a node's id is its rank by value.
// Edges are node-centric: X -> Y iff X[1..k) = Y[0..k-1) and both are in V.  The four successor candidates
// ((X << 2) & mask) | c are consecutive integers, so one lower-bound search and four compares find them all
// (unitig_link_kernel).  X -> Y is compacted iff outdeg(X) = 1, indeg(Y) = 1 and X != Y: next / prev follow those
// edges only (unitig_prev_kernel, unitig_next_kernel).
// Ranking: pointer jumping over prev (Wyllie) gives every node its head J and its distance D to it, in about log2(L)
// synchronous rounds for the longest unitig of L nodes.  A round whose number of unresolved nodes (J not yet a head)
// does not fall has resolved every linear path: what remains lies on cycles of compacted edges.  Those are found and
// cut by doubling over next with a running minimum of the node value (unitig_cycle_step_kernel, until a round changes
// nothing: then every window covers its cycle), cut before their minimum (unitig_cut_kernel), and ranked by more rounds.
// Emission: each tail scatters its unitig's length to the head, each node adds its count to the head's sum (integer
// atomics: deterministic), exclusive scans over node ids (= ascending first k-mer) give the symbol offsets and the
// unitig numbers, and every node writes its last symbol at offset(head) + k - 1 + D; a head writes its whole k-mer.
// Canonical mode keeps a linear unitig U iff first(U) <= rc(last(U)) and a cycle C iff min(C) <= min(rc C).
// The kernels use no warp collectives: counts are summed through shared memory, as in spectrum.cu.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include <cstdlib>
#include <cstring>

#include "../../include/msbwt_gpu.h"
#include "kernel_common.cuh"

namespace msbwt {

namespace {

constexpr uint32_t kNone = 0xffffffffu;
constexpr int kMaxRounds = 80;  // pointer-jumping rounds of a call: each of its two phases needs at most 33

__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t *__restrict__ keys, uint32_t n, uint64_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (keys[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// the per-thread counts of a CTA summed through shared memory, one atomic per CTA (a same-address atomic per thread
// would be aggregated across the warp by ptxas: a vote and a reduction)
__device__ __forceinline__ void cta_count(uint32_t *smem, uint32_t mine, unsigned long long *out) {
    smem[threadIdx.x] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int t = 0; t < kCountThreads; t++) sum += smem[t];
        if (sum) atomicAdd(out, sum);
    }
}

#define UNITIG_LOOP(i, n) for (uint32_t i = blockIdx.x * kCountThreads + threadIdx.x; i < (n); i += gridDim.x * kCountThreads)

// canonical mode: rc of every listed canonical k-mer, flagged unless it is a palindrome
__global__ void __launch_bounds__(kCountThreads)
unitig_revcomp_kernel(const uint64_t *__restrict__ keys, uint32_t n, uint32_t k, uint64_t *__restrict__ rc,
                      uint8_t *__restrict__ flag) {
    UNITIG_LOOP(i, n) {
        const uint64_t v = keys[i], r = revcomp_kmer(v, k);
        rc[i] = r;
        flag[i] = r != v;
    }
}

// one thread per node X: its successors in V; succ[X] = the one successor when outdeg(X) = 1, else kNone.  Every
// edge X -> Y adds 1 to indeg[Y] and writes pred[Y] = X, which is read only where indeg[Y] = 1 (a single writer).
__global__ void __launch_bounds__(kCountThreads)
unitig_link_kernel(const uint64_t *__restrict__ keys, uint32_t n, uint64_t mask, uint32_t *__restrict__ succ,
                   uint32_t *__restrict__ indeg, uint32_t *__restrict__ pred) {
    UNITIG_LOOP(i, n) {
        const uint64_t base = (keys[i] << 2) & mask;
        uint32_t j = lower_bound_u64(keys, n, base), outdeg = 0, s = kNone;
#pragma unroll
        for (uint32_t c = 0; c < 4; c++) {
            if (j < n && keys[j] == base + c) {
                outdeg++;
                s = j;
                atomicAdd(&indeg[j], 1u);
                pred[j] = i;
                j++;
            }
        }
        succ[i] = outdeg == 1 ? s : kNone;
    }
}

// prev[Y] = X along a compacted edge X -> Y (in place over pred)
__global__ void __launch_bounds__(kCountThreads)
unitig_prev_kernel(uint32_t n, const uint32_t *__restrict__ succ, const uint32_t *__restrict__ indeg,
                   uint32_t *__restrict__ pred) {
    UNITIG_LOOP(i, n) {
        uint32_t p = kNone;
        if (indeg[i] == 1) {
            const uint32_t x = pred[i];
            if (x != i && succ[x] == i) p = x;
        }
        pred[i] = p;
    }
}

// next[X] = Y along a compacted edge X -> Y (in place over succ; after unitig_prev_kernel has read succ)
__global__ void __launch_bounds__(kCountThreads)
unitig_next_kernel(uint32_t n, const uint32_t *__restrict__ indeg, uint32_t *__restrict__ succ) {
    UNITIG_LOOP(i, n) {
        const uint32_t s = succ[i];
        succ[i] = (s != kNone && s != i && indeg[s] == 1) ? s : kNone;
    }
}

// J = prev (a head points to itself), D = 1 (0 for a head); *unresolved += nodes whose J is not a head
__global__ void __launch_bounds__(kCountThreads)
unitig_rank_init_kernel(uint32_t n, const uint32_t *__restrict__ prev, uint32_t *__restrict__ J, uint32_t *__restrict__ D,
                        unsigned long long *__restrict__ unresolved) {
    __shared__ uint32_t smem[kCountThreads];
    uint32_t mine = 0;
    UNITIG_LOOP(i, n) {
        const uint32_t p = prev[i];
        J[i] = p == kNone ? i : p;
        D[i] = p != kNone;
        mine += p != kNone && prev[p] != kNone;
    }
    cta_count(smem, mine, unresolved);
}

// one synchronous Wyllie round: J2 = J o J, D2 = D + D o J
__global__ void __launch_bounds__(kCountThreads)
unitig_rank_step_kernel(uint32_t n, const uint32_t *__restrict__ prev, const uint32_t *__restrict__ J,
                        const uint32_t *__restrict__ D, uint32_t *__restrict__ J2, uint32_t *__restrict__ D2,
                        unsigned long long *__restrict__ unresolved) {
    __shared__ uint32_t smem[kCountThreads];
    uint32_t mine = 0;
    UNITIG_LOOP(i, n) {
        const uint32_t j = J[i];
        uint32_t j2 = j, d2 = D[i];
        if (prev[j] != kNone) {  // J[i] is not a head yet (a head has J = itself and D = 0)
            j2 = J[j];
            d2 += D[j];
            mine += prev[j2] != kNone;
        }
        J2[i] = j2;
        D2[i] = d2;
    }
    cta_count(smem, mine, unresolved);
}

// the nodes left unresolved lie on cycles: W = next on them (kNone elsewhere, in both buffers), M = the node's value
__global__ void __launch_bounds__(kCountThreads)
unitig_cycle_init_kernel(uint32_t n, const uint64_t *__restrict__ keys, const uint32_t *__restrict__ prev,
                         const uint32_t *__restrict__ next, const uint32_t *__restrict__ J, uint32_t *__restrict__ W,
                         uint32_t *__restrict__ W2, uint64_t *__restrict__ M) {
    UNITIG_LOOP(i, n) {
        const uint32_t w = prev[J[i]] != kNone ? next[i] : kNone;
        W[i] = W2[i] = w;
        M[i] = keys[i];
    }
}

// one doubling round over the cycles: W2 = W o W, M2 = min(M, M o W); *changed = 1 when a minimum moved
__global__ void __launch_bounds__(kCountThreads)
unitig_cycle_step_kernel(uint32_t n, const uint32_t *__restrict__ W, const uint64_t *__restrict__ M,
                         uint32_t *__restrict__ W2, uint64_t *__restrict__ M2, uint32_t *__restrict__ changed) {
    UNITIG_LOOP(i, n) {
        const uint32_t w = W[i];
        if (w == kNone) continue;
        const uint64_t m = M[i], mw = M[w];
        W2[i] = W[w];
        M2[i] = m < mw ? m : mw;
        if (mw < m) *changed = 1;
    }
}

// every cycle is cut before its minimum node, which becomes a head (J, D and prev reset; its predecessor a tail);
// the other cycle nodes restart ranking from prev.  keep[head] = whether canonical mode keeps the cycle:
// min(C) <= min(rc C), where rc C is the cycle holding rc(min(C)) (1 in plain mode).
__global__ void __launch_bounds__(kCountThreads)
unitig_cut_kernel(uint32_t n, uint32_t k, int canonical, const uint64_t *__restrict__ keys, const uint32_t *__restrict__ W,
                  const uint64_t *__restrict__ M, uint32_t *__restrict__ prev, uint32_t *__restrict__ next,
                  uint32_t *__restrict__ J, uint32_t *__restrict__ D, uint8_t *__restrict__ keep) {
    UNITIG_LOOP(i, n) {
        if (W[i] == kNone) continue;
        const uint64_t m = M[i];
        if (keys[i] == m) {
            J[i] = i;
            D[i] = 0;
            prev[i] = kNone;
            keep[i] = !canonical || m <= M[lower_bound_u64(keys, n, revcomp_kmer(m, k))];  // V holds rc(m)
        } else {
            J[i] = prev[i];
            D[i] = 1;
        }
        if (keys[next[i]] == m) next[i] = kNone;
    }
}

// each node's count goes to its head's sum; each tail gives its head the unitig's length (0 when canonical mode
// drops it) and its flag.  keep[head] is 2 for a linear unitig, else what unitig_cut_kernel decided.
__global__ void __launch_bounds__(kCountThreads)
unitig_tail_kernel(uint32_t n, uint32_t k, int canonical, const uint64_t *__restrict__ keys,
                   const uint64_t *__restrict__ counts, const uint32_t *__restrict__ next, const uint32_t *__restrict__ J,
                   const uint32_t *__restrict__ D, const uint8_t *__restrict__ keep,
                   unsigned long long *__restrict__ sums, uint64_t *__restrict__ lens, uint32_t *__restrict__ kept) {
    UNITIG_LOOP(i, n) {
        const uint32_t h = J[i];
        atomicAdd(&sums[h], (unsigned long long)counts[i]);
        if (next[i] == kNone) {
            const uint8_t kc = keep[h];
            const bool ok = kc != 2 ? kc != 0 : (!canonical || keys[h] <= revcomp_kmer(keys[i], k));
            lens[h] = ok ? (uint64_t)D[i] + k : 0;
            kept[h] = ok;
        }
    }
}

// the symbols: A,C,G,T = 1,2,3,5 for codes 0..3
__device__ __forceinline__ uint8_t code_sym(uint64_t c) { return (uint8_t)(c + 1 + (c == 3)); }

// every node of a kept unitig writes its last symbol; a head writes its whole k-mer, its offset and count sum
__global__ void __launch_bounds__(kCountThreads)
unitig_emit_kernel(uint32_t n, uint32_t k, const uint64_t *__restrict__ keys, const uint32_t *__restrict__ J,
                   const uint32_t *__restrict__ D, const uint32_t *__restrict__ kept, const uint64_t *__restrict__ offs,
                   const uint32_t *__restrict__ idx, const unsigned long long *__restrict__ sums,
                   uint8_t *__restrict__ syms, uint64_t *__restrict__ out_offsets, uint64_t *__restrict__ out_sums) {
    UNITIG_LOOP(i, n) {
        const uint32_t h = J[i];
        if (!kept[h]) continue;
        const uint64_t o = offs[h], x = keys[i];
        syms[o + k - 1 + D[i]] = code_sym(x & 3);
        if (i == h) {
            for (uint32_t j = 0; j + 1 < k; j++) syms[o + j] = code_sym((x >> (2 * (k - 1 - j))) & 3);
            out_offsets[idx[h]] = o;
            out_sums[idx[h]] = sums[h];
        }
    }
}

#define U_TRY(e) CU_TRY_IN("unitigs: ", e)

// malloc'd host outputs, released unless handed to the caller
struct HostOut {
    uint8_t *syms = nullptr;
    uint64_t *offsets = nullptr, *sums = nullptr;
    ~HostOut() {
        free(syms);
        free(offsets);
        free(sums);
    }
};

}  // namespace

int unitigs_on_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                      uint8_t **syms, uint64_t **offsets, uint64_t **count_sums, uint64_t *n_unitigs) {
    // listed k-mers (canonical: pairs), from a histogram-only pass
    uint64_t listed = 0;
    if (int rc = kmer_spectrum_on_device(device, ix, lanes, canonical, k, min_count, nullptr, 0, nullptr, nullptr, &listed);
        rc != MSBWT_OK)
        return rc;
    if (!listed) return MSBWT_OK;
    const uint64_t cap = canonical ? 2 * listed : listed;
    if (cap >= kNone) return fail(MSBWT_ENOMEM, "unitigs: the graph has 2^32 nodes or more (node ids are 32-bit)");

    HostOut host;  // declared first: released after the stream has drained
    DeviceScratch scratch;
    OwnStream st;
    U_TRY(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    // keys / counts and their sort alternates; after the sort the alternates hold indeg, then the ranking's J / D pairs
    uint64_t *keys[2], *counts[2];
    for (int b = 0; b < 2; b++) {
        U_TRY(scratch.alloc(&keys[b], cap));
        U_TRY(scratch.alloc(&counts[b], cap));
    }
    uint64_t n64 = 0;
    if (int rc = kmer_spectrum_to_device(device, ix, lanes, canonical, k, min_count,
                                         DeviceKmerList{keys[0], counts[0], listed}, &n64);
        rc != MSBWT_OK)
        return rc;
    if (n64 != listed) return fail(MSBWT_ECUDA, "unitigs: the listing and the sizing pass disagree");
    uint32_t n = (uint32_t)listed;

    unsigned long long *d_cnt = nullptr;  // [0] selected, [1 + r] unresolved after ranking round r
    U_TRY(scratch.alloc(&d_cnt, 2 + kMaxRounds));
    U_TRY(cudaMemsetAsync(d_cnt, 0, (2 + kMaxRounds) * sizeof(unsigned long long), st.s));
    uint32_t *succ = nullptr, *pred = nullptr;  // -> next, prev; pred has room for the emission's n + 1 flags
    U_TRY(scratch.alloc(&succ, cap));
    U_TRY(scratch.alloc(&pred, cap + 1));
    auto grid = [&](const void *kern) { return persistent_grid(device, kern, kCountThreads, n, kCountThreads); };

    size_t temp_bytes = 0, need = 0;
    U_TRY(cub::DeviceSelect::Flagged(nullptr, need, (const uint64_t *)nullptr, (const uint8_t *)nullptr, (uint64_t *)nullptr,
                                     (unsigned long long *)nullptr, (uint32_t)cap, st.s));
    temp_bytes = std::max(temp_bytes, need);
    {
        cub::DoubleBuffer<uint64_t> kb(keys[0], keys[1]), cb(counts[0], counts[1]);
        U_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, kb, cb, (uint32_t)cap, 0, 2 * (int)k, st.s));
    }
    temp_bytes = std::max(temp_bytes, need);
    U_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, (uint64_t *)nullptr, (uint64_t *)nullptr, cap + 1, st.s));
    temp_bytes = std::max(temp_bytes, need);
    U_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, (uint32_t *)nullptr, (uint32_t *)nullptr, cap + 1, st.s));
    temp_bytes = std::max(temp_bytes, need);
    void *d_temp = nullptr;
    U_TRY(scratch.alloc((char **)&d_temp, temp_bytes));

    if (canonical) {  // append rc of every non-palindromic canonical k-mer
        uint8_t *flag = (uint8_t *)succ;
        unitig_revcomp_kernel<<<grid((const void *)unitig_revcomp_kernel), kCountThreads, 0, st.s>>>(keys[0], n, k, keys[1], flag);
        U_TRY(cudaGetLastError());
        U_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)keys[1], (const uint8_t *)flag,
                                         keys[0] + n, d_cnt, n, st.s));
        U_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)counts[0], (const uint8_t *)flag,
                                         counts[0] + n, d_cnt, n, st.s));
        g_launches += 5;  // the reverse complements + CUB's init and select kernels, twice
        unsigned long long added = 0;
        U_TRY(cudaMemcpyAsync(&added, d_cnt, sizeof(added), cudaMemcpyDeviceToHost, st.s));
        U_TRY(cudaStreamSynchronize(st.s));
        n += (uint32_t)added;
    }

    // nodes in ascending value: node id = rank
    cub::DoubleBuffer<uint64_t> kb(keys[0], keys[1]), cb(counts[0], counts[1]);
    U_TRY(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, kb, cb, n, 0, 2 * (int)k, st.s));
    g_launches++;  // counted as one call: how many kernels CUB issues depends on n
    const uint64_t *K = kb.Current(), *Cn = cb.Current();
    uint32_t *alt[2] = {(uint32_t *)kb.Alternate(), (uint32_t *)cb.Alternate()};  // 8 bytes per node each: J | D

    // links
    const uint64_t mask = k == 32 ? ~0ull : (1ull << (2 * k)) - 1;
    uint32_t *indeg = alt[0], *next = succ, *prev = pred;
    U_TRY(cudaMemsetAsync(indeg, 0, (uint64_t)n * sizeof(uint32_t), st.s));
    unitig_link_kernel<<<grid((const void *)unitig_link_kernel), kCountThreads, 0, st.s>>>(K, n, mask, succ, indeg, pred);
    U_TRY(cudaGetLastError());
    unitig_prev_kernel<<<grid((const void *)unitig_prev_kernel), kCountThreads, 0, st.s>>>(n, succ, indeg, pred);
    U_TRY(cudaGetLastError());
    unitig_next_kernel<<<grid((const void *)unitig_next_kernel), kCountThreads, 0, st.s>>>(n, indeg, succ);
    U_TRY(cudaGetLastError());
    g_launches += 3;

    // ranking: pair p holds the current J (first n words) and D (next n words)
    int p = 0, round = 0;
    auto J = [&](int b) { return alt[b]; };
    auto D = [&](int b) { return alt[b] + n; };
    auto unresolved_after = [&](int r, unsigned long long *u) -> int {
        U_TRY(cudaMemcpyAsync(u, d_cnt + 1 + r, sizeof(*u), cudaMemcpyDeviceToHost, st.s));
        U_TRY(cudaStreamSynchronize(st.s));
        return MSBWT_OK;
    };
    unitig_rank_init_kernel<<<grid((const void *)unitig_rank_init_kernel), kCountThreads, 0, st.s>>>(n, prev, J(0), D(0), d_cnt + 1);
    U_TRY(cudaGetLastError());
    g_launches++;
    unsigned long long before = 0;
    if (int rc = unresolved_after(0, &before); rc != MSBWT_OK) return rc;
    // rounds until the number of unresolved nodes stops falling (until it is 0 when `exact`)
    auto rank_rounds = [&](bool exact) -> int {
        while (before > 0) {
            if (round + 1 >= kMaxRounds) return fail(MSBWT_ECUDA, "unitigs: list ranking did not converge");
            round++;
            unitig_rank_step_kernel<<<grid((const void *)unitig_rank_step_kernel), kCountThreads, 0, st.s>>>(
                n, prev, J(p), D(p), J(p ^ 1), D(p ^ 1), d_cnt + 1 + round);
            U_TRY(cudaGetLastError());
            g_launches++;
            p ^= 1;
            unsigned long long now = 0;
            if (int rc = unresolved_after(round, &now); rc != MSBWT_OK) return rc;
            if (!exact && now == before) break;
            before = now;
        }
        return MSBWT_OK;
    };
    if (int rc = rank_rounds(false); rc != MSBWT_OK) return rc;

    uint8_t *keep = nullptr;  // per head: 2 = linear, else the cycle's canonical keep flag
    U_TRY(scratch.alloc(&keep, n));
    U_TRY(cudaMemsetAsync(keep, 2, n, st.s));
    if (before > 0) {  // cycles: find each one's minimum, cut before it, rank the cut cycles
        DeviceScratch cyc;
        uint64_t *M[2];
        U_TRY(cyc.alloc(&M[0], n));
        U_TRY(cyc.alloc(&M[1], n));
        uint32_t *W[2] = {J(p ^ 1), D(p ^ 1)}, *d_changed = nullptr;
        U_TRY(cyc.alloc(&d_changed, 1));
        unitig_cycle_init_kernel<<<grid((const void *)unitig_cycle_init_kernel), kCountThreads, 0, st.s>>>(
            n, K, prev, next, J(p), W[0], W[1], M[0]);
        U_TRY(cudaGetLastError());
        g_launches++;
        int c = 0;
        for (int r = 0;; r++) {
            if (r >= kMaxRounds) return fail(MSBWT_ECUDA, "unitigs: cycle minima did not converge");
            uint32_t changed = 0;
            U_TRY(cudaMemsetAsync(d_changed, 0, sizeof(uint32_t), st.s));
            unitig_cycle_step_kernel<<<grid((const void *)unitig_cycle_step_kernel), kCountThreads, 0, st.s>>>(
                n, W[c], M[c], W[c ^ 1], M[c ^ 1], d_changed);
            U_TRY(cudaGetLastError());
            g_launches++;
            c ^= 1;
            U_TRY(cudaMemcpyAsync(&changed, d_changed, sizeof(changed), cudaMemcpyDeviceToHost, st.s));
            U_TRY(cudaStreamSynchronize(st.s));
            if (!changed) break;
        }
        unitig_cut_kernel<<<grid((const void *)unitig_cut_kernel), kCountThreads, 0, st.s>>>(
            n, k, canonical, K, W[c], M[c], prev, next, J(p), D(p), keep);
        U_TRY(cudaGetLastError());
        g_launches++;
        U_TRY(cudaStreamSynchronize(st.s));  // before the cycle scratch is freed
        before = 1;  // the cut cycles' nodes are unresolved again
        if (int rc = rank_rounds(true); rc != MSBWT_OK) return rc;
    }

    // emission.  The free J / D pair takes the count sums; prev (ranking is done) the kept-head flags.
    const uint32_t *Jf = J(p), *Df = D(p);
    unsigned long long *sums = (unsigned long long *)alt[p ^ 1];
    uint32_t *kept = prev, *idx = nullptr;
    uint64_t *lens = nullptr;
    U_TRY(scratch.alloc(&lens, (uint64_t)n + 1));
    U_TRY(scratch.alloc(&idx, (uint64_t)n + 1));
    U_TRY(cudaMemsetAsync(sums, 0, (uint64_t)n * sizeof(uint64_t), st.s));
    U_TRY(cudaMemsetAsync(lens, 0, ((uint64_t)n + 1) * sizeof(uint64_t), st.s));
    U_TRY(cudaMemsetAsync(kept, 0, ((uint64_t)n + 1) * sizeof(uint32_t), st.s));
    unitig_tail_kernel<<<grid((const void *)unitig_tail_kernel), kCountThreads, 0, st.s>>>(
        n, k, canonical, K, Cn, next, Jf, Df, keep, sums, lens, kept);
    U_TRY(cudaGetLastError());
    U_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, lens, (uint64_t)n + 1, st.s));  // in place: offsets
    U_TRY(cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, (const uint32_t *)kept, idx, (uint64_t)n + 1, st.s));
    g_launches += 5;  // the tail kernel + CUB's init and scan kernels, twice
    uint64_t total = 0;
    uint32_t n_out = 0;
    U_TRY(cudaMemcpyAsync(&total, lens + n, sizeof(total), cudaMemcpyDeviceToHost, st.s));
    U_TRY(cudaMemcpyAsync(&n_out, idx + n, sizeof(n_out), cudaMemcpyDeviceToHost, st.s));
    U_TRY(cudaStreamSynchronize(st.s));
    if (!n_out) return MSBWT_OK;  // canonical mode keeps one of every pair: never empty when V is not
    scratch.release((void *)Cn);  // the counts are summed
    uint8_t *d_syms = nullptr;
    uint64_t *d_off = nullptr, *d_sums = nullptr;
    U_TRY(scratch.alloc(&d_syms, total));
    U_TRY(scratch.alloc(&d_off, (uint64_t)n_out + 1));
    U_TRY(scratch.alloc(&d_sums, n_out));
    unitig_emit_kernel<<<grid((const void *)unitig_emit_kernel), kCountThreads, 0, st.s>>>(
        n, k, K, Jf, Df, kept, lens, idx, sums, d_syms, d_off, d_sums);
    U_TRY(cudaGetLastError());
    g_launches++;
    U_TRY(cudaMemcpyAsync(d_off + n_out, &total, sizeof(total), cudaMemcpyHostToDevice, st.s));

    host.syms = (uint8_t *)malloc(total);
    host.offsets = (uint64_t *)malloc(((uint64_t)n_out + 1) * sizeof(uint64_t));
    host.sums = (uint64_t *)malloc((uint64_t)n_out * sizeof(uint64_t));
    if (!host.syms || !host.offsets || !host.sums) return fail(MSBWT_ENOMEM, "unitigs: host buffers for the result");
    U_TRY(cudaMemcpyAsync(host.syms, d_syms, total, cudaMemcpyDeviceToHost, st.s));
    U_TRY(cudaMemcpyAsync(host.offsets, d_off, ((uint64_t)n_out + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    U_TRY(cudaMemcpyAsync(host.sums, d_sums, (uint64_t)n_out * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    U_TRY(cudaStreamSynchronize(st.s));
    *syms = host.syms;
    *offsets = host.offsets;
    *count_sums = host.sums;
    host.syms = nullptr;
    host.offsets = host.sums = nullptr;
    *n_unitigs = n_out;
    return MSBWT_OK;
}

}  // namespace msbwt
