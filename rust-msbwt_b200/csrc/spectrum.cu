// spectrum.cu -- the k-mer spectrum of an index and its solid k-mers (msbwt_kmer_spectrum).
//
// The index holds every k-mer of its read set with its count, and an FM-index lists them natively: a backward search
// from the empty string extends every surviving range by A, C, G and T (rank_fanout4, device_rank.cuh: the blocks
// holding l and h are fetched once for the four symbols) and drops a child whose width is below min_count.  The drop
// is exact because constrain_range never widens a range.  A node at depth d is a range [l, h) and the string X of its
// d symbols (X is a suffix of the k-mers below it); with the list requested it also carries X as 2-bit codes,
// v = sum of code(X_j) << 2 (d - 1 - j), so a child that prepends symbol c has value v | c << 2d.
//
// Traversal: depth first over slices, with a bounded frontier.
//   buffers : one per depth d = 0..k-1, each holding the children of ONE slice of depth d-1 (at most 4 B of them;
//             depth 0 is the root [0, N)).
//   host    : take the next slice of <= B nodes from the deepest buffer that is not exhausted, expand it with one
//             kernel (four children + a survivor flag each) and stable-compact the survivors over buffer d + 1 (CUB
//             DeviceSelect::Flagged), which was exhausted; read back how many there are.  At d + 1 == k the survivors
//             are emitted instead: histogram (per-CTA bins in shared memory, flushed with atomics) and, when asked
//             for, (k-mer, count) compacted into a device staging buffer that is copied to a growing host buffer
//             whenever it could not take another slice.
//   order   : children are laid out parent-major, A < C < G < T, the compaction keeps their order, and all
//             descendants of a slice are emitted before the next slice of its depth is taken: the list comes out in
//             co-lexicographic order (by the last symbol first) without a sort.
//   memory  : independent of N and of the number of k-mers (see msbwt_gpu.h).  Nodes at one depth are disjoint ranges
//             of width >= min_count, so no buffer needs more than N / min_count entries either: small indexes
//             allocate little.
// Only the one-step blocks are read, which every index has, whatever other images it carries.
//
// Canonical spectrum (msbwt_kmer_spectrum_canonical): the same walk with the k-mer values, pruned at
// ceil(min_count / 2), stages every k-mer Y it lists.  Each full staging buffer (and the last one) is resolved on the
// device: rc(Y) of every staged Y, count_kmer(rc Y) through the query path (launch_seed_u64 + launch_count_packed,
// so every image of the index is read there), then canonical_resolve_kernel keeps one member of every pair
// {Y, rc Y} whose summed count reaches min_count.  Batches of up to 2^22 lookups keep the query kernels at their
// bulk rate, where the walk's slices can be small.
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/msbwt_gpu.h"
#include "device_rank.cuh"
#include "kernel_common.cuh"

namespace msbwt {

namespace {

constexpr uint64_t kSliceParents = 1ull << 20;  // B: parents expanded per launch
constexpr uint64_t kStagingKmers = 1ull << 22;  // emitted (k-mer, count) pairs held on the device between host copies
constexpr uint32_t kSmemBins = 4096;            // histogram bins privatized per CTA (the rest go to global atomics)

template <class P, bool LIST> struct Node { P l, h; uint64_t v; };
template <class P> struct Node<P, false> { P l, h; };

// one thread per parent: its four children and their survivor flags (one 4-byte store of flags per parent)
template <bool WIDE, bool LIST>
__global__ void __launch_bounds__(kCountThreads, 4)
spectrum_expand_kernel(IndexView ix, const Node<typename Pos<WIDE>::type, LIST> *__restrict__ parents, uint32_t n,
                       uint32_t shift, uint64_t min_count, Node<typename Pos<WIDE>::type, LIST> *__restrict__ child,
                       uint32_t *__restrict__ keep) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    for (uint32_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += threads) {
        const Node<P, LIST> p = parents[i];
        P ol[4], oh[4];
        rank_fanout4<WIDE>(ix, cb, p.l, p.h, ol, oh);
        uint32_t flags = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            Node<P, LIST> c;
            c.l = ol[j];
            c.h = oh[j];
            if constexpr (LIST) c.v = p.v | ((uint64_t)j << shift);
            child[4 * (uint64_t)i + j] = c;
            flags |= (uint32_t)((uint64_t)(oh[j] - ol[j]) >= min_count) << (8 * j);
        }
        keep[i] = flags;
    }
}

// the last step: survivors are k-mers.  bins[0, smem_bins) = this CTA's histogram entries below smem_bins (the rest
// go straight to global atomics); with LIST every child's (k-mer, count) and flag go out for the compaction
template <bool WIDE, bool LIST>
__global__ void __launch_bounds__(kCountThreads, 4)
spectrum_emit_kernel(IndexView ix, const Node<typename Pos<WIDE>::type, LIST> *__restrict__ parents, uint32_t n,
                     uint32_t shift, uint64_t min_count, uint32_t nbins, uint32_t smem_bins,
                     unsigned long long *__restrict__ hist, unsigned long long *__restrict__ n_kmers,
                     uint64_t *__restrict__ kmer_out, uint64_t *__restrict__ count_out, uint32_t *__restrict__ keep) {
    using P = typename Pos<WIDE>::type;
    extern __shared__ uint32_t bins[];
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    __shared__ uint32_t survivors[kCountThreads];
    for (uint32_t t = threadIdx.x; t < smem_bins; t += blockDim.x) bins[t] = 0;
    __syncthreads();
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    uint32_t mine = 0;
    for (uint32_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += threads) {
        const Node<P, LIST> p = parents[i];
        P ol[4], oh[4];
        rank_fanout4<WIDE>(ix, cb, p.l, p.h, ol, oh);
        uint32_t flags = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint64_t cnt = (uint64_t)(oh[j] - ol[j]);
            const bool ok = cnt >= min_count;
            if (ok) {
                mine++;
                if (nbins) {
                    const uint32_t b = (uint32_t)min(cnt, (uint64_t)(nbins - 1));
                    if (b < smem_bins) atomicAdd(&bins[b], 1u);
                    else atomicAdd(&hist[b], 1ull);
                }
            }
            if constexpr (LIST) {
                kmer_out[4 * (uint64_t)i + j] = p.v | ((uint64_t)j << shift);
                count_out[4 * (uint64_t)i + j] = cnt;
                flags |= (uint32_t)ok << (8 * j);
            }
        }
        if constexpr (LIST) keep[i] = flags;
    }
    // survivors summed through shared memory, not with a same-address atomic: ptxas would aggregate that one across
    // the warp (a vote and a reduction after the divergent loop), and the kernels here keep no warp collectives
    survivors[threadIdx.x] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int t = 0; t < kCountThreads; t++) sum += survivors[t];
        if (sum) atomicAdd(n_kmers, sum);
    }
    for (uint32_t t = threadIdx.x; t < smem_bins; t += blockDim.x)
        if (bins[t]) atomicAdd(&hist[t], (unsigned long long)bins[t]);
}

__global__ void __launch_bounds__(kCountThreads)
canonical_revcomp_kernel(const uint64_t *__restrict__ kmers, uint32_t n, uint32_t k, uint64_t *__restrict__ rc) {
    for (uint32_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += gridDim.x * kCountThreads)
        rc[i] = revcomp_kmer(kmers[i], k);
}

// One staged batch of the canonical spectrum: Y = kmers[i] with count_kmer(Y) = counts[i] >= half, and
// rc_counts[i] = count_kmer(rc Y).  Y stands for its pair {Y, rc Y} when it is the canonical member, or when rc Y
// was not listed (count below half), so exactly one listed member of every pair stands for it.  Its canonical count
// C is c_Y + c_rc, or c_Y alone for a palindrome.  With C >= min_count the pair is binned (as in spectrum_emit_kernel)
// and counted, and with `keep` it is written in place over rc_kmers[i] / rc_counts[i] as (canon Y, C) and flagged
// for the compaction.
__global__ void __launch_bounds__(kCountThreads)
canonical_resolve_kernel(const uint64_t *__restrict__ kmers, const uint64_t *__restrict__ counts, uint32_t n, uint32_t k,
                         uint64_t half, uint64_t min_count, uint32_t nbins, uint32_t smem_bins,
                         unsigned long long *__restrict__ hist, unsigned long long *__restrict__ n_kmers,
                         uint64_t *__restrict__ rc_kmers, uint64_t *__restrict__ rc_counts, uint8_t *__restrict__ keep) {
    extern __shared__ uint32_t bins[];
    __shared__ uint32_t survivors[kCountThreads];
    for (uint32_t t = threadIdx.x; t < smem_bins; t += blockDim.x) bins[t] = 0;
    __syncthreads();
    uint32_t mine = 0;
    for (uint32_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += gridDim.x * kCountThreads) {
        const uint64_t y = kmers[i], r = revcomp_kmer(y, k), c_rc = rc_counts[i];
        const uint64_t c = y == r ? counts[i] : counts[i] + c_rc;
        const bool ok = (y <= r || c_rc < half) && c >= min_count;
        if (ok) {
            mine++;
            if (nbins) {
                const uint32_t b = (uint32_t)min(c, (uint64_t)(nbins - 1));
                if (b < smem_bins) atomicAdd(&bins[b], 1u);
                else atomicAdd(&hist[b], 1ull);
            }
        }
        if (keep) {
            rc_kmers[i] = min(y, r);
            rc_counts[i] = c;
            keep[i] = ok;
        }
    }
    survivors[threadIdx.x] = mine;  // summed through shared memory, as in spectrum_emit_kernel
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int t = 0; t < kCountThreads; t++) sum += survivors[t];
        if (sum) atomicAdd(n_kmers, sum);
    }
    for (uint32_t t = threadIdx.x; t < smem_bins; t += blockDim.x)
        if (bins[t]) atomicAdd(&hist[t], (unsigned long long)bins[t]);
}

#define S_TRY(e) CU_TRY_IN("kmer spectrum: ", e)

// a malloc'd host array that grows by doubling; released unless handed to the caller
struct HostU64 {
    uint64_t *p = nullptr;
    uint64_t cap = 0;
    ~HostU64() { free(p); }
    bool reserve(uint64_t n) {
        if (n <= cap) return true;
        const uint64_t want = std::max<uint64_t>(n, 2 * cap);
        void *q = realloc(p, want * sizeof(uint64_t));
        if (!q) return false;
        p = (uint64_t *)q;
        cap = want;
        return true;
    }
};

uint64_t slice_parents() {
    // MSBWT_SPECTRUM_SLICE: a smaller B, so that tests reach many slices at several depths on small indexes
    if (const char *env = getenv("MSBWT_SPECTRUM_SLICE")) {
        const long long v = atoll(env);
        if (v >= 1 && (uint64_t)v <= kSliceParents) return (uint64_t)v;
    }
    return kSliceParents;
}

// `canonical` (LIST only): the walk lists every k-mer with count >= walk_min and stages it; each staged batch is then
// resolved into canonical pairs (canonical_resolve_kernel), which alone are binned, counted and, with `kmers`, listed
// `sink` (LIST only): the list goes to these device arrays instead of host buffers (kmers stays null)
template <bool WIDE, bool LIST>
int spectrum_run(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                 uint64_t *hist, uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers,
                 const DeviceKmerList *sink = nullptr) {
    using P = typename Pos<WIDE>::type;
    using NodeT = Node<P, LIST>;
    const uint64_t B = slice_parents();
    const bool want_list = kmers != nullptr || sink != nullptr;
    // A pair with C >= min_count has a member with count >= ceil(min_count / 2); a pair whose members both count less
    // has C <= min_count - 1.  So the canonical walk prunes at ceil(min_count / 2), exactly.
    const uint64_t walk_min = canonical ? min_count / 2 + (min_count & 1) : min_count;  // (min_count + 1) / 2 wraps at 2^64 - 1
    // survivors of one slice: at most 4 per parent, and at most N / walk_min (disjoint ranges of that width)
    const uint64_t cap = std::max<uint64_t>(1, std::min<uint64_t>(4 * B, ix.total / walk_min));
    const uint64_t staging = LIST ? std::max(cap, std::min(kStagingKmers, ix.total / walk_min)) : 0;
    const uint32_t smem_bins = std::min(nbins, kSmemBins);
    // the walk's emission bins nothing in canonical mode: the resolve kernel does
    const uint32_t emit_bins = canonical ? 0 : nbins, emit_smem_bins = canonical ? 0 : smem_bins;

    HostU64 out_kmers, out_counts;  // declared first: released after the stream has drained
    DeviceScratch scratch;
    OwnStream st;
    S_TRY(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    std::vector<NodeT *> level(k, nullptr);  // level[d]: the nodes of depth d (d >= 1: the children of one slice)
    S_TRY(scratch.alloc(&level[0], 1));
    for (uint32_t d = 1; d < k; d++) S_TRY(scratch.alloc(&level[d], cap));
    // one slice's children before the compaction (or, at the last step, its k-mers and counts), and their flags
    void *d_children = nullptr;
    uint32_t *d_keep = nullptr;
    const uint64_t child_bytes = 4 * std::min(B, cap) * std::max(sizeof(NodeT), LIST ? 2 * sizeof(uint64_t) : 0);
    S_TRY(scratch.alloc((char **)&d_children, child_bytes));
    S_TRY(scratch.alloc(&d_keep, std::min(B, cap)));
    unsigned long long *d_hist = nullptr, *d_count = nullptr;
    S_TRY(scratch.alloc(&d_hist, std::max<uint32_t>(nbins, 1)));
    // [0] k-mers emitted, [1] survivors of the last compaction, [2] k-mers the canonical walk staged
    S_TRY(scratch.alloc(&d_count, 3));
    uint64_t *d_stage_kmers = nullptr, *d_stage_counts = nullptr;
    if (LIST) {
        S_TRY(scratch.alloc(&d_stage_kmers, staging));
        S_TRY(scratch.alloc(&d_stage_counts, staging));
    }
    // canonical: the staged k-mers' reverse complements and their counts (then the resolved pairs, in place), the
    // resolve flags and the query path's scratch for one staged batch
    uint64_t *d_rc_kmers = nullptr, *d_rc_counts = nullptr, *d_packed = nullptr;
    uint8_t *d_resolved = nullptr;
    if (canonical) {
        S_TRY(scratch.alloc(&d_rc_kmers, staging));
        S_TRY(scratch.alloc(&d_rc_counts, staging));
        S_TRY(scratch.alloc(&d_resolved, staging));
        S_TRY(scratch.alloc(&d_packed, packed_layout(ix, k, staging).total()));
    }
    size_t temp_bytes = 0, need = 0;
    const int max_items = (int)(4 * std::min(B, cap));
    S_TRY(cub::DeviceSelect::Flagged(nullptr, need, (const NodeT *)nullptr, (const uint8_t *)nullptr, (NodeT *)nullptr,
                                     (unsigned long long *)nullptr, max_items, st.s));
    temp_bytes = std::max(temp_bytes, need);
    if (LIST) {
        S_TRY(cub::DeviceSelect::Flagged(nullptr, need, (const uint64_t *)nullptr, (const uint8_t *)nullptr,
                                         (uint64_t *)nullptr, (unsigned long long *)nullptr,
                                         canonical ? std::max(max_items, (int)staging) : max_items, st.s));
        temp_bytes = std::max(temp_bytes, need);
    }
    void *d_temp = nullptr;
    S_TRY(scratch.alloc((char **)&d_temp, temp_bytes));

    NodeT root{};
    root.l = 0;
    root.h = (P)ix.total;
    S_TRY(cudaMemcpyAsync(level[0], &root, sizeof(NodeT), cudaMemcpyHostToDevice, st.s));
    S_TRY(cudaMemsetAsync(d_hist, 0, std::max<uint32_t>(nbins, 1) * sizeof(unsigned long long), st.s));
    S_TRY(cudaMemsetAsync(d_count, 0, 3 * sizeof(unsigned long long), st.s));

    const unsigned grid_expand = persistent_grid(device, (const void *)spectrum_expand_kernel<WIDE, LIST>, kCountThreads,
                                                 std::min(B, cap), kCountThreads);
    const unsigned grid_emit = persistent_grid(device, (const void *)spectrum_emit_kernel<WIDE, LIST>, kCountThreads,
                                               std::min(B, cap), kCountThreads);
    const unsigned grid_resolve = canonical ? persistent_grid(device, (const void *)canonical_resolve_kernel,
                                                              kCountThreads, staging, kCountThreads) : 0;
    const size_t emit_smem = std::max<uint32_t>(emit_smem_bins, 1) * sizeof(uint32_t);
    const size_t resolve_smem = std::max<uint32_t>(smem_bins, 1) * sizeof(uint32_t);
    const bool with_b = canonical && packed_batch_needs_list_b(ix, k);
    std::vector<uint64_t> fill(k, 0), next(k, 0);
    fill[0] = 1;
    uint64_t staged = 0, listed = 0;
    auto flush = [&]() -> int {
        if (!staged) return MSBWT_OK;
        if (sink) {
            if (listed + staged > sink->cap) return fail(MSBWT_ECUDA, "kmer spectrum: more k-mers than the sizing pass found");
            S_TRY(cudaMemcpyAsync(sink->kmers + listed, d_stage_kmers, staged * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st.s));
            S_TRY(cudaMemcpyAsync(sink->counts + listed, d_stage_counts, staged * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st.s));
            S_TRY(cudaStreamSynchronize(st.s));  // the staging buffers are refilled next
            listed += staged;
            staged = 0;
            return MSBWT_OK;
        }
        if (!out_kmers.reserve(listed + staged) || !out_counts.reserve(listed + staged))
            return fail(MSBWT_ENOMEM, "kmer spectrum: host buffer for the k-mer list");
        S_TRY(cudaMemcpyAsync(out_kmers.p + listed, d_stage_kmers, staged * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
        S_TRY(cudaMemcpyAsync(out_counts.p + listed, d_stage_counts, staged * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
        S_TRY(cudaStreamSynchronize(st.s));
        listed += staged;
        staged = 0;
        return MSBWT_OK;
    };
    // canonical: count the staged k-mers' reverse complements on the query path, resolve the pairs, and with the list
    // compact the emitted ones into the staging buffers for flush()
    auto resolve = [&]() -> int {
        if (!staged) return MSBWT_OK;
        const uint32_t n = (uint32_t)staged;
        staged = 0;
        const unsigned g = std::min<unsigned>(grid_resolve, (n + kCountThreads - 1) / kCountThreads);
        canonical_revcomp_kernel<<<g, kCountThreads, 0, st.s>>>(d_stage_kmers, n, k, d_rc_kmers);
        S_TRY(cudaGetLastError());
        S_TRY(launch_seed_u64(ix, d_rc_kmers, k, n, d_packed, d_rc_counts, st.s));
        S_TRY(launch_count_packed(device, ix, lanes, d_packed, k, n, d_rc_counts, st.s, with_b));
        canonical_resolve_kernel<<<g, kCountThreads, resolve_smem, st.s>>>(
            d_stage_kmers, d_stage_counts, n, k, walk_min, min_count, nbins, smem_bins, d_hist, d_count, d_rc_kmers,
            d_rc_counts, want_list ? d_resolved : nullptr);
        S_TRY(cudaGetLastError());
        g_launches += 2;  // reverse complements, resolve (the seed and search wrappers count theirs)
        if (!want_list) return MSBWT_OK;
        S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)d_rc_kmers, (const uint8_t *)d_resolved,
                                         d_stage_kmers, d_count + 1, (int)n, st.s));
        S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)d_rc_counts, (const uint8_t *)d_resolved,
                                         d_stage_counts, d_count + 1, (int)n, st.s));
        g_launches += 4;
        unsigned long long emitted = 0;
        S_TRY(cudaMemcpyAsync(&emitted, d_count + 1, sizeof(emitted), cudaMemcpyDeviceToHost, st.s));
        S_TRY(cudaStreamSynchronize(st.s));
        staged = emitted;
        return flush();
    };
    auto drain = [&]() { return canonical ? resolve() : flush(); };
    for (;;) {
        int d = (int)k - 1;
        while (d >= 0 && next[d] == fill[d]) d--;
        if (d < 0) break;
        const uint32_t m = (uint32_t)std::min(B, fill[d] - next[d]);
        const NodeT *slice = level[d] + next[d];
        next[d] += m;
        const uint32_t shift = 2u * (uint32_t)d;
        const unsigned grid = std::min<unsigned>(grid_expand, (m + kCountThreads - 1) / kCountThreads);
        if ((uint32_t)d + 1 < k) {
            NodeT *children = (NodeT *)d_children;
            spectrum_expand_kernel<WIDE, LIST><<<grid, kCountThreads, 0, st.s>>>(ix, slice, m, shift, walk_min, children, d_keep);
            S_TRY(cudaGetLastError());
            S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const NodeT *)children, (const uint8_t *)d_keep,
                                             level[d + 1], d_count + 1, (int)(4 * m), st.s));
            g_launches += 3;  // the expansion + CUB's init and select kernels
            unsigned long long survivors = 0;
            S_TRY(cudaMemcpyAsync(&survivors, d_count + 1, sizeof(survivors), cudaMemcpyDeviceToHost, st.s));
            S_TRY(cudaStreamSynchronize(st.s));
            fill[d + 1] = survivors;
            next[d + 1] = 0;
        } else {
            uint64_t *ck = (uint64_t *)d_children, *cc = ck + 4 * (uint64_t)m;
            const unsigned g = std::min<unsigned>(grid_emit, (m + kCountThreads - 1) / kCountThreads);
            spectrum_emit_kernel<WIDE, LIST><<<g, kCountThreads, emit_smem, st.s>>>(
                ix, slice, m, shift, walk_min, emit_bins, emit_smem_bins, d_hist, canonical ? d_count + 2 : d_count, ck, cc,
                d_keep);
            S_TRY(cudaGetLastError());
            g_launches++;
            if (LIST) {
                const uint64_t most = std::min<uint64_t>(4 * (uint64_t)m, cap);  // survivors this slice can have
                if (staged + most > staging)
                    if (int rc = drain(); rc != MSBWT_OK) return rc;
                S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)ck, (const uint8_t *)d_keep,
                                                 d_stage_kmers + staged, d_count + 1, (int)(4 * m), st.s));
                S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)cc, (const uint8_t *)d_keep,
                                                 d_stage_counts + staged, d_count + 1, (int)(4 * m), st.s));
                g_launches += 4;
                unsigned long long survivors = 0;
                S_TRY(cudaMemcpyAsync(&survivors, d_count + 1, sizeof(survivors), cudaMemcpyDeviceToHost, st.s));
                S_TRY(cudaStreamSynchronize(st.s));
                staged += survivors;
            }
        }
    }
    if (LIST)
        if (int rc = drain(); rc != MSBWT_OK) return rc;
    unsigned long long total_kmers = 0;
    S_TRY(cudaMemcpyAsync(&total_kmers, d_count, sizeof(total_kmers), cudaMemcpyDeviceToHost, st.s));
    if (nbins) S_TRY(cudaMemcpyAsync(hist, d_hist, nbins * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    S_TRY(cudaStreamSynchronize(st.s));
    if (want_list && listed != total_kmers) return fail(MSBWT_ECUDA, "kmer spectrum: the list and the histogram disagree");
    *n_kmers = total_kmers;
    if (kmers) {
        *kmers = listed ? out_kmers.p : nullptr;
        *counts = listed ? out_counts.p : nullptr;
        if (listed) out_kmers.p = out_counts.p = nullptr;
    }
    return MSBWT_OK;
}

}  // namespace

int kmer_spectrum_to_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                            const DeviceKmerList &sink, uint64_t *n_kmers) {
    return index_is_wide(ix)
               ? spectrum_run<true, true>(device, ix, lanes, canonical, k, min_count, nullptr, 0, nullptr, nullptr, n_kmers, &sink)
               : spectrum_run<false, true>(device, ix, lanes, canonical, k, min_count, nullptr, 0, nullptr, nullptr, n_kmers, &sink);
}

int kmer_spectrum_on_device(int device, const IndexView &ix, int lanes, bool canonical, uint32_t k, uint64_t min_count,
                            uint64_t *hist, uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers) {
    // the canonical walk always carries the k-mer values: the pairs are resolved from them
    const bool list = canonical || kmers != nullptr;
    if (index_is_wide(ix))
        return list ? spectrum_run<true, true>(device, ix, lanes, canonical, k, min_count, hist, nbins, kmers, counts, n_kmers)
                    : spectrum_run<true, false>(device, ix, lanes, false, k, min_count, hist, nbins, kmers, counts, n_kmers);
    return list ? spectrum_run<false, true>(device, ix, lanes, canonical, k, min_count, hist, nbins, kmers, counts, n_kmers)
                : spectrum_run<false, false>(device, ix, lanes, false, k, min_count, hist, nbins, kmers, counts, n_kmers);
}

}  // namespace msbwt
