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

#define S_TRY(expr)                                                                        \
    do {                                                                                   \
        cudaError_t e_ = (expr);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            why = std::string("kmer spectrum: ") + #expr + ": " + cudaGetErrorString(e_);  \
            return e_ == cudaErrorMemoryAllocation ? MSBWT_ENOMEM : MSBWT_ECUDA;           \
        }                                                                                  \
    } while (0)

// the call's own stream: drained and destroyed on every way out, before the scratch it used is freed
struct OwnStream {
    cudaStream_t s = nullptr;
    ~OwnStream() {
        if (s) {
            cudaStreamSynchronize(s);
            cudaStreamDestroy(s);
        }
    }
};

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

template <bool WIDE, bool LIST>
int spectrum_run(int device, const IndexView &ix, uint32_t k, uint64_t min_count, uint64_t *hist, uint32_t nbins,
                 uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers, std::string &why, int *launches) {
    using P = typename Pos<WIDE>::type;
    using NodeT = Node<P, LIST>;
    const uint64_t B = slice_parents();
    // survivors of one slice: at most 4 per parent, and at most N / min_count (disjoint ranges of that width)
    const uint64_t cap = std::max<uint64_t>(1, std::min<uint64_t>(4 * B, ix.total / min_count));
    const uint64_t staging = LIST ? std::max(cap, std::min(kStagingKmers, ix.total / min_count)) : 0;
    const uint32_t smem_bins = std::min(nbins, kSmemBins);

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
    S_TRY(scratch.alloc(&d_count, 2));  // [0] k-mers emitted, [1] survivors of the last compaction
    uint64_t *d_stage_kmers = nullptr, *d_stage_counts = nullptr;
    if (LIST) {
        S_TRY(scratch.alloc(&d_stage_kmers, staging));
        S_TRY(scratch.alloc(&d_stage_counts, staging));
    }
    size_t temp_bytes = 0, need = 0;
    const int max_items = (int)(4 * std::min(B, cap));
    S_TRY(cub::DeviceSelect::Flagged(nullptr, need, (const NodeT *)nullptr, (const uint8_t *)nullptr, (NodeT *)nullptr,
                                     (unsigned long long *)nullptr, max_items, st.s));
    temp_bytes = std::max(temp_bytes, need);
    if (LIST) {
        S_TRY(cub::DeviceSelect::Flagged(nullptr, need, (const uint64_t *)nullptr, (const uint8_t *)nullptr,
                                         (uint64_t *)nullptr, (unsigned long long *)nullptr, max_items, st.s));
        temp_bytes = std::max(temp_bytes, need);
    }
    void *d_temp = nullptr;
    S_TRY(scratch.alloc((char **)&d_temp, temp_bytes));

    NodeT root{};
    root.l = 0;
    root.h = (P)ix.total;
    S_TRY(cudaMemcpyAsync(level[0], &root, sizeof(NodeT), cudaMemcpyHostToDevice, st.s));
    S_TRY(cudaMemsetAsync(d_hist, 0, std::max<uint32_t>(nbins, 1) * sizeof(unsigned long long), st.s));
    S_TRY(cudaMemsetAsync(d_count, 0, 2 * sizeof(unsigned long long), st.s));

    const unsigned grid_expand = persistent_grid(device, (const void *)spectrum_expand_kernel<WIDE, LIST>, kCountThreads,
                                                 std::min(B, cap), kCountThreads);
    const unsigned grid_emit = persistent_grid(device, (const void *)spectrum_emit_kernel<WIDE, LIST>, kCountThreads,
                                               std::min(B, cap), kCountThreads);
    const size_t emit_smem = std::max<uint32_t>(smem_bins, 1) * sizeof(uint32_t);
    std::vector<uint64_t> fill(k, 0), next(k, 0);
    fill[0] = 1;
    uint64_t staged = 0, listed = 0;
    auto flush = [&]() -> int {
        if (!staged) return MSBWT_OK;
        if (!out_kmers.reserve(listed + staged) || !out_counts.reserve(listed + staged)) {
            why = "kmer spectrum: host buffer for the k-mer list";
            return MSBWT_ENOMEM;
        }
        S_TRY(cudaMemcpyAsync(out_kmers.p + listed, d_stage_kmers, staged * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
        S_TRY(cudaMemcpyAsync(out_counts.p + listed, d_stage_counts, staged * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
        S_TRY(cudaStreamSynchronize(st.s));
        listed += staged;
        staged = 0;
        return MSBWT_OK;
    };
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
            spectrum_expand_kernel<WIDE, LIST><<<grid, kCountThreads, 0, st.s>>>(ix, slice, m, shift, min_count, children, d_keep);
            S_TRY(cudaGetLastError());
            S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const NodeT *)children, (const uint8_t *)d_keep,
                                             level[d + 1], d_count + 1, (int)(4 * m), st.s));
            if (launches) *launches += 3;  // the expansion + CUB's init and select kernels
            unsigned long long survivors = 0;
            S_TRY(cudaMemcpyAsync(&survivors, d_count + 1, sizeof(survivors), cudaMemcpyDeviceToHost, st.s));
            S_TRY(cudaStreamSynchronize(st.s));
            fill[d + 1] = survivors;
            next[d + 1] = 0;
        } else {
            uint64_t *ck = (uint64_t *)d_children, *cc = ck + 4 * (uint64_t)m;
            const unsigned g = std::min<unsigned>(grid_emit, (m + kCountThreads - 1) / kCountThreads);
            spectrum_emit_kernel<WIDE, LIST><<<g, kCountThreads, emit_smem, st.s>>>(
                ix, slice, m, shift, min_count, nbins, smem_bins, d_hist, d_count, ck, cc, d_keep);
            S_TRY(cudaGetLastError());
            if (launches) (*launches)++;
            if (LIST) {
                const uint64_t most = std::min<uint64_t>(4 * (uint64_t)m, cap);  // survivors this slice can have
                if (staged + most > staging)
                    if (int rc = flush(); rc != MSBWT_OK) return rc;
                S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)ck, (const uint8_t *)d_keep,
                                                 d_stage_kmers + staged, d_count + 1, (int)(4 * m), st.s));
                S_TRY(cub::DeviceSelect::Flagged(d_temp, temp_bytes, (const uint64_t *)cc, (const uint8_t *)d_keep,
                                                 d_stage_counts + staged, d_count + 1, (int)(4 * m), st.s));
                if (launches) *launches += 4;
                unsigned long long survivors = 0;
                S_TRY(cudaMemcpyAsync(&survivors, d_count + 1, sizeof(survivors), cudaMemcpyDeviceToHost, st.s));
                S_TRY(cudaStreamSynchronize(st.s));
                staged += survivors;
            }
        }
    }
    if (LIST)
        if (int rc = flush(); rc != MSBWT_OK) return rc;
    unsigned long long total_kmers = 0;
    S_TRY(cudaMemcpyAsync(&total_kmers, d_count, sizeof(total_kmers), cudaMemcpyDeviceToHost, st.s));
    if (nbins) S_TRY(cudaMemcpyAsync(hist, d_hist, nbins * sizeof(uint64_t), cudaMemcpyDeviceToHost, st.s));
    S_TRY(cudaStreamSynchronize(st.s));
    if (LIST && listed != total_kmers) {
        why = "kmer spectrum: the list and the histogram disagree";
        return MSBWT_ECUDA;
    }
    *n_kmers = total_kmers;
    if (LIST) {
        *kmers = listed ? out_kmers.p : nullptr;
        *counts = listed ? out_counts.p : nullptr;
        if (listed) out_kmers.p = out_counts.p = nullptr;
    }
    return MSBWT_OK;
}

}  // namespace

int kmer_spectrum_on_device(int device, const IndexView &ix, uint32_t k, uint64_t min_count, uint64_t *hist,
                            uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers, std::string &why,
                            int *launches) {
    const bool list = kmers != nullptr;
    if (index_is_wide(ix))
        return list ? spectrum_run<true, true>(device, ix, k, min_count, hist, nbins, kmers, counts, n_kmers, why, launches)
                    : spectrum_run<true, false>(device, ix, k, min_count, hist, nbins, kmers, counts, n_kmers, why, launches);
    return list ? spectrum_run<false, true>(device, ix, k, min_count, hist, nbins, kmers, counts, n_kmers, why, launches)
                : spectrum_run<false, false>(device, ix, k, min_count, hist, nbins, kmers, counts, n_kmers, why, launches);
}

}  // namespace msbwt
