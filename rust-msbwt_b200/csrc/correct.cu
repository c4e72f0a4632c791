// correct.cu -- read correction against an index in the manner of fmlrc (msbwt_correct_reads): weak runs of a read's
// k-mer windows are bridged through the de Bruijn graph of the solid k-mers.  include/msbwt_gpu.h holds the definition;
// oracle/correct.py restates it on the CPU.
//
// Reads are taken in chunks of whole reads of about kChunkSyms symbols, so device memory does not grow with the batch.
// Positions p of a chunk index its symbols; the window of read r that starts at p is window p - off[r].
//   windows   : one thread per position writes the window's k-mer and its reverse complement as u64 queries (0 when
//               the window holds N or runs past the read); the query path (launch_seed_u64 + launch_count_packed, as
//               the canonical spectrum) counts them and count2 sums the strands.
//   threshold : CUB segmented sort of every read's count2 values; one thread per read takes the upper median of the
//               non-zero ones past a binary search for the first non-zero.
//   weak runs : one thread per position: a run starts where a window is weak and its left neighbour is not; the
//               thread scans to the run's end, counts the run and flags it when it is eligible.  CUB compacts the
//               flagged positions into gaps (position order: by read, then by window).
//   BFS       : every gap of the chunk at once, one symbol per round.  The frontier is gap-major and, within a gap, in
//               lexicographic order of the walks: each walk's four children are laid out A < C < G < T and CUB
//               compacts them stably.  Each round counts 4 children x 2 strands through the query path, adds each
//               gap's solid children to its work (integer atomics: order independent), keeps the children that go on
//               and lists the bridges.  A walk is stored as one parent link per expanded walk: the child c of
//               expanded walk e is node 4 e + c, so a node's symbol is its low two bits and its parent is par[node / 4].
//   scoring   : bridges are listed round by round and in frontier order, so within a gap their list order is
//               (|E|, E) ascending, the tie order.  One thread per bridge rebuilds E backwards from the parent links,
//               computes Levenshtein(rev E, rev P) with one row of P in global scratch, and takes the atomic minimum
//               of (distance, list index) over its gap: the first bridge at the least distance wins.
//   assembly  : per replaced gap, delta[position of Y] = |E| - |P| and P's positions are marked; an inclusive scan
//               of delta gives every kept symbol's shift, and the new read offsets.  One thread per position scatters
//               the kept symbols, one per replaced gap writes E.  The chunk's result is copied out once.
// The kernels use no warp collectives: per-CTA counts go through shared memory.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include <algorithm>
#include <cstring>
#include <vector>

#include "../../include/msbwt_gpu.h"
#include "kernel_common.cuh"

namespace msbwt {

namespace {

constexpr uint64_t kChunkSyms = 1ull << 22;   // symbols of a chunk of reads (a longer read is a chunk of its own)
constexpr uint64_t kQueryPiece = 1ull << 24;  // queries per seed + count launch pair
constexpr uint32_t kRoot = 0xffffffffu;       // parent link of a gap's seed X
constexpr uint64_t kNoBridge = ~0ull;
constexpr uint64_t kScoreRowWords = 1ull << 26;  // DP row words of one scoring launch

struct Gap {
    uint64_t x, y;     // seed window a - 1 and target window b, as k-mers
    uint64_t T;        // the read's threshold
    uint64_t budget;   // branch_limit * (k + Emax)
    uint64_t ypos;     // chunk position of window b (P is [ypos - L0, ypos))
    uint32_t L0, emax;
};

struct Walk {
    uint64_t z;    // newest window (a bridge in the list: its round)
    uint32_t gap;
    uint32_t node; // 4 e + c, or kRoot
};

#define CORRECT_LOOP(i, n) for (uint64_t i = blockIdx.x * (uint64_t)kCountThreads + threadIdx.x; i < (n); i += (uint64_t)gridDim.x * kCountThreads)

// per-thread counts summed through shared memory, one atomic per CTA (ends with a barrier so smem may be reused)
__device__ __forceinline__ void cta_add(uint32_t *smem, uint32_t mine, unsigned long long *out) {
    smem[threadIdx.x] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int t = 0; t < kCountThreads; t++) sum += smem[t];
        if (sum) atomicAdd(out, sum);
    }
    __syncthreads();
}

__device__ __forceinline__ uint64_t read_of(const uint64_t *__restrict__ off, uint64_t n_reads, uint64_t p) {
    uint64_t lo = 0, hi = n_reads;  // the last r with off[r] <= p (off[0] = 0 <= p < off[n_reads])
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (off[mid] <= p) lo = mid;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint8_t code_sym(uint32_t c) { return (uint8_t)(c + 1 + (c == 3)); }  // A,C,G,T = 1,2,3,5

// the window starting at p: fwd / rc k-mers as queries 2p / 2p + 1, ok[p] = it lies in its read and holds no N
__global__ void __launch_bounds__(kCountThreads)
correct_windows_kernel(const uint8_t *__restrict__ syms, const uint64_t *__restrict__ off, uint64_t n_reads, uint64_t n,
                       uint32_t k, uint64_t *__restrict__ q, uint8_t *__restrict__ ok) {
    CORRECT_LOOP(p, n) {
        const uint64_t r = read_of(off, n_reads, p);
        bool good = p + k <= off[r + 1];
        uint64_t v = 0;
        for (uint32_t j = 0; good && j < k; j++) {
            const uint8_t s = syms[p + j];
            good = s != 4;
            v = (v << 2) | (uint64_t)(s == 5 ? 3 : s - 1);
        }
        if (!good) v = 0;
        q[2 * p] = v;
        q[2 * p + 1] = revcomp_kmer(v, k);
        ok[p] = good;
    }
}

// count2 of every window (0 without one); the segments of the threshold's sort are [off[r], off[r] + nwin)
__global__ void __launch_bounds__(kCountThreads)
correct_count2_kernel(const uint64_t *__restrict__ cnt, const uint8_t *__restrict__ ok, uint64_t n,
                      uint64_t *__restrict__ c2) {
    CORRECT_LOOP(p, n) c2[p] = ok[p] ? cnt[2 * p] + cnt[2 * p + 1] : 0;
}

__global__ void __launch_bounds__(kCountThreads)
correct_segments_kernel(const uint64_t *__restrict__ off, uint64_t n_reads, uint32_t k, uint64_t *__restrict__ seg_end) {
    CORRECT_LOOP(r, n_reads) {
        const uint64_t len = off[r + 1] - off[r];
        seg_end[r] = off[r] + (len >= k ? len - k + 1 : 0);
    }
}

// T[r] = max(min_count, floor(v[m / 2] * frac / 1000)) over the sorted non-zero count2 values v; 0 = leave the read
__global__ void __launch_bounds__(kCountThreads)
correct_threshold_kernel(const uint64_t *__restrict__ off, const uint64_t *__restrict__ seg_end,
                         const uint64_t *__restrict__ sorted, uint64_t n_reads, uint32_t k, uint64_t min_count,
                         uint32_t frac, uint64_t *__restrict__ T) {
    CORRECT_LOOP(r, n_reads) {
        const uint64_t b = off[r], e = seg_end[r];
        uint64_t t = 0;
        if (off[r + 1] - b >= (uint64_t)k + 2) {
            uint64_t lo = b, hi = e;  // first non-zero
            while (lo < hi) {
                const uint64_t mid = lo + ((hi - lo) >> 1);
                if (sorted[mid] == 0) lo = mid + 1;
                else hi = mid;
            }
            if (lo < e) {
                const uint64_t v = sorted[lo + (e - lo) / 2];
                t = max(min_count, (v / 1000) * frac + (v % 1000) * frac / 1000);  // floor(v * frac / 1000), exactly
            }
        }
        T[r] = t;
    }
}

// one thread per window that starts a weak run: scan to the run's end b, count it, flag it when eligible
__global__ void __launch_bounds__(kCountThreads)
correct_runs_kernel(const uint64_t *__restrict__ off, const uint64_t *__restrict__ seg_end, uint64_t n_reads,
                    const uint64_t *__restrict__ c2, const uint64_t *__restrict__ T, uint64_t n, uint32_t k,
                    uint8_t *__restrict__ flag, uint64_t *__restrict__ run_end, unsigned long long *__restrict__ stats) {
    __shared__ uint32_t smem[kCountThreads];
    uint32_t weak = 0, eligible = 0;
    CORRECT_LOOP(p, n) {
        const uint64_t r = read_of(off, n_reads, p), t = T[r], e = seg_end[r];
        bool f = false;
        if (t && p < e && c2[p] < t && (p == off[r] || c2[p - 1] >= t)) {
            uint64_t b = p + 1;
            while (b < e && c2[b] < t) b++;
            weak++;
            f = p > off[r] && b < e && b - p + 1 >= k;
            eligible += f;
            run_end[p] = b;
        }
        flag[p] = f;
    }
    cta_add(smem, weak, stats);
    cta_add(smem, eligible, stats + 1);
}

// the gaps, and the BFS's first frontier (each gap's X); *l0max = the longest P
__global__ void __launch_bounds__(kCountThreads)
correct_gap_init_kernel(const uint64_t *__restrict__ pos, uint64_t n_gaps, const uint64_t *__restrict__ off,
                        uint64_t n_reads, const uint64_t *__restrict__ run_end, const uint64_t *__restrict__ q,
                        const uint64_t *__restrict__ T, uint32_t k, uint64_t branch_limit, Gap *__restrict__ gaps,
                        Walk *__restrict__ front, unsigned long long *__restrict__ work,
                        unsigned long long *__restrict__ best, unsigned int *__restrict__ l0max) {
    __shared__ uint32_t smem[kCountThreads];
    uint32_t mine = 0;
    CORRECT_LOOP(g, n_gaps) {
        const uint64_t p = pos[g], b = run_end[p];
        Gap G;
        G.x = q[2 * (p - 1)];
        G.y = q[2 * b];
        G.T = T[read_of(off, n_reads, p)];
        G.L0 = (uint32_t)(b - p + 1 - k);
        G.emax = (uint32_t)(13ull * G.L0 / 10 + 2);
        G.budget = branch_limit * (uint64_t)(k + G.emax);
        G.ypos = b;
        gaps[g] = G;
        front[g] = Walk{G.x, (uint32_t)g, kRoot};
        work[g] = 0;
        best[g] = kNoBridge;
        mine = max(mine, G.L0);
    }
    smem[threadIdx.x] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t m = 0;
        for (int t = 0; t < kCountThreads; t++) m = max(m, smem[t]);
        atomicMax(l0max, m);
    }
}

// one round, step 1: expanded walk i is node group base + i; its four children and their reverse complements as
// queries 8 i + 2 c (+ 1)
__global__ void __launch_bounds__(kCountThreads)
correct_expand_kernel(const Walk *__restrict__ front, uint64_t n, uint64_t base, uint64_t mask, uint32_t k,
                      uint32_t *__restrict__ par, uint64_t *__restrict__ q) {
    CORRECT_LOOP(i, n) {
        const Walk w = front[i];
        par[base + i] = w.node;
#pragma unroll
        for (uint32_t c = 0; c < 4; c++) {
            const uint64_t y = ((w.z << 2) | c) & mask;
            q[8 * i + 2 * c] = y;
            q[8 * i + 2 * c + 1] = revcomp_kmer(y, k);
        }
    }
}

// step 2, one thread per child: solid children add to their gap's work; a solid child whose window is Y at round
// t >= k is a bridge (listed with z = t), any other goes on while t < k + Emax
__global__ void __launch_bounds__(kCountThreads)
correct_classify_kernel(const Walk *__restrict__ front, uint64_t n_child, uint64_t base, const uint64_t *__restrict__ q,
                        const uint64_t *__restrict__ cnt, const Gap *__restrict__ gaps, uint32_t t, uint32_t k,
                        unsigned long long *__restrict__ work, Walk *__restrict__ child, uint8_t *__restrict__ ext,
                        uint8_t *__restrict__ bridge) {
    CORRECT_LOOP(j, n_child) {
        const uint32_t g = front[j >> 2].gap;
        const Gap &G = gaps[g];
        const uint64_t y = q[2 * j];
        const bool solid = cnt[2 * j] + cnt[2 * j + 1] >= G.T;
        const bool br = solid && t >= k && y == G.y;
        if (solid) atomicAdd(&work[g], 1ull);
        child[j] = Walk{br ? (uint64_t)t : y, g, (uint32_t)(4 * (base + (j >> 2)) + (j & 3))};
        ext[j] = solid && !br && t < k + G.emax;
        bridge[j] = br;
    }
}

// step 3, after every atomic of the round: a gap whose work passed its budget is abandoned and expands no further
__global__ void __launch_bounds__(kCountThreads)
correct_abandon_kernel(const Walk *__restrict__ child, uint64_t n_child, const Gap *__restrict__ gaps,
                       const unsigned long long *__restrict__ work, uint8_t *__restrict__ ext) {
    CORRECT_LOOP(j, n_child) {
        if (!ext[j]) continue;
        const uint32_t g = child[j].gap;
        if (work[g] > gaps[g].budget) ext[j] = 0;
    }
}

// Levenshtein(E, P) of bridge i0 + ib through the reversed strings, one row over P in rows[ib * stride ..]; best[gap]
// keeps the least (distance, i)
__global__ void __launch_bounds__(kCountThreads)
correct_score_kernel(const Walk *__restrict__ br, uint64_t i0, uint64_t n_br, const uint32_t *__restrict__ par,
                     const Gap *__restrict__ gaps, const unsigned long long *__restrict__ work,
                     const uint8_t *__restrict__ syms, uint32_t k, uint64_t stride, uint32_t *__restrict__ rows,
                     unsigned long long *__restrict__ best) {
    CORRECT_LOOP(ib, n_br) {
        const uint64_t i = i0 + ib;
        const Walk b = br[i];
        const Gap G = gaps[b.gap];
        if (work[b.gap] > G.budget) continue;
        const uint32_t elen = (uint32_t)b.z - k;
        uint32_t node = b.node;
        for (uint32_t s = 0; s < k; s++) node = par[node >> 2];  // past Y
        uint32_t *row = rows + ib * stride;
        const uint8_t *P = syms + G.ypos - G.L0;
        for (uint32_t j = 0; j <= G.L0; j++) row[j] = j;
        for (uint32_t e = 1; e <= elen; e++) {
            const uint8_t s = code_sym(node & 3);
            node = par[node >> 2];
            uint32_t diag = row[0];
            row[0] = e;
            for (uint32_t j = 1; j <= G.L0; j++) {
                const uint32_t up = row[j];
                row[j] = min(min(up, row[j - 1]) + 1, diag + (s != P[G.L0 - j]));
                diag = up;
            }
        }
        atomicMin(&best[b.gap], ((unsigned long long)row[G.L0] << 40) | i);
    }
}

// stats [2..4]; a replaced gap puts |E| - L0 at Y's position and marks P's positions
__global__ void __launch_bounds__(kCountThreads)
correct_decide_kernel(const Gap *__restrict__ gaps, uint64_t n_gaps, const unsigned long long *__restrict__ work,
                      const unsigned long long *__restrict__ best, const Walk *__restrict__ br, uint32_t k,
                      long long *__restrict__ delta, uint8_t *__restrict__ dead, unsigned long long *__restrict__ stats) {
    __shared__ uint32_t smem[kCountThreads];
    uint32_t bridged = 0, abandoned = 0, none = 0;
    CORRECT_LOOP(g, n_gaps) {
        const Gap G = gaps[g];
        if (work[g] > G.budget) { abandoned++; continue; }
        if (best[g] == kNoBridge) { none++; continue; }
        bridged++;
        const uint64_t i = best[g] & ((1ull << 40) - 1);
        delta[G.ypos] = (long long)((uint32_t)br[i].z - k) - (long long)G.L0;
        for (uint64_t p = G.ypos - G.L0; p < G.ypos; p++) dead[p] = 1;
    }
    cta_add(smem, bridged, stats + 2);
    cta_add(smem, abandoned, stats + 3);
    cta_add(smem, none, stats + 4);
}

// new read offsets: off[r] + the shift of everything before the read
__global__ void __launch_bounds__(kCountThreads)
correct_offsets_kernel(const uint64_t *__restrict__ off, uint64_t n_reads, const long long *__restrict__ shift,
                       uint64_t *__restrict__ out_off) {
    CORRECT_LOOP(r, n_reads + 1) out_off[r] = off[r] + (off[r] ? shift[off[r] - 1] : 0);
}

__global__ void __launch_bounds__(kCountThreads)
correct_scatter_kernel(const uint8_t *__restrict__ syms, const uint8_t *__restrict__ dead,
                       const long long *__restrict__ shift, uint64_t n, uint8_t *__restrict__ out) {
    CORRECT_LOOP(p, n) if (!dead[p]) out[p + shift[p]] = syms[p];
}

// E of every replaced gap, written backwards from the node before Y
__global__ void __launch_bounds__(kCountThreads)
correct_write_kernel(const Gap *__restrict__ gaps, uint64_t n_gaps, const unsigned long long *__restrict__ work,
                     const unsigned long long *__restrict__ best, const Walk *__restrict__ br,
                     const uint32_t *__restrict__ par, const long long *__restrict__ shift, uint32_t k,
                     uint8_t *__restrict__ out) {
    CORRECT_LOOP(g, n_gaps) {
        const Gap G = gaps[g];
        if (work[g] > G.budget || best[g] == kNoBridge) continue;
        const Walk b = br[best[g] & ((1ull << 40) - 1)];
        uint32_t node = b.node;
        for (uint32_t s = 0; s < k; s++) node = par[node >> 2];
        const uint64_t end = G.ypos + shift[G.ypos];
        for (uint32_t e = 1; e <= (uint32_t)b.z - k; e++) {
            out[end - e] = code_sym(node & 3);
            node = par[node >> 2];
        }
    }
}

#define C_TRY(e) CU_TRY_IN("correct_reads: ", e)

// a device buffer that grows by half again; with `keep`, what it held is copied over
struct Grow {
    void *p = nullptr;
    size_t cap = 0;
    ~Grow() { cudaFree(p); }
    template <class T> T *as() const { return (T *)p; }
    cudaError_t reserve(size_t bytes, cudaStream_t st, size_t keep = 0) {
        if (bytes <= cap) return cudaSuccess;
        const size_t want = std::max(bytes, cap + cap / 2);
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, want);
        if (e != cudaSuccess) return e;
        if (keep) e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        cudaFree(p);
        p = q;
        cap = want;
        return e;
    }
};

struct Run {
    int device;
    const IndexView &ix;
    int lanes;
    const CorrectParams &prm;
    cudaStream_t st;
    bool with_b;
    uint64_t mask;
    Grow syms, off, q, cnt, packed, ok, c2, sorted, seg_end, T, flag, run_end, pos, gaps, work, best, front, child, ext,
        brf, br, par, rows, delta, out, out_off, temp;
    unsigned long long *d_stats = nullptr, *d_n = nullptr;
    unsigned int *d_l0 = nullptr;
    uint64_t launches = 0;

    unsigned grid(const void *kern, uint64_t n) const {
        return persistent_grid(device, kern, kCountThreads, n, kCountThreads);
    }
    template <class F> int cub_call(F &&f) {  // size the temp storage, grow it, run
        size_t need = 0;
        C_TRY(f((void *)nullptr, need));
        C_TRY(temp.reserve(need, st));
        size_t have = temp.cap;
        C_TRY(f(temp.p, have));
        return MSBWT_OK;
    }
    // count2 inputs: counts of n queries through the query path, in pieces
    int count(uint64_t n) {
        const uint64_t piece = std::min(n, kQueryPiece);
        C_TRY(packed.reserve(packed_layout(ix, prm.k, piece).total() * sizeof(uint64_t), st));
        for (uint64_t b = 0; b < n; b += piece) {
            const uint64_t m = std::min(piece, n - b);
            C_TRY(launch_seed_u64(ix, q.as<uint64_t>() + b, prm.k, m, packed.as<uint64_t>(), cnt.as<uint64_t>() + b, st));
            C_TRY(launch_count_packed(device, ix, lanes, packed.as<uint64_t>(), prm.k, m, cnt.as<uint64_t>() + b, st, with_b));
        }
        return MSBWT_OK;
    }
    int read_u64(const void *src, uint64_t *v) {
        C_TRY(cudaMemcpyAsync(v, src, sizeof(*v), cudaMemcpyDeviceToHost, st));
        C_TRY(cudaStreamSynchronize(st));
        return MSBWT_OK;
    }
    int chunk(const uint8_t *h_syms, const uint64_t *h_off, uint64_t n_reads, std::vector<uint8_t> &out_syms,
              std::vector<uint64_t> &out_lens);
};

int Run::chunk(const uint8_t *h_syms, const uint64_t *h_off, uint64_t nr, std::vector<uint8_t> &out_syms,
               std::vector<uint64_t> &out_lens) {
    const uint64_t n = h_off[nr] - h_off[0];
    const uint32_t k = prm.k;
    if (!n) {
        out_lens.insert(out_lens.end(), nr, 0);
        return MSBWT_OK;
    }
    std::vector<uint64_t> rel(nr + 1);
    for (uint64_t r = 0; r <= nr; r++) rel[r] = h_off[r] - h_off[0];
    C_TRY(syms.reserve(n, st));
    C_TRY(off.reserve((nr + 1) * sizeof(uint64_t), st));
    C_TRY(cudaMemcpyAsync(syms.p, h_syms + h_off[0], n, cudaMemcpyHostToDevice, st));
    C_TRY(cudaMemcpyAsync(off.p, rel.data(), (nr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    for (Grow *b : {&q, &cnt}) C_TRY(b->reserve(2 * n * sizeof(uint64_t), st));
    for (Grow *b : {&c2, &sorted, &run_end}) C_TRY(b->reserve(n * sizeof(uint64_t), st));
    C_TRY(delta.reserve(n * sizeof(long long), st));
    for (Grow *b : {&ok, &flag}) C_TRY(b->reserve(n, st));
    for (Grow *b : {&seg_end, &T}) C_TRY(b->reserve(nr * sizeof(uint64_t), st));
    const uint64_t *d_off = off.as<uint64_t>();

    // windows and their count2
    correct_windows_kernel<<<grid((const void *)correct_windows_kernel, n), kCountThreads, 0, st>>>(
        syms.as<uint8_t>(), d_off, nr, n, k, q.as<uint64_t>(), ok.as<uint8_t>());
    C_TRY(cudaGetLastError());
    if (int rc = count(2 * n); rc != MSBWT_OK) return rc;
    correct_count2_kernel<<<grid((const void *)correct_count2_kernel, n), kCountThreads, 0, st>>>(
        cnt.as<uint64_t>(), ok.as<uint8_t>(), n, c2.as<uint64_t>());
    C_TRY(cudaGetLastError());
    // thresholds
    correct_segments_kernel<<<grid((const void *)correct_segments_kernel, nr), kCountThreads, 0, st>>>(
        d_off, nr, k, seg_end.as<uint64_t>());
    C_TRY(cudaGetLastError());
    if (int rc = cub_call([&](void *tp, size_t &tb) {
            return cub::DeviceSegmentedSort::SortKeys(tp, tb, c2.as<uint64_t>(), sorted.as<uint64_t>(), (int64_t)n,
                                                      (int64_t)nr, d_off, seg_end.as<uint64_t>(), st);
        });
        rc != MSBWT_OK)
        return rc;
    correct_threshold_kernel<<<grid((const void *)correct_threshold_kernel, nr), kCountThreads, 0, st>>>(
        d_off, seg_end.as<uint64_t>(), sorted.as<uint64_t>(), nr, k, prm.min_count, prm.frac_permille, T.as<uint64_t>());
    C_TRY(cudaGetLastError());
    // weak runs -> gaps
    correct_runs_kernel<<<grid((const void *)correct_runs_kernel, n), kCountThreads, 0, st>>>(
        d_off, seg_end.as<uint64_t>(), nr, c2.as<uint64_t>(), T.as<uint64_t>(), n, k, flag.as<uint8_t>(),
        run_end.as<uint64_t>(), d_stats);
    C_TRY(cudaGetLastError());
    C_TRY(pos.reserve(n * sizeof(uint64_t), st));
    if (int rc = cub_call([&](void *tp, size_t &tb) {
            return cub::DeviceSelect::Flagged(tp, tb, cub::CountingInputIterator<uint64_t>(0), flag.as<uint8_t>(),
                                              pos.as<uint64_t>(), d_n, (int64_t)n, st);
        });
        rc != MSBWT_OK)
        return rc;
    launches += 6;  // windows, count2, segments, threshold, runs + the segmented sort, counted as one
    launches += 2;  // CUB's select: init + kernel
    uint64_t n_gaps = 0;
    if (int rc = read_u64(d_n, &n_gaps); rc != MSBWT_OK) return rc;

    uint64_t n_br = 0;
    if (n_gaps) {
        for (Grow *b : {&work, &best}) C_TRY(b->reserve(n_gaps * sizeof(unsigned long long), st));
        C_TRY(gaps.reserve(n_gaps * sizeof(Gap), st));
        C_TRY(front.reserve(n_gaps * sizeof(Walk), st));
        C_TRY(cudaMemsetAsync(d_l0, 0, sizeof(unsigned int), st));
        correct_gap_init_kernel<<<grid((const void *)correct_gap_init_kernel, n_gaps), kCountThreads, 0, st>>>(
            pos.as<uint64_t>(), n_gaps, d_off, nr, run_end.as<uint64_t>(), q.as<uint64_t>(), T.as<uint64_t>(), k,
            prm.branch_limit, gaps.as<Gap>(), front.as<Walk>(), work.as<unsigned long long>(),
            best.as<unsigned long long>(), d_l0);
        C_TRY(cudaGetLastError());
        launches++;
        // rounds: F walks expand into 4 F children; par gains F links
        uint64_t F = n_gaps, base = 0;
        for (uint32_t t = 1; F; t++) {
            if (4 * (base + F) >= kRoot)
                return fail(MSBWT_ENOMEM, "correct_reads: the walks of one chunk need 2^32 node ids or more");
            C_TRY(par.reserve((base + F) * sizeof(uint32_t), st, base * sizeof(uint32_t)));
            C_TRY(br.reserve((n_br + 4 * F) * sizeof(Walk), st, n_br * sizeof(Walk)));
            for (Grow *b : {&q, &cnt}) C_TRY(b->reserve(8 * F * sizeof(uint64_t), st));
            C_TRY(child.reserve(4 * F * sizeof(Walk), st));
            for (Grow *b : {&ext, &brf}) C_TRY(b->reserve(4 * F, st));
            correct_expand_kernel<<<grid((const void *)correct_expand_kernel, F), kCountThreads, 0, st>>>(
                front.as<Walk>(), F, base, mask, k, par.as<uint32_t>(), q.as<uint64_t>());
            C_TRY(cudaGetLastError());
            if (int rc = count(8 * F); rc != MSBWT_OK) return rc;
            correct_classify_kernel<<<grid((const void *)correct_classify_kernel, 4 * F), kCountThreads, 0, st>>>(
                front.as<Walk>(), 4 * F, base, q.as<uint64_t>(), cnt.as<uint64_t>(), gaps.as<Gap>(), t, k,
                work.as<unsigned long long>(), child.as<Walk>(), ext.as<uint8_t>(), brf.as<uint8_t>());
            C_TRY(cudaGetLastError());
            correct_abandon_kernel<<<grid((const void *)correct_abandon_kernel, 4 * F), kCountThreads, 0, st>>>(
                child.as<Walk>(), 4 * F, gaps.as<Gap>(), work.as<unsigned long long>(), ext.as<uint8_t>());
            C_TRY(cudaGetLastError());
            C_TRY(front.reserve(4 * F * sizeof(Walk), st));
            if (int rc = cub_call([&](void *tp, size_t &tb) {
                    return cub::DeviceSelect::Flagged(tp, tb, child.as<Walk>(), brf.as<uint8_t>(), br.as<Walk>() + n_br,
                                                      d_n + 1, (int64_t)(4 * F), st);
                });
                rc != MSBWT_OK)
                return rc;
            if (int rc = cub_call([&](void *tp, size_t &tb) {
                    return cub::DeviceSelect::Flagged(tp, tb, child.as<Walk>(), ext.as<uint8_t>(), front.as<Walk>(), d_n,
                                                      (int64_t)(4 * F), st);
                });
                rc != MSBWT_OK)
                return rc;
            launches += 7;  // expand, classify, abandon + CUB's two selects (init + kernel each)
            unsigned long long got[2];
            C_TRY(cudaMemcpyAsync(got, d_n, sizeof(got), cudaMemcpyDeviceToHost, st));
            C_TRY(cudaStreamSynchronize(st));
            base += F;
            F = got[0];
            n_br += got[1];
        }
        // scoring
        if (n_br) {
            uint64_t l0max = 0;
            unsigned int l0 = 0;
            C_TRY(cudaMemcpyAsync(&l0, d_l0, sizeof(l0), cudaMemcpyDeviceToHost, st));
            C_TRY(cudaStreamSynchronize(st));
            l0max = l0;
            const uint64_t batch = std::max<uint64_t>(1, kScoreRowWords / (l0max + 1));  // bridges per launch
            C_TRY(rows.reserve(std::min(n_br, batch) * (l0max + 1) * sizeof(uint32_t), st));
            for (uint64_t i0 = 0; i0 < n_br; i0 += batch) {
                const uint64_t m = std::min(batch, n_br - i0);
                correct_score_kernel<<<grid((const void *)correct_score_kernel, m), kCountThreads, 0, st>>>(
                    br.as<Walk>(), i0, m, par.as<uint32_t>(), gaps.as<Gap>(), work.as<unsigned long long>(),
                    syms.as<uint8_t>(), k, l0max + 1, rows.as<uint32_t>(), best.as<unsigned long long>());
                C_TRY(cudaGetLastError());
                launches++;
            }
        }
    }

    // assembly
    C_TRY(cudaMemsetAsync(delta.p, 0, n * sizeof(long long), st));
    C_TRY(cudaMemsetAsync(flag.p, 0, n, st));  // now: P's positions of the replaced gaps
    if (n_gaps) {
        correct_decide_kernel<<<grid((const void *)correct_decide_kernel, n_gaps), kCountThreads, 0, st>>>(
            gaps.as<Gap>(), n_gaps, work.as<unsigned long long>(), best.as<unsigned long long>(), br.as<Walk>(), k,
            delta.as<long long>(), flag.as<uint8_t>(), d_stats);
        C_TRY(cudaGetLastError());
        launches++;
    }
    if (int rc = cub_call([&](void *tp, size_t &tb) {
            return cub::DeviceScan::InclusiveSum(tp, tb, delta.as<long long>(), delta.as<long long>(), (int64_t)n, st);
        });
        rc != MSBWT_OK)
        return rc;
    long long last = 0;
    C_TRY(cudaMemcpyAsync(&last, delta.as<long long>() + n - 1, sizeof(last), cudaMemcpyDeviceToHost, st));
    C_TRY(cudaStreamSynchronize(st));
    const uint64_t n_out = n + last;
    C_TRY(out.reserve(n_out, st));
    C_TRY(out_off.reserve((nr + 1) * sizeof(uint64_t), st));
    correct_offsets_kernel<<<grid((const void *)correct_offsets_kernel, nr + 1), kCountThreads, 0, st>>>(
        d_off, nr, delta.as<long long>(), out_off.as<uint64_t>());
    C_TRY(cudaGetLastError());
    correct_scatter_kernel<<<grid((const void *)correct_scatter_kernel, n), kCountThreads, 0, st>>>(
        syms.as<uint8_t>(), flag.as<uint8_t>(), delta.as<long long>(), n, out.as<uint8_t>());
    C_TRY(cudaGetLastError());
    launches += 4;  // CUB's scan (init + kernel), offsets, scatter
    if (n_gaps) {
        correct_write_kernel<<<grid((const void *)correct_write_kernel, n_gaps), kCountThreads, 0, st>>>(
            gaps.as<Gap>(), n_gaps, work.as<unsigned long long>(), best.as<unsigned long long>(), br.as<Walk>(),
            par.as<uint32_t>(), delta.as<long long>(), k, out.as<uint8_t>());
        C_TRY(cudaGetLastError());
        launches++;
    }
    const size_t s0 = out_syms.size(), l0 = out_lens.size();
    std::vector<uint64_t> offs(nr + 1);
    out_syms.resize(s0 + n_out);
    C_TRY(cudaMemcpyAsync(out_syms.data() + s0, out.p, n_out, cudaMemcpyDeviceToHost, st));
    C_TRY(cudaMemcpyAsync(offs.data(), out_off.p, (nr + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    C_TRY(cudaStreamSynchronize(st));
    out_lens.resize(l0 + nr);
    for (uint64_t r = 0; r < nr; r++) out_lens[l0 + r] = offs[r + 1] - offs[r];
    return MSBWT_OK;
}

}  // namespace

int correct_reads_on_device(int device, const IndexView &ix, int lanes, const uint8_t *syms, const uint64_t *offsets,
                            uint64_t n_reads, const CorrectParams &prm, std::vector<uint8_t> &out_syms,
                            std::vector<uint64_t> &out_lens, uint64_t stats[5]) {
    DeviceScratch scratch;
    Run run{device, ix, lanes, prm, nullptr, packed_batch_needs_list_b(ix, prm.k),
            prm.k == 32 ? ~0ull : (1ull << (2 * prm.k)) - 1};
    OwnStream st;  // declared after the buffers: drained before they are freed
    C_TRY(cudaStreamCreateWithFlags(&st.s, cudaStreamNonBlocking));
    run.st = st.s;
    C_TRY(scratch.alloc(&run.d_stats, 5));
    C_TRY(scratch.alloc(&run.d_n, 2));
    C_TRY(scratch.alloc(&run.d_l0, 1));
    C_TRY(cudaMemsetAsync(run.d_stats, 0, 5 * sizeof(unsigned long long), st.s));
    uint64_t r = 0;
    int rc = MSBWT_OK;
    while (rc == MSBWT_OK && r < n_reads) {
        uint64_t e = r + 1;  // whole reads, at least one
        while (e < n_reads && offsets[e + 1] - offsets[r] <= kChunkSyms) e++;
        rc = run.chunk(syms, offsets + r, e - r, out_syms, out_lens);
        r = e;
    }
    g_launches += run.launches;
    if (rc != MSBWT_OK) return rc;
    unsigned long long s[5];
    C_TRY(cudaMemcpyAsync(s, run.d_stats, sizeof(s), cudaMemcpyDeviceToHost, st.s));
    C_TRY(cudaStreamSynchronize(st.s));
    for (int i = 0; i < 5; i++) stats[i] = s[i];
    return MSBWT_OK;
}

}  // namespace msbwt
