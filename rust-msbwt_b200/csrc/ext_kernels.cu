// ext_kernels.cu -- batched queries built on the backward-search step, for the direct callers of the path
// (SURVEY 8f N3): what a read-correction / assembly loop around msbwt2 does with count_kmer and
// constrain_range, as batches.
//
//   constrain_fanout_kernel : for every range [l,h) the FOUR calls RleBWT::constrain_range(sym, ..) for
//                             sym = A,C,G,T (src/rle_bwt.rs:202-287) from ONE fetch of the index blocks that
//                             hold l and h;
//   expand_read_kmers_kernel: the k-mers of every window of every read -- and their reverse complements
//                             (string_util::reverse_complement_i, src/string_util.rs:45-50) -- laid out as the
//                             n*k symbol bytes BWT::count_kmer batches take (src/msbwt_core.rs:125-161), so that
//                             a pileup along a read costs read_len bytes over PCIe instead of k per window;
//   sum_strands_kernel      : count(kmer) + count(revcomp(kmer)) per window.
#include "device_rank.cuh"
#include "engine.h"
#include "kernel_common.cuh"

namespace msbwt {

template <bool WIDE>
__global__ void __launch_bounds__(kCountThreads, 4)
constrain_fanout_kernel(IndexView ix, const uint64_t *__restrict__ l, const uint64_t *__restrict__ h, uint32_t n,
                        uint64_t *__restrict__ out_l, uint64_t *__restrict__ out_h) {
    using P = typename Pos<WIDE>::type;
    __shared__ uint64_t cb_smem[WIDE ? kMaxSuperInSmem * 8 : 4];
    const CBase<WIDE> cb = stage_cbase<WIDE>(ix, cb_smem);
    const uint32_t threads = gridDim.x * kCountThreads;
    for (uint64_t i = blockIdx.x * kCountThreads + threadIdx.x; i < n; i += threads) {
        P ol[4], oh[4];
        rank_fanout4<WIDE>(ix, cb, (P)l[i], (P)h[i], ol, oh);
        // 4 consecutive u64 per range: two 16-byte stores per array
        reinterpret_cast<ulonglong2 *>(out_l)[2 * i] = make_ulonglong2(ol[0], ol[1]);
        reinterpret_cast<ulonglong2 *>(out_l)[2 * i + 1] = make_ulonglong2(ol[2], ol[3]);
        reinterpret_cast<ulonglong2 *>(out_h)[2 * i] = make_ulonglong2(oh[0], oh[1]);
        reinterpret_cast<ulonglong2 *>(out_h)[2 * i + 1] = make_ulonglong2(oh[2], oh[3]);
    }
}

// Query (r * windows + w) * strands + s  <-  read r, offset w; strand 0: the window itself, strand 1: its
// reverse complement ($ACGNT -> $TGCNA; values >= 6 are passed on for the pack stage to refuse).  The output
// is one linear byte array (query-major, k bytes each); every thread produces 16 consecutive bytes of it
// with one vector store, walking (read, query, symbol) counters across query and read boundaries; the read
// bytes come through L1 (each is used k * strands times).
__global__ void __launch_bounds__(256)
expand_read_kmers_kernel(const uint8_t *__restrict__ reads, uint32_t read_len, uint64_t n_reads, uint32_t k,
                         uint32_t strands, uint8_t *__restrict__ syms) {
    const uint32_t windows = read_len - k + 1;
    const uint32_t per_read_q = windows * strands;           // queries per read
    const uint64_t per_read = (uint64_t)per_read_q * k;      // output bytes per read
    const uint64_t total = n_reads * per_read;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x * 16u;
    for (uint64_t o = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16u; o < total; o += step) {
        uint64_t r = o / per_read;
        uint32_t qq, i;                                       // query within the read, symbol within the query
        if (per_read >> 32) {  // one read's windows pass 2^32 bytes (e.g. a 22 Mbp read at k = 100, both strands)
            const uint64_t p = o - r * per_read;
            qq = (uint32_t)(p / k);
            i = (uint32_t)(p - (uint64_t)qq * k);
        } else {               // the usual case keeps the cheaper 32-bit division
            const uint32_t p = (uint32_t)(o - r * per_read);
            qq = p / k;
            i = p - qq * k;
        }
        const uint8_t *rd = reads + r * read_len;
        uint32_t word[4] = {0u, 0u, 0u, 0u};
        const uint32_t nb = (uint32_t)(total - o < 16u ? total - o : 16u);
        for (uint32_t b = 0; b < nb; b++) {
            const uint32_t w = qq / strands, s = qq - w * strands;
            uint32_t c;
            if (s == 0) {
                c = rd[w + i];
            } else {
                c = rd[w + k - 1 - i];
                c = c < 6u ? ((0x142350u >> (4u * c)) & 7u) : c;  // 0,5,3,2,4,1
            }
            word[b >> 2] |= c << (8u * (b & 3u));
            if (++i == k) {
                i = 0;
                if (++qq == per_read_q) { qq = 0; rd += read_len; }
            }
        }
        if (nb == 16u) {
            *reinterpret_cast<uint4 *>(syms + o) = make_uint4(word[0], word[1], word[2], word[3]);
        } else {
            for (uint32_t b = 0; b < nb; b++) syms[o + b] = (uint8_t)(word[b >> 2] >> (8u * (b & 3u)));
        }
    }
}

__global__ void __launch_bounds__(256)
sum_strands_kernel(const uint64_t *__restrict__ per_query, uint64_t n_windows, uint64_t *__restrict__ out) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_windows; i += step) {
        const ulonglong2 v = reinterpret_cast<const ulonglong2 *>(per_query)[i];
        out[i] = v.x + v.y;
    }
}

// counts of an index below 2^32 symbols fit 32 bits: halves the bytes of the copy back to the host
__global__ void __launch_bounds__(256)
narrow_counts_kernel(const uint64_t *__restrict__ in, uint64_t n, uint32_t *__restrict__ out) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) out[i] = (uint32_t)in[i];
}

cudaError_t launch_narrow_counts(int device, const uint64_t *d_in, uint64_t n, uint32_t *d_out, cudaStream_t st) {
    if (!n) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)sm_count(device) * 16);
    g_launches++;
    narrow_counts_kernel<<<grid, 256, 0, st>>>(d_in, n, d_out);
    return cudaGetLastError();
}

cudaError_t launch_constrain_fanout(int device, const IndexView &ix, const uint64_t *d_l, const uint64_t *d_h,
                                    uint64_t n, uint64_t *d_out_l, uint64_t *d_out_h, cudaStream_t st) {
    for (uint64_t q0 = 0; q0 < n; q0 += kMaxPerLaunch) {
        const uint32_t m = (uint32_t)((n - q0) < kMaxPerLaunch ? (n - q0) : kMaxPerLaunch);
        if (index_is_wide(ix)) {
            const unsigned grid = persistent_grid(device, (const void *)constrain_fanout_kernel<true>, kCountThreads, m, kCountThreads);
            constrain_fanout_kernel<true><<<grid, kCountThreads, 0, st>>>(ix, d_l + q0, d_h + q0, m, d_out_l + 4 * q0, d_out_h + 4 * q0);
        } else {
            const unsigned grid = persistent_grid(device, (const void *)constrain_fanout_kernel<false>, kCountThreads, m, kCountThreads);
            constrain_fanout_kernel<false><<<grid, kCountThreads, 0, st>>>(ix, d_l + q0, d_h + q0, m, d_out_l + 4 * q0, d_out_h + 4 * q0);
        }
        g_launches++;
        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_expand_read_kmers(int device, const uint8_t *d_reads, uint32_t read_len, uint64_t n_reads, uint32_t k,
                                     uint32_t strands, uint8_t *d_syms, cudaStream_t st) {
    const uint64_t total = n_reads * (uint64_t)(read_len - k + 1) * strands;
    if (!total) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((total * k / 16 + 256) / 256, (uint64_t)sm_count(device) * 16);
    g_launches++;
    expand_read_kmers_kernel<<<grid, 256, 0, st>>>(d_reads, read_len, n_reads, k, strands, d_syms);
    return cudaGetLastError();
}

cudaError_t launch_sum_strands(int device, const uint64_t *d_per_query, uint64_t n_windows, uint64_t *d_out, cudaStream_t st) {
    if (!n_windows) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n_windows + 255) / 256, (uint64_t)sm_count(device) * 16);
    g_launches++;
    sum_strands_kernel<<<grid, 256, 0, st>>>(d_per_query, n_windows, d_out);
    return cudaGetLastError();
}

}  // namespace msbwt
