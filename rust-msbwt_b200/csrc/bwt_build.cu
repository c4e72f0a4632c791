// bwt_build.cu -- multi-string BWT construction for a set of reads (any lengths), on the device.
//
// Replaces what `msbwt2-build` does through DynamicBWT
// (src/bin/msbwt2-build.rs:19-114, src/dynamic_bwt.rs:305-381,453-473: one serial insert per symbol):
// the BWT of the string collection in "sorted insert" order, i.e. exactly naive_bwt's order
// (src/bwt_util.rs:154-171; equivalence tested by the reference at src/dynamic_bwt.rs:515-525) --
// suffixes compared symbol by symbol with '$' smallest, equal suffixes ordered by the lexicographic
// rank of the whole read -- emitted in the msbwt RLE byte format (src/bwt_converter.rs:52-56).
// It feeds the query path (the loader of capi.cu takes these bytes) and is how the 3 Gsymbol
// configuration is manufactured; nothing on the query path depends on it.
//
//   1. pack  : reads -> 3-bit symbols, 21 per u64 word (first symbol in the top bits, bit 63 clear), the
//              '$' terminator and the padding are zero, so integer order == lexicographic order.
//   2. reads : LSD radix sort of read ids over the words, last word first (CUB radix sort: plumbing).
//   3. suffix: ids (rank of the read) * (L+1) + offset start in tie-break order; LSD over the suffix's
//              21-symbol key words, extracted from the packed read by a funnel shift.
//   4. emit  : BWT[i] = the symbol before suffix i ('$' for offset 0); run heads -> run table -> RLE bytes.
//              (the last three steps are encode_rle_on_device, which the merge of bwt_merge.cu shares)
// Reads of different lengths (create_from_fastx takes any, src/dynamic_bwt.rs:453-473) use the same padded layout
// -- max length + 1 symbols per read, zeros after the '$' -- and simply list only the suffixes that exist (offsets
// 0..len of every read): a shorter suffix ends in '$' = 0 followed by zeros, which is exactly how naive_bwt's
// doubled rotations order it ('$' smallest, then the whole read, i.e. the read's rank).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/msbwt_gpu.h"
#include "engine.h"

namespace msbwt {

namespace {

constexpr uint32_t kKeySyms = 21;  // 3-bit symbols per key word
constexpr uint64_t kKeyMask = (1ull << 63) - 1;

__global__ void pack_reads_kernel(const uint8_t *__restrict__ reads, uint64_t n_reads, uint32_t len, uint32_t words,
                                  uint64_t *__restrict__ packed, uint32_t *__restrict__ bad) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_reads * words) return;
    const uint64_t r = t / words;
    const uint32_t w = (uint32_t)(t % words);
    const uint8_t *src = reads + r * len;
    uint64_t v = 0;
    for (uint32_t i = 0; i < kKeySyms; i++) {
        const uint32_t at = w * kKeySyms + i;
        uint32_t sy = 0;
        if (at < len) {
            sy = src[at];
            if (sy == 0 || sy >= (uint32_t)kAlphabet) { atomicOr(bad, 1u); sy = 1; }  // '$' inside a read / not a symbol
        }
        v |= (uint64_t)sy << (60 - 3 * i);
    }
    packed[t] = v;
}

// the same for reads of any length: read r is syms[offsets[r] .. offsets[r + 1])
__global__ void pack_ragged_kernel(const uint8_t *__restrict__ syms, const uint64_t *__restrict__ offsets, uint64_t n_reads,
                                   uint32_t words, uint64_t *__restrict__ packed, uint32_t *__restrict__ bad) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_reads * words) return;
    const uint64_t r = t / words;
    const uint32_t w = (uint32_t)(t % words);
    const uint8_t *src = syms + offsets[r];
    const uint64_t len = offsets[r + 1] - offsets[r];
    uint64_t v = 0;
    for (uint32_t i = 0; i < kKeySyms; i++) {
        const uint32_t at = w * kKeySyms + i;
        uint32_t sy = 0;
        if (at < len) {
            sy = src[at];
            if (sy == 0 || sy >= (uint32_t)kAlphabet) { atomicOr(bad, 1u); sy = 1; }
        }
        v |= (uint64_t)sy << (60 - 3 * i);
    }
    packed[t] = v;
}

// suffixes per read (length + 1: the '$' rotation included), in the reads' SORTED order
__global__ void sorted_suffix_counts_kernel(const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ ids, uint64_t n_reads,
                                            uint64_t *__restrict__ counts) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_reads) counts[r] = offsets[(uint64_t)ids[r] + 1] - offsets[ids[r]] + 1;
}

// suffix ids of the sorted read r: r * l1 + o, o = 0 .. length(r), at starts[r] ..
template <class IdT>
__global__ void fill_suffix_ids_kernel(const uint64_t *__restrict__ starts, const uint64_t *__restrict__ counts, uint64_t n_reads,
                                       uint32_t l1, IdT *__restrict__ sids) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += step) {
        IdT *dst = sids + starts[r];
        const uint64_t c = counts[r];
        for (uint64_t o = 0; o < c; o++) dst[o] = (IdT)(r * l1 + o);
    }
}

// key word w of read ids[i]
__global__ void read_keys_kernel(const uint64_t *__restrict__ packed, const uint32_t *__restrict__ ids, uint64_t n_reads,
                                 uint32_t words, uint32_t w, uint64_t *__restrict__ keys) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_reads) keys[i] = packed[(uint64_t)ids[i] * words + w];
}

__global__ void permute_reads_kernel(const uint64_t *__restrict__ packed, const uint32_t *__restrict__ ids, uint64_t n_reads,
                                     uint32_t words, uint64_t *__restrict__ sorted) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_reads * words) return;
    sorted[t] = packed[(uint64_t)ids[t / words] * words + t % words];
}

template <class IdT>
__global__ void iota_kernel(IdT *__restrict__ ids, uint64_t n) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) ids[i] = (IdT)i;
}

// key word w (symbols o + 21w .. o + 21w + 20) of suffix sid = read * l1 + o; `sorted` has words + 1 zero-padded
// words per read so that the funnel shift may touch the word after the last
template <class IdT>
__global__ void suffix_keys_kernel(const uint64_t *__restrict__ sorted, const IdT *__restrict__ sids, uint64_t n,
                                   uint32_t l1, uint32_t stride_words, uint32_t w, uint64_t *__restrict__ keys) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const uint64_t sid = (uint64_t)sids[i];
        const uint64_t r = sid / l1;
        const uint32_t o = (uint32_t)(sid - r * l1);
        const uint32_t first = o + w * kKeySyms;  // first symbol of this key word within the read
        uint64_t key = 0;
        if (first < l1) {
            const uint32_t q = first / kKeySyms, sh = 3u * (first % kKeySyms);
            const uint64_t *p = sorted + r * stride_words + q;
            key = (p[0] << sh) & kKeyMask;
            if (sh) key |= p[1] >> (63u - sh);
        }
        keys[i] = key;
    }
}

template <class IdT>
__global__ void emit_bwt_kernel(const uint64_t *__restrict__ sorted, const IdT *__restrict__ sids, uint64_t n,
                                uint32_t l1, uint32_t stride_words, uint8_t *__restrict__ bwt) {
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const uint64_t sid = (uint64_t)sids[i];
        const uint64_t r = sid / l1;
        const uint32_t o = (uint32_t)(sid - r * l1);
        uint8_t sy = 0;  // the rotation that starts at the read's first symbol is preceded by its '$'
        if (o) {
            const uint32_t at = o - 1;
            sy = (uint8_t)((sorted[r * stride_words + at / kKeySyms] >> (60 - 3 * (at % kKeySyms))) & 7u);
        }
        bwt[i] = sy;
    }
}

struct RunHead {
    const uint8_t *bwt;
    __host__ __device__ bool operator()(uint64_t i) const {
#ifdef __CUDA_ARCH__
        return i == 0 || bwt[i] != bwt[i - 1];
#else
        (void)i;
        return false;
#endif
    }
};

// digits of run r (little-endian base 32, src/bwt_converter.rs:52-56)
__global__ void run_digits_kernel(const uint64_t *__restrict__ starts, uint64_t n_runs, uint64_t total,
                                  uint8_t *__restrict__ ndigits) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    uint64_t len = (r + 1 < n_runs ? starts[r + 1] : total) - starts[r];
    uint8_t d = 0;
    while (len) { d++; len >>= 5; }
    ndigits[r] = d;
}

struct WidenDigits {
    __host__ __device__ uint64_t operator()(uint8_t v) const { return v; }
};

__global__ void emit_rle_kernel(const uint8_t *__restrict__ bwt, const uint64_t *__restrict__ starts,
                                const uint64_t *__restrict__ offsets, uint64_t n_runs, uint64_t total,
                                uint8_t *__restrict__ rle) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint64_t s = starts[r];
    uint64_t len = (r + 1 < n_runs ? starts[r + 1] : total) - s;
    const uint8_t sym = bwt[s];
    uint8_t *out = rle + offsets[r];
    while (len) { *out++ = (uint8_t)(sym | ((len & 31u) << 3)); len >>= 5; }
}

#define W_TRY(e) CU_TRY_IN("bwt build: ", e)

constexpr unsigned kGridCap = 148 * 32;
unsigned grid_for(uint64_t n, unsigned threads = 256) {
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + threads - 1) / threads, kGridCap));
}

// sorts (key, id) pairs by the 63 key bits, stably; ids end up in ids.Current()
template <class IdT>
int sort_pass(cub::DoubleBuffer<uint64_t> &keys, cub::DoubleBuffer<IdT> &ids, uint64_t n, void *d_temp, size_t temp_bytes) {
    W_TRY(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, keys, ids, (int64_t)n, 0, 63));
    return MSBWT_OK;
}

// `d_starts` / `d_counts` (reads of different lengths): where the suffixes of sorted read r go and how many it has;
// nullptr: every read has l1 suffixes
template <class IdT>
int suffix_sort_and_emit(const uint64_t *d_sorted, uint64_t n_reads, uint64_t n, uint32_t l1, uint32_t stride_words, uint32_t key_words,
                         const uint64_t *d_starts, const uint64_t *d_counts, uint8_t *d_bwt, DeviceScratch &tmp) {
    uint64_t *k0 = nullptr, *k1 = nullptr;
    IdT *v0 = nullptr, *v1 = nullptr;
    W_TRY(tmp.alloc(&k0, n));
    W_TRY(tmp.alloc(&k1, n));
    W_TRY(tmp.alloc(&v0, n));
    W_TRY(tmp.alloc(&v1, n));
    cub::DoubleBuffer<uint64_t> keys(k0, k1);
    cub::DoubleBuffer<IdT> ids(v0, v1);
    void *d_temp = nullptr;
    size_t temp_bytes = 0;
    W_TRY(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, ids, (int64_t)n, 0, 63));
    W_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
    if (d_starts) fill_suffix_ids_kernel<IdT><<<grid_for(n_reads), 256>>>(d_starts, d_counts, n_reads, l1, ids.Current());
    else iota_kernel<IdT><<<grid_for(n), 256>>>(ids.Current(), n);
    W_TRY(cudaGetLastError());
    for (uint32_t w = key_words; w-- > 0;) {
        suffix_keys_kernel<IdT><<<grid_for(n), 256>>>(d_sorted, ids.Current(), n, l1, stride_words, w, keys.Current());
        W_TRY(cudaGetLastError());
        if (int rc = sort_pass<IdT>(keys, ids, n, d_temp, temp_bytes); rc != MSBWT_OK) return rc;
        g_launches += 2;
    }
    emit_bwt_kernel<IdT><<<grid_for(n), 256>>>(d_sorted, ids.Current(), n, l1, stride_words, d_bwt);
    W_TRY(cudaGetLastError());
    W_TRY(cudaDeviceSynchronize());
    tmp.release(k0); tmp.release(k1); tmp.release(v0); tmp.release(v1); tmp.release(d_temp);
    return MSBWT_OK;
}

}  // namespace

// d_bwt: n symbol bytes on the current device -> *d_rle_out, a cudaMalloc'd buffer of *rle_len msbwt RLE bytes
// (src/bwt_converter.rs:52-56; the caller frees it).  Shared by the builder above and the merge (bwt_merge.cu), so
// both emit the same canonical encoding.
int encode_rle_on_device(const uint8_t *d_bwt, uint64_t n, uint8_t **d_rle_out, uint64_t *rle_len) {
    *d_rle_out = nullptr;
    *rle_len = 0;
    if (!n) return MSBWT_OK;
    DeviceScratch tmp;
    // run heads -> run table (select in chunks of 2^30 positions) -> digits -> RLE bytes
    const uint64_t kChunk = 1ull << 30;
    uint64_t *d_count = nullptr;
    W_TRY(tmp.alloc(&d_count, 1));
    void *d_temp = nullptr;
    size_t temp_bytes = 0, need = 0;
    using HeadIt = cub::TransformInputIterator<bool, RunHead, cub::CountingInputIterator<uint64_t>>;
    using CountIt = cub::TransformInputIterator<uint64_t, RunHead, cub::CountingInputIterator<uint64_t>>;
    {
        cub::CountingInputIterator<uint64_t> idx(0);
        HeadIt heads(idx, RunHead{d_bwt});
        CountIt ones(idx, RunHead{d_bwt});
        W_TRY(cub::DeviceReduce::Sum(nullptr, need, ones, d_count, (int64_t)std::min(kChunk, n)));
        temp_bytes = need;
        W_TRY(cub::DeviceSelect::Flagged(nullptr, need, idx, heads, (uint64_t *)nullptr, d_count, (int64_t)std::min(kChunk, n)));
        temp_bytes = std::max(temp_bytes, need);
    }
    W_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
    uint64_t n_runs = 0;
    std::vector<uint64_t> chunk_runs;
    for (uint64_t b = 0; b < n; b += kChunk) {
        cub::CountingInputIterator<uint64_t> idx(b);
        CountIt ones(idx, RunHead{d_bwt});
        size_t tb = temp_bytes;
        W_TRY(cub::DeviceReduce::Sum(d_temp, tb, ones, d_count, (int64_t)std::min(kChunk, n - b)));
        uint64_t c = 0;
        W_TRY(cudaMemcpy(&c, d_count, sizeof(c), cudaMemcpyDeviceToHost));
        chunk_runs.push_back(c);
        n_runs += c;
    }
    uint64_t *d_starts = nullptr, *d_byte_offsets = nullptr;
    uint8_t *d_ndigits = nullptr;
    W_TRY(tmp.alloc(&d_starts, n_runs));
    uint64_t done = 0;
    for (uint64_t b = 0, ci = 0; b < n; b += kChunk, ci++) {
        cub::CountingInputIterator<uint64_t> idx(b);
        HeadIt heads(idx, RunHead{d_bwt});
        size_t tb = temp_bytes;
        W_TRY(cub::DeviceSelect::Flagged(d_temp, tb, idx, heads, d_starts + done, d_count, (int64_t)std::min(kChunk, n - b)));
        done += chunk_runs[ci];
    }
    W_TRY(tmp.alloc(&d_ndigits, n_runs));
    W_TRY(tmp.alloc(&d_byte_offsets, n_runs + 1));
    run_digits_kernel<<<(unsigned)((n_runs + 255) / 256), 256>>>(d_starts, n_runs, n, d_ndigits);
    W_TRY(cudaGetLastError());
    {
        cub::TransformInputIterator<uint64_t, WidenDigits, const uint8_t *> in(d_ndigits, WidenDigits{});
        void *d_temp2 = nullptr;
        size_t tb = 0;
        W_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, in, d_byte_offsets, (int64_t)n_runs));
        W_TRY(tmp.alloc((uint8_t **)&d_temp2, tb));
        W_TRY(cub::DeviceScan::ExclusiveSum(d_temp2, tb, in, d_byte_offsets, (int64_t)n_runs));
    }
    uint64_t last_off = 0;
    uint8_t last_nd = 0;
    W_TRY(cudaMemcpy(&last_off, d_byte_offsets + (n_runs - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost));
    W_TRY(cudaMemcpy(&last_nd, d_ndigits + (n_runs - 1), 1, cudaMemcpyDeviceToHost));
    const uint64_t bytes = last_off + last_nd;
    uint8_t *d_rle = nullptr;
    W_TRY(cudaMalloc((void **)&d_rle, bytes));
    emit_rle_kernel<<<(unsigned)((n_runs + 255) / 256), 256>>>(d_bwt, d_starts, d_byte_offsets, n_runs, n, d_rle);
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) { cudaFree(d_rle); W_TRY(e); }
    if (cudaError_t e = cudaDeviceSynchronize(); e != cudaSuccess) { cudaFree(d_rle); W_TRY(e); }
    g_launches += 4;
    *d_rle_out = d_rle;
    *rle_len = bytes;
    return MSBWT_OK;
}

// d_reads: symbol bytes (1..5) on the current device -- n_reads * read_len of them (d_offsets == nullptr: reads of one
// length), or read r at d_reads[d_offsets[r] .. d_offsets[r + 1]) with read_len = the longest read (d_offsets: n_reads + 1
// offsets on the device).  On success *d_rle_out is a cudaMalloc'd buffer of *rle_len RLE bytes (the caller frees it)
// and *total = the number of symbols of the BWT (every read's length + 1).
int build_rle_bwt_on_device(const uint8_t *d_reads, const uint64_t *d_offsets, uint64_t n_reads, uint32_t read_len,
                            uint8_t **d_rle_out, uint64_t *rle_len, uint64_t *total) {
    *d_rle_out = nullptr;
    *rle_len = 0;
    *total = 0;
    if (!n_reads) return MSBWT_OK;
    if ((!read_len && !d_offsets) || (read_len && !d_reads)) return fail(MSBWT_EINVAL, "bwt build: empty reads or NULL buffer");
    if (n_reads >> 32) return fail(MSBWT_EINVAL, "bwt build: more than 2^32 reads");
    if (read_len == 0xFFFFFFFFu) return fail(MSBWT_EINVAL, "bwt build: read too long");
    const uint32_t l1 = read_len + 1;
    uint64_t n = n_reads * l1;  // (reads of different lengths: the suffixes that exist, counted below)
    const uint32_t words = (l1 + kKeySyms - 1) / kKeySyms;  // key words per read ('$' included)
    const uint32_t stride_words = words + 1;                // + one zero word for the funnel shift
    DeviceScratch tmp;
    uint64_t *d_packed = nullptr, *d_sorted = nullptr, *d_suffix_counts = nullptr, *d_suffix_starts = nullptr;
    uint32_t *d_bad = nullptr;
    uint8_t *d_bwt = nullptr;

    // 1. pack
    W_TRY(tmp.alloc(&d_packed, n_reads * stride_words));
    W_TRY(tmp.alloc(&d_sorted, n_reads * stride_words));
    W_TRY(tmp.alloc(&d_bad, 1));
    W_TRY(cudaMemset(d_bad, 0, sizeof(uint32_t)));
    if (d_offsets) pack_ragged_kernel<<<(unsigned)((n_reads * stride_words + 255) / 256), 256>>>(d_reads, d_offsets, n_reads, stride_words, d_packed, d_bad);
    else pack_reads_kernel<<<(unsigned)((n_reads * stride_words + 255) / 256), 256>>>(d_reads, n_reads, read_len, stride_words, d_packed, d_bad);
    W_TRY(cudaGetLastError());
    uint32_t bad = 0;
    W_TRY(cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost));
    if (bad) return fail(MSBWT_EINVAL, "bwt build: a read holds '$' (0) or a symbol >= 6");
    g_launches++;

    // 2. sort the reads
    {
        uint64_t *k0 = nullptr, *k1 = nullptr;
        uint32_t *v0 = nullptr, *v1 = nullptr;
        W_TRY(tmp.alloc(&k0, n_reads));
        W_TRY(tmp.alloc(&k1, n_reads));
        W_TRY(tmp.alloc(&v0, n_reads));
        W_TRY(tmp.alloc(&v1, n_reads));
        cub::DoubleBuffer<uint64_t> keys(k0, k1);
        cub::DoubleBuffer<uint32_t> ids(v0, v1);
        void *d_temp = nullptr;
        size_t temp_bytes = 0;
        W_TRY(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, ids, (int64_t)n_reads, 0, 63));
        W_TRY(tmp.alloc((uint8_t **)&d_temp, temp_bytes));
        iota_kernel<uint32_t><<<grid_for(n_reads), 256>>>(ids.Current(), n_reads);
        W_TRY(cudaGetLastError());
        for (uint32_t w = words; w-- > 0;) {
            read_keys_kernel<<<(unsigned)((n_reads + 255) / 256), 256>>>(d_packed, ids.Current(), n_reads, stride_words, w, keys.Current());
            W_TRY(cudaGetLastError());
            if (int rc = sort_pass<uint32_t>(keys, ids, n_reads, d_temp, temp_bytes); rc != MSBWT_OK) return rc;
            g_launches += 2;
        }
        permute_reads_kernel<<<(unsigned)((n_reads * stride_words + 255) / 256), 256>>>(d_packed, ids.Current(), n_reads, stride_words, d_sorted);
        W_TRY(cudaGetLastError());
        if (d_offsets) {  // suffixes per sorted read -> where each read's suffix ids start -> how many there are
            W_TRY(tmp.alloc(&d_suffix_counts, n_reads));
            W_TRY(tmp.alloc(&d_suffix_starts, n_reads));
            sorted_suffix_counts_kernel<<<(unsigned)((n_reads + 255) / 256), 256>>>(d_offsets, ids.Current(), n_reads, d_suffix_counts);
            W_TRY(cudaGetLastError());
            void *d_t2 = nullptr;
            size_t tb = 0;
            W_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_suffix_counts, d_suffix_starts, (int64_t)n_reads));
            W_TRY(tmp.alloc((uint8_t **)&d_t2, tb));
            W_TRY(cub::DeviceScan::ExclusiveSum(d_t2, tb, d_suffix_counts, d_suffix_starts, (int64_t)n_reads));
            uint64_t last_start = 0, last_count = 0;
            W_TRY(cudaMemcpy(&last_start, d_suffix_starts + (n_reads - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost));
            W_TRY(cudaMemcpy(&last_count, d_suffix_counts + (n_reads - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost));
            n = last_start + last_count;
            tmp.release(d_t2);
        }
        W_TRY(cudaDeviceSynchronize());
        tmp.release(k0); tmp.release(k1); tmp.release(v0); tmp.release(v1); tmp.release(d_temp);
        tmp.release(d_packed);
    }

    // 3. sort the suffixes, 4a. emit the BWT symbols
    W_TRY(tmp.alloc(&d_bwt, n));
    // (a suffix id is read rank * l1 + offset in the padded layout, whatever the reads' own lengths)
    const int rc = ((n_reads * l1) >> 32)
                       ? suffix_sort_and_emit<uint64_t>(d_sorted, n_reads, n, l1, stride_words, words, d_suffix_starts, d_suffix_counts, d_bwt, tmp)
                       : suffix_sort_and_emit<uint32_t>(d_sorted, n_reads, n, l1, stride_words, words, d_suffix_starts, d_suffix_counts, d_bwt, tmp);
    if (rc != MSBWT_OK) return rc;
    tmp.release(d_sorted);

    // 4b. run table -> RLE bytes
    if (int rc2 = encode_rle_on_device(d_bwt, n, d_rle_out, rle_len); rc2 != MSBWT_OK) return rc2;
    *total = n;
    return MSBWT_OK;
}

}  // namespace msbwt
