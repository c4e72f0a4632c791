// stats_kernels.cu -- the COUNTING instantiation of the oct search kernel (count_kmers_oct_kernel<true>,
// oct_kernel.cuh): the same walk over live list A that also counts every index line it fetches.  Measurement aid
// for bench.py's roofline accounting (the exact algorithmic traffic of the implemented algorithm on a batch);
// never on a timed path.  A translation unit of its own because ptxas 12.9 crashes on a module that holds two
// instantiations of that kernel.
#include "oct_kernel.cuh"

namespace msbwt {

cudaError_t launch_count_oct_stats(int device, const IndexView &ix, const uint64_t *d_packed, uint32_t k, uint64_t n,
                                   uint64_t *d_out, unsigned long long *d_stats, cudaStream_t st) {
    if (!n) return cudaSuccess;
    if (n > kMaxPerLaunch || !ix.oct || index_is_wide(ix)) return cudaErrorInvalidValue;
    const PackedLayout lay = packed_layout(ix, k, n);
    static bool prepared[64] = {};
    if (device < 0 || device >= 64 || !prepared[device]) {
        if (cudaError_t e = cudaFuncSetAttribute((const void *)count_kmers_oct_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOctSmemPacked); e != cudaSuccess) return e;
        cudaFuncSetAttribute((const void *)count_kmers_oct_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (device >= 0 && device < 64) prepared[device] = true;
    }
    uint32_t *work = reinterpret_cast<uint32_t *>(const_cast<uint64_t *>(d_packed) + lay.work());
    if (cudaError_t e = cudaMemsetAsync(work, 0, sizeof(uint32_t), st); e != cudaSuccess) return e;
    if (cudaError_t e = cudaMemsetAsync(d_stats, 0, kOctStatWords * sizeof(unsigned long long), st); e != cudaSuccess) return e;
    const unsigned grid = oct_grid(device, (const void *)count_kmers_oct_kernel<true>, kOctSmemPacked, lay.n);
    g_launches++;
    count_kmers_oct_kernel<true><<<grid, kCountThreads, kOctSmemPacked, st>>>(ix, d_packed, lay, k, d_out, work, d_stats);
    return cudaGetLastError();
}

}  // namespace msbwt
