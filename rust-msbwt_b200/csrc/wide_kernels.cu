// wide_kernels.cu -- the WIDE instantiation of the oct search kernel (count_kmers_oct_kernel<false, true>,
// oct_kernel.cuh): live list A over the oct and final-step images of an index whose positions need 64 bits -- 2^32
// symbols and more (the reference is u64 throughout: BWTRange src/msbwt_core.rs:18-24, RleBWT src/rle_bwt.rs:14-24),
// or an index cut into several superblocks.  A translation unit of its own because ptxas 12.9 crashes on a module
// that holds two instantiations of that kernel.
//
// Replaces BWT::count_kmer (src/msbwt_core.rs:125-161) on such an index: ten constrain_range steps
// (src/rle_bwt.rs:202-287) per oct line, the last twenty per final-step line, one-symbol steps for what is left.
#include "oct_kernel.cuh"

namespace msbwt {

cudaError_t launch_count_oct_wide(int device, const IndexView &ix, const uint64_t *d_packed, const PackedLayout &lay,
                                  uint32_t k, uint64_t *d_out, cudaStream_t st) {
    const void *kernel = (const void *)count_kmers_oct_kernel<false, true>;
    static bool prepared[64] = {};  // per device: 3 CTAs x 51 KB of staging per SM need the large shared-memory configuration
    if (device < 0 || device >= 64 || !prepared[device]) {
        if (cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kOctSmemWide); e != cudaSuccess) return e;
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (device >= 0 && device < 64) prepared[device] = true;
    }
    uint32_t *work = reinterpret_cast<uint32_t *>(const_cast<uint64_t *>(d_packed) + lay.work());  // engine scratch (quad_kernels.cu)
    if (cudaError_t e = cudaMemsetAsync(work, 0, sizeof(uint32_t), st); e != cudaSuccess) return e;
    const unsigned grid = oct_grid(device, kernel, kOctSmemWide, lay.n);
    count_kmers_oct_kernel<false, true><<<grid, kCountThreads, kOctSmemWide, st>>>(ix, d_packed, lay, k, d_out, work);
    return cudaGetLastError();
}

}  // namespace msbwt
