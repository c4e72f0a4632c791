// handle.h -- what an `msbwt_index` handle owns (per-device replicas, staging lanes, scratch), shared by the
// translation units that implement the C ABI: capi.cu (construction, accessors, device-buffer entry points,
// inspection) and hostpath.cu (host-buffer entry points: the chunk pipelines and the multi-GPU batch split).  Errors
// and launch counts are reported through engine.h, by the function that meets them.
#pragma once
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/msbwt_gpu.h"
#include "engine.h"
#include "hostpack.h"

namespace msbwt {

// grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

// grow-only pinned host buffer
struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// per-device staging for the host-buffer entry points: several lanes so that the host-side packing
// and copy-in of the next chunks overlap the kernels of the current one
constexpr int kPackLanes = 3;  // lanes whose input is packed by the host pool (or every lane of the byte path)
constexpr int kRawLanes = 2;   // hybrid route only: lanes that take their chunk as raw symbol bytes over PCIe
constexpr int kLanes = kPackLanes + kRawLanes;
struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t h2d_done = nullptr;  // the lane's pinned staging buffer may be rewritten after this
    cudaEvent_t d2h_done = nullptr;  // the lane's pinned result buffer holds the counts of its last chunk after this
    DevBuf in_a, in_b, in_c, packed, out_a, out_b;
    PinnedBuf h_stage;               // input staging: host-packed words, or a copy of a PAGEABLE caller buffer's chunk
    PinnedBuf h_out;                 // result staging when the caller's output buffer is pageable
    uint64_t pend_first = 0, pend_count = 0;  // queries whose counts wait in h_out to be copied to the caller (0 = none)
};

struct Replica {
    int device = -1;
    uint4 *d_blocks = nullptr;
    uint32_t *d_aux = nullptr;
    void *d_table = nullptr;   // suffix table of depth table_s (0 = none)
    void *d_table_lower[3] = {nullptr, nullptr, nullptr};  // depths table_s - 1 .. table_s - 3, kept so that a
                                                           // multi-step image always finds a depth that leaves a multiple
                                                           // of its stride (pair: one level, quad: three)
    uint32_t table_s = 0;
    PairImage pair;            // 128-byte pair lines (layout.h), when the index lives in HBM
    QuadImage quad;            // 32-byte quad sectors (layout.h), when the index lives in HBM and the image fits
    OctImage oct;              // 128-byte oct lines (layout.h), next to the quad image when positions are 32-bit
    FinImage fin;              // final-step lines (layout.h), built by default on top of the oct image; final_index = 0
                               // turns them off
    int lanes = 1;           // kernel mapping: 1 = thread per query, 2 = lane pair per query (kernels.cu)
    uint64_t *d_cbase = nullptr;
    IndexView view{};
    std::mutex mu;
    Lane lane[kLanes];
    DevBuf dev_packed;       // scratch for the *_device entry points
    cudaEvent_t dev_packed_free = nullptr;  // recorded after the last kernel that uses dev_packed: the next user's
                                            // stream waits on it (the device entry points are asynchronous and may
                                            // be called on different streams)
    std::unique_ptr<HostPool> pool;  // host-side packers of this replica's chunks (hostpath.cu), created on first use
    uint32_t *d_status = nullptr;  // [0,kLanes): per-lane flags; [kStatusDev]: device entry points
    uint32_t *h_status = nullptr;  // pinned mirror

    ~Replica() {
        if (device < 0) return;
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(device);
        for (auto &ln : lane) {
            if (ln.stream) cudaStreamDestroy(ln.stream);
            if (ln.h2d_done) cudaEventDestroy(ln.h2d_done);
            if (ln.d2h_done) cudaEventDestroy(ln.d2h_done);
            ln.h_stage.release();
            ln.h_out.release();
            ln.in_a.release(); ln.in_b.release(); ln.in_c.release();
            ln.packed.release(); ln.out_a.release(); ln.out_b.release();
        }
        dev_packed.release();
        if (dev_packed_free) cudaEventDestroy(dev_packed_free);
        if (d_status) cudaFree(d_status);
        if (h_status) cudaFreeHost(h_status);
        if (d_blocks) cudaFree(d_blocks);
        if (d_aux) cudaFree(d_aux);
        if (d_table) cudaFree(d_table);
        for (void *t : d_table_lower) if (t) cudaFree(t);
        free_pair_image(pair);
        free_quad_image(quad);
        free_oct_image(oct);
        free_fin_image(fin);
        if (d_cbase) cudaFree(d_cbase);
        cudaSetDevice(cur);
    }
};

struct DeviceGuard {
    int prev = 0;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); cudaSetDevice(dev); }
    ~DeviceGuard() { cudaSetDevice(prev); }
};

constexpr int kStatusWords = 8, kStatusDev = 7;
constexpr int kOctAutoTableS = 14;  // automatic suffix-table depth under an oct image (levels 11..14 are kept)
constexpr uint64_t kChunkQueries = 1ull << 20;  // host-path pipeline granularity (byte route)
constexpr uint64_t kPackedChunkQueries = 1ull << 19;  // packed route: smaller chunks fill / drain the pipeline sooner
constexpr uint64_t kChunkBytes = 1ull << 27;

}  // namespace msbwt

struct msbwt_index {
    uint64_t total = 0;
    uint64_t counts[msbwt::kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t start[msbwt::kAlphabet] = {0, 0, 0, 0, 0, 0};
    std::vector<std::unique_ptr<msbwt::Replica>> reps;
};
