// hostpath.cu -- the host-buffer entry points of the C ABI (include/msbwt_gpu.h): chunk pipelines between the
// caller's host memory and the kernels, and the multi-GPU batch split.
//
// Reference surface: `BWT::count_kmer` / `constrain_range` as implemented by `RleBWT` (src/msbwt_core.rs:125-161,
// src/rle_bwt.rs:202-287) take `&self` on a structure of owned, immutable tables (src/rle_bwt.rs:14-24), so any
// number of queries may run against one index at once.  Here: the index is REPLICATED on every device of the
// handle, a batch is cut into one contiguous slice per device, every slice is driven by its own host thread
// through that replica's lanes (stream + staging buffers: copy-in, kernels and copy-out of consecutive chunks
// overlap), and the results land in disjoint slices of the caller's output -- a host-side gather, no collective.
// There is no CPU fallback: every route ends in kernel launches.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "handle.h"
#include "kernel_common.cuh"

using namespace msbwt;

namespace {

thread_local uint64_t g_last_h2d = 0, g_last_d2h = 0;

// one device's share of a host batch
struct Slice {
    uint64_t begin, end;
    uint64_t len() const { return end - begin; }
};
Slice slice_for(uint64_t n, size_t d, size_t ndev) { return {n * d / ndev, n * (d + 1) / ndev}; }

struct Xfer { uint64_t h2d = 0, d2h = 0; };

// where the counts of a call go: u64 (the reference's type) or, for an index below 2^32 symbols, u32 (half the
// bytes on the way back)
struct CountsOut {
    uint64_t *o64 = nullptr;
    uint32_t *o32 = nullptr;
};

// Runs fn(replica, slice, xfer) for every replica of the handle on its own thread (the caller's for replica 0) with
// that replica's device current, and joins.  Whatever a route does -- including returning early on a CUDA error --
// every lane stream of the replica is drained before its thread leaves, so no copy of this call is still reading
// or writing the caller's buffers when the call returns.  The first failure (by device order) is reported.
// Caller holds the replica locks when fn uses the lanes.
template <class F>
int run_on_replicas(const msbwt_index *idx, uint64_t n, F &&fn) {
    const size_t ndev = idx->reps.size();
    struct Res { int rc = MSBWT_OK; std::string err; Xfer x; };
    std::vector<Res> res(ndev);
    auto body = [&](size_t d) {
        Replica &rep = *idx->reps[d];
        DeviceGuard guard(rep.device);
        const Slice sl = slice_for(n, d, ndev);
        int rc = sl.len() ? fn(rep, sl, res[d].x) : MSBWT_OK;
        for (auto &ln : rep.lane) {
            if (!ln.stream) continue;
            const cudaError_t e = cudaStreamSynchronize(ln.stream);
            if (e != cudaSuccess && rc == MSBWT_OK) rc = fail(MSBWT_ECUDA, std::string("draining the lanes: ") + cudaGetErrorString(e));
        }
        res[d].rc = rc;
        if (rc != MSBWT_OK) res[d].err = g_last_error;
    };
    if (ndev == 1) {
        body(0);
    } else {
        std::vector<std::thread> workers;
        for (size_t d = 1; d < ndev; d++) workers.emplace_back(body, d);
        body(0);
        for (auto &w : workers) w.join();
    }
    int rc = MSBWT_OK;
    for (auto &r : res) {
        g_last_h2d += r.x.h2d;
        g_last_d2h += r.x.d2h;
        if (r.rc != MSBWT_OK && rc == MSBWT_OK) {
            rc = r.rc;
            g_last_error = r.err;
        }
    }
    return rc;
}

// Chunk size of a slice: about eight chunks per slice so that copy-in, kernels and copy-out overlap, never below
// 128 Ki queries (per-chunk launch overhead) nor above `max_chunk` / kChunkBytes of input.
uint64_t pick_chunk(uint64_t slice_len, uint64_t max_chunk, uint64_t in_bytes_per_query) {
    uint64_t c = std::max<uint64_t>(slice_len / 8, 1ull << 17);
    c = std::min(c, max_chunk);
    if (in_bytes_per_query && c * in_bytes_per_query > kChunkBytes) c = std::max<uint64_t>(1, kChunkBytes / in_bytes_per_query);
    return std::max<uint64_t>(1, std::min(c, slice_len));
}

int reset_status(Replica &rep) {
    CU_TRY(cudaMemsetAsync(rep.d_status, 0, kLanes * sizeof(uint32_t), rep.lane[0].stream));
    CU_TRY(cudaStreamSynchronize(rep.lane[0].stream));
    return MSBWT_OK;
}

// after the lanes were drained: did any chunk of this replica see a symbol >= 6 (or a bad range)?
int check_status(Replica &rep, const char *what) {
    CU_TRY(cudaMemcpy(rep.h_status, rep.d_status, kLanes * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (std::any_of(rep.h_status, rep.h_status + kLanes, [](uint32_t v) { return v != 0; }))
        return fail(MSBWT_EINVAL, std::string(what) + ": symbol >= 6 or range out of bounds in the batch");
    return MSBWT_OK;
}

int drain(Replica &rep) {
    for (auto &ln : rep.lane) CU_TRY(cudaStreamSynchronize(ln.stream));
    return MSBWT_OK;
}

// Host threads a replica's packers may use: the process's share of the host (hostpack.cpp) divided by the
// handle's devices, each of which is fed by its own thread.
int replica_pack_threads(size_t ndev) { return std::max(1, host_threads_available() / (int)std::max<size_t>(1, ndev)); }

// true when `p` is page-locked host memory the copy engine can read / write while the host does something else
// (cudaMemcpyAsync on pageable memory stages through the driver and holds the calling thread)
bool is_pinned_host(const void *p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

HostPool &replica_pool(Replica &rep, size_t ndev) {
    const int want = replica_pack_threads(ndev);
    if (!rep.pool || rep.pool->size() != want) rep.pool = std::make_unique<HostPool>(want);
    return *rep.pool;
}

struct PoolSession {  // the workers stay hot for the duration of one call only
    HostPool &p;
    explicit PoolSession(HostPool &pool) : p(pool) { p.begin_session(); }
    ~PoolSession() { p.end_session(); }
};

// PAGEABLE caller buffers (a Rust Vec, a numpy array): the copy engine cannot touch them asynchronously -- measured
// on B200, 117 ms per 100 M packed 31-mers through cudaMemcpyAsync on pageable memory against 18.8 ms on pinned
// memory (profiles/r2p_e2e_probe.log).  So a pageable input chunk is first copied into the lane's pinned staging
// buffer by the replica's worker threads, and a pageable output receives its counts from the lane's pinned result
// buffer the same way once the lane's copy-out has completed; the copy engines keep running underneath.
struct HostStage {
    HostPool *pool = nullptr;
    bool in = false, out = false;
    CountsOut dst;
    size_t out_elem = sizeof(uint64_t);
};

void parallel_copy(HostPool *pool, void *dst, const void *src, size_t bytes) {
    if (!pool || pool->size() == 1 || bytes < (1u << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    pool->run([&](int tid, int nt) {
        const size_t a = bytes * (size_t)tid / (size_t)nt, b = bytes * (size_t)(tid + 1) / (size_t)nt;
        memcpy((char *)dst + a, (const char *)src + a, b - a);
    });
}

HostStage make_stage(Replica &rep, size_t ndev, const void *in_ptr, CountsOut out) {
    HostStage hs;
    hs.dst = out;
    hs.out_elem = out.o32 ? sizeof(uint32_t) : sizeof(uint64_t);
    hs.in = in_ptr && !is_pinned_host(in_ptr);
    hs.out = !is_pinned_host(out.o32 ? (const void *)out.o32 : (const void *)out.o64);
    if (hs.in || hs.out) hs.pool = &replica_pool(rep, ndev);
    for (auto &ln : rep.lane) ln.pend_count = 0;
    return hs;
}

// the counts of the lane's last chunk, waiting in its pinned result buffer -> the caller's (pageable) output
int flush_lane_output(Lane &ln, HostStage &hs) {
    if (!ln.pend_count) return MSBWT_OK;
    CU_TRY(cudaEventSynchronize(ln.d2h_done));
    char *dst = hs.dst.o32 ? (char *)(hs.dst.o32 + ln.pend_first) : (char *)(hs.dst.o64 + ln.pend_first);
    parallel_copy(hs.pool, dst, ln.h_out.p, ln.pend_count * hs.out_elem);
    ln.pend_count = 0;
    return MSBWT_OK;
}

int flush_all_outputs(Replica &rep, HostStage &hs) {
    for (auto &ln : rep.lane)
        if (int rc = flush_lane_output(ln, hs); rc != MSBWT_OK) return rc;
    return MSBWT_OK;
}

// `bytes` of the caller's input for this chunk, where the copy engine may read them: the caller's own (pinned)
// memory, or the lane's staging buffer after a copy (the previous copy-in from that buffer has completed)
int stage_input(Lane &ln, HostStage &hs, const void *src, size_t bytes, const void **where) {
    *where = src;
    if (!hs.in || !bytes) return MSBWT_OK;
    CU_TRY(cudaEventSynchronize(ln.h2d_done));
    parallel_copy(hs.pool, ln.h_stage.p, src, bytes);
    *where = ln.h_stage.p;
    return MSBWT_OK;
}

// search the lane's packed scratch and send the counts of queries [b, b + m) home
int search_and_copy_out(Replica &rep, Lane &ln, uint32_t k, uint64_t b, uint64_t m, HostStage &hs, bool with_b, Xfer &x) {
    CU_TRY(launch_count_packed(rep.device, rep.view, rep.lanes, ln.packed.as<uint64_t>(), k, m, ln.out_a.as<uint64_t>(),
                               ln.stream, with_b));
    const void *d_res = ln.out_a.p;
    if (hs.dst.o32) {
        CU_TRY(launch_narrow_counts(rep.device, ln.out_a.as<uint64_t>(), m, ln.out_b.as<uint32_t>(), ln.stream));
        d_res = ln.out_b.p;
    }
    void *h_res = hs.dst.o32 ? (void *)(hs.dst.o32 + b) : (void *)(hs.dst.o64 + b);
    if (hs.out) h_res = ln.h_out.p;
    CU_TRY(cudaMemcpyAsync(h_res, d_res, m * hs.out_elem, cudaMemcpyDeviceToHost, ln.stream));
    x.d2h += m * hs.out_elem;
    if (hs.out) {
        CU_TRY(cudaEventRecord(ln.d2h_done, ln.stream));
        ln.pend_first = b;
        ln.pend_count = m;
    }
    return MSBWT_OK;
}

int reserve_search_buffers(Replica &rep, Lane &ln, uint32_t k, uint64_t chunk, const HostStage &hs) {
    CU_TRY(ln.packed.reserve(packed_layout(rep.view, k, std::max<uint64_t>(1, chunk)).total() * sizeof(uint64_t)));
    CU_TRY(ln.out_a.reserve(std::max<uint64_t>(1, chunk) * sizeof(uint64_t)));
    if (hs.dst.o32) CU_TRY(ln.out_b.reserve(std::max<uint64_t>(1, chunk) * sizeof(uint32_t)));
    if (hs.out) CU_TRY(ln.h_out.reserve(std::max<uint64_t>(1, chunk) * hs.out_elem));
    return MSBWT_OK;
}

// The byte route: the caller's symbol bytes are copied to the device as they are and packed + validated there
// (pack_seed_kernel / pack_seed_final_kernel).  PCIe carries k bytes per query.
int bytes_route(Replica &rep, size_t ndev, const uint8_t *syms, uint32_t k, Slice sl, CountsOut out, Xfer &x) {
    const uint64_t chunk = pick_chunk(sl.len(), kChunkQueries, k);
    HostStage hs = make_stage(rep, ndev, k ? syms : nullptr, out);
    std::unique_ptr<PoolSession> session;
    if (hs.pool) session = std::make_unique<PoolSession>(*hs.pool);
    for (auto &ln : rep.lane) {
        CU_TRY(cudaStreamSynchronize(ln.stream));
        CU_TRY(ln.in_a.reserve(std::max<uint64_t>(1, chunk * k)));
        if (hs.in) CU_TRY(ln.h_stage.reserve(std::max<uint64_t>(1, chunk * k)));
        if (int rc = reserve_search_buffers(rep, ln, k, chunk, hs); rc != MSBWT_OK) return rc;
    }
    if (int rc = reset_status(rep); rc != MSBWT_OK) return rc;
    uint64_t c = 0;
    for (uint64_t b = sl.begin; b < sl.end; b += chunk, c++) {
        const uint64_t m = std::min(chunk, sl.end - b);
        const int li = (int)(c % kLanes);
        Lane &ln = rep.lane[li];
        if (int rc = flush_lane_output(ln, hs); rc != MSBWT_OK) return rc;
        if (k) {
            const void *src = nullptr;
            if (int rc = stage_input(ln, hs, syms + b * k, m * k, &src); rc != MSBWT_OK) return rc;
            CU_TRY(cudaMemcpyAsync(ln.in_a.p, src, m * k, cudaMemcpyHostToDevice, ln.stream));
            if (hs.in) CU_TRY(cudaEventRecord(ln.h2d_done, ln.stream));
        }
        CU_TRY(launch_pack_seed(rep.view, ln.in_a.as<uint8_t>(), k, m, ln.packed.as<uint64_t>(), ln.out_a.as<uint64_t>(),
                                rep.d_status + li, ln.stream));
        x.h2d += m * k;
        if (int rc = search_and_copy_out(rep, ln, k, b, m, hs, true, x); rc != MSBWT_OK) return rc;
    }
    if (int rc = drain(rep); rc != MSBWT_OK) return rc;
    if (int rc = flush_all_outputs(rep, hs); rc != MSBWT_OK) return rc;
    return check_status(rep, "count_kmers_fixed");
}

// Host-side 2-bit packing pays off when enough host threads can feed it: the byte route moves k bytes per query
// over PCIe (~55 GB/s), the packed route 8 * ceil(k/32) but needs the CPU to read the k bytes.
bool use_host_pack(uint32_t k, uint64_t n, size_t ndev) {
    if (!k || k > max_host_packed_k() || n < 4096) return false;
    if (const char *env = getenv("MSBWT_HOST_PACK")) return atoi(env) != 0;
    return replica_pack_threads(ndev) >= 8;
}

// The packed / hybrid route (hostpack.cpp): the replica's worker threads pack all-ACGT k-mers 2 bits per symbol
// into a lane's pinned staging buffer while earlier chunks are copied and searched; the device receives
// 8 * ceil(k/32) bytes per query (seed_packed_kernel).  K-mers with any other symbol are exceptions: they are
// collected and sent through the byte route afterwards, which validates and counts them.
// HYBRID (the caller's buffer is pinned): the packers are bound by host memory bandwidth (they have to read k bytes
// per query) while the PCIe link idles at 8 bytes per query, so whenever the copy engine has drained the previous
// raw chunk the next chunk goes over the link as it is -- k symbol bytes, packed and validated on the device
// (pack_seed_kernel) -- instead of through the packers.  The split balances itself: a raw lane is taken exactly
// when its last copy-in has completed.
int packed_route(Replica &rep, size_t ndev, const uint8_t *syms, uint32_t k, uint64_t n_total, Slice sl, CountsOut out, Xfer &x) {
    const uint32_t nw = (k + kPairSymsPerWord - 1) / kPairSymsPerWord;
    const uint64_t chunk = pick_chunk(sl.len(), kPackedChunkQueries, 8ull * nw);
    bool hybrid = is_pinned_host(syms);
    if (const char *env = getenv("MSBWT_HYBRID")) hybrid = hybrid && atoi(env) != 0;
    HostPool &pool = replica_pool(rep, ndev);
    PoolSession session(pool);
    // (the packers read the caller's symbol bytes themselves, pageable or not: only the OUTPUT may need staging)
    HostStage hs = make_stage(rep, ndev, nullptr, out);
    hs.pool = &pool;
    std::vector<std::vector<uint64_t>> exc_by_thread((size_t)pool.size());

    for (int li = 0; li < kLanes; li++) {
        Lane &ln = rep.lane[li];
        CU_TRY(cudaStreamSynchronize(ln.stream));
        if (li < kPackLanes) {
            CU_TRY(ln.h_stage.reserve(chunk * nw * sizeof(uint64_t)));
            CU_TRY(ln.in_b.reserve(chunk * nw * sizeof(uint64_t)));
        } else if (hybrid) {
            CU_TRY(ln.in_a.reserve(chunk * k));
        } else {
            continue;
        }
        if (int rc = reserve_search_buffers(rep, ln, k, chunk, hs); rc != MSBWT_OK) return rc;
    }
    if (int rc = reset_status(rep); rc != MSBWT_OK) return rc;
    const bool with_b = packed_batch_needs_list_b(rep.view, k);
    uint64_t packed_turn = 0;
    for (uint64_t b = sl.begin; b < sl.end; b += chunk) {
        const uint64_t m = std::min(chunk, sl.end - b);
        int raw_lane = -1;
        if (hybrid)
            for (int r = 0; r < kRawLanes && raw_lane < 0; r++)
                if (cudaEventQuery(rep.lane[kPackLanes + r].h2d_done) == cudaSuccess) raw_lane = kPackLanes + r;
        if (raw_lane >= 0) {  // the link is idle: this chunk travels as symbol bytes
            Lane &ln = rep.lane[raw_lane];
            if (int rc = flush_lane_output(ln, hs); rc != MSBWT_OK) return rc;
            CU_TRY(cudaMemcpyAsync(ln.in_a.p, syms + b * k, m * k, cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(cudaEventRecord(ln.h2d_done, ln.stream));
            CU_TRY(launch_pack_seed(rep.view, ln.in_a.as<uint8_t>(), k, m, ln.packed.as<uint64_t>(), ln.out_a.as<uint64_t>(),
                                    rep.d_status + raw_lane, ln.stream));
            x.h2d += m * k;
            if (int rc = search_and_copy_out(rep, ln, k, b, m, hs, true, x); rc != MSBWT_OK) return rc;
            continue;
        }
        Lane &ln = rep.lane[packed_turn++ % kPackLanes];
        if (int rc = flush_lane_output(ln, hs); rc != MSBWT_OK) return rc;
        CU_TRY(cudaEventSynchronize(ln.h2d_done));  // the lane's staging buffer is free again
        uint64_t *stage = (uint64_t *)ln.h_stage.p;
        pool.run([&](int tid, int nthreads) {
            const uint64_t q0 = b + m * (uint64_t)tid / (uint64_t)nthreads, q1 = b + m * (uint64_t)(tid + 1) / (uint64_t)nthreads;
            host_pack_range(syms, k, n_total, q0, q1, b, m, stage, exc_by_thread[(size_t)tid]);
        });
        CU_TRY(cudaMemcpyAsync(ln.in_b.p, stage, m * nw * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
        CU_TRY(cudaEventRecord(ln.h2d_done, ln.stream));
        CU_TRY(launch_seed_packed(rep.view, ln.in_b.as<uint64_t>(), k, m, ln.packed.as<uint64_t>(), ln.out_a.as<uint64_t>(), ln.stream));
        x.h2d += m * nw * sizeof(uint64_t);
        if (int rc = search_and_copy_out(rep, ln, k, b, m, hs, with_b, x); rc != MSBWT_OK) return rc;
    }
    if (int rc = drain(rep); rc != MSBWT_OK) return rc;
    if (int rc = flush_all_outputs(rep, hs); rc != MSBWT_OK) return rc;
    if (int rc = check_status(rep, "count_kmers_fixed"); rc != MSBWT_OK) return rc;  // raw chunks validate on the device
    // exceptions: k-mers with a symbol outside ACGT go through the byte route (device-side validation)
    std::vector<uint64_t> exc;
    for (auto &v : exc_by_thread) exc.insert(exc.end(), v.begin(), v.end());
    if (exc.empty()) return MSBWT_OK;
    std::vector<uint8_t> esyms(exc.size() * (size_t)k);
    std::vector<uint64_t> eout(exc.size());
    for (size_t i = 0; i < exc.size(); i++) memcpy(esyms.data() + i * k, syms + exc[i] * k, k);
    CountsOut tmp;
    tmp.o64 = eout.data();
    if (int rc = bytes_route(rep, ndev, esyms.data(), k, Slice{0, exc.size()}, tmp, x); rc != MSBWT_OK) return rc;
    for (size_t i = 0; i < exc.size(); i++) {
        if (out.o32) out.o32[exc[i]] = (uint32_t)eout[i];
        else out.o64[exc[i]] = eout[i];
    }
    return MSBWT_OK;
}

int fixed_route(const msbwt_index *idx, const uint8_t *syms, uint32_t k, uint64_t n, CountsOut out) {
    const size_t ndev = idx->reps.size();
    const bool packed = use_host_pack(k, n, ndev);
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &x) {
        return packed ? packed_route(rep, ndev, syms, k, n, sl, out, x) : bytes_route(rep, ndev, syms, k, sl, out, x);
    });
}

// K-mers the caller already holds as integers (k <= 32): nothing to do on the host, 8 bytes per query over the
// link on the way in and 8 (u64 counts) or 4 (u32 counts) on the way back.  A lane's stream orders copy-in, seed,
// search and copy-out, so its buffers are reused safely by its next chunk.
int u64_route(Replica &rep, size_t ndev, const uint64_t *kmers, uint32_t k, Slice sl, CountsOut out, Xfer &x) {
    const uint64_t chunk = pick_chunk(sl.len(), 1ull << 21, sizeof(uint64_t));
    HostStage hs = make_stage(rep, ndev, kmers, out);
    std::unique_ptr<PoolSession> session;
    if (hs.pool) session = std::make_unique<PoolSession>(*hs.pool);
    for (auto &ln : rep.lane) {
        CU_TRY(cudaStreamSynchronize(ln.stream));
        CU_TRY(ln.in_b.reserve(chunk * sizeof(uint64_t)));
        if (hs.in) CU_TRY(ln.h_stage.reserve(chunk * sizeof(uint64_t)));
        if (int rc = reserve_search_buffers(rep, ln, k, chunk, hs); rc != MSBWT_OK) return rc;
    }
    const bool with_b = packed_batch_needs_list_b(rep.view, k);
    // MSBWT_TRACE_PIPE=1: per-chunk timeline of the lanes (copy-in, kernels, copy-out) on stderr -- a measurement aid
    const bool trace = getenv("MSBWT_TRACE_PIPE") != nullptr;
    struct Marks { cudaEvent_t e[3]; int lane; };
    std::vector<Marks> marks;
    cudaEvent_t t0 = nullptr;
    if (trace) {
        cudaEventCreate(&t0);
        cudaEventRecord(t0, rep.lane[0].stream);
    }
    uint64_t c = 0;
    for (uint64_t b = sl.begin; b < sl.end; b += chunk, c++) {
        const uint64_t m = std::min(chunk, sl.end - b);
        Lane &ln = rep.lane[c % kLanes];
        if (int rc = flush_lane_output(ln, hs); rc != MSBWT_OK) return rc;
        const void *src = nullptr;
        if (int rc = stage_input(ln, hs, kmers + b, m * sizeof(uint64_t), &src); rc != MSBWT_OK) return rc;
        Marks mk{};
        if (trace) {
            for (auto &e : mk.e) cudaEventCreate(&e);
            mk.lane = (int)(c % kLanes);
            cudaEventRecord(mk.e[0], ln.stream);
        }
        CU_TRY(cudaMemcpyAsync(ln.in_b.p, src, m * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
        if (hs.in) CU_TRY(cudaEventRecord(ln.h2d_done, ln.stream));
        if (trace) cudaEventRecord(mk.e[1], ln.stream);
        CU_TRY(launch_seed_u64(rep.view, ln.in_b.as<uint64_t>(), k, m, ln.packed.as<uint64_t>(), ln.out_a.as<uint64_t>(), ln.stream));
        x.h2d += m * sizeof(uint64_t);
        if (int rc = search_and_copy_out(rep, ln, k, b, m, hs, with_b, x); rc != MSBWT_OK) return rc;
        if (trace) {
            cudaEventRecord(mk.e[2], ln.stream);
            marks.push_back(mk);
        }
    }
    if (int rc = drain(rep); rc != MSBWT_OK) return rc;
    if (int rc = flush_all_outputs(rep, hs); rc != MSBWT_OK) return rc;
    if (trace) {
        fprintf(stderr, "[msbwt] u64 route on device %d: %zu chunks of %llu queries\n  chunk lane  h2d_start  h2d_end  d2h_end (ms)\n",
                rep.device, marks.size(), (unsigned long long)chunk);
        for (size_t i = 0; i < marks.size(); i++) {
            float t[3];
            for (int j = 0; j < 3; j++) cudaEventElapsedTime(&t[j], t0, marks[i].e[j]);
            fprintf(stderr, "  %5zu %4d  %9.3f %8.3f %8.3f\n", i, marks[i].lane, t[0], t[1], t[2]);
            for (auto &e : marks[i].e) cudaEventDestroy(e);
        }
        cudaEventDestroy(t0);
    }
    return MSBWT_OK;
}

struct AllLocks {
    std::vector<std::unique_lock<std::mutex>> locks;
    explicit AllLocks(const msbwt_index *idx) {
        for (auto &rep : idx->reps) locks.emplace_back(rep->mu);
    }
};

int check_fixed_args(const msbwt_index *idx, const void *in, uint32_t k, uint64_t n, const void *out, bool narrow) {
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (n && (!out || (k && !in))) return fail(MSBWT_EINVAL, "NULL host buffer");
    if (narrow && idx->total >= (1ull << 32))
        return fail(MSBWT_EINVAL, "32-bit counts need an index below 2^32 symbols (a count can reach total_size)");
    return MSBWT_OK;
}

}  // namespace

extern "C" int msbwt_count_kmers_fixed(const msbwt_index *idx, const uint8_t *syms, uint32_t k, uint64_t n, uint64_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (int rc = check_fixed_args(idx, syms, k, n, out, false); rc != MSBWT_OK) return rc;
    if (!n) return MSBWT_OK;
    AllLocks locks(idx);
    CountsOut o;
    o.o64 = out;
    return fixed_route(idx, syms, k, n, o);
}

extern "C" int msbwt_count_kmers_fixed_u32(const msbwt_index *idx, const uint8_t *syms, uint32_t k, uint64_t n, uint32_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (int rc = check_fixed_args(idx, syms, k, n, out, true); rc != MSBWT_OK) return rc;
    if (!n) return MSBWT_OK;
    AllLocks locks(idx);
    CountsOut o;
    o.o32 = out;
    return fixed_route(idx, syms, k, n, o);
}

extern "C" int msbwt_count_kmers_u64(const msbwt_index *idx, const uint64_t *kmers, uint32_t k, uint64_t n, uint64_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (int rc = check_fixed_args(idx, kmers, 1, n, out, false); rc != MSBWT_OK) return rc;
    if (k == 0 || k > 32) return fail(MSBWT_EINVAL, "count_kmers_u64: k must be 1..32 (one 2-bit-per-symbol word per k-mer)");
    if (!n) return MSBWT_OK;
    AllLocks locks(idx);
    CountsOut o;
    o.o64 = out;
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &x) { return u64_route(rep, idx->reps.size(), kmers, k, sl, o, x); });
}

extern "C" int msbwt_count_kmers_u64_u32(const msbwt_index *idx, const uint64_t *kmers, uint32_t k, uint64_t n, uint32_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (int rc = check_fixed_args(idx, kmers, 1, n, out, true); rc != MSBWT_OK) return rc;
    if (k == 0 || k > 32) return fail(MSBWT_EINVAL, "count_kmers_u64: k must be 1..32 (one 2-bit-per-symbol word per k-mer)");
    if (!n) return MSBWT_OK;
    AllLocks locks(idx);
    CountsOut o;
    o.o32 = out;
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &x) { return u64_route(rep, idx->reps.size(), kmers, k, sl, o, x); });
}

extern "C" void msbwt_last_transfer_bytes(uint64_t *h2d, uint64_t *d2h) {
    if (h2d) *h2d = g_last_h2d;
    if (d2h) *d2h = g_last_d2h;
}

extern "C" int msbwt_host_pack_threads(void) { return host_threads_available(); }

extern "C" int msbwt_count_kmers(const msbwt_index *idx, const uint8_t *syms, const uint64_t *offsets, uint64_t n, uint64_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!n) return MSBWT_OK;
    if (!out || !offsets) return fail(MSBWT_EINVAL, "NULL host buffer");
    for (uint64_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) return fail(MSBWT_EINVAL, "offsets must be non-decreasing");
    if (offsets[n] > offsets[0] && !syms) return fail(MSBWT_EINVAL, "NULL host buffer");
    AllLocks locks(idx);
    // A batch whose k-mers all have the same length -- what `count_kmers(&[Vec<u8>])` is called with in a k-mer
    // counting loop -- is the fixed-k batch laid out contiguously: it takes the packed / table-seeded route.
    {
        const uint64_t k0 = offsets[1] - offsets[0];
        bool uniform = k0 > 0 && k0 <= 0xFFFFFFFFull;
        for (uint64_t i = 1; uniform && i < n; i++) uniform = offsets[i + 1] - offsets[i] == k0;
        if (uniform) {
            CountsOut o;
            o.o64 = out;
            return fixed_route(idx, syms + offsets[0], (uint32_t)k0, n, o);
        }
    }
    // mixed lengths: per device, walk the slice in chunks bounded in both queries and symbol bytes (byte-wise
    // kernel, no suffix table)
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &x) {
        if (int rc = reset_status(rep); rc != MSBWT_OK) return rc;
        uint64_t round = 0;
        for (uint64_t b = sl.begin; b < sl.end; round++) {
            uint64_t e = std::min(sl.end, b + kChunkQueries);
            if (offsets[e] - offsets[b] > kChunkBytes) {
                // largest e with offsets[e]-offsets[b] <= kChunkBytes, at least one query
                const uint64_t *hi = std::upper_bound(offsets + b, offsets + e + 1, offsets[b] + kChunkBytes);
                e = std::max<uint64_t>(b + 1, (uint64_t)(hi - offsets) - 1);
            }
            const uint64_t m = e - b, nbytes = offsets[e] - offsets[b];
            Lane &ln = rep.lane[round & 1];
            CU_TRY(cudaStreamSynchronize(ln.stream));  // buffers may be regrown below
            CU_TRY(ln.in_a.reserve(std::max<uint64_t>(1, nbytes)));
            CU_TRY(ln.in_b.reserve((m + 1) * sizeof(uint64_t)));
            CU_TRY(ln.out_a.reserve(m * sizeof(uint64_t)));
            if (nbytes) CU_TRY(cudaMemcpyAsync(ln.in_a.p, syms + offsets[b], nbytes, cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(cudaMemcpyAsync(ln.in_b.p, offsets + b, (m + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
            // the kernel indexes syms with absolute offsets: bias the base pointer instead of rewriting them
            const uint8_t *biased = ln.in_a.as<uint8_t>() - offsets[b];
            CU_TRY(launch_count_bytes(rep.device, rep.view, biased, ln.in_b.as<uint64_t>(), m, ln.out_a.as<uint64_t>(),
                                      rep.d_status + (round & 1), ln.stream));
            CU_TRY(cudaMemcpyAsync(out + b, ln.out_a.p, m * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
            x.h2d += nbytes + (m + 1) * sizeof(uint64_t);
            x.d2h += m * sizeof(uint64_t);
            b = e;
        }
        if (int rc = drain(rep); rc != MSBWT_OK) return rc;
        return check_status(rep, "count_kmers");
    });
}

extern "C" int msbwt_constrain_ranges(const msbwt_index *idx, const uint8_t *sym, const uint64_t *l, const uint64_t *h,
                                      uint64_t n, uint64_t *out_l, uint64_t *out_h) {
    g_last_error.clear();
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!n) return MSBWT_OK;
    if (!sym || !l || !h || !out_l || !out_h) return fail(MSBWT_EINVAL, "NULL host buffer");
    AllLocks locks(idx);
    // validation first (the reference's constrain_range is unchecked; we refuse bad input before any output is written)
    for (uint64_t i = 0; i < n; i++)
        if (sym[i] >= kAlphabet || l[i] > h[i] || h[i] > idx->total)
            return fail(MSBWT_EINVAL, "constrain_ranges: item " + std::to_string(i) + " has sym >= 6, l > h or h > total_size");
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &) {
        const uint64_t chunk = pick_chunk(sl.len(), kChunkQueries, 17);
        for (int li = 0; li < 2; li++) {
            Lane &ln = rep.lane[li];
            CU_TRY(cudaStreamSynchronize(ln.stream));
            CU_TRY(ln.in_a.reserve(chunk));
            CU_TRY(ln.in_b.reserve(chunk * sizeof(uint64_t)));
            CU_TRY(ln.in_c.reserve(chunk * sizeof(uint64_t)));
            CU_TRY(ln.out_a.reserve(chunk * sizeof(uint64_t)));
            CU_TRY(ln.out_b.reserve(chunk * sizeof(uint64_t)));
        }
        uint64_t c = 0;
        for (uint64_t b = sl.begin; b < sl.end; b += chunk, c++) {
            const uint64_t m = std::min(chunk, sl.end - b);
            Lane &ln = rep.lane[c & 1];
            CU_TRY(cudaMemcpyAsync(ln.in_a.p, sym + b, m, cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(cudaMemcpyAsync(ln.in_b.p, l + b, m * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(cudaMemcpyAsync(ln.in_c.p, h + b, m * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(launch_constrain_ranges(rep.device, rep.view, ln.in_a.as<uint8_t>(), ln.in_b.as<uint64_t>(), ln.in_c.as<uint64_t>(), m,
                                           ln.out_a.as<uint64_t>(), ln.out_b.as<uint64_t>(), ln.stream));
            CU_TRY(cudaMemcpyAsync(out_l + b, ln.out_a.p, m * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
            CU_TRY(cudaMemcpyAsync(out_h + b, ln.out_b.p, m * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
        }
        return drain(rep);
    });
}

// ================================================================ batched callers of the path (SURVEY 8f N3)

extern "C" int msbwt_constrain_ranges_fanout(const msbwt_index *idx, const uint64_t *l, const uint64_t *h, uint64_t n,
                                             uint64_t *out_l, uint64_t *out_h) {
    g_last_error.clear();
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!n) return MSBWT_OK;
    if (!l || !h || !out_l || !out_h) return fail(MSBWT_EINVAL, "NULL host buffer");
    AllLocks locks(idx);
    for (uint64_t i = 0; i < n; i++)
        if (l[i] > h[i] || h[i] > idx->total)
            return fail(MSBWT_EINVAL, "constrain_ranges_fanout: item " + std::to_string(i) + " has l > h or h > total_size");
    return run_on_replicas(idx, n, [&](Replica &rep, Slice sl, Xfer &) {
        const uint64_t chunk = pick_chunk(sl.len(), kChunkQueries, 16);
        for (int li = 0; li < 2; li++) {
            Lane &ln = rep.lane[li];
            CU_TRY(cudaStreamSynchronize(ln.stream));
            CU_TRY(ln.in_b.reserve(chunk * sizeof(uint64_t)));
            CU_TRY(ln.in_c.reserve(chunk * sizeof(uint64_t)));
            CU_TRY(ln.out_a.reserve(4 * chunk * sizeof(uint64_t)));
            CU_TRY(ln.out_b.reserve(4 * chunk * sizeof(uint64_t)));
        }
        uint64_t c = 0;
        for (uint64_t b = sl.begin; b < sl.end; b += chunk, c++) {
            const uint64_t m = std::min(chunk, sl.end - b);
            Lane &ln = rep.lane[c & 1];
            CU_TRY(cudaMemcpyAsync(ln.in_b.p, l + b, m * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(cudaMemcpyAsync(ln.in_c.p, h + b, m * sizeof(uint64_t), cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(launch_constrain_fanout(rep.device, rep.view, ln.in_b.as<uint64_t>(), ln.in_c.as<uint64_t>(), m,
                                           ln.out_a.as<uint64_t>(), ln.out_b.as<uint64_t>(), ln.stream));
            CU_TRY(cudaMemcpyAsync(out_l + 4 * b, ln.out_a.p, 4 * m * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
            CU_TRY(cudaMemcpyAsync(out_h + 4 * b, ln.out_b.p, 4 * m * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
        }
        return drain(rep);
    });
}

extern "C" int msbwt_count_read_kmers(const msbwt_index *idx, const uint8_t *reads, uint32_t read_len, uint64_t n_reads,
                                      uint32_t k, uint32_t strands, uint64_t *out) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!k || k > read_len) return fail(MSBWT_EINVAL, "count_read_kmers: k must be in 1..read_len");
    if (strands != 1 && strands != 2) return fail(MSBWT_EINVAL, "count_read_kmers: strands must be 1 or 2");
    if (!n_reads) return MSBWT_OK;
    if (!reads || !out) return fail(MSBWT_EINVAL, "NULL host buffer");
    const uint64_t windows = (uint64_t)read_len - k + 1, per_read_q = windows * strands;
    // the expand kernel numbers a read's queries in 32 bits
    if (per_read_q >> 32) return fail(MSBWT_EINVAL, "count_read_kmers: a read has 2^32 or more queries (windows x strands)");
    AllLocks locks(idx);
    // symbols are validated where they are packed (count_kmer's own check, src/msbwt_core.rs:127): the pack
    // kernel flags any symbol >= 6 and the call then returns EINVAL
    return run_on_replicas(idx, n_reads, [&](Replica &rep, Slice sl, Xfer &x) {
        const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(sl.len(), 4 * kChunkQueries / per_read_q));  // reads per chunk
        if (int rc = reset_status(rep); rc != MSBWT_OK) return rc;
        for (int li = 0; li < 2; li++) {
            Lane &ln = rep.lane[li];
            CU_TRY(cudaStreamSynchronize(ln.stream));
            CU_TRY(ln.in_a.reserve(chunk * read_len));
            CU_TRY(ln.in_b.reserve(chunk * per_read_q * k + 16));
            CU_TRY(ln.packed.reserve(packed_layout(rep.view, k, chunk * per_read_q).total() * sizeof(uint64_t)));
            CU_TRY(ln.out_a.reserve(chunk * per_read_q * sizeof(uint64_t)));
            CU_TRY(ln.out_b.reserve(chunk * windows * sizeof(uint64_t)));
        }
        uint64_t c = 0;
        for (uint64_t b = sl.begin; b < sl.end; b += chunk, c++) {
            const uint64_t m = std::min(chunk, sl.end - b), nq = m * per_read_q;
            Lane &ln = rep.lane[c & 1];
            uint32_t *flag = rep.d_status + (c & 1);
            CU_TRY(cudaMemcpyAsync(ln.in_a.p, reads + b * read_len, m * read_len, cudaMemcpyHostToDevice, ln.stream));
            CU_TRY(launch_expand_read_kmers(rep.device, ln.in_a.as<uint8_t>(), read_len, m, k, strands, ln.in_b.as<uint8_t>(), ln.stream));
            CU_TRY(launch_pack_seed(rep.view, ln.in_b.as<uint8_t>(), k, nq, ln.packed.as<uint64_t>(), ln.out_a.as<uint64_t>(), flag, ln.stream));
            CU_TRY(launch_count_packed(rep.device, rep.view, rep.lanes, ln.packed.as<uint64_t>(), k, nq, ln.out_a.as<uint64_t>(),
                                       ln.stream));
            const uint64_t *res = ln.out_a.as<uint64_t>();
            if (strands == 2) {
                CU_TRY(launch_sum_strands(rep.device, ln.out_a.as<uint64_t>(), m * windows, ln.out_b.as<uint64_t>(), ln.stream));
                res = ln.out_b.as<uint64_t>();
            }
            CU_TRY(cudaMemcpyAsync(out + b * windows, res, m * windows * sizeof(uint64_t), cudaMemcpyDeviceToHost, ln.stream));
            x.h2d += m * read_len;
            x.d2h += m * windows * sizeof(uint64_t);
        }
        if (int rc = drain(rep); rc != MSBWT_OK) return rc;
        return check_status(rep, "count_read_kmers");
    });
}

extern "C" int msbwt_correct_reads(const msbwt_index *idx, const uint8_t *syms, const uint64_t *offsets, uint64_t n_reads,
                                   uint32_t k, uint64_t min_count, uint32_t frac_permille, uint32_t branch_limit,
                                   uint8_t **out_syms, uint64_t **out_offsets, uint64_t *stats) {
    g_last_error.clear();
    g_last_h2d = g_last_d2h = 0;
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!k || k > 32) return fail(MSBWT_EINVAL, "correct_reads: k must be in 1..32");
    if (!min_count) return fail(MSBWT_EINVAL, "correct_reads: min_count must be at least 1");
    if (frac_permille > 1000) return fail(MSBWT_EINVAL, "correct_reads: frac_permille must be in 0..1000");
    if (!branch_limit) return fail(MSBWT_EINVAL, "correct_reads: branch_limit must be at least 1");
    if (!out_syms || !out_offsets) return fail(MSBWT_EINVAL, "correct_reads: NULL output pointer");
    if (n_reads && (!syms || !offsets)) return fail(MSBWT_EINVAL, "NULL host buffer");
    for (uint64_t r = 0; r < n_reads; r++) {
        if (offsets[r + 1] < offsets[r]) return fail(MSBWT_EINVAL, "correct_reads: offsets decrease at read " + std::to_string(r));
        // a read is sorted as one CUB segment, whose sizes are int
        if (offsets[r + 1] - offsets[r] >= (1ull << 31)) return fail(MSBWT_EINVAL, "correct_reads: a read of 2^31 symbols or more");
    }
    if (n_reads)
        for (uint64_t i = offsets[0]; i < offsets[n_reads]; i++)
            if (syms[i] == 0 || syms[i] >= 6)
                return fail(MSBWT_EINVAL, "correct_reads: symbol " + std::to_string(syms[i]) + " at " + std::to_string(i) +
                                              " (reads hold A, C, G, N, T = 1..5)");
    // each replica corrects one contiguous slice of the reads with its own stream and scratch (no lane: no lock)
    const CorrectParams prm{k, min_count, frac_permille, branch_limit};
    struct Part {
        std::vector<uint8_t> syms;
        std::vector<uint64_t> lens;
        uint64_t stats[5] = {0, 0, 0, 0, 0};
    };
    std::vector<Part> parts(idx->reps.size());
    int rc = run_on_replicas(idx, n_reads, [&](Replica &rep, Slice sl, Xfer &x) {
        size_t d = 0;
        while (idx->reps[d].get() != &rep) d++;
        Part &pt = parts[d];
        const int r = correct_reads_on_device(rep.device, rep.view, rep.lanes, syms, offsets + sl.begin, sl.len(), prm,
                                              pt.syms, pt.lens, pt.stats);
        x.h2d += offsets[sl.end] - offsets[sl.begin] + (sl.len() + 1) * sizeof(uint64_t);
        x.d2h += pt.syms.size() + pt.lens.size() * sizeof(uint64_t);
        return r;
    });
    if (rc != MSBWT_OK) return rc;
    uint64_t total = 0;
    for (const Part &pt : parts) total += pt.syms.size();
    uint8_t *os = (uint8_t *)malloc(std::max<uint64_t>(total, 1));
    uint64_t *oo = (uint64_t *)malloc((n_reads + 1) * sizeof(uint64_t));
    if (!os || !oo) {
        free(os);
        free(oo);
        return fail(MSBWT_ENOMEM, "correct_reads: host buffers for the result");
    }
    uint64_t at = 0, r = 0;
    oo[0] = 0;
    for (const Part &pt : parts) {
        if (!pt.syms.empty()) memcpy(os + at, pt.syms.data(), pt.syms.size());
        at += pt.syms.size();
        for (uint64_t len : pt.lens) {
            oo[r + 1] = oo[r] + len;
            r++;
        }
    }
    if (stats)
        for (int i = 0; i < 5; i++) {
            stats[i] = 0;
            for (const Part &pt : parts) stats[i] += pt.stats[i];
        }
    *out_syms = os;
    *out_offsets = oo;
    return MSBWT_OK;
}
