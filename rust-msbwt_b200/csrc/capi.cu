// capi.cu -- the C ABI declared in include/msbwt_gpu.h: handle management, device
// replicas, host<->device staging pipelines and the multi-GPU batch split.
//
// Reference surface being replaced: the `BWT` trait as implemented by `RleBWT`
// (src/msbwt_core.rs:28-162, src/rle_bwt.rs:44-322).  There is no CPU fallback
// anywhere in this file: every query entry point ends in a kernel launch.
#include <algorithm>
#include <cerrno>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <thread>

#include "handle.h"
#include "kernel_common.cuh"

using namespace msbwt;

namespace msbwt {
thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};
int codec_fail(int code, const std::string &msg) { return fail(code, msg); }  // codec.cpp reports through the same thread-local
}  // namespace msbwt

namespace {

int resolve_devices(const int *devices, int ndev, std::vector<int> &devs) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(MSBWT_ENODEV, std::string("no usable CUDA device (there is no CPU fallback): ") +
                                      (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (ndev <= 0 || !devices) {
        int cur = 0;
        CU_TRY(cudaGetDevice(&cur));
        devs.push_back(cur);
    } else {
        devs.assign(devices, devices + ndev);
    }
    for (int d : devs)
        if (d < 0 || d >= count) return fail(MSBWT_ENODEV, "device ordinal " + std::to_string(d) + " out of range");
    return MSBWT_OK;
}

// Runs body(i) for i in [0, n): on the calling thread when n == 1, else one thread per replica (every replica lives on
// its own device, so the builds of a multi-GPU handle overlap).  A thread's failure text (thread-local) is carried back
// to the caller; the first failure by slot order is returned.
template <class F>
int for_each_replica_slot(size_t n, F &&body) {
    std::vector<int> rc(n, MSBWT_OK);
    std::vector<std::string> err(n);
    auto run = [&](size_t i) {
        rc[i] = body(i);
        if (rc[i] != MSBWT_OK) err[i] = g_last_error;
    };
    if (n == 1) {
        run(0);
    } else {
        std::vector<std::thread> workers;
        for (size_t i = 1; i < n; i++) workers.emplace_back(run, i);
        run(0);
        for (auto &w : workers) w.join();
    }
    for (size_t i = 0; i < n; i++)
        if (rc[i] != MSBWT_OK) return fail(rc[i], err[i]);
    return MSBWT_OK;
}

// The optional-image fields of the view, from what the replica owns: an image that was never built or has been freed
// reads as null / 0.  Called after every build stage that adds or frees an image.
void refresh_view(Replica &rep) {
    IndexView &v = rep.view;
    v.table = rep.d_table;
    v.table2 = rep.d_table_lower[0];
    v.table3 = rep.d_table_lower[1];
    v.table4 = rep.d_table_lower[2];
    v.table_s = rep.table_s;
    v.pair = rep.pair.lines;
    v.c2base = rep.pair.c2base;
    v.npair = rep.pair.npair;
    v.n_super2 = rep.pair.n_super2;
    v.quad = rep.quad.sectors;
    v.c4base = rep.quad.c4base;
    v.nsec4 = rep.quad.nsec4;
    v.n_super4 = rep.quad.n_super4;
    v.sb_shift4 = rep.quad.sb_shift4;
    v.oct = rep.oct.lines;
    v.nbuck8 = rep.oct.nbuck8;
    v.oct_shift = (uint32_t)rep.oct.shift;
    v.fin = rep.fin.lines;
    v.fin_shift = (uint32_t)rep.fin.shift;
    v.fin_lb = (uint32_t)rep.fin.lb;
}

// Device memory of the images one replica holds (msbwt_index_bytes)
uint64_t replica_bytes(const Replica &rep) {
    const IndexView &v = rep.view;
    uint64_t b = v.nblocks * kBlockBytes + v.nblocks * 2 * sizeof(uint32_t) + (uint64_t)v.n_super * 8 * sizeof(uint64_t);
    b += rep.pair.npair * kPairBytes + (rep.pair.c2base ? (uint64_t)rep.pair.n_super2 * 16 * sizeof(uint64_t) : 0);
    b += (uint64_t)kQuadCodes * rep.quad.nsec4 * kQuadSectorBytes +
         (rep.quad.c4base ? (uint64_t)rep.quad.n_super4 * kQuadCodes * sizeof(uint64_t) : 0);
    b += (uint64_t)kOctCodes * rep.oct.nbuck8 * kOctLineBytes;
    b += rep.fin.nlines * (uint64_t)kFinLineBytes;
    const uint64_t eb = index_is_wide(v) ? 16 : 8;
    if (rep.d_table) b += (1ull << (2 * rep.table_s)) * eb;
    for (int j = 1; j <= 3; j++)
        if (rep.d_table_lower[j - 1]) b += (1ull << (2 * (rep.table_s - j))) * eb;
    return b;
}

// The block image is built on each device from the RLE bytes (builder.cu).
int build_replicas_on_device(msbwt_index *idx, const uint8_t *rle, uint64_t len, uint32_t sb_shift, const int *devices,
                             int ndev) {
    std::vector<int> devs;
    if (int rc = resolve_devices(devices, ndev, devs); rc != MSBWT_OK) return rc;
    idx->reps.resize(devs.size());
    int rc = for_each_replica_slot(devs.size(), [&](size_t i) -> int {
        DeviceGuard guard(devs[i]);
        DeviceImage img;
        if (int r = build_image_on_device(rle, len, sb_shift, img); r != MSBWT_OK) { free_device_image(img); return r; }
        auto rep = std::make_unique<Replica>();
        rep->device = devs[i];
        rep->d_blocks = img.blocks;
        rep->d_aux = img.aux;
        rep->d_cbase = img.cbase;
        if (i == 0) {
            idx->total = img.total;
            for (int s = 0; s < kAlphabet; s++) { idx->counts[s] = img.counts[s]; idx->start[s] = img.start[s]; }
        }
        CU_TRY(cudaMalloc((void **)&rep->d_status, kStatusWords * sizeof(uint32_t)));
        CU_TRY(cudaMemset(rep->d_status, 0, kStatusWords * sizeof(uint32_t)));
        CU_TRY(cudaHostAlloc((void **)&rep->h_status, kStatusWords * sizeof(uint32_t), cudaHostAllocDefault));
        memset(rep->h_status, 0, kStatusWords * sizeof(uint32_t));
        for (auto &ln : rep->lane) {
            CU_TRY(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
            CU_TRY(cudaEventCreateWithFlags(&ln.h2d_done, cudaEventDisableTiming));
            CU_TRY(cudaEventCreateWithFlags(&ln.d2h_done, cudaEventDisableTiming));
        }
        rep->view.blocks = rep->d_blocks;
        rep->view.cbase = rep->d_cbase;
        rep->view.aux = rep->d_aux;
        rep->view.total = img.total;
        rep->view.nblocks = img.nblocks;
        rep->view.n_super = img.n_super;
        rep->view.sb_shift = img.sb_shift;
        idx->reps[i] = std::move(rep);
        return MSBWT_OK;
    });
    if (rc != MSBWT_OK) idx->reps.clear();
    return rc;
}

// Suffix table (layout.h): level j+1 from level j with one constrain_range per entry, on the
// replica's own device.  s < 0 picks ceil(log4(N / 32)) capped to kAutoMaxTableS: about the
// depth at which a read set's BWT ranges stop being shared between unrelated k-mers.
constexpr int kAutoMaxTableS = 13;

struct Options {
    uint32_t sb_shift = 0;
    int table_s = -1;   // -1 auto
    int pair = -1;      // -1 auto, 0 off, 1 on
    int quad = -1;      // -1 auto, 0 off, 1 on (builds the pair image on the way and drops it)
    int oct = -1;       // -1 auto (with an automatic or requested quad image), 0 off, 1 on (implies quad)
    int oct_shift = 0;  // 0 auto, else the oct image's bucket shift
    int keep_quad = -1; // under an oct image: -1 auto, 0 drop the quad image once the other images are built, 1 keep it
    int fin = -1;       // final-step image on top of the oct image: -1 auto (on), 0 off, 1 on (fail if it cannot be built)
    int fin_shift = 0;  // 0 = 16
    int fin_lb = 0;     // 0 auto (13 = 16 B/symbol when that fits 30 % of the device, else 12 = 8 B/symbol)
    int lanes = 0;      // 0 auto, 1, 2
};

// The environment fills the layout knobs the caller left automatic, before the layout is planned: each variable means
// what the same value of its msbwt_options field means (include/msbwt_gpu.h)
void fill_from_env(Options &o) {
    auto env_int = [](const char *name, int fallback) { const char *e = getenv(name); return e ? atoi(e) : fallback; };
    const char *e;
    if (o.table_s < 0 && (e = getenv("MSBWT_SUFFIX_TABLE_S"))) o.table_s = std::clamp(atoi(e), 0, kMaxTableS);
    if (o.lanes != 1 && o.lanes != 2 && (e = getenv("MSBWT_LANES"))) o.lanes = atoi(e) == 2 ? 2 : 1;
    if (o.pair == -1 && (e = getenv("MSBWT_PAIR_INDEX"))) o.pair = atoi(e) != 0;
    if (o.quad == -1 && (e = getenv("MSBWT_QUAD_INDEX"))) o.quad = atoi(e) != 0;
    if (o.oct == -1 && (e = getenv("MSBWT_OCT_INDEX"))) o.oct = atoi(e) != 0;
    if (o.keep_quad == -1) o.keep_quad = env_int("MSBWT_KEEP_QUAD", -1);
    if (o.fin == -1) o.fin = env_int("MSBWT_FINAL_INDEX", -1);
    if (!o.fin_shift) o.fin_shift = env_int("MSBWT_FINAL_BUCKET_SHIFT", 16);
    if (!o.fin_lb) o.fin_lb = env_int("MSBWT_FINAL_LINES_LOG2", 0);
    if (!o.oct_shift) o.oct_shift = env_int("MSBWT_OCT_BUCKET_SHIFT", 0);
}

// What the policy reads of a device: its L2 size and its memory before any optional image is built
struct DeviceSizes {
    uint64_t l2 = 0, free = 0, total = 0;
};

DeviceSizes device_sizes(int device) {
    int l2 = 0;
    size_t free_b = 0, total_b = 0;
    if (cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device) != cudaSuccess || l2 <= 0) l2 = 96 << 20;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = total_b = 0;
    return {(uint64_t)l2, free_b, total_b};
}

// Free memory of the current device as a build stage finds it (0 when it cannot be read)
uint64_t free_bytes_now() {
    size_t free_b = 0, total_b = 0;
    return cudaMemGetInfo(&free_b, &total_b) == cudaSuccess ? free_b : 0;
}

// The images a replica gets, its suffix-table depth and its kernel lanes (msbwt_debug_plan_layout writes these fields)
struct Layout {
    int table_s = 0;            // before the deepening for HBM (deepen_table_for_hbm)
    bool explicit_s = false;    // the caller or the environment fixed the depth: it is not deepened
    bool hbm = false;           // one-step blocks + suffix table > 2 x L2
    bool wide_oct = false;      // 64-bit positions: oct (and final-step) lines by walking LF, no quad image
    bool quad = false;          // the quad route (pair -> quad [-> oct -> final-step]), when no wide images were built
    bool oct = false;           // oct lines on top of the quad image
    bool fin = false;           // final-step lines on top of the oct lines
    bool pair = false;          // the pair image alone
    bool keep_quad = false;     // the quad image stays once the oct lines exist
    bool oct_required = false;  // oct_index = 1: no 8 GB reserve beside the oct lines; the wide route must succeed
    bool fin_required = false;  // final_index = 1: create fails without the final-step lines
    int fin_lb = 0;             // log2 of the final-step lines per bucket
    int lanes = 1;
    int oct_shift = 0, fin_shift = 0;
};

// The layout policy: a function of the options (the environment folded in), the index's size, the bytes of its bare
// replica (block image) and the device's sizes, and nothing else.
Layout plan_layout(const Options &opt, uint64_t N, bool wide, uint64_t block_bytes, const DeviceSizes &dev) {
    Layout p;
    p.explicit_s = opt.table_s >= 0;
    p.table_s = p.explicit_s ? std::min(opt.table_s, kMaxTableS) : 0;
    while (!p.explicit_s && p.table_s < kAutoMaxTableS && (1ull << (2 * p.table_s)) < N / 32) p.table_s++;
    const uint64_t one_step = block_bytes + (p.table_s > 0 ? (1ull << (2 * p.table_s)) * (wide ? 16 : 8) : 0);
    // Kernel mapping (kernels.cu): one thread per query while blocks + table are (mostly) L2-resident,
    // a lane pair per query -- one coalesced 64-byte request per block -- once they live in HBM.
    p.hbm = one_step > 2 * dev.l2;
    p.lanes = opt.lanes == 1 || opt.lanes == 2 ? opt.lanes : (p.hbm ? 2 : 1);

    // 64-bit positions: the oct and final-step images when the index lives in HBM, the caller pinned no other layout,
    // and the two images at their coarsest settings plus the builders' scratch fit the free device memory.
    p.oct_required = opt.oct == 1;
    p.wide_oct = wide && (opt.oct == 1 || (opt.oct != 0 && opt.pair == -1 && opt.quad == -1 && p.hbm && (N >> 40) == 0 &&
                                           oct_image_bytes(N, kOctMaxShift) + fin_image_bytes(N, 16, 12) + 12 * N +
                                                   (8ull << 30) <= dev.free));

    // The quad image (layout.h: one 32-byte sector per FOUR steps, 256 * N / 7 bytes) halves the line fills of the pair
    // image again.  Automatic choice: the one-step index does not fit L2 (measured on the 151 Msymbol BWT, 1.7 x L2:
    // 10.2 G queries/s through quad sectors + a depth-15 table in HBM against 7.3 G through the mostly L2-resident
    // one-step blocks), the image stays below 64 GB (measured, profiles/r1_gather_big.json: random reads keep 93 % of
    // their rate over a 64 GB buffer and lose three quarters of it over 128 GB) and below half of the free device
    // memory.  When the oct image will sit on top (32-bit positions, not switched off) the quad image only serves
    // fallbacks and remainders, the randomly read footprint is the oct image + the suffix table, and the quad image may
    // take up to 65 % of the free memory (110 GB for configs[4]'s 3.02 Gsymbol BWT).  A pinned pair_index pins the
    // layout: no quad image.
    const bool narrow_oct = !wide && opt.oct != 0;
    const uint64_t quad_bytes = quad_image_bytes(N);
    if (opt.oct == 1 || opt.quad == 1) p.quad = true;
    else if (opt.quad == 0 || opt.pair == 0 || opt.pair == 1) p.quad = false;
    else p.quad = one_step > dev.l2 && (narrow_oct ? quad_bytes <= dev.free / 100 * 65
                                                   : quad_bytes <= (64ull << 30) && quad_bytes <= dev.free / 2);
    // The oct image (layout.h: one 128-byte line per kOctSyms = 10 steps) rides on the quad image, 32-bit positions
    // only; the final-step image rides on the oct image.
    p.oct = p.quad && narrow_oct;
    p.fin = (p.oct || p.wide_oct) && opt.fin != 0;
    p.fin_required = opt.fin == 1;
    // The pair image (layout.h: one 128-byte line per two steps) pays off once the index lives in HBM;
    // an L2-resident index is served faster by the 64-byte one-step blocks (smaller footprint).
    p.pair = !p.quad && (opt.pair == 0 || opt.pair == 1 ? opt.pair == 1 : p.hbm);
    // Under the oct image the quad image only serves remainders of 4..9 symbols and the rare fallbacks of the oct
    // kernel, which one-symbol ranks answer as well: it is kept when quad + 40 B/symbol for the other two images fit
    // 70 % of the device (55 GB at 1.51 Gsymbols), dropped otherwise (110 GB at 3.02 Gsymbols).
    p.keep_quad = opt.keep_quad != -1 ? opt.keep_quad != 0 : quad_bytes + 40 * N <= dev.total / 10 * 7;
    // Lines per final-step bucket: 2^13, 16 bytes per symbol (0.8 % of the read-sampled 31-mers find their line
    // overflowed and take the oct steps), when that fits 30 % of the device (48 GB at 3.02 Gsymbols), else 2^12, 8 bytes
    // per symbol (6.5 %)
    p.fin_lb = opt.fin_lb ? opt.fin_lb : (fin_image_bytes(N, opt.fin_shift, 13) <= dev.total / 10 * 3 ? 13 : 12);
    p.oct_shift = opt.oct_shift;
    p.fin_shift = opt.fin_shift;
    return p;
}

// An index that lives in HBM pays one 128-byte line fill per pair step whatever it does, and HBM is
// large: every two further table levels remove one of those steps from every query.  Deepen the
// automatic choice while the tables (depth s and s-1) stay below 4x the block and multi-step images and a
// quarter of the free device memory once those images exist.
int deepen_table_for_hbm(int s, uint64_t image_bytes, size_t entry_bytes, uint64_t free_bytes) {
    const uint64_t budget = std::min<uint64_t>(4 * image_bytes, free_bytes / 4);
    while (s < kMaxTableS) {
        const uint64_t next = ((1ull << (2 * (s + 1))) + (1ull << (2 * s))) * entry_bytes;
        if (next > budget) break;
        s++;
    }
    return s;
}

int build_pair(msbwt_index *idx, Replica &rep, uint8_t **keep_codes = nullptr) {
    DeviceGuard guard(rep.device);
    if (int rc = build_pair_image_on_device(rep.device, rep.view, idx->start, rep.pair, keep_codes); rc != MSBWT_OK) {
        free_pair_image(rep.pair);
        return rc;
    }
    refresh_view(rep);
    return MSBWT_OK;
}

// Out of device memory for an image the caller did not require: the index works without it.  Clears the CUDA error and
// the builder's message, so that the create still succeeds with an empty msbwt_last_error().
bool absorb_oom(int rc, bool required) {
    if (rc != MSBWT_ENOMEM || required) return false;
    cudaGetLastError();
    g_last_error.clear();
    return true;
}

void build_trace(const char *what) {
    static const bool on = getenv("MSBWT_TRACE") != nullptr;
    if (!on) return;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    fprintf(stderr, "[msbwt] index build: %s (%.1f GB of device memory free)\n", what, (double)free_b / 1e9);
}

// The final-step lines on top of the oct image, from the 20-symbol codes (owned by the builder from here on).  Running out
// of device memory leaves the index without this image unless the caller required it.
int build_fin(Replica &rep, const Layout &p, uint64_t *codes20) {
    if (int rc = build_fin_lines_on_device(rep.device, rep.view.total, codes20, p.fin_shift, p.fin_lb, rep.fin); rc != MSBWT_OK) {
        free_fin_image(rep.fin);
        return absorb_oom(rc, p.fin_required) ? MSBWT_OK : rc;
    }
    refresh_view(rep);
    build_trace("multi-step images done");
    return MSBWT_OK;
}

// The multi-step images of an index that lives in HBM, built on the replica's device in stages so that the peak
// footprint stays below the device's memory even for a 3 Gsymbol BWT:
//   pair image + pair codes -> quad image + quad codes (pair image dropped) -> 10-symbol codes (quad codes dropped)
//   -> 20-symbol codes -> [quad image dropped unless it is kept] -> oct lines -> final-step lines.
// The quad image is what the builders walk LF^4 with; afterwards it only serves remainders of 4..9 symbols and the
// rare fallbacks (overflowed line, range over two buckets) of the oct kernel.  It is dropped unless `keep_quad` -- and
// always kept when there is no oct image on top (N >= 2^32, or switched off): then it is the search image.
int build_multi_step(msbwt_index *idx, Replica &rep, const Layout &p) {
    uint8_t *codes2 = nullptr;
    if (int rc = build_pair(idx, rep, &codes2); rc != MSBWT_OK) return rc;
    DeviceGuard guard(rep.device);
    DevicePtr<uint8_t> codes2_owner(codes2);
    uint16_t *codes4 = nullptr;
    build_trace("quad image");
    int rc = build_quad_image_on_device(rep.device, rep.view, codes2, rep.quad, p.oct ? &codes4 : nullptr);
    free_pair_image(rep.pair);
    if (rc != MSBWT_OK) { free_quad_image(rep.quad); if (codes4) cudaFree(codes4); return rc; }
    refresh_view(rep);
    if (!p.oct) return MSBWT_OK;

    const uint64_t N = rep.view.total;
    // 10-symbol codes (4 B per position), then 20-symbol codes (8 B per position): both walk LF^4 through the quad image
    uint32_t *codes10 = nullptr;
    build_trace("10-symbol codes");
    rc = build_oct_codes_on_device(rep.device, rep.view, codes4, codes2, &codes10);  // frees codes4
    if (rc != MSBWT_OK) return rc;
    DevicePtr<uint32_t> codes10_owner(codes10);
    codes2_owner.reset();
    uint64_t *codes20 = nullptr;
    if (p.fin) {  // no room for the codes: codes20 stays null and the index works without this image
        rc = build_fin_codes_on_device(rep.device, rep.view, codes10, &codes20);
        if (rc != MSBWT_OK && !absorb_oom(rc, p.fin_required)) return rc;
    }
    DevicePtr<uint64_t> codes20_owner(codes20);
    if (!p.keep_quad) {
        build_trace("dropping the quad image");
        free_quad_image(rep.quad);
        refresh_view(rep);
    }

    // oct lines: what is left after the final-step lines, their sort scratch (about 16 B per position, of which the
    // 12 B per position of the two code arrays are free again by then) and 8 GB for the suffix table and the query
    // pipeline; the builder picks coarser buckets, or builds nothing, beyond that
    const uint64_t free_b = free_bytes_now();
    const uint64_t fin_need = codes20 ? fin_image_bytes(N, p.fin_shift, p.fin_lb) + 4 * N : 0;
    const uint64_t reserve = fin_need + (p.oct_required ? 0 : (8ull << 30));
    const uint64_t budget = free_b > reserve ? free_b - reserve : 0;
    build_trace("oct lines");
    rc = build_oct_lines_on_device(rep.device, rep.view, codes10, p.oct_shift, budget, rep.oct);
    codes10_owner.reset();
    if (rc != MSBWT_OK) { free_oct_image(rep.oct); return rc; }
    if (!rep.oct.lines) {  // no room at all: the quad image serves alone and must stay
        if (!rep.view.quad) return fail(MSBWT_ENOMEM, "no room for the oct image after the quad image was dropped (MSBWT_KEEP_QUAD=1 keeps it)");
        return MSBWT_OK;
    }
    refresh_view(rep);
    if (codes20) return build_fin(rep, p, codes20_owner.release());
    build_trace("multi-step images done");
    return MSBWT_OK;
}

// The same two images for an index whose positions need 64 bits (N >= 2^32: the reference is u64 throughout,
// src/msbwt_core.rs:18-24, src/rle_bwt.rs:14-24; or several superblocks).  A quad image of such an index (36.6 B per
// position: 157 GB at 2^32) has no room, so nothing is built on the way: the builders walk LF through the one-step
// blocks (oct_builder.cu build_oct_codes_by_walk, fin_builder.cu build_fin_codes_by_walk), and the search kernel
// (wide_kernels.cu) takes remainders and fallbacks as one-symbol steps.
//   10-symbol codes -> oct lines -> 20-symbol codes (10-symbol codes dropped) -> final-step lines.
// Unless `oct_required`, running out of device memory leaves the index without these images (*built = false,
// MSBWT_OK) and the caller falls back to the quad or pair route.
int build_multi_step_wide(Replica &rep, const Layout &p, bool *built) {
    *built = false;
    DeviceGuard guard(rep.device);
    const uint64_t N = rep.view.total;
    uint32_t *codes10 = nullptr;
    build_trace("10-symbol codes (walk)");
    int rc = build_oct_codes_by_walk(rep.device, rep.view, &codes10);
    if (rc != MSBWT_OK) return absorb_oom(rc, p.oct_required) ? MSBWT_OK : rc;
    DevicePtr<uint32_t> codes10_owner(codes10);

    const uint64_t free_b = free_bytes_now();
    // what the final-step image will need after the oct lines exist: its lines, the 20-symbol codes (8 B per
    // position) and the run records + sort scratch (4 B per position once the codes are gone)
    const uint64_t fin_need = p.fin ? fin_image_bytes(N, p.fin_shift, p.fin_lb) + 12 * N : 0;
    const uint64_t reserve = fin_need + (p.oct_required ? 0 : (8ull << 30));
    const uint64_t budget = free_b > reserve ? free_b - reserve : 0;
    build_trace("oct lines");
    rc = build_oct_lines_on_device(rep.device, rep.view, codes10, p.oct_shift, budget, rep.oct);
    if (rc != MSBWT_OK) {
        free_oct_image(rep.oct);
        return absorb_oom(rc, p.oct_required) ? MSBWT_OK : rc;
    }
    if (!rep.oct.lines) {
        if (p.oct_required) return fail(MSBWT_ENOMEM, "no room for the oct image of this index");
        return MSBWT_OK;
    }
    refresh_view(rep);
    *built = true;
    if (!p.fin) return MSBWT_OK;

    uint64_t *codes20 = nullptr;
    rc = build_fin_codes_by_walk(rep.device, rep.view, codes10, &codes20);
    codes10_owner.reset();
    if (rc != MSBWT_OK) return absorb_oom(rc, p.fin_required) ? MSBWT_OK : rc;
    return build_fin(rep, p, codes20);
}

int build_suffix_table(Replica &rep, int s) {
    if (s <= 0) return MSBWT_OK;
    DeviceGuard guard(rep.device);
    const bool wide = index_is_wide(rep.view);
    const size_t eb = wide ? 16 : 8;
    // levels kept: s, and the (stride - 1) below it that a multi-step image may start from
    const int keep_lower = (rep.view.quad || rep.view.oct) ? 3 : (rep.view.pair ? 1 : 0);
    const int lowest_kept = std::max(1, s - keep_lower);
    std::vector<void *> level((size_t)s + 1, nullptr);
    void *scratch[2] = {nullptr, nullptr};
    auto cleanup = [&](bool all) {
        for (void *p : scratch) if (p) cudaFree(p);
        if (all) for (int j = lowest_kept; j <= s; j++) if (level[(size_t)j]) cudaFree(level[(size_t)j]);
    };
    cudaError_t e = cudaSuccess;
    for (int j = lowest_kept; j <= s && e == cudaSuccess; j++) e = cudaMalloc(&level[(size_t)j], (1ull << (2 * j)) * eb);
    if (lowest_kept > 0 && e == cudaSuccess) {  // levels below the kept ones ping-pong through two scratch buffers
        const uint64_t big = 1ull << (2 * (lowest_kept - 1));
        e = cudaMalloc(&scratch[0], big * eb);
        if (e == cudaSuccess) e = cudaMalloc(&scratch[1], std::max<uint64_t>(1, big / 4) * eb);
        for (int j = lowest_kept - 1, t = 0; j >= 0; j--, t ^= 1) level[(size_t)j] = scratch[t];
    }
    if (e != cudaSuccess) {
        cleanup(true);
        return fail(MSBWT_ENOMEM, std::string("suffix table: ") + cudaGetErrorString(e));
    }
    uint64_t root[2] = {0, rep.view.total};
    uint32_t root32[2] = {0, (uint32_t)rep.view.total};
    e = cudaMemcpy(level[0], wide ? (const void *)root : (const void *)root32, eb, cudaMemcpyHostToDevice);
    for (int j = 0; j < s && e == cudaSuccess; j++) {
        e = launch_table_extend(rep.device, rep.view, level[(size_t)j], level[(size_t)j + 1], (uint32_t)(1ull << (2 * (j + 1))), nullptr);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cleanup(true);
        return fail(MSBWT_ECUDA, std::string("suffix table build: ") + cudaGetErrorString(e));
    }
    cleanup(false);
    rep.d_table = level[(size_t)s];
    for (int b = 1; b <= 3 && s - b >= lowest_kept; b++) rep.d_table_lower[b - 1] = level[(size_t)(s - b)];
    rep.table_s = (uint32_t)s;
    refresh_view(rep);
    return MSBWT_OK;
}

msbwt_index *create_common(const uint8_t *rle, uint64_t len, const int *devices, int ndev, Options opt, int *err) {
    fill_from_env(opt);
    g_last_error.clear();
    auto idx = std::make_unique<msbwt_index>();
    int rc = validate_rle(rle, len);
    if (rc == MSBWT_OK) rc = build_replicas_on_device(idx.get(), rle, len, opt.sb_shift, devices, ndev);
    if (rc == MSBWT_OK) {
        rc = for_each_replica_slot(idx->reps.size(), [&](size_t slot) -> int {
            Replica &rep = *idx->reps[slot];
            DeviceGuard guard(rep.device);
            const uint64_t N = rep.view.total;
            const bool wide = index_is_wide(rep.view);
            // Planned from the device's free memory before any optional image exists.  A wide build that runs out of
            // memory frees everything it allocated, and cudaMalloc / cudaFree keep no cache, so the quad route after it
            // meets the same free memory.
            const Layout p = plan_layout(opt, N, wide, replica_bytes(rep), device_sizes(rep.device));
            bool wide_oct = false;
            if (p.wide_oct) {
                if (int r = build_multi_step_wide(rep, p, &wide_oct); r != MSBWT_OK) return r;
            }
            if (!wide_oct && (p.quad || p.pair)) {
                if (int r = p.quad ? build_multi_step(idx.get(), rep, p) : build_pair(idx.get(), rep); r != MSBWT_OK) return r;
            }
            int s = p.table_s;
            if (!p.explicit_s && (wide_oct || p.quad || (p.pair && p.hbm))) {
                const uint64_t multi = wide_oct ? oct_image_bytes(N, rep.oct.shift) : p.quad ? quad_image_bytes(N) : rep.view.npair * kPairBytes;
                s = deepen_table_for_hbm(s, rep.view.nblocks * kBlockBytes + multi, wide ? 16 : 8, free_bytes_now());
                // with ten symbols per oct line a 31-mer wants the depth-11 level (33 MB, L2-resident): the
                // deepest of the four kept levels need not go beyond 14 (2.1 GB instead of 8.6 GB at 15)
                if (rep.view.oct) s = std::min(s, kOctAutoTableS);
            }
            if (int r = build_suffix_table(rep, s); r != MSBWT_OK) return r;
            rep.lanes = p.lanes;
            return MSBWT_OK;
        });
    }
    if (err) *err = rc;
    if (rc != MSBWT_OK) return nullptr;
    return idx.release();
}

}  // namespace

// ================================================================ construction

extern "C" msbwt_index *msbwt_index_create_from_rle(const uint8_t *rle, uint64_t len, const int *devices, int ndev,
                                                   int *err) {
    return create_common(rle, len, devices, ndev, Options{}, err);
}

extern "C" msbwt_index *msbwt_index_create_ex(const uint8_t *rle, uint64_t len, const int *devices, int ndev,
                                             uint32_t superblock_shift, int suffix_table_s, int *err) {
    Options o;
    o.sb_shift = superblock_shift;
    o.table_s = suffix_table_s;
    return create_common(rle, len, devices, ndev, o, err);
}

namespace {
int parse_options(const msbwt_options *opts, Options &o) {
    if (opts) {
        if (opts->struct_size < offsetof(msbwt_options, quad_index))  // the ABI-2 struct ended before quad_index
            return fail(MSBWT_EINVAL, "msbwt_options.struct_size is smaller than the oldest msbwt_options this library accepts");
        o.sb_shift = opts->superblock_shift;
        o.table_s = opts->suffix_table_s;
        o.pair = opts->pair_index;
        o.lanes = opts->kernel_lanes;
        if (opts->struct_size >= offsetof(msbwt_options, quad_index) + sizeof(int32_t)) o.quad = opts->quad_index;
        if (opts->struct_size >= offsetof(msbwt_options, oct_index) + sizeof(int32_t)) o.oct = opts->oct_index;
        if (opts->struct_size >= offsetof(msbwt_options, oct_bucket_shift) + sizeof(int32_t)) o.oct_shift = opts->oct_bucket_shift;
        if (opts->struct_size >= offsetof(msbwt_options, final_lines_log2) + sizeof(int32_t)) {  // the four ABI-4 fields
            o.keep_quad = opts->keep_quad_index;
            o.fin = opts->final_index;
            o.fin_shift = opts->final_bucket_shift;
            o.fin_lb = opts->final_lines_log2;
        }
    }
    return MSBWT_OK;
}

}  // namespace

extern "C" msbwt_index *msbwt_index_create_opts(const uint8_t *rle, uint64_t len, const int *devices, int ndev,
                                               const msbwt_options *opts, int *err) {
    Options o;
    if (int rc = parse_options(opts, o); rc != MSBWT_OK) {
        if (err) *err = rc;
        return nullptr;
    }
    return create_common(rle, len, devices, ndev, o, err);
}

extern "C" msbwt_index *msbwt_index_create_from_npy(const char *path, const int *devices, int ndev, int *err) {
    g_last_error.clear();
    std::vector<uint8_t> payload;
    if (int rc = read_npy_payload(path, payload); rc != MSBWT_OK) {
        if (err) *err = rc;
        return nullptr;
    }
    return create_common(payload.data(), payload.size(), devices, ndev, Options{}, err);
}

extern "C" msbwt_index *msbwt_index_create_from_npy_opts(const char *path, const int *devices, int ndev,
                                                        const msbwt_options *opts, int *err) {
    g_last_error.clear();
    Options o;
    if (int rc = parse_options(opts, o); rc != MSBWT_OK) {
        if (err) *err = rc;
        return nullptr;
    }
    std::vector<uint8_t> payload;
    if (int rc = read_npy_payload(path, payload); rc != MSBWT_OK) {
        if (err) *err = rc;
        return nullptr;
    }
    return create_common(payload.data(), payload.size(), devices, ndev, o, err);
}

extern "C" void msbwt_index_destroy(msbwt_index *idx) { delete idx; }

// ================================================================ accessors

extern "C" uint64_t msbwt_total_size(const msbwt_index *idx) { return idx ? idx->total : 0; }
extern "C" uint64_t msbwt_symbol_count(const msbwt_index *idx, uint8_t sym) {
    return (idx && sym < kAlphabet) ? idx->counts[sym] : 0;
}
extern "C" uint64_t msbwt_start_index(const msbwt_index *idx, uint8_t sym) {
    if (!idx) return 0;
    return sym < kAlphabet ? idx->start[sym] : idx->total;
}
extern "C" int msbwt_device_count(const msbwt_index *idx) { return idx ? (int)idx->reps.size() : 0; }
extern "C" int msbwt_device_ordinal(const msbwt_index *idx, int slot) {
    return (idx && slot >= 0 && slot < (int)idx->reps.size()) ? idx->reps[slot]->device : -1;
}
extern "C" uint64_t msbwt_index_bytes(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? replica_bytes(*idx->reps[0]) : 0; }
extern "C" int msbwt_suffix_table_s(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? (int)idx->reps[0]->view.table_s : 0; }
extern "C" int msbwt_kernel_lanes(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? idx->reps[0]->lanes : 0; }
extern "C" int msbwt_pair_index(const msbwt_index *idx) { return (idx && !idx->reps.empty() && idx->reps[0]->view.pair) ? 1 : 0; }
extern "C" int msbwt_quad_index(const msbwt_index *idx) { return (idx && !idx->reps.empty() && idx->reps[0]->view.quad) ? 1 : 0; }
extern "C" int msbwt_oct_index(const msbwt_index *idx) { return (idx && !idx->reps.empty() && idx->reps[0]->view.oct) ? 1 : 0; }
extern "C" uint64_t msbwt_oct_overflow_lines(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? idx->reps[0]->oct.overflow_lines : 0; }
extern "C" uint64_t msbwt_oct_overflow_occurrences(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? idx->reps[0]->oct.overflow_occurrences : 0; }
extern "C" uint64_t msbwt_oct_runs(const msbwt_index *idx) { return (idx && !idx->reps.empty()) ? idx->reps[0]->oct.runs : 0; }
extern "C" int msbwt_oct_symbols(void) { return kOctSyms; }
// final-step image (layout.h): built by default on top of the oct image; final_index = 0 turns it off
extern "C" int msbwt_final_index(const msbwt_index *idx) {
    return (idx && !idx->reps.empty() && idx->reps[0]->view.fin) ? 1 : 0;
}
extern "C" int msbwt_debug_copy_final_image(const msbwt_index *idx, int slot, uint64_t *nlines, uint32_t *bucket_shift,
                                            uint32_t *lines_log2, uint64_t *overflow_lines, uint32_t *lines) {
    g_last_error.clear();
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    Replica &rep = *idx->reps[(size_t)slot];
    if (!rep.fin.lines) return fail(MSBWT_EINVAL, "this index has no final-step image");
    if (nlines) *nlines = rep.fin.nlines;
    if (bucket_shift) *bucket_shift = (uint32_t)rep.fin.shift;
    if (lines_log2) *lines_log2 = (uint32_t)rep.fin.lb;
    if (overflow_lines) *overflow_lines = rep.fin.overflow_lines;
    if (lines) {
        DeviceGuard guard(rep.device);
        CU_TRY(cudaMemcpy(lines, rep.fin.lines, rep.fin.nlines * (size_t)kFinLineBytes, cudaMemcpyDeviceToHost));
    }
    return MSBWT_OK;
}
// the depth policy on its own (no device needed): `steps` = symbols per step of the image that serves list A
// (1 one-step blocks, 2 pair lines, 4 quad sectors, kOctSyms oct lines)
extern "C" int msbwt_debug_table_depth(uint32_t k, uint32_t table_s, uint32_t steps) {
    if (steps == (uint32_t)kOctSyms) return (int)oct_table_depth(k, table_s);
    if (steps == 1 || steps == 2 || steps == 4) return (int)acgt_table_depth(k, table_s, steps);
    return -1;
}
// the layout policy on its own (no device needed): what create plans for a replica from these options, the environment
// and these sizes
extern "C" int msbwt_debug_plan_layout(const msbwt_options *opts, uint64_t total, int wide, uint64_t block_bytes,
                                       uint64_t l2_bytes, uint64_t free_bytes, uint64_t device_bytes, int32_t *plan, int nplan) {
    g_last_error.clear();
    Options o;
    if (int rc = parse_options(opts, o); rc != MSBWT_OK) return rc;
    fill_from_env(o);
    const Layout p = plan_layout(o, total, wide != 0, block_bytes, DeviceSizes{l2_bytes, free_bytes, device_bytes});
    const int32_t v[] = {p.table_s,   p.explicit_s,   p.hbm,          p.wide_oct, p.quad,  p.oct,       p.fin,      p.pair,
                         p.keep_quad, p.oct_required, p.fin_required, p.fin_lb,   p.lanes, p.oct_shift, p.fin_shift};
    if (!plan || nplan < (int)std::size(v)) return fail(MSBWT_EINVAL, "plan_layout: plan must hold 15 values");
    std::copy(std::begin(v), std::end(v), plan);
    return MSBWT_OK;
}
extern "C" int msbwt_table_depth_for_k(const msbwt_index *idx, uint32_t k) {
    return (idx && !idx->reps.empty()) ? (int)list_a_table_depth(idx->reps[0]->view, k) : 0;
}
extern "C" int msbwt_oct_bucket_shift(const msbwt_index *idx) { return (idx && !idx->reps.empty() && idx->reps[0]->view.oct) ? (int)idx->reps[0]->view.oct_shift : 0; }
extern "C" uint64_t msbwt_launch_count(void) { return g_launches.load(); }
extern "C" const char *msbwt_last_error(void) { return g_last_error.c_str(); }
extern "C" int msbwt_abi_version(void) { return MSBWT_ABI_VERSION; }

extern "C" void *msbwt_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        g_last_error = "cudaHostAlloc failed";
        return nullptr;
    }
    return p;
}
extern "C" void msbwt_host_free(void *p) { if (p) cudaFreeHost(p); }

// ================================================================ device-buffer entry points

extern "C" int msbwt_count_kmers_fixed_device(const msbwt_index *idx, int slot, const uint8_t *d_syms, uint32_t k,
                                              uint64_t n, uint64_t *d_out, uint32_t *d_status, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_out || (k && !d_syms))) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    std::lock_guard<std::mutex> lock(rep.mu);
    DeviceGuard guard(rep.device);
    cudaStream_t st = (cudaStream_t)stream;
    const uint64_t per = std::min<uint64_t>(n, kMaxPerLaunch);
    uint32_t *flag = d_status ? d_status : rep.d_status + kStatusDev;
    // The call is asynchronous and its pack / seed scratch is the replica's: a later call on ANOTHER stream must not
    // start rewriting the scratch while this one's kernels still read it.  Every call records an event after its last
    // launch and makes its own stream wait for the previous call's event first (a no-op on the same stream).
    if (!rep.dev_packed_free) CU_TRY(cudaEventCreateWithFlags(&rep.dev_packed_free, cudaEventDisableTiming));
    else CU_TRY(cudaStreamWaitEvent(st, rep.dev_packed_free, 0));
    CU_TRY(cudaMemsetAsync(flag, 0, sizeof(uint32_t), st));
    CU_TRY(rep.dev_packed.reserve(packed_layout(rep.view, k, per).total() * sizeof(uint64_t)));
    for (uint64_t q0 = 0; q0 < n; q0 += per) {  // sub-batches reuse the scratch in stream order
        const uint64_t m = std::min(per, n - q0);
        CU_TRY(launch_pack_seed(rep.view, d_syms + q0 * k, k, m, rep.dev_packed.as<uint64_t>(), d_out + q0, flag, st));
        CU_TRY(launch_count_packed(rep.device, rep.view, rep.lanes, rep.dev_packed.as<uint64_t>(), k, m, d_out + q0, st));
    }
    CU_TRY(cudaEventRecord(rep.dev_packed_free, st));
    return MSBWT_OK;
}

extern "C" uint64_t msbwt_packed_bytes(const msbwt_index *idx, uint32_t k, uint64_t n) {
    return (idx && !idx->reps.empty()) ? packed_layout(idx->reps[0]->view, k, n).total() * sizeof(uint64_t) : 0;
}

extern "C" int msbwt_pack_kmers_device(const msbwt_index *idx, int slot, const uint8_t *d_syms, uint32_t k, uint64_t n,
                                       uint64_t *d_packed, uint64_t *d_out, uint32_t *d_status, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_packed || !d_out || !d_status || (k && !d_syms))) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (n > kMaxPerLaunch) return fail(MSBWT_EINVAL, "more than 2^30 queries per pack/count pair: split the batch");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    CU_TRY(launch_pack_seed(rep.view, d_syms, k, n, d_packed, d_out, d_status, (cudaStream_t)stream));
    return MSBWT_OK;
}

// the pack stage for k-mers the caller holds on the device as 2-bit-per-symbol integers (msbwt_count_kmers_u64's format)
extern "C" int msbwt_seed_kmers_u64_device(const msbwt_index *idx, int slot, const uint64_t *d_kmers, uint32_t k, uint64_t n,
                                           uint64_t *d_packed, uint64_t *d_out, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_packed || !d_out || !d_kmers)) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (k == 0 || k > 32) return fail(MSBWT_EINVAL, "k must be 1..32 (one 2-bit-per-symbol word per k-mer)");
    if (n > kMaxPerLaunch) return fail(MSBWT_EINVAL, "more than 2^30 queries per pack/count pair: split the batch");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    CU_TRY(launch_seed_u64(rep.view, d_kmers, k, n, d_packed, d_out, (cudaStream_t)stream));
    return MSBWT_OK;
}

extern "C" int msbwt_count_kmers_packed_device(const msbwt_index *idx, int slot, const uint64_t *d_packed, uint32_t k,
                                               uint64_t n, uint64_t *d_out, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_out || !d_packed)) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (n > kMaxPerLaunch) return fail(MSBWT_EINVAL, "more than 2^30 queries per pack/count pair: split the batch");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    CU_TRY(launch_count_packed(rep.device, rep.view, rep.lanes, d_packed, k, n, d_out, (cudaStream_t)stream));
    return MSBWT_OK;
}

// Measurement aid: what the last msbwt_pack_kmers_device call on this scratch left for the search kernels and what
// its one-request path did (synchronises the device).  out[0] = live list A, [1] = live list B, [2] = final-step
// lines fetched by the pack stage, [3] = of which had overflowed, [4] = ranges over two buckets, [5] = k-mers the
// suffix table already answered with an empty range ([2..5] are zero when the one-request path did not apply).
extern "C" int msbwt_debug_pack_stats(const msbwt_index *idx, int slot, const uint64_t *d_packed, uint32_t k, uint64_t n,
                                      uint64_t *out6) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size() || !d_packed || !out6) return fail(MSBWT_EINVAL, "bad handle, slot or buffer");
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    const PackedLayout lay = packed_layout(rep.view, k, n);
    uint64_t tmp[8];
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(tmp, d_packed + lay.live(), sizeof(tmp), cudaMemcpyDeviceToHost));
    out6[0] = tmp[0]; out6[1] = tmp[1];
    for (int i = 0; i < 4; i++) out6[2 + i] = tmp[4 + i];
    return MSBWT_OK;
}

// Measurement aid: msbwt_count_kmers_packed_device over list A with the counting instantiation of the oct kernel
// (stats_kernels.cu).  d_stats: 8 u64 on the device -- oct lines, final-step lines, of which overflowed, quad steps,
// 128-byte lines those read, one-symbol steps, 64-byte blocks those read, queries walked.  EINVAL without an oct image.
extern "C" int msbwt_count_kmers_packed_stats_device(const msbwt_index *idx, int slot, const uint64_t *d_packed, uint32_t k,
                                                     uint64_t n, uint64_t *d_out, uint64_t *d_stats, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_out || !d_packed || !d_stats)) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (n > kMaxPerLaunch) return fail(MSBWT_EINVAL, "more than 2^30 queries per pack/count pair: split the batch");
    Replica &rep = *idx->reps[slot];
    if (!rep.view.oct) return fail(MSBWT_EINVAL, "this index has no oct image");
    if (index_is_wide(rep.view)) return fail(MSBWT_EINVAL, "the counting build of the oct kernel exists for 32-bit positions only");
    if (!n) return MSBWT_OK;
    DeviceGuard guard(rep.device);
    CU_TRY(launch_count_oct_stats(rep.device, rep.view, d_packed, k, n, d_out, (unsigned long long *)d_stats, (cudaStream_t)stream));
    return MSBWT_OK;
}

extern "C" int msbwt_constrain_ranges_device(const msbwt_index *idx, int slot, const uint8_t *d_sym,
                                             const uint64_t *d_l, const uint64_t *d_h, uint64_t n,
                                             uint64_t *d_out_l, uint64_t *d_out_h, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_sym || !d_l || !d_h || !d_out_l || !d_out_h)) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    CU_TRY(launch_constrain_ranges(rep.device, rep.view, d_sym, d_l, d_h, n, d_out_l, d_out_h, (cudaStream_t)stream));
    return MSBWT_OK;
}

extern "C" int msbwt_l2_fetch_granularity(int device, int bytes) {
    DeviceGuard guard(device);
    if (bytes > 0) {
        cudaError_t e = cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes);
        if (e != cudaSuccess) return -fail(MSBWT_ECUDA, std::string("cudaDeviceSetLimit: ") + cudaGetErrorString(e));
    }
    size_t v = 0;
    cudaError_t e = cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity);
    if (e != cudaSuccess) return -fail(MSBWT_ECUDA, std::string("cudaDeviceGetLimit: ") + cudaGetErrorString(e));
    return (int)v;
}

// ================================================================ inspection

extern "C" int msbwt_debug_build_image(const uint8_t *rle, uint64_t len, uint32_t superblock_shift, uint64_t *nblocks,
                                       uint32_t *n_super, uint32_t *blocks, uint32_t *aux, uint64_t *cbase) {
    g_last_error.clear();
    if (!nblocks || !n_super) return fail(MSBWT_EINVAL, "NULL size outputs");
    HostImage img;
    if (int rc = build_image_from_rle(rle, len, superblock_shift, img); rc != MSBWT_OK) return rc;
    *nblocks = img.nblocks;
    *n_super = img.n_super;
    if (blocks) memcpy(blocks, img.blocks.data(), img.blocks.size() * sizeof(uint32_t));
    if (aux) memcpy(aux, img.aux.data(), img.aux.size() * sizeof(uint32_t));
    if (cbase) memcpy(cbase, img.cbase.data(), img.cbase.size() * sizeof(uint64_t));
    return MSBWT_OK;
}

extern "C" int msbwt_debug_copy_image(const msbwt_index *idx, int slot, uint64_t *nblocks, uint32_t *n_super,
                                      uint32_t *blocks, uint32_t *aux, uint64_t *cbase) {
    g_last_error.clear();
    if (!idx || slot < 0 || slot >= (int)idx->reps.size() || !nblocks || !n_super) return fail(MSBWT_EINVAL, "bad handle, slot or size outputs");
    const Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    *nblocks = rep.view.nblocks;
    *n_super = rep.view.n_super;
    if (blocks) CU_TRY(cudaMemcpy(blocks, rep.d_blocks, rep.view.nblocks * kBlockBytes, cudaMemcpyDeviceToHost));
    if (aux) CU_TRY(cudaMemcpy(aux, rep.d_aux, rep.view.nblocks * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (cbase) CU_TRY(cudaMemcpy(cbase, rep.d_cbase, (size_t)rep.view.n_super * 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return MSBWT_OK;
}

extern "C" int msbwt_debug_host_pack(const uint8_t *syms, uint32_t k, uint64_t n, int threads, uint64_t *words,
                                     uint64_t *exceptions, uint64_t max_exceptions, uint64_t *n_exceptions) {
    g_last_error.clear();
    if (!k || (n && (!syms || !words)) || !n_exceptions) return fail(MSBWT_EINVAL, "host_pack: k == 0 or NULL buffer");
    if (threads < 1) threads = 1;
    HostPool pool(threads);
    std::vector<std::vector<uint64_t>> exc((size_t)threads);
    pool.begin_session();
    pool.run([&](int tid, int nthreads) {
        host_pack_range(syms, k, n, n * (uint64_t)tid / (uint64_t)nthreads, n * (uint64_t)(tid + 1) / (uint64_t)nthreads, 0, n,
                        words, exc[(size_t)tid]);
    });
    pool.end_session();
    uint64_t total = 0;
    for (auto &v : exc)
        for (uint64_t q : v) {
            if (exceptions && total < max_exceptions) exceptions[total] = q;
            total++;
        }
    *n_exceptions = total;
    return MSBWT_OK;
}

extern "C" int msbwt_debug_copy_pair_image(const msbwt_index *idx, int slot, uint64_t *npair, uint32_t *n_super2,
                                           uint32_t *lines, uint64_t *c2base) {
    g_last_error.clear();
    if (!idx || slot < 0 || slot >= (int)idx->reps.size() || !npair || !n_super2) return fail(MSBWT_EINVAL, "bad handle, slot or size outputs");
    const Replica &rep = *idx->reps[slot];
    if (!rep.view.pair) return fail(MSBWT_EINVAL, "this index has no pair image");
    DeviceGuard guard(rep.device);
    *npair = rep.view.npair;
    *n_super2 = rep.view.c2base ? rep.view.n_super2 : 0;
    if (lines) CU_TRY(cudaMemcpy(lines, rep.view.pair, rep.view.npair * kPairBytes, cudaMemcpyDeviceToHost));
    if (c2base && rep.view.c2base) CU_TRY(cudaMemcpy(c2base, rep.view.c2base, (size_t)rep.view.n_super2 * 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return MSBWT_OK;
}

extern "C" int msbwt_debug_copy_quad_image(const msbwt_index *idx, int slot, uint64_t *nsec4, uint32_t *n_super4,
                                           uint32_t *sectors, uint64_t *c4base) {
    g_last_error.clear();
    if (!idx || slot < 0 || slot >= (int)idx->reps.size() || !nsec4 || !n_super4) return fail(MSBWT_EINVAL, "bad handle, slot or size outputs");
    const Replica &rep = *idx->reps[slot];
    if (!rep.view.quad) return fail(MSBWT_EINVAL, "this index has no quad image");
    DeviceGuard guard(rep.device);
    *nsec4 = rep.view.nsec4;
    *n_super4 = rep.view.c4base ? rep.view.n_super4 : 0;
    if (sectors) CU_TRY(cudaMemcpy(sectors, rep.view.quad, (size_t)kQuadCodes * rep.view.nsec4 * kQuadSectorBytes, cudaMemcpyDeviceToHost));
    if (c4base && rep.view.c4base) CU_TRY(cudaMemcpy(c4base, rep.view.c4base, (size_t)rep.view.n_super4 * kQuadCodes * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return MSBWT_OK;
}

extern "C" int msbwt_debug_copy_oct_image(const msbwt_index *idx, int slot, uint64_t *nbuck8, uint32_t *lines) {
    g_last_error.clear();
    if (!idx || slot < 0 || slot >= (int)idx->reps.size() || !nbuck8) return fail(MSBWT_EINVAL, "bad handle, slot or size output");
    const Replica &rep = *idx->reps[slot];
    if (!rep.view.oct) return fail(MSBWT_EINVAL, "this index has no oct image");
    DeviceGuard guard(rep.device);
    *nbuck8 = rep.view.nbuck8;
    if (lines) CU_TRY(cudaMemcpy(lines, rep.view.oct, (size_t)kOctCodes * rep.view.nbuck8 * kOctLineBytes, cudaMemcpyDeviceToHost));
    return MSBWT_OK;
}

// ================================================================ batched callers of the path (SURVEY 8f N3)

extern "C" int msbwt_constrain_ranges_fanout_device(const msbwt_index *idx, int slot, const uint64_t *d_l,
                                                    const uint64_t *d_h, uint64_t n, uint64_t *d_out_l,
                                                    uint64_t *d_out_h, void *stream) {
    if (!idx || slot < 0 || slot >= (int)idx->reps.size()) return fail(MSBWT_EINVAL, "bad handle or slot");
    if (n && (!d_l || !d_h || !d_out_l || !d_out_h)) return fail(MSBWT_EINVAL, "NULL device buffer");
    if (!n) return MSBWT_OK;
    Replica &rep = *idx->reps[slot];
    DeviceGuard guard(rep.device);
    CU_TRY(launch_constrain_fanout(rep.device, rep.view, d_l, d_h, n, d_out_l, d_out_h, (cudaStream_t)stream));
    return MSBWT_OK;
}

// ================================================================ construction of the BWT itself

namespace {
int check_device(int device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(MSBWT_ENODEV, "no usable CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= count) return fail(MSBWT_ENODEV, "device ordinal out of range");
    return MSBWT_OK;
}

// `len` RLE bytes on the current device -> *rle, a malloc'd host copy (the caller frees it with msbwt_buffer_free)
int rle_to_host(const uint8_t *d_rle, uint64_t len, uint8_t **rle) {
    uint8_t *host = (uint8_t *)malloc(len ? len : 1);
    if (!host) return fail(MSBWT_ENOMEM, "host buffer for the RLE bytes");
    if (len) {
        if (cudaError_t e = cudaMemcpy(host, d_rle, len, cudaMemcpyDeviceToHost); e != cudaSuccess) {
            free(host);
            return fail(MSBWT_ECUDA, std::string("copying the RLE bytes: ") + cudaGetErrorString(e));
        }
    }
    *rle = host;
    return MSBWT_OK;
}

// reads (and, for reads of different lengths, their n_reads + 1 offsets) on the host or already on `device` ->
// RLE bytes of their multi-string BWT in a malloc'd host buffer
int build_rle_bwt_common(const uint8_t *reads, const uint64_t *offsets, uint64_t n_reads, uint32_t read_len, uint64_t n_syms,
                         int on_device, int device, uint8_t **rle, uint64_t *rle_len, uint64_t *total) {
    if (int rc = check_device(device); rc != MSBWT_OK) return rc;
    DeviceGuard guard(device);
    DevicePtr<uint8_t> reads_copy;
    DevicePtr<uint64_t> offsets_copy;
    const uint8_t *d_reads = reads;
    const uint64_t *d_offsets = offsets;
    if (!on_device && n_reads) {
        if (n_syms) {
            uint8_t *p = nullptr;
            CU_TRY(cudaMalloc(&p, n_syms));
            reads_copy.reset(p);
            CU_TRY(cudaMemcpy(p, reads, n_syms, cudaMemcpyHostToDevice));
        }
        d_reads = reads_copy.get();
        if (offsets) {
            uint64_t *p = nullptr;
            CU_TRY(cudaMalloc(&p, (n_reads + 1) * sizeof(uint64_t)));
            offsets_copy.reset(p);
            CU_TRY(cudaMemcpy(p, offsets, (n_reads + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice));
            d_offsets = p;
        }
    }
    uint8_t *d_rle = nullptr;
    int rc = build_rle_bwt_on_device(d_reads, d_offsets, n_reads, read_len, &d_rle, rle_len, total);
    DevicePtr<uint8_t> d_rle_owner(d_rle);
    if (rc != MSBWT_OK) return rc;
    return rle_to_host(d_rle, *rle_len, rle);
}
}  // namespace

extern "C" int msbwt_build_rle_bwt(const uint8_t *reads, uint64_t n_reads, uint32_t read_len, int reads_on_device,
                                   int device, uint8_t **rle, uint64_t *rle_len, uint64_t *total) {
    g_last_error.clear();
    if (!rle || !rle_len || !total) return fail(MSBWT_EINVAL, "NULL output pointer");
    *rle = nullptr;
    *rle_len = 0;
    *total = 0;
    if (n_reads && (!reads || !read_len)) return fail(MSBWT_EINVAL, "NULL reads or read_len == 0");
    return build_rle_bwt_common(reads, nullptr, n_reads, read_len, n_reads * read_len, reads_on_device, device, rle, rle_len, total);
}

extern "C" int msbwt_build_rle_bwt_ragged(const uint8_t *syms, const uint64_t *offsets, uint64_t n_reads, int device,
                                          uint8_t **rle, uint64_t *rle_len, uint64_t *total) {
    g_last_error.clear();
    if (!rle || !rle_len || !total) return fail(MSBWT_EINVAL, "NULL output pointer");
    *rle = nullptr;
    *rle_len = 0;
    *total = 0;
    if (!n_reads) return MSBWT_OK;
    if (!offsets) return fail(MSBWT_EINVAL, "NULL offsets");
    uint64_t longest = 0;
    for (uint64_t r = 0; r < n_reads; r++) {
        if (offsets[r + 1] < offsets[r]) return fail(MSBWT_EINVAL, "offsets must be non-decreasing");
        longest = std::max(longest, offsets[r + 1] - offsets[r]);
    }
    if (longest >= 0xFFFFFFFFull) return fail(MSBWT_EINVAL, "a read is longer than 2^32 - 2 symbols");
    const uint64_t n_syms = offsets[n_reads] - offsets[0];
    if (n_syms && !syms) return fail(MSBWT_EINVAL, "NULL symbols");
    // the kernels index the symbols with the caller's absolute offsets: copy from the first read's first symbol and
    // bias the device pointer instead of rewriting the offsets
    if (offsets[0] == 0)
        return build_rle_bwt_common(syms, offsets, n_reads, (uint32_t)longest, n_syms, 0, device, rle, rle_len, total);
    std::vector<uint64_t> rebased(offsets, offsets + n_reads + 1);
    for (auto &o : rebased) o -= offsets[0];
    return build_rle_bwt_common(syms + offsets[0], rebased.data(), n_reads, (uint32_t)longest, n_syms, 0, device, rle, rle_len, total);
}

extern "C" int msbwt_merge_rle_bwts(const uint8_t *rle_a, uint64_t len_a, const uint8_t *rle_b, uint64_t len_b, int device,
                                    uint8_t **rle, uint64_t *rle_len, uint64_t *total, uint32_t *iterations) {
    g_last_error.clear();
    if (!rle || !rle_len || !total) return fail(MSBWT_EINVAL, "NULL output pointer");
    *rle = nullptr;
    *rle_len = 0;
    *total = 0;
    if (iterations) *iterations = 0;
    if ((len_a && !rle_a) || (len_b && !rle_b)) return fail(MSBWT_EINVAL, "NULL input with a length above 0");
    if (int rc = check_device(device); rc != MSBWT_OK) return rc;
    DeviceGuard guard(device);
    uint8_t *d_rle = nullptr;
    uint64_t len = 0, n = 0;
    uint32_t passes = 0;
    int rc = merge_rle_bwts_on_device(rle_a, len_a, rle_b, len_b, &d_rle, &len, &n, &passes);
    DevicePtr<uint8_t> d_rle_owner(d_rle);
    if (rc != MSBWT_OK) return rc;
    if (int r = rle_to_host(d_rle, len, rle); r != MSBWT_OK) return r;
    *rle_len = len;
    *total = n;
    if (iterations) *iterations = passes;
    return MSBWT_OK;
}

static int kmer_spectrum_call(const msbwt_index *idx, bool canonical, uint32_t k, uint64_t min_count, uint64_t *hist,
                              uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers) {
    g_last_error.clear();
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!k || k > 32) return fail(MSBWT_EINVAL, "kmer_spectrum: k must be in 1..32");
    if (!min_count) return fail(MSBWT_EINVAL, "kmer_spectrum: min_count must be at least 1");
    if (!n_kmers) return fail(MSBWT_EINVAL, "kmer_spectrum: NULL n_kmers");
    if (nbins && !hist) return fail(MSBWT_EINVAL, "kmer_spectrum: NULL hist with nbins > 0");
    if (nbins == 1 || nbins > (1u << 20)) return fail(MSBWT_EINVAL, "kmer_spectrum: nbins must be 0 or in 2..2^20");
    if (!kmers != !counts) return fail(MSBWT_EINVAL, "kmer_spectrum: kmers and counts must be both NULL or both set");
    *n_kmers = 0;
    if (kmers) *kmers = *counts = nullptr;
    // replica 0's images are read-only after create; the call has its own stream and scratch (the canonical lookups
    // too: no lane of the replica), so it takes no lock and runs beside the query entry points
    const Replica &rep = *idx->reps[0];
    DeviceGuard guard(rep.device);
    return kmer_spectrum_on_device(rep.device, rep.view, rep.lanes, canonical, k, min_count, hist, nbins, kmers, counts,
                                   n_kmers);
}

extern "C" int msbwt_kmer_spectrum(const msbwt_index *idx, uint32_t k, uint64_t min_count, uint64_t *hist, uint32_t nbins,
                                   uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers) {
    return kmer_spectrum_call(idx, false, k, min_count, hist, nbins, kmers, counts, n_kmers);
}

extern "C" int msbwt_kmer_spectrum_canonical(const msbwt_index *idx, uint32_t k, uint64_t min_count, uint64_t *hist,
                                             uint32_t nbins, uint64_t **kmers, uint64_t **counts, uint64_t *n_kmers) {
    return kmer_spectrum_call(idx, true, k, min_count, hist, nbins, kmers, counts, n_kmers);
}

extern "C" int msbwt_unitigs(const msbwt_index *idx, uint32_t k, uint64_t min_count, int canonical, uint8_t **syms,
                             uint64_t **offsets, uint64_t **count_sums, uint64_t *n_unitigs) {
    g_last_error.clear();
    if (!idx || idx->reps.empty()) return fail(MSBWT_EINVAL, "bad handle");
    if (!k || k > 32) return fail(MSBWT_EINVAL, "unitigs: k must be in 1..32");
    if (!min_count) return fail(MSBWT_EINVAL, "unitigs: min_count must be at least 1");
    if (canonical != 0 && canonical != 1) return fail(MSBWT_EINVAL, "unitigs: canonical must be 0 or 1");
    if (!syms || !offsets || !count_sums || !n_unitigs) return fail(MSBWT_EINVAL, "unitigs: NULL output pointer");
    *syms = nullptr;
    *offsets = *count_sums = nullptr;
    *n_unitigs = 0;
    // as the spectrum: replica 0's images are read-only after create and the call has its own stream and scratch
    const Replica &rep = *idx->reps[0];
    DeviceGuard guard(rep.device);
    return unitigs_on_device(rep.device, rep.view, rep.lanes, canonical == 1, k, min_count, syms, offsets, count_sums,
                             n_unitigs);
}

extern "C" void msbwt_buffer_free(uint8_t *p) { free(p); }

// ================================================================ measurement aid

extern "C" int msbwt_gather_bench(int device, const void *d_buf, uint64_t buf_bytes, uint32_t granule,
                                  uint64_t n_gathers, uint64_t seed, uint64_t *d_sink, void *stream) {
    if (!d_buf || !d_sink) return fail(MSBWT_EINVAL, "NULL device buffer");
    DeviceGuard guard(device);
    CU_TRY(launch_gather(device, d_buf, buf_bytes, granule, n_gathers, seed, d_sink, (cudaStream_t)stream));
    return MSBWT_OK;
}
