// msbwt_gpu.hpp -- header-only C++ host layer over the C ABI (msbwt_gpu.h), mirroring the
// reference's `RleBWT` + `BWT` trait: same names, argument meaning and error behaviour
// (src/rle_bwt.rs:44-322, src/msbwt_core.rs:18-162).  Where the reference panics this
// throws msbwt::Panic; where it returns Err(io::Error) this throws msbwt::IoError.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <array>
#include <string>
#include <vector>

#include "msbwt_gpu.h"

namespace msbwt {

constexpr int VC_LEN = 6;  // src/msbwt_core.rs:4  ($ A C G N T)

struct BWTRange {  // src/msbwt_core.rs:18-24
    uint64_t l = 0, h = 0;
    bool operator==(const BWTRange &o) const { return l == o.l && h == o.h; }
};

struct Panic : std::runtime_error { int code; Panic(int c, const std::string &m) : std::runtime_error(m), code(c) {} };
struct IoError : std::runtime_error { using std::runtime_error::runtime_error; };

// string_util.rs:15-32 / 63-67
inline uint8_t string_to_int(char c) {
    switch (c) {
        case '$': return 0;
        case 'A': case 'a': return 1;
        case 'C': case 'c': return 2;
        case 'G': case 'g': return 3;
        case 'T': case 't': return 5;
        default: return 4;
    }
}
inline std::vector<uint8_t> convert_stoi(const std::string &s) {
    std::vector<uint8_t> v(s.size());
    for (size_t i = 0; i < s.size(); i++) v[i] = string_to_int(s[i]);
    return v;
}

// bwt_converter.rs:26-80 / 102-130: text BWT -> RLE bytes; RLE bytes -> msbwt2's .npy container
inline std::vector<uint8_t> convert_to_vec(const std::string &text) {
    uint8_t *rle = nullptr;
    uint64_t n = 0;
    const int rc = msbwt_convert_to_rle(reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rle, &n);
    if (rc != MSBWT_OK) throw Panic(rc, msbwt_last_error());
    std::vector<uint8_t> out(rle, rle + n);
    msbwt_buffer_free(rle);
    return out;
}
inline void save_bwt_numpy(const std::vector<uint8_t> &rle, const std::string &filename) {
    const int rc = msbwt_save_rle_npy(rle.data(), rle.size(), filename.c_str());
    if (rc == MSBWT_EIO) throw IoError(msbwt_last_error());
    if (rc != MSBWT_OK) throw Panic(rc, msbwt_last_error());
}

class RleBWT {
  public:
    RleBWT() = default;                                            // RleBWT::new()
    static RleBWT with_bin_power(uint8_t) { return RleBWT(); }     // accepted for parity; no effect on results
    explicit RleBWT(std::vector<int> devices) : devices_(std::move(devices)) {}
    RleBWT(const RleBWT &) = delete;
    RleBWT &operator=(const RleBWT &) = delete;
    RleBWT(RleBWT &&o) noexcept : h_(o.h_), devices_(std::move(o.devices_)) { o.h_ = nullptr; }
    ~RleBWT() { msbwt_index_destroy(h_); }

    void load_vector(const std::vector<uint8_t> &bwt) {            // src/rle_bwt.rs:59-66
        int err = 0;
        msbwt_index *h = msbwt_index_create_from_rle(bwt.data(), bwt.size(), devices_.data(), (int)devices_.size(), &err);
        if (!h) raise(err);
        reset(h);
    }
    void load_numpy_file(const std::string &filename) {            // src/rle_bwt.rs:81-155
        int err = 0;
        msbwt_index *h = msbwt_index_create_from_npy(filename.c_str(), devices_.data(), (int)devices_.size(), &err);
        if (!h) raise(err);
        reset(h);
    }
    uint64_t get_symbol_count(uint8_t symbol) const { return msbwt_symbol_count(h_, symbol); }
    uint64_t get_total_size() const { return msbwt_total_size(h_); }

    BWTRange constrain_range(uint8_t sym, const BWTRange &in) const {  // src/rle_bwt.rs:202-287
        BWTRange out;
        check(msbwt_constrain_ranges(h_, &sym, &in.l, &in.h, 1, &out.l, &out.h));
        return out;
    }
    uint64_t count_kmer(const std::vector<uint8_t> &kmer) const {      // src/msbwt_core.rs:125-161
        const uint64_t offs[2] = {0, kmer.size()};
        uint64_t out = 0;
        check(msbwt_count_kmers(h_, kmer.data(), offs, 1, &out));
        return out;
    }
    // the batched entry point BASELINE.json adds: count_kmers(&[Vec<u8>]) -> Vec<u64>
    std::vector<uint64_t> count_kmers(const std::vector<std::vector<uint8_t>> &kmers) const {
        std::vector<uint64_t> offs(kmers.size() + 1, 0), out(kmers.size());
        std::vector<uint8_t> flat;
        for (size_t i = 0; i < kmers.size(); i++) {
            flat.insert(flat.end(), kmers[i].begin(), kmers[i].end());
            offs[i + 1] = flat.size();
        }
        check(msbwt_count_kmers(h_, flat.data(), offs.data(), kmers.size(), out.data()));
        return out;
    }
    std::vector<uint64_t> count_kmers_fixed(const std::vector<uint8_t> &syms, uint32_t k) const {
        if (!k || syms.size() % k) throw Panic(MSBWT_EINVAL, "len(syms) must be a positive multiple of k");
        std::vector<uint64_t> out(syms.size() / k);
        check(msbwt_count_kmers_fixed(h_, syms.data(), k, out.size(), out.data()));
        return out;
    }
    // k-mers held as integers (k <= 32, first symbol in the most significant of the 2k bits; A,C,G,T = 0..3)
    std::vector<uint64_t> count_kmers_u64(const std::vector<uint64_t> &kmers, uint32_t k) const {
        std::vector<uint64_t> out(kmers.size());
        check(msbwt_count_kmers_u64(h_, kmers.data(), k, kmers.size(), out.data()));
        return out;
    }
    // the same with 32-bit counts (index below 2^32 symbols): 4 bytes per query on the way back
    std::vector<uint32_t> count_kmers_u64_u32(const std::vector<uint64_t> &kmers, uint32_t k) const {
        std::vector<uint32_t> out(kmers.size());
        check(msbwt_count_kmers_u64_u32(h_, kmers.data(), k, kmers.size(), out.data()));
        return out;
    }
    // the four constrain_range calls (A, C, G, T) of one extension step, from one fetch of the index blocks
    std::array<BWTRange, 4> constrain_range_fanout(const BWTRange &in) const {
        uint64_t l[4], h[4];
        check(msbwt_constrain_ranges_fanout(h_, &in.l, &in.h, 1, l, h));
        std::array<BWTRange, 4> out;
        for (int j = 0; j < 4; j++) { out[j].l = l[j]; out[j].h = h[j]; }
        return out;
    }
    // count_kmer of every k-mer window of every read (reads: n * read_len symbol bytes); both_strands adds the
    // count of each window's reverse complement (string_util::reverse_complement_i)
    std::vector<uint64_t> count_read_kmers(const std::vector<uint8_t> &reads, uint32_t read_len, uint32_t k,
                                           bool both_strands = false) const {
        if (!read_len || reads.size() % read_len || !k || k > read_len) throw Panic(MSBWT_EINVAL, "bad read_len / k");
        const uint64_t n = reads.size() / read_len;
        std::vector<uint64_t> out(n * (read_len - k + 1));
        check(msbwt_count_read_kmers(h_, reads.data(), read_len, n, k, both_strands ? 2 : 1, out.data()));
        return out;
    }
    // the k-mer spectrum (hist: nbins entries, the last one = count >= nbins - 1) and, with want_list, the k-mers with
    // count >= min_count and their counts in co-lexicographic order (k <= 32; msbwt_count_kmers_u64's encoding);
    // canonical: both strands, once per pair {X, rc X} (msbwt_kmer_spectrum_canonical; the list in no promised order)
    struct KmerSpectrum {
        std::vector<uint64_t> hist, kmers, counts;
        uint64_t n_kmers = 0;
    };
    KmerSpectrum kmer_spectrum(uint32_t k, uint64_t min_count = 1, uint32_t nbins = 10001, bool want_list = false,
                               bool canonical = false) const {
        KmerSpectrum out;
        out.hist.assign(nbins, 0);
        uint64_t *km = nullptr, *cn = nullptr;
        check((canonical ? msbwt_kmer_spectrum_canonical : msbwt_kmer_spectrum)(
            h_, k, min_count, nbins ? out.hist.data() : nullptr, nbins, want_list ? &km : nullptr,
            want_list ? &cn : nullptr, &out.n_kmers));
        if (km) {
            out.kmers.assign(km, km + out.n_kmers);
            out.counts.assign(cn, cn + out.n_kmers);
        }
        msbwt_buffer_free(reinterpret_cast<uint8_t *>(km));
        msbwt_buffer_free(reinterpret_cast<uint8_t *>(cn));
        return out;
    }
    // the unitigs of the compacted de Bruijn graph of the solid k-mers (msbwt_unitigs): sequences (msbwt alphabet)
    // concatenated, n + 1 offsets, per-unitig sums of the k-window counts; ascending by first k-mer
    struct Unitigs {
        std::vector<uint8_t> syms;
        std::vector<uint64_t> offsets{0}, count_sums;
    };
    Unitigs unitigs(uint32_t k, uint64_t min_count = 2, bool canonical = false) const {
        Unitigs out;
        uint8_t *s = nullptr;
        uint64_t *o = nullptr, *c = nullptr, n = 0;
        check(msbwt_unitigs(h_, k, min_count, canonical ? 1 : 0, &s, &o, &c, &n));
        if (n) {
            out.syms.assign(s, s + o[n]);
            out.offsets.assign(o, o + n + 1);
            out.count_sums.assign(c, c + n);
        }
        msbwt_buffer_free(s);
        msbwt_buffer_free(reinterpret_cast<uint8_t *>(o));
        msbwt_buffer_free(reinterpret_cast<uint8_t *>(c));
        return out;
    }
    // reads corrected in the manner of fmlrc (msbwt_correct_reads): weak interior runs of k-mer windows bridged
    // through the solid k-mers; `stats` (optional) receives the call's five counters
    std::vector<std::vector<uint8_t>> correct_reads(const std::vector<std::vector<uint8_t>> &reads, uint32_t k,
                                                    uint64_t min_count = 5, uint32_t frac_permille = 100,
                                                    uint32_t branch_limit = 4, uint64_t *stats = nullptr) const {
        std::vector<uint8_t> flat;
        std::vector<uint64_t> offsets{0};
        for (const auto &r : reads) {
            flat.insert(flat.end(), r.begin(), r.end());
            offsets.push_back(flat.size());
        }
        uint8_t *s = nullptr;
        uint64_t *o = nullptr;
        check(msbwt_correct_reads(h_, flat.data(), offsets.data(), reads.size(), k, min_count, frac_permille,
                                  branch_limit, &s, &o, stats));
        std::vector<std::vector<uint8_t>> out(reads.size());
        for (size_t r = 0; r < reads.size(); r++) out[r].assign(s + o[r], s + o[r + 1]);
        msbwt_buffer_free(s);
        msbwt_buffer_free(reinterpret_cast<uint8_t *>(o));
        return out;
    }
    const msbwt_index *handle() const { return h_; }

  private:
    void reset(msbwt_index *h) { msbwt_index_destroy(h_); h_ = h; }
    static void raise(int rc) {
        const std::string msg = msbwt_last_error();
        if (rc == MSBWT_EIO) throw IoError(msg);
        throw Panic(rc, msg);
    }
    static void check(int rc) { if (rc != MSBWT_OK) raise(rc); }
    msbwt_index *h_ = nullptr;
    std::vector<int> devices_;
};

}  // namespace msbwt
