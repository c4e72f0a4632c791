// loader.cu -- host side of index construction: msbwt RLE byte stream (or the .npy
// that wraps it) -> block image described in layout.h.
//
// Replaces, for the device layout, the reference's load path: load_vector /
// load_numpy_file (src/rle_bwt.rs:59-66,81-155) -> standard_init ->
// calculate_totals + construct_fmindex (src/rle_bwt.rs:324-467).  The reference's
// sampled tables are not reproduced: the block image is a different exact rank
// structure (see layout.h).
#include <cstdio>
#include <cstring>

#include "../../include/msbwt_gpu.h"
#include "engine.h"

namespace msbwt {

namespace {

struct ImageWriter {
    HostImage &img;
    uint64_t pos = 0;
    uint64_t running[kAlphabet] = {0, 0, 0, 0, 0, 0};
    uint64_t super_base[kAlphabet] = {0, 0, 0, 0, 0, 0};

    explicit ImageWriter(HostImage &i) : img(i) { open_block(0); }

    void open_block(uint64_t blk) {
        const uint64_t per_super = (uint64_t)1 << img.sb_shift;
        if ((blk & (per_super - 1)) == 0) {
            const uint64_t sb = blk >> img.sb_shift;
            for (int s = 0; s < kAlphabet; s++) {
                super_base[s] = running[s];
                img.cbase[sb * 8 + s] = img.start[s] + running[s];
            }
        }
        uint32_t *w = &img.blocks[blk * kWordsPerBlock];
        for (int s : {1, 2, 3, 5}) {
            const int slot = ckpt_slot(s);  // half = slot >> 1, word = slot & 1
            w[(slot >> 1) * 8 + (slot & 1)] = (uint32_t)(running[s] - super_base[s]);
        }
        img.aux[blk * 2 + 0] = (uint32_t)(running[0] - super_base[0]);  // $
        img.aux[blk * 2 + 1] = (uint32_t)(running[4] - super_base[4]);  // N
    }

    // set symbol `sym` at block offsets [off, off+take) of block blk
    void fill(uint64_t blk, uint32_t off, uint32_t take, uint32_t sym) {
        uint32_t *w = &img.blocks[blk * kWordsPerBlock];
        const uint32_t end = off + take;
        for (uint32_t j = off >> 5; j <= (end - 1) >> 5; j++) {
            const uint32_t lo = off > (j << 5) ? off - (j << 5) : 0;
            const uint32_t hi = end < ((j + 1) << 5) ? end - (j << 5) : 32;
            const uint32_t m = (hi == 32 ? ~0u : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
            uint32_t *hw = w + (j >> 1) * 8 + (j & 1);  // half j/2, word j%2 within each plane pair
            if (sym & 1u) hw[2] |= m;
            if (sym & 2u) hw[4] |= m;
            if (sym & 4u) hw[6] |= m;
        }
    }

    void run(uint32_t sym, uint64_t len) {
        while (len) {
            const uint64_t blk = pos >> kBlockShift;
            const uint32_t off = (uint32_t)(pos & (kBlockSyms - 1));
            const uint32_t take = (uint32_t)(len < (uint64_t)(kBlockSyms - off) ? len : (uint64_t)(kBlockSyms - off));
            fill(blk, off, take, sym);
            running[sym] += take;
            pos += take;
            len -= take;
            if ((pos & (kBlockSyms - 1)) == 0) open_block(pos >> kBlockShift);
        }
    }

    void finish() {
        const uint32_t off = (uint32_t)(pos & (kBlockSyms - 1));
        fill(pos >> kBlockShift, off, kBlockSyms - off, 7u);  // padding matches no symbol
    }
};

}  // namespace

// Format check shared by both builders, done on the host before any device is touched so that a
// malformed stream is MSBWT_EFORMAT regardless of the machine: symbol >= 6 (the reference panics
// indexing symbol_counts, src/rle_bwt.rs:371) or a single run of 13+ bytes (>= 2^60 symbols).
int validate_rle(const uint8_t *rle, uint64_t len) {
    if (len && !rle) return fail(MSBWT_EINVAL, "rle is NULL");
    uint8_t prev = 255;
    int digits = 0;
    uint64_t total = 0;  // every addend is below 2^60 and the sum is checked after each: it cannot wrap unnoticed
    for (uint64_t i = 0; i < len; i++) {
        const uint8_t c = rle[i] & 7u;
        if (c >= kAlphabet)
            return fail(MSBWT_EFORMAT, "RLE byte " + std::to_string(i) + " has symbol " + std::to_string(c) + " (>= 6)");
        digits = (c == prev) ? digits + 1 : 0;
        prev = c;
        if (digits >= 12) return fail(MSBWT_EFORMAT, "run longer than 2^60 symbols");
        total += (uint64_t)(rle[i] >> 3) << (5 * digits);
        if (total >> 62) return fail(MSBWT_EFORMAT, "BWT longer than 2^62 symbols");  // (the device builder's u64 prefix sums stay exact)
    }
    return MSBWT_OK;
}

int build_image_from_rle(const uint8_t *rle, uint64_t len, uint32_t sb_shift, HostImage &img) {
    if (len && !rle) return fail(MSBWT_EINVAL, "rle is NULL");
    if (sb_shift == 0) sb_shift = kDefaultSuperShift;
    if (sb_shift > (uint32_t)kDefaultSuperShift) return fail(MSBWT_EINVAL, "superblock_shift > 25 would overflow the u32 block counters");

    // pass 1: symbol totals (the C array) -- src/rle_bwt.rs:352-384
    uint8_t prev = 255;
    int digits = 0;
    uint64_t total = 0;
    for (uint64_t i = 0; i < len; i++) {
        const uint8_t v = rle[i], c = v & 7u;
        if (c >= kAlphabet)
            return fail(MSBWT_EFORMAT, "RLE byte " + std::to_string(i) + " has symbol " + std::to_string(c) + " (>= 6)");
        digits = (c == prev) ? digits + 1 : 0;
        prev = c;
        if (digits >= 12) return fail(MSBWT_EFORMAT, "run longer than 2^60 symbols");
        const uint64_t add = (uint64_t)(v >> 3) << (5 * digits);
        img.counts[c] += add;
        total += add;
        if (total >> 62) return fail(MSBWT_EFORMAT, "BWT longer than 2^62 symbols");
    }
    uint64_t sum = 0;
    for (int s = 0; s < kAlphabet; s++) { img.start[s] = sum; sum += img.counts[s]; }
    img.total = total;
    img.sb_shift = sb_shift;
    img.nblocks = (total >> kBlockShift) + 1;
    img.n_super = (uint32_t)(((img.nblocks - 1) >> sb_shift) + 1);
    try {
        img.blocks.assign(img.nblocks * kWordsPerBlock, 0u);
        img.aux.assign(img.nblocks * 2, 0u);
        img.cbase.assign((size_t)img.n_super * 8, 0ull);
    } catch (const std::bad_alloc &) {
        return fail(MSBWT_ENOMEM, "out of host memory for the block image");
    }

    // pass 2: runs -> blocks
    ImageWriter wr(img);
    prev = 255;
    digits = 0;
    uint64_t run_len = 0;
    for (uint64_t i = 0; i < len; i++) {
        const uint8_t v = rle[i], c = v & 7u;
        if (c == prev) {
            digits++;
            run_len += (uint64_t)(v >> 3) << (5 * digits);
        } else {
            if (run_len) wr.run(prev, run_len);
            prev = c;
            digits = 0;
            run_len = v >> 3;
        }
    }
    if (run_len) wr.run(prev, run_len);
    wr.finish();
    return MSBWT_OK;
}

// ---------------------------------------------------------------- .npy reader

namespace {

// Reads the `shape` tuple's first entry out of a numpy header dict.  Accepts what the
// reference accepts (src/rle_bwt.rs:115-125: the dict, after quote/paren/False
// substitutions, must be valid JSON whose "shape"[0] is an unsigned integer).
struct DictReader {
    const char *p, *end;
    bool have_shape = false;
    uint64_t shape0 = 0;

    void ws() { while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) p++; }
    bool lit(const char *w) { size_t n = strlen(w); if ((size_t)(end - p) >= n && !memcmp(p, w, n)) { p += n; return true; } return false; }
    bool str(std::string &out) {
        if (p >= end || (*p != '\'' && *p != '"')) return false;
        p++;  // the reference maps ' to " so either quote closes either
        const char *s = p;
        while (p < end && *p != '\'' && *p != '"') { if (*p == '\\') p++; p++; }
        if (p >= end) return false;
        out.assign(s, p);
        p++;
        return true;
    }
    bool number(bool &is_uint, uint64_t &v) {
        const char *s = p;
        bool neg = false, frac = false;
        if (p < end && *p == '-') { neg = true; p++; }
        const char *d = p;
        v = 0;
        while (p < end && *p >= '0' && *p <= '9') { v = v * 10 + (uint64_t)(*p - '0'); p++; }
        if (p == d) { p = s; return false; }
        if (p - d > 1 && *d == '0') return false;
        if (p < end && *p == '.') { frac = true; p++; const char *f = p; while (p < end && *p >= '0' && *p <= '9') p++; if (p == f) return false; }
        if (p < end && (*p == 'e' || *p == 'E')) { frac = true; p++; if (p < end && (*p == '+' || *p == '-')) p++; const char *e = p; while (p < end && *p >= '0' && *p <= '9') p++; if (p == e) return false; }
        is_uint = !neg && !frac;
        return true;
    }
    // `, }` `, ]` `,]` are tolerated by the reference's substitutions; a bare `,}` is not
    bool value(int depth, bool is_shape) {
        ws();
        if (p >= end || depth > 32) return false;
        if (*p == '{') return dict(depth + 1);
        if (*p == '(' || *p == '[') {
            p++;
            ws();
            if (p < end && (*p == ')' || *p == ']')) { p++; return true; }
            for (int idx = 0;; idx++) {
                ws();
                bool isu; uint64_t v; const char *s = p;
                if (number(isu, v)) { if (is_shape && idx == 0 && isu) { have_shape = true; shape0 = v; } }
                else { p = s; if (!value(depth + 1, false)) return false; }
                ws();
                if (p < end && *p == ',') {
                    p++;
                    const char *after = p;
                    if (p < end && *p == ' ') p++;
                    if (p < end && (*p == ')' || *p == ']')) { p++; return true; }
                    p = after;
                    continue;
                }
                if (p < end && (*p == ')' || *p == ']')) { p++; return true; }
                return false;
            }
        }
        if (*p == '\'' || *p == '"') { std::string s; return str(s); }
        if (lit("False") || lit("false") || lit("true") || lit("null")) return true;
        bool isu; uint64_t v;
        return number(isu, v);
    }
    bool dict(int depth) {
        p++;  // '{'
        ws();
        if (p < end && *p == '}') { p++; return true; }
        for (;;) {
            ws();
            std::string key;
            if (!str(key)) return false;
            ws();
            if (p >= end || *p != ':') return false;
            p++;
            const bool is_shape = (depth == 1 && key == "shape");
            if (is_shape) have_shape = false;
            if (!value(depth, is_shape)) return false;
            ws();
            if (p < end && *p == ',') {
                p++;
                const char *after = p;
                if (p < end && *p == ' ') { p++; if (p < end && *p == '}') { p++; return true; } }
                p = after;
                continue;
            }
            if (p < end && *p == '}') { p++; return true; }
            return false;
        }
    }
    bool parse() {
        ws();
        if (p >= end || *p != '{') return false;
        if (!dict(1)) return false;
        ws();
        return p == end && have_shape;
    }
};

}  // namespace

int read_npy_payload(const char *path, std::vector<uint8_t> &payload) {
    if (!path) return fail(MSBWT_EINVAL, "path is NULL");
    FILE *f = fopen(path, "rb");
    if (!f) return fail(MSBWT_EIO, std::string("cannot open ") + path + ": " + strerror(errno));
    struct Closer { FILE *f; ~Closer() { fclose(f); } } closer{f};
    if (fseek(f, 0, SEEK_END) != 0) return fail(MSBWT_EIO, "cannot seek");
    const long long full = ftell(f);
    rewind(f);
    uint8_t fixed[10];
    if (fread(fixed, 1, 10, f) != 10) return fail(MSBWT_EFORMAT, "file shorter than the 10-byte npy preamble");
    // magic and version deliberately unchecked (src/rle_bwt.rs:96)
    const size_t header_len = (size_t)fixed[8] + 256u * (size_t)fixed[9];
    size_t skip = 10 + header_len;
    if (skip % 16) skip = (skip / 16 + 1) * 16;
    std::vector<char> hdr(skip - 10);
    if (fread(hdr.data(), 1, hdr.size(), f) != hdr.size())
        return fail(MSBWT_EIO, "could not read bytes 10-" + std::to_string(skip) + " of the header");
    DictReader rd{hdr.data(), hdr.data() + hdr.size()};
    if (!rd.parse()) return fail(MSBWT_EFORMAT, "could not parse the npy header dict / shape");
    const uint64_t disk = (uint64_t)full - skip;
    if (rd.shape0 != disk)
        return fail(MSBWT_EIO, "header indicates shape of " + std::to_string(rd.shape0) + ", but remaining file size is " +
                                   std::to_string(disk));
    try { payload.resize(disk); } catch (const std::bad_alloc &) { return fail(MSBWT_ENOMEM, "out of host memory"); }
    if (disk && fread(payload.data(), 1, disk, f) != disk) return fail(MSBWT_EIO, "short read of the BWT body");
    return MSBWT_OK;
}

}  // namespace msbwt
