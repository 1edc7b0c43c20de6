// jpgpu_host.cpp — host side of the drop-in boundary: the marker/header parser that
// stands in for JPEGImage::parse (reference src/jpeg/mod.rs:202-414), geometry
// (decoder.rs:164-192), Huffman/quantisation table preparation and batch planning.
// Pure host code; the image data itself is only ever touched by the CUDA kernels.
#include "jpgpu_host.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <stdio.h>

#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <new>

namespace jpgpu {

namespace {

struct ParseError {
    int code;
};

struct Cursor {  // Rust-style bounds-checked view of the file (index OOB -> reference panic)
    const uint8_t* p;
    size_t len;
    uint8_t at(size_t i) const {
        if (i >= len) throw ParseError{JPGPU_PANIC_INDEX_OOB};
        return p[i];
    }
    void range(size_t a, size_t b) const {
        if (b > len || a > b) throw ParseError{JPGPU_PANIC_INDEX_OOB};
    }
    uint16_t be16(size_t i) const { return (uint16_t)((at(i) << 8) + at(i + 1)); }  // mod.rs:9-13
};

}  // namespace

int compute_geometry(const jpgpu_image_desc& d, Geometry& g) {
    g = Geometry();
    if (d.ncomp != 1 && d.ncomp != 3) return JPGPU_PANIC_COMPONENT_COUNT;  // decoder.rs:330
    if (d.width == 0 || d.height == 0) return JPGPU_ERR_UNSUPPORTED;
    for (uint32_t c = 0; c < d.ncomp; c++) {
        const jpgpu_component& k = d.comp[c];
        if (k.h < 1 || k.h > 2 || k.v < 1 || k.v > 2) return JPGPU_ERR_UNSUPPORTED;  // mod.rs:275-277
        g.h[c] = k.h;
        g.v[c] = k.v;
    }
    // In the order the reference meets them: the first MCU looks up every component's AC, then DC table
    // (decoder.rs:197-198 -> 154-160); the quantization tables come after the entropy decode (decoder.rs:222-224).
    for (uint32_t c = 0; c < d.ncomp; c++) {
        const jpgpu_component& k = d.comp[c];
        if (k.ta >= 4) return JPGPU_PANIC_INDEX_OOB;
        if (!d.ac_present[k.ta]) return JPGPU_PANIC_MISSING_TABLE;
        if (k.td >= 4) return JPGPU_PANIC_INDEX_OOB;
        if (!d.dc_present[k.td]) return JPGPU_PANIC_MISSING_TABLE;
    }
    for (uint32_t c = 0; c < d.ncomp; c++) {
        const jpgpu_component& k = d.comp[c];
        if (k.tq >= 4) return JPGPU_PANIC_INDEX_OOB;
        if (!d.qt_present[k.tq]) return JPGPU_PANIC_MISSING_TABLE;
    }
    if (d.layout != JPGPU_LAYOUT_REF && d.ncomp == 1) { g.h[0] = 1; g.v[0] = 1; }  // T.81 A.2.2
    g.hmax = g.vmax = 1;
    g.blocks_per_mcu = 0;
    for (uint32_t c = 0; c < d.ncomp; c++) {
        g.hmax = std::max(g.hmax, g.h[c]);
        g.vmax = std::max(g.vmax, g.v[c]);
        g.blocks_per_mcu += g.h[c] * g.v[c];
    }
    g.mcux = (d.width + 8 * g.hmax - 1) / (8 * g.hmax);
    g.mcuy = (d.height + 8 * g.vmax - 1) / (8 * g.vmax);
    const uint32_t nbx = (d.width + 7) / 8, nby = (d.height + 7) / 8;
    if (d.layout == JPGPU_LAYOUT_REF) {
        const uint32_t skip = (uint32_t)g.hmax * g.vmax;
        g.units = (nbx * nby + skip - 1) / skip;  // decoder.rs:191-192
    } else {
        g.units = g.mcux * g.mcuy;
    }
    for (uint32_t c = 0; c < d.ncomp; c++) g.nblocks[c] = g.units * g.h[c] * g.v[c];

    // which fused colour kernel, if any
    g.kind = kKindGeneric;
    if (d.ncomp == 1 && g.h[0] == 1 && g.v[0] == 1) g.kind = kKindGray;
    if (d.ncomp == 3 && g.h[1] == 1 && g.v[1] == 1 && g.h[2] == 1 && g.v[2] == 1) {
        if (g.h[0] == 1 && g.v[0] == 1) g.kind = kKind444;
        else if (g.h[0] == 2 && g.v[0] == 1) g.kind = kKind422;
        else if (g.h[0] == 2 && g.v[0] == 2) g.kind = kKind420;
        else if (g.h[0] == 1 && g.v[0] == 2) g.kind = kKind440;
    }
    if (d.layout == JPGPU_LAYOUT_SPEC) {
        g.fused_ok = g.kind != kKindGeneric;
    } else if (d.layout == JPGPU_LAYOUT_SPEC_FANCY) {
        // without sub-sampled chroma there is nothing to interpolate: the fused kernels serve gray and 4:4:4
        g.fused_ok = g.kind == kKindGray || g.kind == kKind444;
        g.compose = !g.fused_ok && g.kind != kKindGeneric;
        if (!g.fused_ok && !g.compose) return JPGPU_ERR_UNSUPPORTED;
    } else {
        // REF == SPEC exactly for these shape classes (SURVEY.md §8 parity policy)
        g.fused_ok = (g.kind == kKindGray && d.width % 8 == 0) || (g.kind == kKind444 && d.width % 8 == 0) ||
                     (g.kind == kKind422 && d.width % 16 == 0);
        if (g.fused_ok && g.units != g.mcux * g.mcuy) g.fused_ok = false;
    }
    return JPGPU_OK;
}

int build_huff_lut(const uint8_t bits[16], const uint8_t* vals, int nvals, bool is_dc, HuffLut& out) {
    memset(&out, 0, sizeof out);
    out.is_dc = is_dc ? 1u : 0u;
    int total = 0;
    for (int i = 0; i < 16; i++) total += bits[i];
    if (total > 256 || total > nvals) return JPGPU_ERR_BAD_HUFFMAN_TABLE;
    memcpy(out.vals, vals, (size_t)total);
    // canonical codes (huffman.rs:80-98 = T.81 Fig. C.2)
    struct Code { uint32_t code; int len; uint8_t val; };
    std::vector<Code> codes;
    uint32_t code = 0;
    int k = 0;
    for (int l = 1; l <= 16; l++) {
        const int n = bits[l - 1];
        out.maxcode[l] = -1;
        out.valoff[l] = k - (int32_t)code;
        for (int i = 0; i < n; i++, k++, code++) {
            if (code >= (1u << l)) return JPGPU_ERR_BAD_HUFFMAN_TABLE;  // not a prefix code
            codes.push_back(Code{code, l, vals[k]});
        }
        if (n) out.maxcode[l] = (int32_t)code - 1;
        code <<= 1;
    }
    out.maxcode[0] = -1;
    out.maxcode[17] = 0x7fffffff;
    // DC symbols naming a size category > 16 (huffman.rs:202 assert) stay out of both LUT levels: the canonical
    // walk finds them and reports them, so the per-symbol path never has to look at that flag.  So does category 16,
    // whose difference the walk's caller corrects to the reference's i16 value (dc16_correction).
    if (is_dc) codes.erase(std::remove_if(codes.begin(), codes.end(), [](const Code& c) { return c.val >= 16; }), codes.end());
    // first level: codes of length <= kLutBits fill 2^(kLutBits-len) entries each
    for (const Code& c : codes) {
        if (c.len > kLutBits) continue;
        const uint32_t first = c.code << (kLutBits - c.len), cnt = 1u << (kLutBits - c.len);
        for (uint32_t e = 0; e < cnt; e++) out.fast[first + e] = make_entry(c.val, (uint32_t)c.len, is_dc);
    }
    // second level: one sub-table per kLutBits-prefix that starts longer codes, as wide as its longest code up to
    // kLutBits+7 bits; what does not fit the pool (or is longer) is left to the canonical walk (entry 0).
    uint8_t maxlen_of[kLutSize] = {0};
    for (const Code& c : codes)
        if (c.len > kLutBits) {
            uint8_t& m = maxlen_of[c.code >> (c.len - kLutBits)];
            m = std::max<uint8_t>(m, (uint8_t)c.len);
        }
    uint32_t pool_used = 0;
    int32_t base_of[kLutSize], nb_of[kLutSize];
    for (uint32_t prefix = 0; prefix < (uint32_t)kLutSize; prefix++) {   // pools are handed out in prefix order
        base_of[prefix] = -1;
        if (!maxlen_of[prefix]) continue;
        const int nb = std::min((int)maxlen_of[prefix] - kLutBits, 7);
        if (pool_used + (1u << nb) > (uint32_t)kPoolSize) continue;
        base_of[prefix] = (int32_t)pool_used;
        nb_of[prefix] = nb;
        pool_used += 1u << nb;
        out.fast[prefix] = kLinkBit | (uint32_t)base_of[prefix] | ((uint32_t)nb << 9);
    }
    for (const Code& c : codes) {
        if (c.len <= kLutBits) continue;
        const uint32_t prefix = c.code >> (c.len - kLutBits);
        if (base_of[prefix] < 0 || c.len > kLutBits + nb_of[prefix]) continue;
        const int nb = nb_of[prefix], rest = c.len - kLutBits;  // bits of the code inside the sub-table index
        const uint32_t first = (c.code & ((1u << rest) - 1u)) << (nb - rest), cnt = 1u << (nb - rest);
        for (uint32_t e = 0; e < cnt; e++) out.pool[(uint32_t)base_of[prefix] + first + e] = make_entry(c.val, (uint32_t)c.len, is_dc);
    }
    return JPGPU_OK;
}

void build_multi_lut(const uint8_t bits[16], const uint8_t* vals, bool is_dc, std::vector<uint32_t>& out) {
    // canonical code ranges (T.81 Fig. C.2 / F.2.2.3), as build_huff_lut
    int32_t maxcode[17], valoff[17];
    uint32_t code = 0;
    int k = 0;
    for (int l = 1; l <= 16; l++) {
        maxcode[l] = -1;
        valoff[l] = k - (int32_t)code;
        k += bits[l - 1];
        code += bits[l - 1];
        if (bits[l - 1]) maxcode[l] = (int32_t)code - 1;
        code <<= 1;
    }
    const int K = is_dc ? kMultiBitsDc : kMultiBitsAc;
    const size_t base = out.size();
    out.resize(base + ((size_t)1 << K), 0u);
    for (uint32_t w = 0; w < (1u << K); w++) {
        int pos = 0, nsym = 0;
        uint32_t tb_all = 0, adv_all = 0, adv_pre = 0, tb1 = 0, adv1 = 0;
        while (pos < K) {
            // the code starting at window bit `pos`, if the window holds all of it
            int len = 0, sym = -1;
            for (int l = 1; l <= 16 && pos + l <= K; l++) {
                const int32_t c = (int32_t)((w >> (K - pos - l)) & ((1u << l) - 1u));
                if (c <= maxcode[l]) { len = l; sym = vals[(valoff[l] + c) & 255]; break; }
            }
            if (sym < 0) break;
            uint32_t size, adv;
            bool eob = false;
            if (is_dc) { if (sym >= 16) break; size = (uint32_t)sym; adv = 1; }    // size 16: dc16_correction; > 16: huffman.rs:202 (single-symbol path)
            else if (sym == 0x00) { size = 0; adv = 64; eob = true; }
            else if (sym == 0xf0) { size = 0; adv = 16; }
            else { size = (uint32_t)sym & 15u; adv = ((uint32_t)sym >> 4) + 1u; }
            if (nsym > 0 && adv_all + (eob ? 0u : adv) > 63u) break;   // would not fit one block whatever z is
            adv_pre = adv_all;
            adv_all += adv;
            tb_all += (uint32_t)len + size;
            if (nsym == 0) { tb1 = tb_all; adv1 = adv; }
            nsym++;
            pos += len + (int)size;
            if (eob || is_dc) break;
        }
        if (nsym == 0) continue;   // 0: single-symbol path
        out[base + w] = multi_entry(tb_all, adv_all, adv_pre, tb1, adv1);
        if (is_dc) {
            // one symbol: the code length goes where AC entries keep adv_pre
            int len = 0;
            for (int l = 1; l <= 16 && l <= K; l++) {
                const int32_t c = (int32_t)((w >> (K - l)) & ((1u << l) - 1u));
                if (c <= maxcode[l]) { len = l; break; }
            }
            out[base + w] = multi_entry(tb_all, 1u, (uint32_t)len, tb1, 1u);
        }
    }
}

void build_qt_multipliers(const uint16_t qt_zigzag[64], float out[64]) {
    for (int k = 0; k < 64; k++) {
        const int nat = kZigzagNaturalHost[k], u = nat & 7, v = nat >> 3;
        out[u * 8 + v] = (float)((double)qt_zigzag[k] * kAanScale[u] * kAanScale[v] / 8.0);
    }
}

namespace {
struct LutCacheEntry {
    HuffLut lut;
    std::vector<uint32_t> mlut;
};
// Process-wide, never shrinking below its entries (pointers handed out stay valid); bounded: a stream of files with
// ever new optimised tables stops being cached after kLutCacheMax entries and builds its tables per plan.
constexpr size_t kLutCacheMax = 1024;
int cached_luts(const std::string& key, const uint8_t bits[16], const uint8_t* vals, int nvals, bool is_dc, const LutCacheEntry** out) {
    static std::mutex mu;
    static std::map<std::string, std::unique_ptr<LutCacheEntry>> cache;
    static thread_local LutCacheEntry overflow;   // uncached build
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) { *out = it->second.get(); return JPGPU_OK; }
    }
    std::unique_ptr<LutCacheEntry> e(new LutCacheEntry());
    const int st = build_huff_lut(bits, vals, nvals, is_dc, e->lut);
    if (st != JPGPU_OK) return st;
    build_multi_lut(bits, vals, is_dc, e->mlut);
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second.get(); return JPGPU_OK; }
    if (cache.size() >= kLutCacheMax) { overflow = std::move(*e); *out = &overflow; return JPGPU_OK; }
    *out = cache.emplace(key, std::move(e)).first->second.get();
    return JPGPU_OK;
}
}  // namespace

uint32_t choose_subseq_bits(uint64_t total_scan_bytes) {
    if (const char* e = getenv("JPGPU_SUBSEQ_BITS")) {
        const long v = atol(e);
        if (v >= kMinSubseqBits && v <= kMaxSubseqBits && (v & (v - 1)) == 0) return (uint32_t)v;
    }
    // 8192-bit subsequences when that still gives ~1.3 decode threads per hardware thread slot (148 SMs x 1536); a
    // smaller batch trades threads for less look-back and verification per decoded bit: halve only while fewer than
    // ~120 k threads would be left (256 x 1080p: 4096 bits / 153 k threads beat 2048 bits / 306 k by 11 %).
    const uint64_t bits = total_scan_bytes * 8;
    uint32_t s = kDefaultMaxSubseqBits;
    if (bits / s >= 300000) return s;
    s >>= 1;
    while (s > (uint32_t)kMinSubseqBits && bits / s < 120000) s >>= 1;
    return s;
}

// Cold-start distance of the synchronisation pass.  A batch that fills the machine with 8192-bit subsequences pays
// for every look-back bit (1024: 12.5 % more decoding, ~15 % of the links left to the repair walks).  A small batch
// leaves most of the machine idle, and there the rounds of repair walks are what the caller waits for - with 4:2:0,
// whose six-block MCUs (two table sets in a 4+1+1 pattern) lock in slowly (a single 4096 x 4096 4:2:0 image: 9.5 ms
// with 1024 bits, 1.3 ms with 8192; MCUs of up to four blocks synchronise within 1024 bits and gain nothing).
uint32_t choose_lookback_bits(uint64_t total_scan_bytes, uint32_t sub_bits, uint32_t max_blocks_per_mcu) {
    if (const char* e = getenv("JPGPU_LOOKBACK_BITS")) {
        const long v = atol(e);
        if (v >= 0 && v <= (1 << 20)) return (uint32_t)v;
    }
    const uint64_t threads = total_scan_bytes * 8 / sub_bits;
    if (max_blocks_per_mcu < 6 || (sub_bits >= (uint32_t)kDefaultMaxSubseqBits && threads >= 300000)) return kDefaultLookbackBits;
    if (sub_bits >= 4096) return 2048u;          // measured: 256 / 512 x 1080p
    // measured: 64 x 1080p (2048-bit subsequences) 2048: 1.01 ms, 4096: 1.17 ms with the multi-symbol repair walks of
    // round 2 (round 1, symbol by symbol: 4096); 16 / 1 x 1080p, 1 x 4096 x 4096: 8192
    return threads >= 40000 ? 2048u : 8192u;
}

int build_plan(const jpgpu_image_desc* descs, size_t n, HostPlan& plan, uint32_t sub_bits) {
    plan = HostPlan();
    if (sub_bits == 0) {
        uint64_t tot = 0;
        for (size_t i = 0; i < n; i++) tot += descs[i].scan_len;
        sub_bits = choose_subseq_bits(tot);
    }
    plan.sub_bits = sub_bits;
    plan.lookback_bits = kDefaultLookbackBits;   // settled below, once the MCU structure of the images is known
    plan.seg_bits = std::max<uint32_t>(kMinSegBits, sub_bits / 8);
    if (const char* e = getenv("JPGPU_SEG_BITS")) {
        const long v = atol(e);
        if (v >= 64 && v <= (long)sub_bits && (v & (v - 1)) == 0) plan.seg_bits = (uint32_t)v;
    }
    // the write pass cuts every subsequence into units at checkpoint boundaries (decode_write_kernel)
    {
        uint32_t parts = kDefaultWriteParts;
        if (const char* e = getenv("JPGPU_WRITE_PARTS")) { const long v = atol(e); if (v >= 1 && v <= 64 && (v & (v - 1)) == 0) parts = (uint32_t)v; }
        while (parts > 1 && (parts > sub_bits / plan.seg_bits || sub_bits / parts < (uint32_t)kMinSubseqBits)) parts >>= 1;
        plan.wp_shift = 0;
        while ((1u << plan.wp_shift) < parts) plan.wp_shift++;
    }
    uint32_t lw = 0;
    while ((32u << lw) < sub_bits) lw++;
    plan.lw = lw;
    const uint64_t group_words = (uint64_t)32 << lw;  // one warp's 32 subsequences, lane-interleaved
    plan.imgs.resize(n);
    plan.status.assign(n, JPGPU_OK);
    plan.out_w.assign(n, 0);
    plan.out_h.assign(n, 0);
    plan.frame_part.assign(n, 0);
    for (size_t i = 0; i < n; i++) plan.frame_part[i] = (uint8_t)std::min<uint32_t>(descs[i].frame_part, 3u);
    std::map<std::string, uint32_t> lut_ids;
    std::map<std::string, uint32_t> qt_ids;
    std::map<std::string, uint64_t> map_ids;
    std::string cur_lutset;
    long cur_frame = -1;   // the frame whose scans are being planned (index into plan.frames), -1: none
    // groups: contiguous image ranges of about equal scan bytes
    uint64_t tot_bytes = 0;
    for (size_t i = 0; i < n; i++) tot_bytes += descs[i].scan_len;
    uint32_t want_groups = n >= 192 ? 3u : (n >= 128 ? 2u : 1u);   // few, large groups: small kernels lose more in their tails than overlap wins
    if (const char* e = getenv("JPGPU_GROUPS")) { const long v = atol(e); if (v >= 1 && v <= 64) want_groups = (uint32_t)v; }
    if (want_groups > n) want_groups = n ? (uint32_t)n : 1u;
    const uint64_t group_bytes = tot_bytes / want_groups + 1;
    uint64_t acc_bytes = 0;
    uint32_t max_bpm = 0;
    constexpr uint32_t kJobsPerCta = 8;   // write kernel CTAs take 8 warp jobs, sync kernel CTAs 4: pad to the larger
    auto close_group = [&](size_t next_img) {
        while (plan.seqs.size() % kJobsPerCta != 0) plan.seqs.push_back(SeqDesc{0xffffffffu, 0u});
        if (!plan.groups.empty()) {
            GroupPlan& g = plan.groups.back();
            g.nimg = (uint32_t)next_img - g.img0;
            g.njobs = (uint32_t)plan.seqs.size() - g.job0;
            for (int k = 0; k < kNumKinds; k++) g.kind_hi[k] = (uint32_t)plan.kind_imgs[k].size();
            g.frame_hi = (uint32_t)plan.frames.size();
        }
    };
    auto open_group = [&](size_t img) {
        GroupPlan g;
        g.img0 = (uint32_t)img;
        g.job0 = (uint32_t)plan.seqs.size();
        for (int k = 0; k < kNumKinds; k++) g.kind_lo[k] = (uint32_t)plan.kind_imgs[k].size();
        g.frame_lo = (uint32_t)plan.frames.size();
        plan.groups.push_back(g);
        cur_lutset.clear();
    };
    open_group(0);
    auto align_up = [](uint64_t x, uint64_t a) { return (x + a - 1) / a * a; };

    for (size_t i = 0; i < n; i++) {
        const jpgpu_image_desc& d = descs[i];
        ImgDev& im = plan.imgs[i];
        memset(&im, 0, sizeof im);
        if (i > 0 && acc_bytes >= (uint64_t)plan.groups.size() * group_bytes && plan.groups.size() < want_groups &&
            d.frame_part != 2) {   // the scans of one frame stay in one group: its pixels are put together there
            close_group(i);
            open_group(i);
        }
        acc_bytes += d.scan_len;
        Geometry g;
        int st = compute_geometry(d, g);
        if (st == JPGPU_OK && d.frame_part) {
            // one non-interleaved scan of a frame (jpgpu_parse_scans): entropy-decoded as the one-component image it
            // is, its pixels come from the compose path once all scans of the frame are there
            if (d.frame_part > 2 || d.ncomp != 1 || d.layout == JPGPU_LAYOUT_REF || d.frame_ncomp != 3 || d.frame_comp > 2 ||
                (d.frame_part == 2 && (i == 0 || cur_frame < 0 || plan.status[i - 1] != JPGPU_OK)))
                st = JPGPU_ERR_INVALID_ARG;
            g.fused_ok = false;
            g.compose = true;
        }
        if (st == JPGPU_OK && d.frame_part && (uint64_t)d.frame_width * d.frame_height * 3 > 0xffffffffull) st = JPGPU_ERR_UNSUPPORTED;
        if (st != JPGPU_OK || d.frame_part != 2) cur_frame = -1;
        if (st == JPGPU_OK && (d.scan == nullptr || d.scan_len < 4)) st = JPGPU_PANIC_INDEX_OOB;  // huffman.rs:127-128
        if (st == JPGPU_OK && d.scan_len > 0x1ff00000ull) st = JPGPU_ERR_UNSUPPORTED;             // bit positions are 32-bit
        if (st == JPGPU_OK && (uint64_t)g.units * g.blocks_per_mcu * 64 >= (uint64_t)kPosSat) st = JPGPU_ERR_UNSUPPORTED;   // positions saturate there (fold_advance)
        if (st == JPGPU_OK && (uint64_t)d.width * d.height * 3 > 0xffffffffull) st = JPGPU_ERR_UNSUPPORTED;   // 32-bit byte offsets inside an image's output
        // The header's claim is tied to the bytes that came with it: no block is shorter than two bits (a 1-bit DC
        // code and a 1-bit EOB), so a scan of scan_len bytes holds at most 4 * scan_len blocks.  A file claiming more
        // can only end as JPGPU_ERR_TRUNCATED, and is turned away here before anything is sized by its header (a 90 KB
        // file declaring 30001 x 30001 would otherwise reserve 10 GB of placement map, coefficients and RGB).
        if (st == JPGPU_OK && (uint64_t)g.units * g.blocks_per_mcu > (uint64_t)d.scan_len * 4 + 8) st = JPGPU_ERR_TRUNCATED;

        // Huffman tables -> slots
        uint32_t slot_lut[kMaxLutSlots];
        int nslots = 0;
        uint8_t dc_slot[4] = {0, 0, 0, 0}, ac_slot[4] = {0, 0, 0, 0};
        for (uint32_t c = 0; st == JPGPU_OK && c < d.ncomp; c++) {
            for (int cls = 0; cls < 2; cls++) {
                const int tid = cls == 0 ? d.comp[c].td : d.comp[c].ta;
                const uint8_t* bits = cls == 0 ? d.dc_bits[tid] : d.ac_bits[tid];
                const uint8_t* vals = cls == 0 ? d.dc_vals[tid] : d.ac_vals[tid];
                const int nvals = cls == 0 ? d.dc_nvals[tid] : d.ac_nvals[tid];
                std::string key(cls == 0 ? "D" : "A");
                key.append((const char*)bits, 16);
                key.append((const char*)vals, (size_t)std::min(nvals, 256));
                auto it = lut_ids.find(key);
                uint32_t id;
                if (it == lut_ids.end()) {
                    // device tables of this DHT table: built once per process (most files carry the Annex-K tables, and a
                    // multi-symbol table costs ~50 us to build - more than the rest of a single-image plan)
                    const LutCacheEntry* ce = nullptr;
                    st = cached_luts(key, bits, vals, nvals, cls == 0, &ce);
                    if (st != JPGPU_OK) break;
                    id = (uint32_t)plan.luts.size();
                    plan.luts.push_back(ce->lut);
                    plan.mlut_off.push_back((uint32_t)plan.mluts.size());
                    plan.mluts.insert(plan.mluts.end(), ce->mlut.begin(), ce->mlut.end());
                    lut_ids.emplace(key, id);
                } else {
                    id = it->second;
                }
                int s = 0;
                while (s < nslots && slot_lut[s] != id) s++;
                if (s == nslots) slot_lut[nslots++] = id;
                (cls == 0 ? dc_slot : ac_slot)[c] = (uint8_t)s;
            }
        }
        // gather path: placement map per distinct shape
        uint64_t map_off = 0;
        const uint32_t map_plane = (uint32_t)align_up((uint64_t)d.width * d.height, 4);
        if (st == JPGPU_OK && d.layout > JPGPU_LAYOUT_SPEC_FANCY) st = JPGPU_ERR_INVALID_ARG;
        if (st == JPGPU_OK && !g.fused_ok && !g.compose) {
            // the host-built placement map is 4 bytes per pixel and component, built pixel by pixel: 64 Mpixel at most
            if ((uint64_t)d.width * d.height > kMaxGatherPixels) st = JPGPU_ERR_UNSUPPORTED;
            char key[64];
            const int kl = snprintf(key, sizeof key, "%u,%u,%u,%u|%u%u,%u%u,%u%u", d.width, d.height, d.ncomp, d.layout,
                                    g.h[0], g.v[0], g.h[1], g.v[1], g.h[2], g.v[2]);
            auto it = st == JPGPU_OK ? map_ids.find(std::string(key, kl)) : map_ids.end();
            if (st == JPGPU_OK && it == map_ids.end()) {
                std::vector<uint32_t> m;
                st = build_gather_map(d, g, map_plane, m);
                if (st == JPGPU_OK) {
                    map_off = plan.gmap.size();
                    plan.gmap.insert(plan.gmap.end(), m.begin(), m.end());
                    map_ids.emplace(std::string(key, kl), map_off);
                }
            } else if (st == JPGPU_OK) {
                map_off = it->second;
            }
        }
        plan.status[i] = st;
        if (st != JPGPU_OK) {
            // Skipped image: zero work, but its own (tiny) arena slices so that the per-image
            // kernels, which still visit it, never touch another image's memory.
            im.stream_off = plan.stream_words;
            im.stream_cap_words = (uint32_t)group_words;
            plan.stream_words += group_words;
            im.raw_off = plan.raw_bytes;
            plan.raw_bytes += 16;
            im.nseg_cap = 1;
            im.seg_off = (uint32_t)plan.seg_entries;
            plan.seg_entries += 3;
            im.sub_off = (uint32_t)plan.sub_entries;
            im.seq_first = (uint32_t)plan.seqs.size();
            im.coef_off = plan.coef_elems;
            im.rgb_off = plan.rgb_bytes;
            im.blocks_per_mcu = 1;
            continue;
        }

        im.width = d.width; im.height = d.height;
        im.raw_len = (uint32_t)d.scan_len;
        im.ncomp = (uint8_t)d.ncomp;
        im.blocks_per_mcu = (uint8_t)g.blocks_per_mcu;
        max_bpm = std::max<uint32_t>(max_bpm, g.blocks_per_mcu);
        im.hmax = g.hmax; im.vmax = g.vmax;
        im.mcux = g.mcux; im.mcuy = g.mcuy; im.units = g.units;
        im.kind = g.fused_ok ? g.kind : (uint8_t)kKindGeneric; im.layout = (uint8_t)d.layout;
        im.restart_interval = d.restart_interval;
        im.seg_units = d.restart_interval * g.blocks_per_mcu * 64u;
        im.total_coefs = g.units * g.blocks_per_mcu * 64u;
        im.nslots = (uint8_t)nslots;
        plan.max_slots = std::max<uint32_t>(plan.max_slots, (uint32_t)nslots);
        for (int s = 0; s < nslots; s++) im.slot_lut[s] = slot_lut[s];
        {
            uint32_t words = 0;
            for (int s = 0; s < nslots; s++) words += 1u << (plan.luts[slot_lut[s]].is_dc ? kMultiBitsDc : kMultiBitsAc);
            plan.max_mlut_words = std::max(plan.max_mlut_words, words);
        }
        int blk = 0;
        for (uint32_t c = 0; c < d.ncomp; c++) {
            im.h[c] = g.h[c]; im.v[c] = g.v[c];
            for (int k = 0; k < g.h[c] * g.v[c]; k++, blk++) {
                im.blk_comp[blk] = (uint8_t)c;
                im.blk_dc_slot[blk] = dc_slot[c];
                im.blk_ac_slot[blk] = ac_slot[c];
                im.blk_info[blk] = (uint32_t)dc_slot[c] | ((uint32_t)ac_slot[c] << 8) | (c << 16);
            }
            // quantisation multipliers (deduplicated)
            const uint16_t* q = d.qt[d.comp[c].tq];
            std::string key((const char*)q, 128);
            auto it = qt_ids.find(key);
            if (it == qt_ids.end()) {
                const uint32_t off = (uint32_t)plan.qt.size();
                plan.qt.resize(off + 64);
                build_qt_multipliers(q, plan.qt.data() + off);
                it = qt_ids.emplace(key, off).first;
            }
            im.qt_off[c] = it->second;
        }
        // arenas
        im.raw_off = plan.raw_bytes;
        plan.raw_bytes += align_up((uint64_t)im.raw_len + 16, 16);
        im.stream_off = plan.stream_words;
        im.stream_cap_words = (uint32_t)align_up((uint64_t)(im.raw_len + 3) / 4 + 1 + kStreamPadWords, group_words);
        plan.stream_words += im.stream_cap_words;
        im.nseg_cap = d.restart_interval ? (g.units + d.restart_interval - 1) / d.restart_interval : 1u;
        if (im.nseg_cap == 0) im.nseg_cap = 1;
        // Restart intervals of at most 2.5 subsequences (measured crossover on B200: between 2 and 4): a decode thread finds an interval start (a known
        // state) near the start of its subsequence, so the image skips the synchronisation and verification passes.
        im.interval_mode = d.restart_interval && (uint64_t)im.raw_len * 8 / im.nseg_cap * 2 <= (uint64_t)sub_bits * 5 ? 1u : 0u;
        if (const char* e = getenv("JPGPU_INTERVAL_MODE")) im.interval_mode = d.restart_interval && atoi(e) ? 1u : 0u;
        if (!im.interval_mode) { plan.nsync++; plan.groups.back().nsync++; }
        im.seg_off = (uint32_t)plan.seg_entries;
        plan.seg_entries += im.nseg_cap + 2;
        {
            const uint32_t nchunks = (im.raw_len + 4095u) / 4096u;   // kPreChunk of jpgpu_kernels.cu
            im.chunk_off = (uint32_t)plan.chunk_entries;
            plan.chunk_entries += nchunks;
            plan.max_chunks = std::max(plan.max_chunks, nchunks);
            plan.groups.back().max_chunks = std::max(plan.groups.back().max_chunks, nchunks);
        }
        im.nsub_cap = std::max<uint32_t>(1u, (uint32_t)(((uint64_t)im.raw_len * 8 + sub_bits - 1) / sub_bits));
        im.sub_off = (uint32_t)plan.sub_entries;
        plan.sub_entries += im.nsub_cap;
        // warp jobs: 32 consecutive subsequences each; a CTA takes kSeqThreads/32 consecutive jobs, which may belong
        // to different images as long as those use the same Huffman tables (the CTA keeps one copy in shared memory)
        {
            std::string lutset((const char*)slot_lut, sizeof(uint32_t) * (size_t)nslots);
            if (lutset != cur_lutset && plan.seqs.size() % kJobsPerCta != 0)
                while (plan.seqs.size() % kJobsPerCta != 0) plan.seqs.push_back(SeqDesc{0xffffffffu, 0u});
            cur_lutset = lutset;
        }
        im.nseq = (im.nsub_cap + 31) / 32;
        im.seq_first = (uint32_t)plan.seqs.size();
        for (uint32_t q = 0; q < im.nseq; q++) plan.seqs.push_back(SeqDesc{(uint32_t)i, q * 32u});
        im.coef_off = plan.coef_elems;
        plan.coef_elems += im.total_coefs;
        // output: an image's own size; for the scans of a frame the first one owns the frame's pixels, the others nothing
        uint32_t ow = im.width, oh = im.height;
        if (d.frame_part == 1) { ow = d.frame_width; oh = d.frame_height; }
        if (d.frame_part == 2) { ow = oh = 0; }
        plan.out_w[i] = ow; plan.out_h[i] = oh;
        im.out_pixels = ow * oh;
        im.rgb_off = d.frame_part == 2 ? plan.frames[(size_t)cur_frame].rgb_off : plan.rgb_bytes;
        plan.rgb_bytes += align_up((uint64_t)ow * oh * 3, 256);
        const uint32_t mcus_per_tile = 128u / (8u * g.hmax);
        im.tiles_x = (g.mcux + mcus_per_tile - 1) / mcus_per_tile;
        im.tiles_y = g.mcuy;
        plan.kind_imgs[im.kind].push_back((uint32_t)i);
        plan.kind_max_tiles[im.kind] = std::max(plan.kind_max_tiles[im.kind], im.tiles_x * im.tiles_y);
        plan.groups.back().kind_max_tiles[im.kind] = std::max(plan.groups.back().kind_max_tiles[im.kind], im.tiles_x * im.tiles_y);
        if (g.compose && d.frame_part) {
            // compose path, frame of non-interleaved scans: this scan is one plane of it
            if (d.frame_part == 1) {
                FrameDev f;
                memset(&f, 0, sizeof f);
                f.width = d.frame_width; f.height = d.frame_height; f.ncomp = d.frame_ncomp;
                f.fancy = d.layout == JPGPU_LAYOUT_SPEC_FANCY ? 1u : 0u;
                f.rgb_off = im.rgb_off;
                plan.frames.push_back(f);
                cur_frame = (long)plan.frames.size() - 1;
                const uint32_t quads = (uint32_t)(((uint64_t)f.width * f.height + 3) / 4);
                plan.frame_max_quads = std::max(plan.frame_max_quads, quads);
                plan.groups.back().frame_max_quads = std::max(plan.groups.back().frame_max_quads, quads);
            }
            PlaneRef& r = plan.frames[(size_t)cur_frame].pl[d.frame_comp];
            r.smp_off = plan.sample_floats;
            r.mcux = g.mcux; r.bpm = 1; r.first = 0; r.h = r.v = 1;
            r.wc = d.width; r.hc = d.height;
            r.fx = std::max<uint32_t>(1u, d.frame_hmax / std::max<uint32_t>(1u, d.frame_h));
            r.fy = std::max<uint32_t>(1u, d.frame_vmax / std::max<uint32_t>(1u, d.frame_v));
            r.bias = d.frame_comp == 0 ? 0.0f : -128.0f;   // block_idct_kernel level-shifts every one-component image
            im.frame = (uint32_t)cur_frame + 1u;
        } else if (g.compose) {
            // compose path: one frame of this image's own three components, chroma interpolated (jpgpu_core.h)
            FrameDev f;
            memset(&f, 0, sizeof f);
            f.width = d.width; f.height = d.height; f.ncomp = d.ncomp; f.fancy = 1u;
            f.rgb_off = im.rgb_off;
            uint32_t first = 0;
            for (uint32_t c = 0; c < d.ncomp; c++) {
                PlaneRef& r = f.pl[c];
                r.smp_off = plan.sample_floats;
                r.mcux = g.mcux; r.bpm = g.blocks_per_mcu; r.first = first;
                r.h = g.h[c]; r.v = g.v[c];
                r.fx = g.hmax / g.h[c]; r.fy = g.vmax / g.v[c];
                r.wc = (d.width * g.h[c] + g.hmax - 1) / g.hmax;
                r.hc = (d.height * g.v[c] + g.vmax - 1) / g.vmax;
                r.bias = 0.0f;     // block_idct_kernel level-shifts component 0 only
                first += g.h[c] * g.v[c];
            }
            plan.frames.push_back(f);
            im.frame = (uint32_t)plan.frames.size();
            const uint32_t quads = (uint32_t)(((uint64_t)d.width * d.height + 3) / 4);
            plan.frame_max_quads = std::max(plan.frame_max_quads, quads);
            plan.groups.back().frame_max_quads = std::max(plan.groups.back().frame_max_quads, quads);
        }
        if (im.kind == kKindGeneric) {
            const uint32_t nblk = g.units * g.blocks_per_mcu;
            im.map_off = map_off;
            im.map_plane = g.compose ? 0u : map_plane;
            im.smp_off = plan.sample_floats;
            plan.sample_floats += (uint64_t)nblk * 64;
            plan.gather_max_blocks = std::max(plan.gather_max_blocks, nblk);
            plan.gather_max_quads = std::max(plan.gather_max_quads, im.map_plane / 4);
            plan.groups.back().gather_max_blocks = std::max(plan.groups.back().gather_max_blocks, nblk);
            plan.groups.back().gather_max_quads = std::max(plan.groups.back().gather_max_quads, im.map_plane / 4);
        }

        plan.tot_scan_bytes += im.raw_len;
        plan.tot_blocks += (uint64_t)g.units * g.blocks_per_mcu;
        plan.tot_pixels += (uint64_t)ow * oh;
        plan.tot_rgb_bytes += (uint64_t)ow * oh * 3;
    }
    close_group(n);
    plan.lookback_bits = choose_lookback_bits(tot_bytes, sub_bits, max_bpm);
    if (plan.sub_entries > 0xffffffffull || plan.seg_entries > 0xffffffffull) return JPGPU_ERR_UNSUPPORTED;
    return JPGPU_OK;
}

int build_gather_map(const jpgpu_image_desc& d, const Geometry& g, uint32_t plane, std::vector<uint32_t>& out) {
    const size_t W = d.width, H = d.height, npix = W * H;
    out.assign((size_t)plane * d.ncomp, kMapNone);
    uint32_t first_blk[4] = {0, 0, 0, 0};
    for (uint32_t c = 1; c < d.ncomp; c++) first_blk[c] = first_blk[c - 1] + g.h[c - 1] * g.v[c - 1];
    const uint32_t bpm = g.blocks_per_mcu;
    if (d.layout == JPGPU_LAYOUT_SPEC) {
        for (uint32_t c = 0; c < d.ncomp; c++) {
            uint32_t* m = out.data() + (size_t)c * plane;
            const uint32_t hc = g.h[c], vc = g.v[c], fx = g.hmax / hc, fy = g.vmax / vc;  // replication factors
            for (size_t y = 0; y < H; y++)
                for (size_t x = 0; x < W; x++) {
                    const uint32_t xs = (uint32_t)x / fx, ys = (uint32_t)y / fy, bx = xs >> 3, by = ys >> 3;
                    const uint32_t mcu = (by / vc) * g.mcux + bx / hc;
                    if (mcu >= g.units) continue;
                    const uint32_t blk = mcu * bpm + first_blk[c] + (by % vc) * hc + bx % hc;
                    m[y * W + x] = (blk << 6) | ((ys & 7) << 3) | (xs & 7);
                }
        }
        return JPGPU_OK;
    }
    // REF: decoder.rs:238-312 + 347-379 replayed on indices
    const size_t nbx = (W + 7) / 8, nby = (H + 7) / 8;
    for (uint32_t c = 0; c < d.ncomp; c++) {
        uint32_t* m = out.data() + (size_t)c * plane;
        const float x_i = ceilf((float)W * ((float)g.h[c] / (float)g.hmax));   // decoder.rs:237-243
        const float y_i = ceilf((float)H * ((float)g.v[c] / (float)g.vmax));
        const size_t xf = (size_t)ceilf((float)W / x_i), yf = (size_t)ceilf((float)H / y_i);  // decoder.rs:247-248
        if (xf == 0 || yf == 0) return JPGPU_PANIC_ARITH;
        const size_t hv = (size_t)g.h[c] * g.v[c], nblocks = (size_t)g.units * hv;
        size_t block_i = 0;
        for (size_t y = 0; y < nby / yf; y++)
            for (size_t x = 0; x < nbx / xf; x++, block_i++) {
                size_t bx = x, by = y;                                           // get_indices, decoder.rs:259-288
                if (g.vmax > 1 && yf == 1) {
                    if (g.hmax > 1 && xf == 1) {
                        if ((y & 1) == 0) {
                            if ((x / 2) & 1) { bx = x / 2 - 1 + (x & 1); by = y + 1; }
                            else { bx = x / 2 + (x & 1); by = y; }
                        } else {
                            if (((x / 2) & 1) == 0) { bx = nbx / 2 + x / 2 - 1 + (x & 1); by = y; }
                            else { bx = nbx / 2 + x / 2 + (x & 1); by = y - 1; }
                        }
                    } else {
                        if ((y & 1) == 0) { bx = x / 2; by = y + (x & 1); }
                        else { bx = x / 2 + nbx / 2; by = y - (x & 1); }
                    }
                }
                if (block_i >= nblocks) return JPGPU_PANIC_INDEX_OOB;            // component_blocks[block_i], decoder.rs:303
                const uint32_t blk = (uint32_t)((block_i / hv) * bpm + first_blk[c] + block_i % hv);
                const size_t start_x = bx * 8 * xf;                              // fill_block_in_array, decoder.rs:347-379
                if (W < start_x) continue;
                for (size_t line = 0; line < 8; line++) {
                    const size_t start_i = by * 8 * yf * W + line * W + start_x;
                    for (size_t ind = 0; ind < 8 * xf; ind++) {
                        const size_t i = ind + start_i;
                        for (size_t j = 0; j < yf; j++) {
                            if (i + j * W < npix) {                              // decoder.rs:371
                                const size_t idx = i + j * W * 8;                // decoder.rs:372
                                if (idx >= npix) return JPGPU_PANIC_INDEX_OOB;
                                m[idx] = (blk << 6) | (uint32_t)(line * 8 + ind / xf);
                            }
                        }
                    }
                }
            }
    }
    return JPGPU_OK;
}

void export_reference_order(const ImgDev& im, const int16_t* arena, int16_t* out, uint32_t nblocks[4]) {
    uint8_t pos[64];
    for (int k = 0; k < 64; k++) pos[k] = (uint8_t)zigzag_to_colmajor(k, kZigzagNaturalHost);
    size_t comp_off[4] = {0, 0, 0, 0};
    size_t acc = 0;
    for (int c = 0; c < 4; c++) {
        nblocks[c] = c < im.ncomp ? im.units * im.h[c] * im.v[c] : 0;
        comp_off[c] = acc;
        acc += (size_t)nblocks[c] * 64;
    }
    size_t written[4] = {0, 0, 0, 0};
    for (uint32_t m = 0; m < im.units; m++)
        for (uint32_t b = 0; b < im.blocks_per_mcu; b++) {
            const int c = im.blk_comp[b];
            const int16_t* src = arena + ((size_t)m * im.blocks_per_mcu + b) * 64;
            int16_t* dst = out + comp_off[c] + written[c] * 64;
            for (int k = 0; k < 64; k++) dst[k] = src[pos[k]];
            written[c]++;
        }
}

}  // namespace jpgpu

// =============================================================== C ABI, host-only part
using namespace jpgpu;

extern "C" int jpgpu_abi_version(void) { return JPGPU_ABI_VERSION; }

extern "C" const char* jpgpu_status_string(int s) {
    switch (s) {
        case JPGPU_OK: return "ok";
        case JPGPU_PANIC_UNHANDLED_MARKER: return "Unhandled byte marker (mod.rs:457)";
        case JPGPU_PANIC_DRI: return "got to restart interval def (mod.rs:427)";
        case JPGPU_PANIC_APP12_14: return "got ApplicationSegment12/14 (mod.rs:446,449)";
        case JPGPU_PANIC_DQT_PRECISION: return "Unknown precision of quantization table (mod.rs:258)";
        case JPGPU_PANIC_SAMPLING_ASSERT: return "sampling factor assertion failed (mod.rs:275-277)";
        case JPGPU_PANIC_INDEX_OOB: return "index out of bounds";
        case JPGPU_PANIC_NO_FRAME_HEADER: return "SOS before SOF0 (mod.rs:388 unwrap on None)";
        case JPGPU_PANIC_MISSING_TABLE: return "missing Huffman or quantization table (decoder.rs:155,159,224)";
        case JPGPU_PANIC_DC_LOOKUP: return "DC lookup fail (huffman.rs:156)";
        case JPGPU_PANIC_AC_LOOKUP: return "ILLEGAL STATE! (huffman.rs:162)";
        case JPGPU_PANIC_COMPONENT_COUNT: return "component count is neither 1 nor 3 (decoder.rs:330)";
        case JPGPU_PANIC_READ_BITS_ASSERT: return "Should not read more than 16 bits at a time! (huffman.rs:202)";
        case JPGPU_PANIC_SCAN_COMPONENT: return "scan component not found (decoder.rs:148)";
        case JPGPU_NO_SCAN: return "no SOS segment: image_data is None";
        case JPGPU_PANIC_ARITH: return "arithmetic overflow (debug build panic)";
        case JPGPU_ERR_INVALID_ARG: return "invalid argument";
        case JPGPU_ERR_NO_DEVICE: return "no usable CUDA device (there is no CPU fallback)";
        case JPGPU_ERR_CUDA: return "CUDA runtime error";
        case JPGPU_ERR_UNSUPPORTED: return "outside the supported subset";
        case JPGPU_ERR_BAD_HUFFMAN_TABLE: return "BITS/HUFFVAL do not describe a prefix code";
        case JPGPU_ERR_TRUNCATED: return "entropy-coded data ended early";
        case JPGPU_ERR_BAD_CODE: return "bit pattern is no code of the selected Huffman table";
        case JPGPU_ERR_RESTART: return "restart markers missing or out of sequence";
        case JPGPU_ERR_OOM: return "out of memory";
        default: return "unknown status";
    }
}

// The reference's own panic text for statuses 1..15 (the literal part of its message, without formatted arguments):
// what a strict drop-in shim passes to panic!() so that callers and tests matching on the message see what they saw
// before.  NULL for statuses that are not reference panics.
extern "C" const char* jpgpu_panic_message(int s) {
    switch (s) {
        case JPGPU_PANIC_UNHANDLED_MARKER: return "Unhandled byte marker";                                   // mod.rs:457
        case JPGPU_PANIC_DRI: return "got to restart interval def";                                          // mod.rs:427
        case JPGPU_PANIC_APP12_14: return "got ApplicationSegment";                                          // mod.rs:446,449 ("got {:?}")
        case JPGPU_PANIC_DQT_PRECISION: return "Unknown precision of quantization table";                    // mod.rs:258
        case JPGPU_PANIC_SAMPLING_ASSERT: return "assertion failed: horizontal_sampling_factor > 0";         // mod.rs:275-277
        case JPGPU_PANIC_INDEX_OOB: return "index out of bounds";
        case JPGPU_PANIC_NO_FRAME_HEADER: return "called `Option::unwrap()` on a `None` value";             // mod.rs:388
        case JPGPU_PANIC_MISSING_TABLE: return "Did not find quantization table for";                        // decoder.rs:224 (155,159: unwrap on None)
        case JPGPU_PANIC_DC_LOOKUP: return "called `Option::unwrap()` on a `None` value";                   // huffman.rs:156
        case JPGPU_PANIC_AC_LOOKUP: return "ILLEGAL STATE!";                                                 // huffman.rs:162
        case JPGPU_PANIC_COMPONENT_COUNT: return "asd";                                                      // decoder.rs:330
        case JPGPU_PANIC_READ_BITS_ASSERT: return "Should not read more than 16 bits at a time!";            // huffman.rs:202
        case JPGPU_PANIC_SCAN_COMPONENT: return "called `Option::unwrap()` on a `None` value";              // decoder.rs:148
        case JPGPU_PANIC_ARITH: return "attempt to subtract with overflow";                                  // mod.rs:218 (debug build)
        default: return nullptr;
    }
}

// JPEGImage::parse, mod.rs:202-414 — marker walk up to (not including) decode().
// `scans` == nullptr: the reference's walk, which ends at the first SOS with the rest of the file as scan data.
// Otherwise (jpgpu_parse_scans): every SOS appends a descriptor whose scan data ends at the next marker, and the walk
// goes on; `out` is the running state (tables, frame) the descriptors are cut from.
static int parse_walk(const uint8_t* file, size_t len, uint32_t ext, uint32_t layout, jpgpu_image_desc* out,
                      std::vector<jpgpu_image_desc>* scans) {
    memset(out, 0, sizeof *out);
    out->layout = layout;
    const Cursor f{file, len};
    struct FrameComp { uint8_t id, h, v, tq; };
    std::vector<FrameComp> frame;
    bool have_frame = false;
    try {
        size_t i = 0;
        while (i < len) {
            // bytes_to_marker, mod.rs:157-181 (including its "n == 0 -> look one byte further" quirk)
            if (f.at(i) != 0xff) { (void)f.at(i + 1); return JPGPU_PANIC_UNHANDLED_MARKER; }
            uint8_t m = f.at(i + 1);
            if (m == 0) m = f.at(i + 2);
            const bool known = m == 0xc0 || m == 0xc4 || m == 0xd8 || m == 0xd9 || m == 0xda || m == 0xdb ||
                               m == 0xdd || m == 0xe0 || m == 0xec || m == 0xee || m == 0xfe;
            const bool skippable = (ext & JPGPU_EXT_SKIP_APPN) && ((m >= 0xe1 && m <= 0xef) || (m >= 0xf0 && m <= 0xfd));
            if (!known && !skippable) return JPGPU_PANIC_UNHANDLED_MARKER;  // mod.rs:456-462
            if (m == 0xd8 || m == 0xd9) { i += 2; continue; }                // mod.rs:208-214
            const uint16_t seglen = f.be16(i + 2);
            if (seglen < 2) return JPGPU_PANIC_ARITH;                        // mod.rs:218
            const size_t dl = (size_t)seglen - 2;
            i += 4;
            switch (m) {
                case 0xfe: f.range(i, i + dl); break;                        // COM, mod.rs:222-227
                case 0xdb: {                                                 // DQT, mod.rs:228-261
                    size_t idx = i;
                    while (idx < i + dl) {
                        const uint8_t pqtq = f.at(idx);
                        const unsigned pq = pqtq >> 4, tq = pqtq & 15;
                        if (pq == 0) {
                            f.range(idx + 1, idx + 65);
                            if (tq >= 4) return JPGPU_PANIC_INDEX_OOB;
                            for (int k = 0; k < 64; k++) out->qt[tq][k] = file[idx + 1 + k];
                            out->qt_present[tq] = 1;
                            idx += 65;
                        } else if (pq == 1) {
                            f.range(idx + 1, idx + 129);
                            if (tq >= 4) return JPGPU_PANIC_INDEX_OOB;
                            for (int k = 0; k < 64; k++)
                                out->qt[tq][k] = (uint16_t)((file[idx + 1 + 2 * k] << 8) | file[idx + 2 + 2 * k]);
                            out->qt_present[tq] = 1;
                            idx += 129;
                        } else {
                            return JPGPU_PANIC_DQT_PRECISION;
                        }
                    }
                    break;
                }
                case 0xc0: {                                                 // SOF0, mod.rs:262-298
                    (void)f.at(i);
                    const uint16_t lines = f.be16(i + 1), spl = f.be16(i + 3);
                    const uint8_t nc = f.at(i + 5);
                    frame.clear();
                    size_t idx = i + 6;
                    for (unsigned c = 0; c < nc; c++, idx += 3) {
                        FrameComp fc;
                        fc.id = f.at(idx);
                        const uint8_t hv = f.at(idx + 1);
                        fc.h = hv >> 4; fc.v = hv & 15;
                        if (!(fc.h > 0 && fc.h < 3) || !(fc.v > 0 && fc.v < 3)) return JPGPU_PANIC_SAMPLING_ASSERT;
                        fc.tq = f.at(idx + 2);
                        frame.push_back(fc);
                    }
                    out->width = spl; out->height = lines;
                    have_frame = true;
                    break;
                }
                case 0xc4: {                                                 // DHT, mod.rs:299-336
                    size_t idx = i;
                    const size_t end = i + dl;
                    while (idx < end) {
                        const uint8_t tcth = f.at(idx);
                        const unsigned tc = tcth >> 4, th = tcth & 15;
                        idx += 1;
                        f.range(idx, idx + 16);
                        const uint8_t* bits = file + idx;
                        idx += 16;
                        size_t ncodes = 0;
                        for (int k = 0; k < 16; k++) ncodes += bits[k];
                        f.range(idx, idx + ncodes);
                        if (ncodes == 0) return JPGPU_PANIC_INDEX_OOB;       // huffman.rs:85 sizes[0]
                        if (th >= 4) return JPGPU_PANIC_INDEX_OOB;
                        if (ncodes > 256) return JPGPU_ERR_BAD_HUFFMAN_TABLE;
                        uint8_t* dbits = tc == 0 ? out->dc_bits[th] : out->ac_bits[th];
                        uint8_t* dvals = tc == 0 ? out->dc_vals[th] : out->ac_vals[th];
                        memcpy(dbits, bits, 16);
                        memset(dvals, 0, 256);
                        memcpy(dvals, file + idx, ncodes);
                        (tc == 0 ? out->dc_nvals : out->ac_nvals)[th] = (uint16_t)ncodes;
                        (tc == 0 ? out->dc_present : out->ac_present)[th] = 1;
                        idx += ncodes;
                    }
                    break;
                }
                case 0xda: {                                                 // SOS, mod.rs:337-414
                    const uint8_t ns = f.at(i);
                    struct ScanComp { uint8_t id, td, ta; };
                    std::vector<ScanComp> scan;
                    for (unsigned c = 0; c < ns; c++) {
                        ScanComp sc;
                        sc.id = f.at(i + 1);
                        const uint8_t t = f.at(i + 2);
                        sc.td = t >> 4; sc.ta = t & 15;
                        scan.push_back(sc);
                        i += 2;
                    }
                    (void)f.at(i + 1); (void)f.at(i + 2); (void)f.at(i + 3);
                    i += 4;
                    if (!scans && i < len && file[len - 1] == 0xff)
                        return JPGPU_PANIC_INDEX_OOB;                        // mod.rs:378: vec[i + 1] past the end
                    if (!have_frame) return JPGPU_PANIC_NO_FRAME_HEADER;     // mod.rs:388
                    // builder semantics of decoder.rs:83-152: first matching id wins, scan order kept
                    if (scan.size() > 4) return JPGPU_PANIC_COMPONENT_COUNT;
                    out->ncomp = (uint32_t)scan.size();
                    for (size_t c = 0; c < scan.size(); c++) {
                        const FrameComp* fc = nullptr;  // decoder.rs:86-95: a later frame entry with the same id overwrites
                        for (const FrameComp& k : frame) if (k.id == scan[c].id) fc = &k;
                        // decoder.rs:116-123 updates the selectors in scan order: the last entry with this id wins
                        uint8_t td = scan[c].td, ta = scan[c].ta;
                        bool first = true;
                        for (size_t k = 0; k < scan.size(); k++) {
                            if (scan[k].id != scan[c].id) continue;
                            // decoder.rs:126-136: a component the frame does not know enters with its selectors swapped
                            if (!fc && first) { td = scan[k].ta; ta = scan[k].td; } else { td = scan[k].td; ta = scan[k].ta; }
                            first = false;
                        }
                        if (!fc) {
                            // Its sampling factors are 0xff: the product overflows in the first MCU (decoder.rs:200-201, debug
                            // build) - unless a table lookup of this or an earlier scan component panics before that.
                            for (size_t e = 0; e <= c; e++) {
                                const uint8_t e_td = e < c ? out->comp[e].td : td, e_ta = e < c ? out->comp[e].ta : ta;
                                if (e_ta >= 4) return JPGPU_PANIC_INDEX_OOB;
                                if (!out->ac_present[e_ta]) return JPGPU_PANIC_MISSING_TABLE;
                                if (e_td >= 4) return JPGPU_PANIC_INDEX_OOB;
                                if (!out->dc_present[e_td]) return JPGPU_PANIC_MISSING_TABLE;
                            }
                            return JPGPU_PANIC_ARITH;
                        }
                        out->comp[c] = jpgpu_component{fc->id, fc->h, fc->v, fc->tq, td, ta};
                    }
                    out->scan = i <= len ? file + i : file + len;
                    out->scan_len = i <= len ? len - i : 0;
                    if (!scans) return JPGPU_OK;                             // mod.rs:415: decode() happens on the GPU
                    {
                        // multi-scan walk: this scan's entropy-coded data ends at the next marker that is neither a
                        // stuffed FF00, a restart marker nor a fill byte
                        size_t end = std::min(i, len);
                        while (end < len) {
                            if (file[end] == 0xff && end + 1 < len && file[end + 1] != 0x00 && file[end + 1] != 0xff &&
                                !(file[end + 1] >= 0xd0 && file[end + 1] <= 0xd7)) break;
                            end++;
                        }
                        jpgpu_image_desc d = *out;
                        d.scan_len = end - std::min(i, len);
                        if (scan.size() == frame.size()) {
                            d.frame_part = 0;                                // every component interleaved: an image of its own
                        } else if (scan.size() == 1) {
                            // one component, non-interleaved (T.81 A.2.2): a one-component image of the component's own size
                            int k = -1, hmax = 1, vmax = 1;
                            for (size_t c = 0; c < frame.size(); c++) {
                                if (frame[c].id == scan[0].id) k = (int)c;
                                hmax = std::max<int>(hmax, frame[c].h);
                                vmax = std::max<int>(vmax, frame[c].v);
                            }
                            if (k < 0 || frame.size() != 3) return JPGPU_ERR_UNSUPPORTED;
                            d.frame_part = 2;
                            d.frame_width = out->width; d.frame_height = out->height;
                            d.frame_ncomp = (uint8_t)frame.size(); d.frame_comp = (uint8_t)k;
                            d.frame_h = frame[(size_t)k].h; d.frame_v = frame[(size_t)k].v;
                            d.frame_hmax = (uint8_t)hmax; d.frame_vmax = (uint8_t)vmax;
                            d.width = (out->width * d.frame_h + hmax - 1) / hmax;
                            d.height = (out->height * d.frame_v + vmax - 1) / vmax;
                            d.comp[0].h = d.comp[0].v = 1;
                            if (d.layout == JPGPU_LAYOUT_REF) d.layout = JPGPU_LAYOUT_SPEC;   // the reference never gets here
                        } else {
                            return JPGPU_ERR_UNSUPPORTED;                    // partly interleaved scans
                        }
                        scans->push_back(d);
                        i = end;
                        continue;
                    }
                }
                case 0xdd:                                                   // DRI, mod.rs:424-428
                    if (!(ext & JPGPU_EXT_DRI)) return JPGPU_PANIC_DRI;
                    out->restart_interval = f.be16(i);
                    break;
                case 0xe0:                                                   // APP0, mod.rs:429-444 (absolute offsets)
                    f.range(i, i + 6);
                    (void)f.at(7); (void)f.at(8); (void)f.at(13); f.range(10, 12); f.range(12, 14); (void)f.at(14); (void)f.at(15);
                    break;
                case 0xec: case 0xee:                                        // APP12 / APP14, mod.rs:445-450
                    if (!(ext & JPGPU_EXT_SKIP_APPN)) return JPGPU_PANIC_APP12_14;
                    break;
                default: break;                                              // skipped extension segment
            }
            i += dl;                                                         // mod.rs:455
        }
    } catch (const ParseError& e) {
        return e.code;
    } catch (const std::bad_alloc&) {   // no C++ exception crosses the C ABI
        return JPGPU_ERR_OOM;
    } catch (...) {
        return JPGPU_ERR_INVALID_ARG;
    }
    return JPGPU_NO_SCAN;                                                    // mod.rs:464
}

extern "C" int jpgpu_parse(const uint8_t* file, size_t len, uint32_t ext, uint32_t layout, jpgpu_image_desc* out) {
    if (!file || !out) return JPGPU_ERR_INVALID_ARG;
    return parse_walk(file, len, ext & ~(uint32_t)JPGPU_EXT_MULTISCAN, layout, out, nullptr);
}

extern "C" int jpgpu_parse_scans(const uint8_t* file, size_t len, uint32_t ext, uint32_t layout, jpgpu_image_desc* out,
                                 size_t max_out, size_t* n) try {
    if (n) *n = 0;
    if (!file || !out || !n || !max_out || !(ext & JPGPU_EXT_MULTISCAN)) return JPGPU_ERR_INVALID_ARG;
    std::vector<jpgpu_image_desc> scans;
    jpgpu_image_desc state;
    const int st = parse_walk(file, len, ext, layout, &state, &scans);
    if (st != JPGPU_NO_SCAN) return st;                  // the multi-scan walk only ends by running out of markers
    if (scans.empty()) return JPGPU_NO_SCAN;
    if (scans.size() == 1 && scans[0].frame_part == 0) {
        // the ordinary file: as jpgpu_parse, except that the scan data ends at EOI instead of the end of the file
        out[0] = scans[0];
        *n = 1;
        return JPGPU_OK;
    }
    // a frame of non-interleaved scans: every component exactly once, nothing else in the file
    const size_t nc = scans[0].frame_ncomp;
    if (scans.size() != nc || nc > max_out) return scans.size() > max_out ? JPGPU_ERR_INVALID_ARG : JPGPU_ERR_UNSUPPORTED;
    uint32_t seen = 0;
    for (size_t k = 0; k < nc; k++) {
        if (scans[k].frame_part != 2 || scans[k].frame_ncomp != nc) return JPGPU_ERR_UNSUPPORTED;
        seen |= 1u << scans[k].frame_comp;
    }
    if (seen != (1u << nc) - 1u) return JPGPU_ERR_UNSUPPORTED;
    scans[0].frame_part = 1;
    for (size_t k = 0; k < nc; k++) out[k] = scans[k];
    *n = nc;
    return JPGPU_OK;
} catch (const std::bad_alloc&) {
    return JPGPU_ERR_OOM;
} catch (...) {
    return JPGPU_ERR_INVALID_ARG;
}

extern "C" int jpgpu_geometry(const jpgpu_image_desc* desc, uint32_t* mcus, uint32_t* blocks_per_mcu, uint32_t nblocks[4]) {
    if (!desc) return JPGPU_ERR_INVALID_ARG;
    Geometry g;
    const int st = compute_geometry(*desc, g);
    if (st != JPGPU_OK) return st;
    if (mcus) *mcus = g.units;
    if (blocks_per_mcu) *blocks_per_mcu = g.blocks_per_mcu;
    if (nblocks) for (int c = 0; c < 4; c++) nblocks[c] = g.nblocks[c];
    return JPGPU_OK;
}

// What the planner decides for a set of images (host only; the decisions DESIGN.md 4.2 / 4.5 describe, testable
// without a GPU).
extern "C" int jpgpu_plan_info(const jpgpu_image_desc* descs, size_t n, uint64_t info[8]) try {
    if ((!descs && n) || !info) return JPGPU_ERR_INVALID_ARG;
    HostPlan plan;
    const int st = build_plan(descs, n, plan, 0);
    if (st != JPGPU_OK) return st;
    uint64_t by_interval = 0;
    for (size_t i = 0; i < n; i++) by_interval += plan.status[i] == JPGPU_OK && plan.imgs[i].interval_mode ? 1u : 0u;
    info[0] = plan.sub_bits;
    info[1] = plan.lookback_bits;
    info[2] = plan.seg_bits;
    info[3] = 1ull << plan.wp_shift;
    info[4] = plan.groups.size();
    info[5] = by_interval;
    info[6] = plan.seqs.size();
    info[7] = plan.raw_bytes + plan.stream_words * 4 + plan.coef_elems * 2 + plan.rgb_bytes;
    return JPGPU_OK;
} catch (const std::bad_alloc&) {
    return JPGPU_ERR_OOM;
} catch (...) {
    return JPGPU_ERR_INVALID_ARG;
}
