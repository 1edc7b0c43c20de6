// jpgpu_core.h — data layout and the per-thread decode core shared by the CUDA
// kernels (jpgpu_kernels.cu) and, for host-side unit tests of the algorithm, by a
// CPU simulation harness under tests/ (never by the product path).
//
// Reference semantics restated here (file:line in martinhath/jpeg-rust):
//   huffman.rs:146-195  next_block       -> decode_symbol(): DC size/EXTEND, EOB, ZRL, (run,size)
//   huffman.rs:211-227  next_code        -> two-level LUT + huff_slow(): canonical prefix decode
//   huffman.rs:256-268  value_correction -> extend()
//   decoder.rs:195-215  MCU loop + DC prediction -> g/c bookkeeping + dc predictors
// The parallel formulation (look-back synchronisation of subsequences) is new; see DESIGN.md.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define JPGPU_HD __host__ __device__ __forceinline__
#else
#define JPGPU_HD inline
#endif

namespace jpgpu {

// ------------------------------------------------------------------ constants
constexpr int kLutBits = 9;                // first-level Huffman LUT index width
constexpr int kLutSize = 1 << kLutBits;
constexpr int kPoolSize = 256;             // second-level entries (sub-tables for codes longer than kLutBits)
constexpr int kMaxBlocksPerMcu = 12;       // 3 components x (H,V in {1,2})
constexpr int kMaxLutSlots = 6;            // distinct (DC, AC) tables one image can reference
#ifndef JPGPU_SEQ_THREADS
#define JPGPU_SEQ_THREADS 128
#endif
// Bits per subsequence (one decode thread each) are a per-batch plan parameter
// (BatchDev::sub_bits), a power of two in [kMinSubseqBits, kMaxSubseqBits]: larger means less
// look-back overhead per decoded bit, smaller means more threads for small batches.
constexpr int kMinSubseqBits = 1024;
constexpr int kMaxSubseqBits = 32768;
constexpr int kDefaultMaxSubseqBits = 8192;   // what the planner picks for large batches
constexpr int kDefaultLookbackBits = 1024;   // cold-start distance before a subsequence for machine-filling batches (choose_lookback_bits)
constexpr int kDefaultWriteParts = 1;       // write-pass units per subsequence (BatchDev::wp_shift), never shorter than kMinSubseqBits
constexpr int kMinSegBits = 512;           // smallest checkpoint distance inside a subsequence (BatchDev::seg_bits)
constexpr int kSeqThreads = JPGPU_SEQ_THREADS;  // subsequences per sequence (= CTA size of the sync/write kernels)
constexpr int kStreamPadWords = 8;         // zero words readable past every image's stream
constexpr int kWriteBufs = 1;              // coefficient block buffers per lane in the write kernel
#ifndef JPGPU_PHASE_SYMBOLS
#define JPGPU_PHASE_SYMBOLS 5
#endif
constexpr int kPhaseSymbols = JPGPU_PHASE_SYMBOLS;  // symbols a lane decodes between two cooperative flushes

// status bits accumulated per image on the device (mapped to JPGPU_* by the host)
enum : uint32_t {
    kStBadCode = 1u,       // a bit pattern matched no code (true decode path only)
    kStDone = 2u,          // all MCUs were decoded
    kStRestart = 4u,       // RST markers out of sequence / wrong count
    kStDcSize = 8u         // DC size category > 16 (reference: huffman.rs:202 assert)
};

// One Huffman table in device format.
// Packed decode entry: byte 0 total bits (code + value bits), byte 1 code length, byte 2
// zigzag advance (1 for DC; run+1; 16 for ZRL; 64 for EOB), bit 24 DC size category > 16
// (huffman.rs:202 assert).  With `advance`, next_block's three cases (huffman.rs:164-189)
// collapse into nz = min(z + advance, 64).  A first-level entry with bit 31 set links to a
// second-level sub-table: bits 0-8 pool offset, bits 9-11 its index width (1..7 bits after
// the first kLutBits).  0 = no code here (walk the canonical tables).
struct HuffLut {
    uint32_t fast[kLutSize];
    uint32_t pool[kPoolSize];
    int32_t maxcode[18];      // largest code of length l (right aligned), -1 if none; l = 1..16
    int32_t valoff[18];       // index of first symbol of length l minus its smallest code
    uint8_t vals[256];        // HUFFVAL
    uint32_t is_dc;
    uint32_t pad[3];
};
constexpr uint32_t kLinkBit = 1u << 31;

JPGPU_HD uint32_t make_entry(uint32_t sym, uint32_t len, bool is_dc) {
    uint32_t size, adv, big = 0;
    if (is_dc) { size = sym; adv = 1; if (size > 16) { size = 16; big = 1; } }
    else if (sym == 0x00) { size = 0; adv = 64; }
    else if (sym == 0xf0) { size = 0; adv = 16; }
    else { size = sym & 15; adv = (sym >> 4) + 1; }
    return (len + size) | (len << 8) | (adv << 16) | (big << 24);
}
constexpr uint32_t kBadEntry = 16u | (16u << 8) | (64u << 16);  // unknown code: 16 bits, ends the block

// ---- multi-symbol tables of the synchronisation pass
// The synchronisation pass only tracks state (bit position, zigzag index, block in the MCU, DC sums): for AC symbols
// it needs no values, only how many bits and zigzag positions they take.  Its AC lookups therefore go through a wider
// table whose entry covers EVERY symbol whose code lies inside the next kMultiBitsAc bits (the benchmark corpus averages
// 4.65 bits per symbol: 1.7 symbols per lookup).  Entry, for the bits of the window decoded greedily from the left:
//   bits  0-4   tb_all   bits consumed by all symbols of the entry (codes + value bits; the last one's value bits may
//                        reach past the window: <= kMultiBitsAc + 15)
//   bits  5-11  adv_all  zigzag positions they advance (an EOB, always last, counts 64)
//   bits 12-17  adv_pre  the same without the entry's last symbol; the entry holds for a decoder at zigzag index z iff
//                        z + adv_pre <= 63 (no symbol before the last one completes the block - what follows a
//                        completed block is a DC symbol of another table)
//   bits 18-22  tb1      |
//   bits 23-29  adv1     | the first symbol alone: what to take when the entry does not hold
// DC tables have the same format with one symbol per entry, index width kMultiBitsDc, and the code LENGTH in the
// adv_pre field (the DC difference must be extracted; z = 0 there, so the entry always holds).  0 = no symbol can be
// determined from the window (code longer than the window, no such code, DC size >= 16): single-symbol path.
#ifndef JPGPU_MULTI_BITS
#define JPGPU_MULTI_BITS 12
#endif
constexpr int kMultiBitsAc = JPGPU_MULTI_BITS;
constexpr int kMultiBitsDc = 9;
JPGPU_HD uint32_t multi_entry(uint32_t tb_all, uint32_t adv_all, uint32_t adv_pre, uint32_t tb1, uint32_t adv1) {
    return tb_all | (adv_all << 5) | (adv_pre << 12) | (tb1 << 18) | (adv1 << 23);
}

// Per-image plan, written by the host, read by every kernel.
struct ImgDev {
    uint32_t width, height;
    uint32_t raw_len;         // stuffed scan bytes
    uint32_t stream_cap_words;
    uint64_t raw_off;         // byte offset into the raw arena (16-byte aligned)
    uint64_t stream_off;      // word offset into the compacted stream arena (32-word aligned)
    uint64_t coef_off;        // int16 offset into the coefficient arena
    uint64_t rgb_off;         // byte offset into the RGB arena (256-byte aligned)
    uint32_t seg_off;         // offset into the segment table (entries: start bit of each restart interval)
    uint32_t nseg_cap;        // expected number of intervals (1 without DRI)
    uint32_t sub_off;         // offset into the subsequence-info array
    uint32_t nsub_cap;        // capacity in subsequences (from raw_len)
    uint32_t chunk_off;       // offset of this image's entries in the pre-pass chunk table
    uint32_t interval_mode;   // 1: restart intervals are short against a subsequence: decode threads start at interval
                              // boundaries, which are known states - no synchronisation pass for this image (DESIGN.md 4.2)
    uint32_t seq_first;       // index of this image's first sequence in the global sequence list
    uint32_t nseq;
    uint32_t mcux, mcuy;      // MCU grid (SPEC geometry)
    uint32_t units;           // MCUs to decode (decoder.rs:192 for REF, mcux*mcuy for SPEC)
    uint32_t restart_interval;
    uint32_t seg_units;       // restart_interval * blocks_per_mcu * 64 (coefficient positions per interval)
    uint32_t total_coefs;     // units * blocks_per_mcu * 64
    uint8_t ncomp, blocks_per_mcu, hmax, vmax;
    uint8_t h[4], v[4];
    uint8_t blk_comp[kMaxBlocksPerMcu];   // component of block c inside an MCU
    uint8_t blk_dc_slot[kMaxBlocksPerMcu];
    uint8_t blk_ac_slot[kMaxBlocksPerMcu];
    uint32_t blk_info[kMaxBlocksPerMcu];  // DC slot | AC slot << 8 | component << 16 (what the decoder loads per block)
    uint8_t nslots, kind, layout, pad0;   // kind: colour kernel variant (see ImgKind)
    uint32_t slot_lut[kMaxLutSlots];      // index into the global HuffLut array
    uint32_t qt_off[4];                   // per component: offset (in floats) of its 64 pre-scaled multipliers
    uint32_t tiles_x, tiles_y;            // colour-kernel tiles (128 px x 8*vmax rows)
    // gather path only (kind == kKindGeneric): REF placement / generic sampling
    uint64_t map_off;                     // u32 offset of this shape's placement map (ncomp planes of map_plane entries)
    uint64_t smp_off;                     // float offset of this image's per-block IDCT samples
    uint32_t map_plane;                   // entries per component plane (W*H rounded up to 4)
    uint32_t frame;                       // compose path: index + 1 of the FrameDev this image's samples feed (0: none)
    uint32_t out_pixels;                  // pixels of the output this image owns in the RGB arena (a frame's first scan: the frame's; further scans: 0)
    uint32_t pad2;
};

// ---- compose path: per-block IDCT samples (block_idct_kernel) -> pixels, plane by plane.  Serves what the fused
// kernels do not: libjpeg-style "fancy" (triangle filter) chroma up-sampling, and frames whose components arrive in
// separate non-interleaved scans (each scan is entropy-decoded as a one-component image of its own).
struct PlaneRef {          // where the samples of one component of a frame are
    uint64_t smp_off;      // float offset of the owning image's per-block samples ([block][row * 8 + col])
    uint32_t mcux, bpm;    // the owning image's MCUs per row and blocks per MCU
    uint32_t first;        // first block of this component inside an MCU
    uint32_t h, v;         // its blocks per MCU, horizontally / vertically
    uint32_t wc, hc;       // samples per line / lines of the component (T.81 A.1.1: ceil(X * H / Hmax), ceil(Y * V / Vmax))
    uint32_t fx, fy;       // up-sampling factors to the frame (Hmax / H, Vmax / V): 1 or 2
    float bias;            // added to every sample (chroma decoded as a one-component image carries a +128 it must lose)
    uint32_t pad;
};
struct FrameDev {
    uint32_t width, height, ncomp;
    uint32_t fancy;        // 0: box replication (the reference's fill_block_in_array, decoder.rs:347-379), 1: triangle filter
    uint64_t rgb_off;      // byte offset of the frame's output in the RGB arena (before the format's sample size)
    PlaneRef pl[3];
};
constexpr uint32_t kMapNone = 0xffffffffu;  // placement-map entry of a pixel no block was ever written to

enum ImgKind : uint8_t { kKindGray = 0, kKind444 = 1, kKind422 = 2, kKind420 = 3, kKind440 = 4, kKindGeneric = 5 };

// Written by the pre-pass for each image.
struct ImgDyn {
    uint32_t stream_bits;   // length of the compacted (unstuffed, marker-free) stream
    uint32_t nseg;          // restart intervals found (RST markers + 1)
    uint32_t status;        // kSt* bits
    uint32_t bits_consumed; // bit position after the last decoded MCU -> bytes_read
    // Without kStDone (data ended early): coefficient positions [0, coef_end) are what this decode produced; the blocks
    // from there on were never written and read as zeros (the arenas are reused wave after wave and never cleared, so
    // they hold an earlier image's coefficients): zero_tail_kernel fills them in after the write pass.
    uint32_t coef_end;
    uint32_t pad[3];
};
// Blocks of an image the IDCT stage may read from the coefficient arena; blocks at or past it are zeros.
JPGPU_HD uint32_t coef_block_limit(const ImgDyn& d) { return (d.status & kStDone) ? 0xffffffffu : d.coef_end >> 6; }

// Synchronisation record of one subsequence j (bits [j*S, (j+1)*S) of the compacted stream).
// A = state at the first symbol starting at or after j*S, reached from a cold start
// lookback_bits earlier; B = state at the first symbol starting at or after (j+1)*S.
// The chain is consistent where A(j) == B(j-1).
struct RepairJob {     // a broken link: decode subsequence `sub` again from (p, cz) = B of its predecessor
    uint32_t sub, p, cz;
};

// A subsequence is recorded in S/C segments of C bits (C = BatchDev::seg_bits): the state at
// the first symbol at or after each C-bit boundary plus what was counted inside the segment.
// A repair walker that reaches a boundary in the recorded state can stop there: from that
// point on the recorded decode was already the true one.
struct SegRec {
    uint32_t p;        // bit position at the end of the segment
    uint32_t cz;       // bits 0-5 z, 6-9 c at the end; bit 30: a restart interval began inside (n/dc absolute)
    int32_t n;         // coefficient positions advanced inside the segment (or absolute position at its end)
    int32_t dc[3];     // sum of DC differences per component inside the segment (or absolute predictors)
    uint32_t pad[2];
};

struct SubInfo {
    uint32_t pA, pB;   // bit positions
    uint32_t cz;       // bits 0-5 z(A), 6-9 c(A), 10-15 z(B), 16-19 c(B), 30 absolute (a restart
                       // interval began inside: n/dc below are absolute, not relative to A), 31 bad
    int32_t n;         // sync pass: coefficient positions advanced A -> B (or absolute position at B);
                       // after the scan: absolute coefficient position at A
    int32_t dc[3];     // same for the sum of DC differences / the DC predictors per component
    uint32_t pad;
};
constexpr uint32_t kCzMask = 0x3ffu;
constexpr uint32_t kCrossed = 1u << 30;

// ------------------------------------------------------------ zigzag mappings
// decoder.rs:404-407: ZIGZAG_INDICES[k] = natural (row-major v*8+u) index of zigzag position k.
#ifdef __CUDACC__
#define JPGPU_CONST_TABLE __device__ __constant__
#else
#define JPGPU_CONST_TABLE static const
#endif

static const uint8_t kZigzagNaturalHost[64] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// Coefficients live in HBM in "column-major natural" order: position u*8+v holds
// F[v][u] (u = horizontal frequency), so that the 16 bytes one lane loads are one
// column — the input of the vertical IDCT pass.  The mapping from zigzag index is
// folded into the entropy decoder's store address.
JPGPU_HD int zigzag_to_colmajor(int k, const uint8_t* zz_nat) {
    int nat = zz_nat[k];
    return ((nat & 7) << 3) | (nat >> 3);
}

// ------------------------------------------------------------------ bit reader
// The compacted stream is stored as 32-bit words holding 4 stream bytes each, first byte
// in the most significant position, so a word IS the next 32 bits.  Words are laid out
// LANE-INTERLEAVED in pieces of kPieceWords words (32 bytes = one memory sector): with
// W = S/32 words per subsequence, a group of 32 consecutive subsequences (one warp of decode
// threads) occupies 32*W words; word k of subsequence l sits at
//     (k / kPieceWords) * 32 * kPieceWords + l * kPieceWords + k % kPieceWords
// inside it.  A lane reads its own sector front to back (eight refills from one 32-byte
// sector, whatever the other lanes do), the 32 lanes of a warp at similar depths share
// 1 KiB row blocks, and the pre-pass writes whole sectors.
#ifndef JPGPU_PIECE_SHIFT
#define JPGPU_PIECE_SHIFT 3
#endif
constexpr uint32_t kPieceShift = JPGPU_PIECE_SHIFT;
constexpr uint32_t kPieceWords = 1u << kPieceShift;
JPGPU_HD uint32_t stream_phys(uint32_t i, uint32_t lw) {  // lw = log2(W)
    const uint32_t k = i & ((1u << lw) - 1u);
    return (i & ~((32u << lw) - 1u)) | ((k & ~(kPieceWords - 1u)) << 5) | (((i >> lw) & 31u) << kPieceShift) | (k & (kPieceWords - 1u));
}

struct BitReader {
    const uint32_t* w;
    uint32_t lw;     // log2(words per subsequence)
    uint32_t widx;   // next (linear) word to load
    uint32_t avail;  // valid bits at the top of buf
    uint64_t buf;

    JPGPU_HD uint32_t load(uint32_t i) const { return w[stream_phys(i, lw)]; }
    JPGPU_HD void seek(uint32_t p) {
        widx = p >> 5;
        const uint32_t off = p & 31;
        const uint64_t a = load(widx), b = load(widx + 1);
        buf = ((a << 32) | b) << off;
        avail = 64 - off;
        widx += 2;
    }
    JPGPU_HD uint32_t peek() const { return (uint32_t)(buf >> 32); }
    JPGPU_HD void skip(uint32_t n) { buf <<= n; avail -= n; }  // n <= 32
    JPGPU_HD void refill() {
        if (avail <= 32) {
            buf |= (uint64_t)load(widx++) << (32 - avail);
            avail += 32;
        }
    }
};

// huffman.rs:211-227 next_code for codes the LUT levels do not hold: canonical prefix decode
// (T.81 F.2.2.3). Returns a packed entry, 0 if no code matches.
JPGPU_HD uint32_t huff_slow(const HuffLut& t, uint32_t peek32) {
    const uint32_t code16 = peek32 >> 16;
#pragma unroll 1
    for (int l = 1; l <= 16; l++) {
        const int32_t code = (int32_t)(code16 >> (16 - l));
        if (code <= t.maxcode[l]) return make_entry(t.vals[(t.valoff[l] + code) & 255], (uint32_t)l, t.is_dc != 0);
    }
    return 0;
}

// huffman.rs:256-268 value_correction (T.81 F.2.2.1 EXTEND).  `top` = the bits following the
// code, left aligned; `v` = the first `size` of them.
JPGPU_HD int32_t extend(uint32_t v, uint32_t top, uint32_t size) {
    const uint32_t neg = (uint32_t)((int32_t)~top >> 31);   // all ones when the first value bit is 0
    return (int32_t)v - (int32_t)(neg & ((1u << size) - 1u));
}

// The reference's value_correction works in i16, so a DC difference of size category 16 is its 16 raw bits read as
// an i16, where T.81 EXTEND gives raw - 65535 (first bit 0) or raw (first bit 1).  What to add to extend() for such
// a symbol; `top` as there.  Only the canonical walk decodes DC category 16 (build_huff_lut, build_multi_lut), so
// the per-symbol paths never look at it.
JPGPU_HD int32_t dc16_correction(uint32_t top) { return (top >> 31) ? -65536 : 65535; }

// The reference keeps the DC predictor in f32 and stores it `as i16`, which saturates (decoder.rs:208-210); the
// predictor itself is not saturated.
JPGPU_HD int32_t sat_i16(int32_t v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); }

// ------------------------------------------------------------ decoder state
struct DecCtx {               // per-image constants of the entropy decoder
    const uint32_t* words;    // compacted stream of this image (lane-interleaved)
    uint32_t lw;              // log2(words per subsequence)
    const uint32_t* seg;      // seg[k] = first bit of restart interval k; seg[nseg] = stream_bits
    uint32_t nseg;
    uint32_t stream_bits;
    uint32_t seg_units;
    int32_t nblk;             // blocks per MCU
    const HuffLut* luts;      // slot array
    const uint32_t* blk_info; // per block of an MCU: DC slot | AC slot << 8 | component << 16
    const uint32_t* const* mluts;  // per slot: its multi-symbol table (synchronisation pass), or nullptr: symbol by symbol
};

struct DecState {
    BitReader br;
    uint32_t p;       // bit position of the next symbol
    int32_t g;        // coefficient position: (block index << 6) | zigzag index; relative or absolute
    int32_t c;        // block index within the MCU
    uint32_t seg;     // current restart interval
    uint32_t seg_end; // its end bit
    int32_t dc0, dc1, dc2;  // DC sums / predictors per component
    uint32_t flags;   // kCrossed | kSt* bits
    const HuffLut* tdc;     // tables and component of block c
    const HuffLut* tac;
    int32_t comp;
};

JPGPU_HD void load_block_tables(const DecCtx& cx, DecState& st) {
    const uint32_t info = cx.blk_info[st.c];
    st.tdc = cx.luts + (info & 255u);
    st.tac = cx.luts + ((info >> 8) & 255u);
    st.comp = (int32_t)(info >> 16);
}

// Largest k with seg[k] <= p.
JPGPU_HD uint32_t find_segment(const DecCtx& cx, uint32_t p) {
    uint32_t lo = 0, hi = cx.nseg;  // invariant: seg[lo] <= p < seg[hi] (seg[nseg] = stream_bits, p < stream_bits)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (cx.seg[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// Smallest k with seg[k] >= bit (k = nseg when there is none; seg[nseg] = stream_bits).
JPGPU_HD uint32_t first_interval_from(const uint32_t* seg, uint32_t nseg, uint32_t bit) {
    uint32_t lo = 0, hi = nseg;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (seg[mid] >= bit) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// Establish a decoder at bit p with block/zigzag state (c, z) and predictors.
// A decoder standing exactly on the first bit of a restart interval is in a
// known absolute state whatever it was told (predictors 0, MCU boundary).
JPGPU_HD void init_state(const DecCtx& cx, DecState& st, uint32_t p, int32_t g, int32_t c, int32_t d0, int32_t d1,
                         int32_t d2) {
    st.flags = 0;
    st.br.w = cx.words;
    st.br.lw = cx.lw;
    st.p = p;
    if (p >= cx.stream_bits) {  // nothing to decode
        st.seg = cx.nseg ? cx.nseg - 1 : 0;
        st.seg_end = cx.stream_bits;
        st.br.widx = (p >> 5) + 2; st.br.avail = 64 - (p & 31); st.br.buf = 0;
        st.g = g; st.c = c; st.dc0 = d0; st.dc1 = d1; st.dc2 = d2;
        load_block_tables(cx, st);
        return;
    }
    const uint32_t k = find_segment(cx, p);
    st.seg = k;
    st.seg_end = cx.seg[k + 1];
    st.br.seek(p);
    if (cx.seg[k] == p) {
        st.g = (int32_t)(k * cx.seg_units);
        st.c = 0;
        st.dc0 = st.dc1 = st.dc2 = 0;
        st.flags = kCrossed;
    } else {
        st.g = g; st.c = c; st.dc0 = d0; st.dc1 = d1; st.dc2 = d2;
    }
    load_block_tables(cx, st);
}

// Events decode_symbol reports to its caller.
enum : uint32_t {
    kEvBlock = 1u,   // the symbol completed a block (EOB, ZRL/run past the end, or coefficient 63)
    kEvCross = 2u,   // no symbol decoded: moved to the start of the next restart interval
    kEvEnd = 4u      // no symbol decoded: end of the entropy-coded data
};

// Position of coefficient `pos` (column-major, see zigzag_to_colmajor) inside a block buffer whose
// 16-byte pieces are XOR-swizzled by `swz` (0 for plain memory).
JPGPU_HD int buf_index(int pos, uint32_t swz) { return (int)((((uint32_t)pos >> 3) ^ swz) << 3) | (pos & 7); }

// Decode ONE symbol at st.p (huffman.rs:146-195 unrolled into single steps).
// WRITE = false: synchronisation pass, only state (and DC sums) are tracked.
// WRITE = true : when store_on, coefficients go to blk[buf_index(store_pos[k], swz)] (buffer pre-zeroed).
template <bool WRITE>
JPGPU_HD uint32_t decode_symbol(const DecCtx& cx, DecState& st, int16_t* blk, uint32_t swz, const uint8_t* store_pos,
                                bool store_on) {
    st.br.refill();
    if (st.p + 8 > st.seg_end) {  // fewer than 8 bits left in this restart interval (or already past it)
        bool cross = st.p >= st.seg_end;
        if (!cross) {
            const uint32_t rem = st.seg_end - st.p;  // 1..7 pad bits must all be 1 (T.81 F.1.2.3)
            cross = (st.br.peek() >> (32 - rem)) == ((1u << rem) - 1u);
        }
        if (cross) {
            st.p = st.seg_end;
            st.br.seek(st.p);
            if (st.seg + 1 >= cx.nseg) return kEvEnd;  // end of the entropy-coded data
            st.seg += 1;
            st.seg_end = cx.seg[st.seg + 1];
            st.g = (int32_t)(st.seg * cx.seg_units);
            st.c = 0;
            load_block_tables(cx, st);
            st.dc0 = st.dc1 = st.dc2 = 0;
            st.flags |= kCrossed;
            return kEvCross;
        }
    }
    const uint32_t peek = st.br.peek();
    const int32_t z = st.g & 63;
    const HuffLut* t = z ? st.tac : st.tdc;
    uint32_t e = t->fast[peek >> (32 - kLutBits)];
    if (e & kLinkBit) e = t->pool[(e & 511u) + ((peek << kLutBits) >> (32 - ((e >> 9) & 7u)))];
    int32_t fix = 0;
    if (e == 0) {
        e = huff_slow(*t, peek);
        if (e == 0) { st.flags |= kStBadCode; e = kBadEntry; }  // huffman.rs:156/162 panic
        else if ((e & 255u) - ((e >> 8) & 255u) == 16u) fix = dc16_correction(peek << ((e >> 8) & 255u));  // AC sizes are <= 15
    }
    const uint32_t tb = e & 255u, len = (e >> 8) & 255u;
    const int32_t adv = (int32_t)((e >> 16) & 255u);
    if (WRITE || z == 0) {
        const uint32_t size = tb - len;
        const uint32_t top = peek << len;
#ifdef __CUDA_ARCH__
        const uint32_t v = __funnelshift_l(top, 0u, size);
#else
        const uint32_t v = size ? top >> (32 - size) : 0u;
#endif
        const int32_t val = extend(v, top, size) + fix;
        if (z == 0) {  // DC difference -> predictor (decoder.rs:208-210)
            if (e & (1u << 24)) st.flags |= kStDcSize;
            int32_t pred;
            if (st.comp == 0) { st.dc0 += val; pred = st.dc0; } else if (st.comp == 1) { st.dc1 += val; pred = st.dc1; } else { st.dc2 += val; pred = st.dc2; }
            if (WRITE && store_on) blk[buf_index(store_pos[0], swz)] = (int16_t)sat_i16(pred);
        } else if (WRITE && store_on && val != 0) {  // huffman.rs:183-189: min(run, 64 - len - 1) zeros, then the value
            const int32_t pos = z + adv - 1 < 63 ? z + adv - 1 : 63;
            blk[buf_index(store_pos[pos], swz)] = (int16_t)val;
        }
    }
    st.br.skip(tb);
    st.p += tb;
    if (z + adv >= 64) {  // block complete
        st.g = (st.g | 63) + 1;
        st.c += 1;
        if (st.c == cx.nblk) st.c = 0;
        load_block_tables(cx, st);
        return kEvBlock;
    }
    st.g += adv;
    return 0u;
}

// Synchronisation pass, one lookup in the multi-symbol table of the current block's DC / AC slot (format above):
// every symbol whose code lies inside the window, as far as they stay inside the block.  The caller guarantees
// st.p + 32 <= the bit it decodes to and <= seg_end - 7 (an entry consumes at most kMultiBitsAc + 15 bits), so no
// symbol of the entry starts past either.  The kernels' form is fast_mstep() (jpgpu_kernels.cu).
JPGPU_HD void multi_symbol(const DecCtx& cx, DecState& st) {
    st.br.refill();
    const uint32_t peek = st.br.peek();
    const uint32_t z = (uint32_t)st.g & 63u;
    const bool is_dc = z == 0u;
    const uint32_t* tab = cx.mluts[(is_dc ? st.tdc : st.tac) - cx.luts];
    const uint32_t e = tab[peek >> (32 - (is_dc ? kMultiBitsDc : kMultiBitsAc))];
    if (e == 0u) { decode_symbol<false>(cx, st, nullptr, 0u, nullptr, false); return; }
    const uint32_t pre = (e >> 12) & 63u;
    const bool ok = z + pre <= 63u;
    const uint32_t tb = (ok ? e : e >> 18) & 31u;
    const uint32_t adv = (ok ? e >> 5 : e >> 23) & 127u;
    if (is_dc) {  // DC difference -> running sum (decoder.rs:208-210)
        const uint32_t len = pre, size = tb - len, top = peek << len;
        const uint32_t v = size ? top >> (32 - size) : 0u;
        const int32_t val = extend(v, top, size);
        if (st.comp == 0) st.dc0 += val; else if (st.comp == 1) st.dc1 += val; else st.dc2 += val;
    }
    st.br.skip(tb);
    st.p += tb;
    if (z + adv >= 64u) {  // block complete
        st.g = (st.g | 63) + 1;
        st.c += 1;
        if (st.c == cx.nblk) st.c = 0;
        load_block_tables(cx, st);
    } else {
        st.g += (int32_t)adv;
    }
}

JPGPU_HD uint32_t pack_cz(const DecState& st) { return (uint32_t)(st.g & 63) | ((uint32_t)st.c << 6); }

// Synchronisation decode of one segment: from the state in `st` to the first symbol at or after end_bit.
JPGPU_HD void sync_segment(const DecCtx& cx, DecState& st, uint32_t end_bit, SegRec& r) {
    const int32_t g_base = st.g;
    st.dc0 = st.dc1 = st.dc2 = 0;
    // A decoder standing on the first bit of a restart interval (it was put there, or its last step crossed into
    // it) is in an absolute state: the record must say so even if no crossing happens inside the segment.  (A
    // predecessor whose last symbol ended exactly on the interval's last bit stops there without having crossed.)
    if (st.p == cx.seg[st.seg] && st.p < cx.stream_bits) st.flags |= kCrossed; else st.flags &= ~kCrossed;
    if (end_bit > cx.stream_bits) end_bit = cx.stream_bits;
#pragma unroll 1
    while (st.p < end_bit) {
        // through the multi-symbol tables while no symbol of an entry can start at or past end_bit (or inside the last
        // bits of a restart interval): the state at end_bit stays that of the FIRST symbol at or after it
        if (cx.mluts && st.p + 32u <= end_bit && st.p + 39u <= st.seg_end) { multi_symbol(cx, st); continue; }
        if (decode_symbol<false>(cx, st, nullptr, 0u, nullptr, false) & kEvEnd) break;
    }
    r.p = st.p;
    r.cz = pack_cz(st) | (st.flags & kCrossed);
    r.n = (st.flags & kCrossed) ? st.g : st.g - g_base;
    r.dc[0] = st.dc0; r.dc[1] = st.dc1; r.dc[2] = st.dc2;
    r.pad[0] = r.pad[1] = 0;
}

// Coefficient positions saturate here.  The stream after an image's last MCU is still decoded by the
// synchronisation pass (nobody knows yet where the scan ends), and a crafted file can hold far more "blocks" than its
// header declares (1-bit EOB codes: one block per bit), so the running position over a whole stream does not fit
// 32 bits.  Advances are never negative, so a saturating sum stays associative; the planner keeps total_coefs below
// kPosSat, and one subsequence advances less than 2^31 - kPosSat (32768 bits x 64 positions), so a saturated position
// is "past the scan" for every consumer and never wraps.
constexpr int32_t kPosSat = 0x7f000000;
JPGPU_HD int32_t sat_pos(int64_t v) { return v > (int64_t)kPosSat ? kPosSat : (int32_t)v; }

// Accumulate segment / subsequence advances: a restart interval makes the values absolute.
// DC sums wrap modulo 2^32 (they are values, never addresses).
JPGPU_HD void fold_advance(int32_t acc[4], uint32_t& crossed, uint32_t cz, int32_t n, const int32_t dc[3]) {
    if (cz & kCrossed) { acc[0] = sat_pos(n); acc[1] = dc[0]; acc[2] = dc[1]; acc[3] = dc[2]; crossed = kCrossed; }
    else {
        acc[0] = sat_pos((int64_t)acc[0] + n);
        acc[1] = (int32_t)((uint32_t)acc[1] + (uint32_t)dc[0]);
        acc[2] = (int32_t)((uint32_t)acc[2] + (uint32_t)dc[1]);
        acc[3] = (int32_t)((uint32_t)acc[3] + (uint32_t)dc[2]);
    }
}

// Decode subsequence [own, own + S) from the state in `st` (standing at A; rec.pA / rec.cz(A) set by the
// caller), segment by segment.  compare = false: first decode, every segment is recorded.  compare = true:
// repair walk; stops at the first segment end where it meets the recorded state.  Fills the rest of rec.
JPGPU_HD void sync_subsequence(const DecCtx& cx, DecState& st, uint32_t own, uint32_t S, uint32_t C, SegRec* segs,
                               bool compare, SubInfo& rec) {
    const uint32_t nsegs = S / C;
#pragma unroll 1
    for (uint32_t k = 0; k < nsegs; k++) {
        SegRec r;
        sync_segment(cx, st, own + (k + 1) * C, r);
        const bool met = compare && segs[k].p == r.p && ((segs[k].cz ^ r.cz) & kCzMask) == 0u;
        segs[k] = r;
        if (met) break;
    }
    int32_t acc[4] = {0, 0, 0, 0};
    uint32_t crossed = 0;
    for (uint32_t k = 0; k < nsegs; k++) fold_advance(acc, crossed, segs[k].cz, segs[k].n, segs[k].dc);
    rec.pB = segs[nsegs - 1].p;
    rec.cz = (rec.cz & kCzMask) | ((segs[nsegs - 1].cz & kCzMask) << 10) | crossed;
    rec.n = acc[0]; rec.dc[0] = acc[1]; rec.dc[1] = acc[2]; rec.dc[2] = acc[3];
    rec.pad = 0;
}

// ------------------------------------------------------------------- IDCT
// Scaled 8-point inverse DCT (Arai-Agui-Nakajima factorisation, float): inputs are
// coefficients pre-multiplied by aan[k] (and by 1/8 over the two passes); 5 multiplies.
// Replaces the O(N^4) direct form of transform.rs:55-87; results differ from it only
// by float rounding (<= 1 LSB after truncation, measured in the parity tests).
JPGPU_HD void idct8(float& x0, float& x1, float& x2, float& x3, float& x4, float& x5, float& x6, float& x7) {
    // even part
    float t10 = x0 + x4, t11 = x0 - x4;
    float t13 = x2 + x6;
    float t12 = (x2 - x6) * 1.414213562f - t13;
    float e0 = t10 + t13, e3 = t10 - t13, e1 = t11 + t12, e2 = t11 - t12;
    // odd part
    float z13 = x5 + x3, z10 = x5 - x3, z11 = x1 + x7, z12 = x1 - x7;
    float o7 = z11 + z13;
    float t11o = (z11 - z13) * 1.414213562f;
    float z5 = (z10 + z12) * 1.847759065f;
    float t10o = z5 - z12 * 1.082392200f;
    float t12o = z5 - z10 * 2.613125930f;
    float o6 = t12o - o7;
    float o5 = t11o - o6;
    float o4 = t10o - o5;
    x0 = e0 + o7; x7 = e0 - o7;
    x1 = e1 + o6; x6 = e1 - o6;
    x2 = e2 + o5; x5 = e2 - o5;
    x3 = e3 + o4; x4 = e3 - o4;
}

static const double kAanScale[8] = {1.0, 1.387039845, 1.306562965, 1.175875602, 1.0, 0.785694958, 0.541196100, 0.275899379};

}  // namespace jpgpu
