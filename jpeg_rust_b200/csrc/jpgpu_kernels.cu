// jpgpu_kernels.cu — hand-written sm_100a kernels of the JPEG decode hot path.
//
//   prepass_*_kernel        mod.rs:371-385 (byte unstuffing) as a parallel stream
//                           compaction, plus RSTn detection (no reference counterpart:
//                           mod.rs:424-428 panics on DRI)
//   sync_kernel             |
//   verify_scan_kernel      |  huffman.rs:146-227 + decoder.rs:195-215 (serial MCU loop)
//   decode_write_kernel     |  as look-back synchronised subsequence decoding
//   idct_colour_kernel      decoder.rs:227-235 (dequant, de-zigzag), transform.rs:55-87
//                           (IDCT), decoder.rs:290-331 + 347-402 (placement, replication,
//                           YCbCr->RGB, +128, clamp, truncation)
// See DESIGN.md for the algorithm, the HBM layout and the roofline of each kernel.
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "jpgpu_kernels.cuh"

namespace jpgpu {

__constant__ uint8_t c_store_pos[64];  // zigzag index -> column-major position (see jpgpu_core.h)

cudaError_t init_constants() {
    uint8_t h[64];
    for (int k = 0; k < 64; k++) h[k] = (uint8_t)zigzag_to_colmajor(k, kZigzagNaturalHost);
    return cudaMemcpyToSymbol(c_store_pos, h, 64);
}

// =============================================================== stage 1a: pre-pass
// mod.rs:371-385 (drop the 00 after every FF) as a parallel stream compaction in three small kernels, so that
// no CTA walks an image serially: (1) every 4 KiB chunk counts the bytes it keeps and the RSTn markers it
// holds, (2) one CTA per image turns the counts into offsets and writes the per-image results, (3) every chunk
// compacts its bytes to its final position in the lane-interleaved word stream.
constexpr int kPreThreads = 256;
constexpr int kPreChunk = kPreThreads * 16;  // raw bytes per CTA

// Classification of the 16 raw bytes at offset o (thread-private): which are kept, which start an RSTn marker.
struct PreBytes {
    uint32_t w[4];
    uint32_t keep, rstm, next;
};
// Per-byte masks of a 32-bit word (4 raw bytes, little endian): 0x80 in every byte that fulfils the predicate.
__device__ __forceinline__ uint32_t bytes_eq(uint32_t w, uint32_t pattern) {   // byte == pattern byte
    const uint32_t x = w ^ pattern;                       // 0 where equal
    return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
}
// Gathers the 0x80 marks of four word masks into a 16-bit mask (bit k = byte k of the 16).
__device__ __forceinline__ uint32_t marks16(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    auto pack = [](uint32_t m) { return ((m >> 7) * 0x00204081u >> 21) & 0xfu; };  // bits 7,15,23,31 -> 0..3
    return pack(m0) | (pack(m1) << 4) | (pack(m2) << 8) | (pack(m3) << 12);
}
// What a thread reads from memory for its 16-byte vector at offset o: the vector (zeros past the end) and, for the
// first / last lane of a warp, the byte before / after the warp's 512 bytes (the other lanes get theirs by shuffle).
struct PreRaw { uint4 v; uint32_t edge; };
__device__ __forceinline__ PreRaw pre_load(const uint8_t* __restrict__ in, uint32_t n, uint32_t o) {
    PreRaw r;
    r.v = make_uint4(0u, 0u, 0u, 0u);
    r.edge = 0u;
    if (o < n) {
        const uint32_t lane = threadIdx.x & 31u;
        r.v = *reinterpret_cast<const uint4*>(in + o);  // raw arena is 16-byte padded
        if (lane == 0u && o > 0) r.edge = in[o - 1];
        if (lane == 31u && o + 16 < n) r.edge = in[o + 16];
    }
    return r;
}
// All 32 lanes of a warp come here together, with consecutive vectors.
__device__ __forceinline__ PreBytes pre_classify(const PreRaw& raw, uint32_t n, uint32_t o, bool dri) {
    PreBytes r;
    r.w[0] = raw.v.x; r.w[1] = raw.v.y; r.w[2] = raw.v.z; r.w[3] = raw.v.w;
    r.keep = r.rstm = 0u;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t prev = __shfl_up_sync(0xffffffffu, r.w[3], 1) >> 24;
    r.next = __shfl_down_sync(0xffffffffu, r.w[0], 1) & 0xffu;
    if (lane == 0u) prev = raw.edge;
    if (lane == 31u) r.next = raw.edge;
    if (o + 16 >= n) r.next = 0u;
    if (o >= n) { r.next = 0u; return r; }
    const uint32_t valid = n - o >= 16u ? 0xffffu : (1u << (n - o)) - 1u;
    // byte k is 0xff / 0x00 (bit k), four bytes per word at a time
    const uint32_t ff = marks16(bytes_eq(r.w[0], 0xffffffffu), bytes_eq(r.w[1], 0xffffffffu), bytes_eq(r.w[2], 0xffffffffu),
                                bytes_eq(r.w[3], 0xffffffffu));
    const uint32_t zz = marks16(bytes_eq(r.w[0], 0u), bytes_eq(r.w[1], 0u), bytes_eq(r.w[2], 0u), bytes_eq(r.w[3], 0u));
    const uint32_t prev_ff = ((ff << 1) | (prev == 0xffu ? 1u : 0u)) & 0xffffu;   // the byte before k is 0xff
    uint32_t drop = zz & prev_ff;                            // stuffed zero (mod.rs:378-382)
    if (dri) {  // restart-interval extension: RSTn markers and fill bytes leave the stream
        const uint32_t dx = marks16(bytes_eq(r.w[0] & 0xf8f8f8f8u, 0xd0d0d0d0u), bytes_eq(r.w[1] & 0xf8f8f8f8u, 0xd0d0d0d0u),
                                    bytes_eq(r.w[2] & 0xf8f8f8f8u, 0xd0d0d0d0u), bytes_eq(r.w[3] & 0xf8f8f8f8u, 0xd0d0d0d0u));
        const uint32_t has_next = n - o > 16u ? 0xffffu : valid >> 1;               // byte k+1 exists
        const uint32_t next_dx = ((dx >> 1) | ((r.next & 0xf8u) == 0xd0u ? 0x8000u : 0u)) & has_next;
        const uint32_t next_ff = ((ff >> 1) | (r.next == 0xffu ? 0x8000u : 0u)) & has_next;
        const uint32_t r1 = ff & next_dx;                    // FF of a marker
        const uint32_t r2 = dx & prev_ff;                    // its Dn byte
        const uint32_t fill = ff & next_ff;                  // FF FF: fill byte
        drop |= r1 | r2 | fill;
        r.rstm = r1 & valid;
    }
    r.keep = ~drop & valid;
    return r;
}

// CTA-wide exclusive scan of two counters (kept bytes, markers). Returns the exclusive prefixes and the totals.
__device__ __forceinline__ void pre_scan(uint32_t cnt, uint32_t nr, uint32_t (*s_wsum)[kPreThreads / 32], uint32_t& exc,
                                         uint32_t& exr, uint32_t& totc, uint32_t& totr) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t ic = cnt, ir = nr;  // warp-inclusive scans
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t tc = __shfl_up_sync(0xffffffffu, ic, d);
        const uint32_t tr = __shfl_up_sync(0xffffffffu, ir, d);
        if (lane >= (uint32_t)d) { ic += tc; ir += tr; }
    }
    if (lane == 31) { s_wsum[0][warp] = ic; s_wsum[1][warp] = ir; }
    __syncthreads();
    uint32_t wc = 0, wr = 0;
    totc = totr = 0;
#pragma unroll
    for (int i = 0; i < kPreThreads / 32; i++) {
        const uint32_t a = s_wsum[0][i], r = s_wsum[1][i];
        if ((uint32_t)i < warp) { wc += a; wr += r; }
        totc += a; totr += r;
    }
    exc = wc + ic - cnt;
    exr = wr + ir - nr;
}

// The same for one chunk, whose counters fit 16 bits each (<= 4096 kept bytes, <= 2048 markers): one packed scan.
__device__ __forceinline__ void pre_scan_chunk(uint32_t cnt, uint32_t nr, uint32_t* s_wsum, uint32_t& exc, uint32_t& exr,
                                               uint32_t& totc, uint32_t& totr) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, v = cnt | (nr << 16);
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += t;
    }
    if (lane == 31) s_wsum[warp] = inc;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < kPreThreads / 32; i++) {
        const uint32_t a = s_wsum[i];
        if ((uint32_t)i < warp) before += a;
        tot += a;
    }
    const uint32_t ex = before + inc - v;
    exc = ex & 0xffffu; exr = ex >> 16;
    totc = tot & 0xffffu; totr = tot >> 16;
}

// (1) grid (max chunks of any image, images): counts per chunk.
// A CTA takes kCountChunks consecutive chunks and reads them all before it looks at any (the kernel is a stream of
// short-lived threads: what bounds it is the number of loads in flight).
constexpr int kCountChunks = 4;
__global__ void __launch_bounds__(kPreThreads) prepass_count_kernel(BatchDev b) {
    __shared__ uint32_t s_wsum[kCountChunks][kPreThreads / 32];
    const ImgDev& im = b.imgs[b.img0 + blockIdx.y];
    const uint32_t n = im.raw_len, base = blockIdx.x * (kCountChunks * kPreChunk);
    if (base >= n) return;
    const uint8_t* in = b.raw + im.raw_off;
    const bool dri = im.restart_interval != 0;
    PreRaw raw[kCountChunks];
#pragma unroll
    for (int c = 0; c < kCountChunks; c++) raw[c] = pre_load(in, n, base + c * kPreChunk + threadIdx.x * 16);
#pragma unroll
    for (int c = 0; c < kCountChunks; c++) {
        const PreBytes pb = pre_classify(raw[c], n, base + c * kPreChunk + threadIdx.x * 16, dri);
        // only the chunk's totals are wanted here: kept bytes (<= 4096) and markers (<= 2048) as one packed sum
        const uint32_t wsum = __reduce_add_sync(0xffffffffu, __popc(pb.keep) | (__popc(pb.rstm) << 16));
        if ((threadIdx.x & 31u) == 0u) s_wsum[c][threadIdx.x >> 5] = wsum;
    }
    __syncthreads();
    if (threadIdx.x < kCountChunks && base + threadIdx.x * kPreChunk < n) {
        uint32_t t = 0;
#pragma unroll
        for (int i = 0; i < kPreThreads / 32; i++) t += s_wsum[threadIdx.x][i];
        b.chunk_counts[im.chunk_off + blockIdx.x * kCountChunks + threadIdx.x] = make_uint2(t & 0xffffu, t >> 16);
    }
}

// (2) one CTA per image: exclusive scan of its chunk counts; stream length, interval count, padding.
__global__ void __launch_bounds__(kPreThreads) prepass_scan_kernel(BatchDev b) {
    __shared__ uint32_t s_wsum[2][kPreThreads / 32];
    const uint32_t img = b.img0 + blockIdx.x;
    const ImgDev& im = b.imgs[img];
    const uint32_t nchunks = (im.raw_len + kPreChunk - 1) / kPreChunk;
    uint2* counts = b.chunk_counts + im.chunk_off;
    const uint32_t per = (nchunks + kPreThreads - 1) / kPreThreads;
    const uint32_t lo = threadIdx.x * per, hi = min(nchunks, lo + per);
    uint32_t c = 0, r = 0;
    for (uint32_t i = lo; i < hi; i++) { const uint2 v = counts[i]; c += v.x; r += v.y; }
    uint32_t exc, exr, totc, totr;
    pre_scan(c, r, s_wsum, exc, exr, totc, totr);
    for (uint32_t i = lo; i < hi; i++) {
        const uint2 v = counts[i];
        counts[i] = make_uint2(exc, exr);
        exc += v.x; exr += v.y;
    }
    if (threadIdx.x == 0) {
        uint32_t* out = b.stream + im.stream_off;
        uint32_t* seg = b.segtab + im.seg_off;
        const uint32_t wend = (totc + 3u) >> 2;
        for (int i = 0; i < kStreamPadWords; i++) out[stream_phys(wend + i, b.lw)] = 0u;
        const bool dri = im.restart_interval != 0;
        uint32_t nseg = totr + 1, st = 0;
        if (nseg != im.nseg_cap && dri) st |= kStRestart;
        if (nseg > im.nseg_cap) nseg = im.nseg_cap;
        seg[0] = 0u;
        seg[nseg] = totc * 8u;
        ImgDyn d;
        d.stream_bits = totc * 8u; d.nseg = nseg; d.status = st; d.bits_consumed = 0u;
        d.coef_end = 0u; d.pad[0] = d.pad[1] = d.pad[2] = 0u;
        b.dyn[img] = d;
    }
}

// (3) grid as (1): every chunk writes its kept bytes at its offset. A stream word IS the next 32 bits (first byte
// in the most significant position).  The bytes are staged in shared memory aligned to the 32-byte pieces of the
// stream layout (stream_phys), so a piece the chunk covers entirely leaves as two 16-byte stores (a whole sector);
// the first and last piece are shared with the neighbouring chunks and are written word by word, the words a
// chunk only partly covers byte by byte.
__global__ void __launch_bounds__(kPreThreads) prepass_write_kernel(BatchDev b) {
    __shared__ __align__(16) uint32_t s_stage[kPreChunk / 4 + 2 * kPieceWords];
    __shared__ uint32_t s_wsum[kPreThreads / 32];
    const uint32_t img = b.img0 + blockIdx.y;
    const ImgDev& im = b.imgs[img];
    const uint32_t n = im.raw_len, base = blockIdx.x * kPreChunk;
    if (base >= n) return;
    const uint32_t lw = b.lw, tid = threadIdx.x;
    const PreBytes pb = pre_classify(pre_load(b.raw + im.raw_off, n, base + tid * 16), n, base + tid * 16, im.restart_interval != 0);
    const uint2 start = b.chunk_counts[im.chunk_off + blockIdx.x];   // bytes / markers before this chunk
    uint32_t exc, exr, totc, totr;
    pre_scan_chunk(__popc(pb.keep), __popc(pb.rstm), s_wsum, exc, exr, totc, totr);
    uint8_t* stage_bytes = reinterpret_cast<uint8_t*>(s_stage);
    const uint32_t carry = start.x & (4u * kPieceWords - 1u);       // the chunk's first byte inside its first piece
    uint32_t pos = carry + exc;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        if (pb.keep & (1u << k)) {
            stage_bytes[pos ^ 3u] = (uint8_t)((pb.w[k >> 2] >> (8 * (k & 3))) & 0xffu);
            pos++;
        }
    }
    if (pb.rstm) {
        uint32_t* seg = b.segtab + im.seg_off;
        uint32_t r = start.y + exr;
#pragma unroll 1
        for (int k = 0; k < 16; k++) {
            if (!(pb.rstm & (1u << k))) continue;
            const uint32_t idx = start.x + exc + __popc(pb.keep & ((1u << k) - 1u));
            if (r + 1 < im.nseg_cap) seg[r + 1] = idx * 8u;
            const uint32_t mk = k < 15 ? ((pb.w[(k + 1) >> 2] >> (8 * ((k + 1) & 3))) & 0xffu) : pb.next;
            if ((mk & 7u) != (r & 7u)) atomicOr(&b.dyn[img].status, kStRestart);
            r++;
        }
    }
    __syncthreads();
    uint32_t* out = b.stream + im.stream_off;
    const uint32_t staged = carry + totc;                            // staged bytes, counted from the piece boundary
    const uint32_t w0 = (start.x >> 2) & ~(kPieceWords - 1u);        // stream word of s_stage[0]
    const uint32_t npieces = (staged + 4u * kPieceWords - 1u) / (4u * kPieceWords);
    for (uint32_t t = tid; t < npieces; t += kPreThreads) {
        const uint32_t b0 = t * 4u * kPieceWords;
        uint32_t* dst = out + stream_phys(w0 + t * kPieceWords, lw);
        if (b0 >= carry && b0 + 4u * kPieceWords <= staged) {
            const uint4* src = reinterpret_cast<const uint4*>(s_stage + t * kPieceWords);
#pragma unroll
            for (uint32_t i = 0; i < kPieceWords / 4u; i++) reinterpret_cast<uint4*>(dst)[i] = src[i];
        } else {
#pragma unroll 1
            for (uint32_t i = 0; i < kPieceWords; i++) {
                const uint32_t lo = max(b0 + 4u * i, carry), hi = min(b0 + 4u * i + 4u, staged);
                if (lo >= hi) continue;
                if (hi - lo == 4u) {
                    dst[i] = s_stage[t * kPieceWords + i];
                } else {
                    uint8_t* wb = reinterpret_cast<uint8_t*>(dst + i);
                    for (uint32_t q = lo; q < hi; q++) wb[3u - (q & 3u)] = stage_bytes[q ^ 3u];
                }
            }
        }
    }
}

// jpgpu_batch_set_device_scans(): the raw scan bytes of the images already lie in device memory, image i at
// base + offs[i] (any alignment).  One launch moves them into the batch's raw arena (16-byte aligned per image):
// every thread assembles one aligned 16-byte vector from five aligned source words.
__global__ void __launch_bounds__(kPreThreads) gather_scans_kernel(BatchDev b, const uint8_t* __restrict__ base, const uint64_t* __restrict__ offs) {
    const uint32_t img = b.img0 + blockIdx.y;
    const ImgDev& im = b.imgs[img];
    const uint32_t n = im.raw_len, o = blockIdx.x * kPreChunk + threadIdx.x * 16u;
    if (o >= n) return;
    const uint8_t* sp = base + offs[img] + o;
    uint4 v;
    if (o + 20u <= n) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(sp);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)(a & 3u) * 8u;
        const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2), w3 = __ldg(wp + 3), w4 = __ldg(wp + 4);
        v = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    } else {   // the last bytes of the image: nothing is read past them
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        for (uint32_t k = 0; k < 16u && o + k < n; k++) w[k >> 2] |= (uint32_t)sp[k] << (8u * (k & 3u));
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    *reinterpret_cast<uint4*>(const_cast<uint8_t*>(b.raw) + im.raw_off + o) = v;
}

// ========================================================= stage 1b-1d: entropy decode
constexpr int kJobsPerCta = kSeqThreads / 32;      // sync kernel
constexpr int kWriteThreads = 256;                 // write kernel: more warps share one copy of the Huffman tables
constexpr int kWriteJobsPerCta = kWriteThreads / 32;
template <int JOBS>
struct EntropySmemT {
    ImgDev img[JOBS];            // per warp job (verify_scan_kernel: [0] only)
    uint8_t store_pos[64];
    HuffLut lut[kMaxLutSlots];   // kernels with dynamic shared memory only carve max_slots of these
};
using EntropySmem = EntropySmemT<kJobsPerCta>;

// Cooperative load of the per-image decode context into shared memory: every group of `group` threads loads the
// image of its own job into sm.img[threadIdx.x / group] (kNoImage: nothing).
template <class SM>
__device__ __forceinline__ void load_entropy_img(const BatchDev& b, uint32_t img, SM& sm, int group) {
    const int slot = threadIdx.x / group, t = threadIdx.x % group;
    if (img != kNoImage) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&b.imgs[img]);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&sm.img[slot]);
        for (int i = t; i < (int)(sizeof(ImgDev) / 4); i += group) dst[i] = src[i];
    }
    if (threadIdx.x < 64) sm.store_pos[threadIdx.x] = c_store_pos[threadIdx.x];
    __syncthreads();
}
// The Huffman tables of the CTA: those of job 0 (all jobs of a CTA use the same set, see build_plan).
template <class SM>
__device__ __forceinline__ void load_entropy_luts(const BatchDev& b, SM& sm, int nthreads) {
    const int nslots = sm.img[0].nslots;
    constexpr int kLutVecs = sizeof(HuffLut) / 16;
    for (int s = 0; s < nslots; s++) {
        const uint4* ls = reinterpret_cast<const uint4*>(&b.luts[sm.img[0].slot_lut[s]]);
        uint4* ld = reinterpret_cast<uint4*>(&sm.lut[s]);
        for (int i = threadIdx.x; i < kLutVecs; i += nthreads) ld[i] = __ldg(ls + i);
    }
    __syncthreads();
}

// ------------------------------------------------------------------ fast decode step
// decode_symbol() of jpgpu_core.h (the form the CPU simulation and the repair kernels execute)
// restated for the two bulk kernels with everything on the per-symbol path branch-free or a
// short forward branch: predicated stream refill, Huffman tables / block buffers / DC
// predictors addressed as 32-bit shared-memory offsets, the DC predictor of the current
// component held in a register and swapped through shared memory at block boundaries.
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds32v(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t lds8(uint32_t a) { uint32_t v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint2 lds64(uint32_t a) { uint2 v; asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ void sts32v(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
// stores v saturated to [-32768, 32767]
__device__ __forceinline__ void sts16_sat_if(uint32_t a, int32_t v, bool p) {
    asm volatile("{\n .reg .pred q;\n .reg .b16 h;\n setp.ne.u32 q, %2, 0;\n cvt.sat.s16.s32 h, %1;\n @q st.shared.u16 [%0], h;\n}"
                 :: "r"(a), "r"(v), "r"((uint32_t)p) : "memory");
}
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

#define JPGPU_PIN32(x) asm volatile("" : "+r"(x))
#define JPGPU_PIN64(x) asm volatile("" : "+l"(x))

struct FastCtx {
    const uint32_t* words;   // lane-interleaved stream of the image (global)
    uint32_t lw, wmask5, gmask_inv;   // wmask5 = piece-row bits of a physical word offset
    const uint32_t* seg;
    uint32_t nseg, stream_bits, seg_units;
    uint32_t info_addr;      // shared: FastTables::info
    uint32_t dc_addr;        // shared: this lane's DC slots (component k at dc_addr + k * dc_stride)
    uint32_t dc_stride;      // 4 * threads of the CTA
    uint32_t sp_addr;        // shared: byte offset of zigzag position k inside an unswizzled block buffer
    const HuffLut* luts;     // generic pointer to the shared LUT slots (rare paths)
    uint32_t lut0_addr;
    uint32_t minfo_addr;     // shared: per job and block of an MCU {DC, AC} multi-symbol table addresses; 0 = kernel without them
};

struct FastState {
    uint32_t w0, w1, w2;     // stream words p>>5, +1, +2: the next 32 bits are funnelshift_l(w1, w0, p & 31)
    const uint32_t* kp;      // stream + the group and lane bits of w2's physical word offset (fast_kbase)
    uint32_t p;
    int32_t g;
    uint32_t info_ptr;       // shared address of the FastTables::info entry of the current block-in-MCU
    uint32_t lut_dc, lut_ac, dc_off;
    uint32_t m_dc, m_ac;     // multi-symbol tables of the current block (synchronisation pass, fast_mstep)
    int32_t dcur;
    uint32_t seg, seg_end, seg_lim, flags;   // seg_lim = seg_end - 7 (0 if shorter): at or past it a step must look at the interval end
    uint32_t wrap_lim, lim;                  // wrap_lim: see fast_advance(); lim = min(seg_lim, wrap_lim)
};

// per-CTA tables the fast path reads (filled once after the LUTs are loaded)
template <int THREADS>
struct FastTablesT {
    static constexpr int kThreads = THREADS;
    uint4 info[THREADS / 32][kMaxBlocksPerMcu];  // per job and block of an MCU: {dc lut addr | ac lut addr << 16, DC slot offset, address of the next entry, c}
    uint32_t dc[3 * THREADS];
    uint8_t sp[128];   // byte offset of zigzag position k in a block buffer; k >= 64 (a block's last symbol may step past 63) as 63
};
using FastTables = FastTablesT<kSeqThreads>;

// `group` threads fill the table of job threadIdx.x / group (its image must be loaded; kNoImage jobs skip).
template <class FT, class SM>
__device__ __forceinline__ void fast_tables_init(FT& ft, const SM& sm, bool valid, int group, int nthreads) {
    const int slot = threadIdx.x / group, t = threadIdx.x % group;
    const uint32_t lut0 = smem_addr(&sm.lut[0]), info0 = smem_addr(ft.info[slot]);
    if (valid) {
        const int nblk = sm.img[slot].blocks_per_mcu;
        for (int i = t; i < kMaxBlocksPerMcu; i += group) {
            const uint32_t info = sm.img[slot].blk_info[i < nblk ? i : 0];
            const uint32_t a_dc = lut0 + (info & 255u) * (uint32_t)sizeof(HuffLut), a_ac = lut0 + ((info >> 8) & 255u) * (uint32_t)sizeof(HuffLut);
            ft.info[slot][i] = make_uint4(a_dc | (a_ac << 16), (info >> 16) * 4u * FT::kThreads, info0 + (i + 1 < nblk ? i + 1 : 0) * 16u, (uint32_t)i);
        }
    }
    for (int i = threadIdx.x; i < 128; i += nthreads) {
        const uint32_t pos = sm.store_pos[i < 64 ? i : 63];
        ft.sp[i] = (uint8_t)(((pos >> 3) << 4) | ((pos & 7u) << 1));
    }
}

__device__ __forceinline__ const uint32_t* fast_word_ptr(const FastCtx& cx, uint32_t i) {
    const uint32_t phys = (i & cx.gmask_inv) | ((i << 5) & cx.wmask5) | (((i >> cx.lw) & 31u) << kPieceShift) | (i & (kPieceWords - 1u));
    return cx.words + phys;
}
// The part of a physical word offset that stays the same while the window moves inside one subsequence's words.
__device__ __forceinline__ const uint32_t* fast_kbase(const FastCtx& cx, uint32_t i) { return cx.words + ((i & cx.gmask_inv) | (((i >> cx.lw) & 31u) << kPieceShift)); }
__device__ __forceinline__ uint32_t fast_peek(const FastState& st) { return __funnelshift_l(st.w1, st.w0, st.p); }
__device__ __forceinline__ void fast_set_lim(FastState& st) { st.lim = min(st.seg_lim, st.wrap_lim); }
__device__ __forceinline__ void fast_seek(const FastCtx& cx, FastState& st, uint32_t p) {
    st.p = p;
    const uint32_t i = p >> 5;
    st.w0 = __ldg(fast_word_ptr(cx, i));
    st.w1 = __ldg(fast_word_ptr(cx, i + 1));
    st.w2 = __ldg(fast_word_ptr(cx, i + 2));
    st.kp = fast_kbase(cx, i + 2);
    st.wrap_lim = ((((i + 2u) >> cx.lw) + 1u) << (cx.lw + 5u)) - 64u;
    fast_set_lim(st);
}
// The bit position moved from st.p to pn (at most 32 bits on): when that crosses a word boundary the window
// slides by one word.  The word to fetch, (pn >> 5) + 2, is the next one of this lane's 32-byte piece or, after its
// last, the first of the lane's piece in the next row block: its physical offset (stream_phys) is st.kp plus row
// and in-piece bits that come straight from pn — except once per sub_bits, when the window's last word enters the
// next subsequence and st.kp no longer holds.  That slide (the one that takes the position to wrap_lim or past it)
// fetches the lane's own first word instead and is put right by fast_fix_wrap(), which the caller runs when it sees
// st.p >= st.wrap_lim — before the word can reach the decoder, two slides later.
__device__ __forceinline__ void fast_advance(const FastCtx& cx, FastState& st, uint32_t pn) {
    const bool cross = ((st.p ^ pn) & ~31u) != 0u;
    st.p = pn;
    st.w0 = cross ? st.w1 : st.w0;
    st.w1 = cross ? st.w2 : st.w1;
    const uint32_t t = pn + 64u;   // t >> 5 = index of the window's last word; wmask5 has no bit below 5
    const uint32_t rel = (t & cx.wmask5) | ((t >> 5) & (kPieceWords - 1u));
#ifndef JPGPU_PF_BYTES
#define JPGPU_PF_BYTES (128 << JPGPU_PIECE_SHIFT)   // the lane's piece in the next row block
#endif
    asm("{\n .reg .pred q;\n .reg .u64 a;\n setp.ne.u32 q, %3, 0;\n mad.wide.u32 a, %2, 4, %1;\n @q ld.global.nc.u32 %0, [a];\n"
#if JPGPU_PF_BYTES > 0
        " @q prefetch.global.L1 [a + %4];\n"
#endif
        "}" : "+r"(st.w2) : "l"(st.kp), "r"(rel), "r"((uint32_t)cross), "n"(JPGPU_PF_BYTES));
}
__device__ __forceinline__ void fast_fix_wrap(const FastCtx& cx, FastState& st) {   // st.p >= st.wrap_lim
    st.w2 = __ldg(fast_word_ptr(cx, (st.p >> 5) + 2u));
    st.kp = fast_kbase(cx, (st.p >> 5) + 2u);
    st.wrap_lim += 32u << cx.lw;
    fast_set_lim(st);
}
__device__ __forceinline__ uint32_t fast_c(const FastState& st) { return lds32(st.info_ptr + 12u); }
__device__ __forceinline__ void fast_load_multi(const FastCtx& cx, FastState& st) {
    if (cx.minfo_addr) {   // uniform: only the multi-symbol synchronisation kernel has these tables
        const uint2 m = lds64(cx.minfo_addr + ((st.info_ptr - cx.info_addr) >> 1));
        st.m_dc = m.x; st.m_ac = m.y;
    }
}
__device__ __forceinline__ void fast_load_block(const FastCtx& cx, FastState& st) {  // st.info_ptr changed: tables + DC slot
    fast_load_multi(cx, st);
    uint4 info;
    asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(info.x), "=r"(info.y), "=r"(info.z), "=r"(info.w) : "r"(st.info_ptr));
    sts32v(cx.dc_addr + st.dc_off, (uint32_t)st.dcur);
    st.dc_off = info.y;
    st.dcur = (int32_t)lds32v(cx.dc_addr + st.dc_off);
    st.lut_dc = info.x & 0xffffu;
    st.lut_ac = info.x >> 16;
}
__device__ __forceinline__ void fast_set_dc(const FastCtx& cx, FastState& st, int32_t d0, int32_t d1, int32_t d2) {
    sts32v(cx.dc_addr, (uint32_t)d0);
    sts32v(cx.dc_addr + cx.dc_stride, (uint32_t)d1);
    sts32v(cx.dc_addr + 2u * cx.dc_stride, (uint32_t)d2);
    st.dcur = (int32_t)lds32v(cx.dc_addr + st.dc_off);
}
__device__ __forceinline__ void fast_get_dc(const FastCtx& cx, const FastState& st, int32_t dc[3]) {
    sts32v(cx.dc_addr + st.dc_off, (uint32_t)st.dcur);
    dc[0] = (int32_t)lds32v(cx.dc_addr);
    dc[1] = (int32_t)lds32v(cx.dc_addr + cx.dc_stride);
    dc[2] = (int32_t)lds32v(cx.dc_addr + 2u * cx.dc_stride);
}
__device__ __forceinline__ void fast_set_segment(const FastCtx& cx, FastState& st, uint32_t k) {
    st.seg = k;
    st.seg_end = cx.seg[k + 1];
    st.seg_lim = st.seg_end >= 7u ? st.seg_end - 7u : 0u;
    fast_set_lim(st);
}

// init_state() of jpgpu_core.h
__device__ __forceinline__ void fast_init(const FastCtx& cx, FastState& st, uint32_t p, int32_t g, uint32_t c, int32_t d0,
                                          int32_t d1, int32_t d2) {
    st.flags = 0;
    st.dc_off = 0;
    st.dcur = 0;
    st.wrap_lim = 0xffffffffu;
    if (p >= cx.stream_bits) {
        st.seg = cx.nseg ? cx.nseg - 1 : 0;
        st.seg_end = cx.stream_bits;
        st.seg_lim = st.seg_end >= 7u ? st.seg_end - 7u : 0u;
        st.p = p; st.w0 = st.w1 = st.w2 = 0u;
        st.kp = fast_kbase(cx, (cx.stream_bits >> 5) + 2);   // whatever a step fetches from here on lies inside the image's stream
        st.lim = st.seg_lim;
        st.g = g;
    } else {
        uint32_t lo = 0, hi = cx.nseg;  // find_segment
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (cx.seg[mid] <= p) lo = mid; else hi = mid;
        }
        fast_set_segment(cx, st, lo);
        fast_seek(cx, st, p);
        if (cx.seg[lo] == p) {
            st.g = (int32_t)(lo * cx.seg_units);
            c = 0;
            d0 = d1 = d2 = 0;
            st.flags = kCrossed;
        } else {
            st.g = g;
        }
    }
    st.info_ptr = cx.info_addr + c * 16u;
    const uint4 info = *reinterpret_cast<const uint4*>(__cvta_shared_to_generic(st.info_ptr));
    st.dc_off = info.y;
    st.lut_dc = info.x & 0xffffu;
    st.lut_ac = info.x >> 16;
    st.m_dc = st.m_ac = 0u;
    fast_load_multi(cx, st);
    fast_set_dc(cx, st, d0, d1, d2);
}

// Rare part of a step: fewer than 8 bits left in the restart interval. Returns 0 when decoding simply goes on.
__device__ __forceinline__ uint32_t fast_interval_end(const FastCtx& cx, FastState& st) {
    bool cross = st.p >= st.seg_end;
    if (!cross) {
        const uint32_t rem = st.seg_end - st.p;  // 1..7 pad bits must all be 1 (T.81 F.1.2.3)
        cross = (fast_peek(st) >> (32u - rem)) == ((1u << rem) - 1u);
    }
    if (!cross) return 0u;
    fast_seek(cx, st, st.seg_end);
    if (st.seg + 1 >= cx.nseg) return kEvEnd;
    fast_set_segment(cx, st, st.seg + 1);
    st.g = (int32_t)(st.seg * cx.seg_units);
    st.info_ptr = cx.info_addr;
    fast_load_block(cx, st);
    fast_set_dc(cx, st, 0, 0, 0);
    st.flags |= kCrossed;
    return kEvCross;
}

// Second-level LUT or canonical walk (huffman.rs:211-227) for codes longer than kLutBits.
__device__ __forceinline__ uint32_t fast_long_code(const FastCtx& cx, FastState& st, uint32_t lut, uint32_t e, uint32_t hi) {
    if (e != 0u) e = lds32(lut + (uint32_t)(kLutSize * 4) + (((e & 511u) + ((hi << kLutBits) >> (32u - ((e >> 9) & 7u)))) << 2));
    if (e == 0u) {
        e = huff_slow(cx.luts[(lut - cx.lut0_addr) / (uint32_t)sizeof(HuffLut)], hi);
        if (e == 0u) { st.flags |= kStBadCode; e = kBadEntry; }
        st.flags |= (e >> 21) & kStDcSize;        // bit 24 -> kStDcSize (8): such DC symbols are only in the canonical tables
        // DC category 16, also only here: the caller adds fast_extend()'s T.81 value; make it the reference's i16 one
        const uint32_t len = (e >> 8) & 255u;
        if ((e & 255u) - len == 16u) st.dcur += dc16_correction(hi << len);   // AC sizes are <= 15
    }
    return e;
}

// Per-lane output state of the write kernel: NBUF block buffers (rows of 128 bytes in shared memory) used as a ring.
template <int NBUF>
struct WriteLane {
    static_assert(NBUF >= 1 && NBUF <= 2, "two completion slots");
    enum : uint32_t { kRun = 0, kBlocked = 1, kFinished = 2, kBlockEnd = 3 };
    uint32_t row_swz;          // shared address of the buffer being filled | its piece swizzle (bits 4-6): a coefficient at byte offset `off` goes to row_swz ^ off
    uint32_t rows_addr, row0;  // address of this lane's first row, its row number
    uint32_t cur, ndone;       // ring position, completed (unflushed) buffers
    uint32_t dest0, dest1;     // arena block index of each completed buffer, oldest first (0xffffffff = discard)
    uint32_t end_bit, end_bit_blk;   // where the lane stops: at a restart-interval / at a block boundary at or past this bit
    int32_t total;
    int32_t seg_limit;         // first coefficient position past the current restart interval (= total without DRI)
    uint32_t store_on;         // 0 while finishing a block that started in the previous subsequence, and past seg_limit
    uint32_t state;            // kRun / kBlocked (out of buffers until the next flush) / kFinished
    int16_t* coefs;            // coefficient arena of the image
    __device__ __forceinline__ void select(uint32_t c) {
        cur = c;
        row_swz = (rows_addr + c * 128u) | (((row0 + c) & 7u) << 4);
        JPGPU_PIN32(row_swz);   // one register, not recomputed from threadIdx in every step
    }
    // the buffer being filled is complete (block index d) or to be discarded; z == 0 now
    __device__ __forceinline__ void close_block(uint32_t d, uint32_t p, int32_t g) {
        if (store_on) {
            if (NBUF == 1 || ndone == 0u) dest0 = d; else dest1 = d;
            ndone++;
            if (NBUF > 1) select(cur + 1 == (uint32_t)NBUF ? 0u : cur + 1);
        }
        store_on = g < seg_limit ? 1u : 0u;   // a damaged interval holding more MCUs than it should is decoded, not stored
        // finished: block boundary past the subsequence / scan; blocked: no free buffer
        state = (p >= end_bit_blk || g >= total) ? (uint32_t)kFinished : (ndone == (uint32_t)NBUF ? (uint32_t)kBlocked : (uint32_t)kRun);
    }
    // Rare: the decoder moved to the next restart interval (kEvCross) or reached the end of the data (kEvEnd);
    // g_before = coefficient position before the move, st.g = first position of the new interval.
    // A valid stream changes interval exactly where the previous one is complete.  A damaged one may come short
    // (the missing blocks, a half-written one included, become zeros) or long (the excess was decoded without
    // being stored); both are reported (kStRestart).
    template <class CX, class ST>
    __device__ __forceinline__ void on_interval(uint32_t ev, int32_t g_before, const CX& cx, ST& st) {
        if (ev & kEvEnd) { state = kFinished; return; }
        const int32_t old_limit = seg_limit, gap_from = g_before & ~63;
        seg_limit = min(total, st.g + (int32_t)cx.seg_units);
        if (g_before != old_limit) st.flags |= kStRestart;
        if ((g_before & 63) != 0 && store_on) close_block(0xffffffffu, st.p, st.g);
        for (int32_t g = gap_from; g < old_limit && g < st.g; g += 64) {
            uint4* dst = reinterpret_cast<uint4*>(coefs + (size_t)g);
#pragma unroll
            for (int i = 0; i < 8; i++) dst[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        store_on = 1u;
        if (st.p >= end_bit || st.g >= total) state = kFinished;
        else if (state != kBlocked) state = kRun;
    }
};
struct NoLane { enum : uint32_t { kBlockEnd = 3 }; uint32_t state; };

// base + 4 * i as one multiply-add (the compiler's own shift, mask and add are three instructions on the busier pipe)
__device__ __forceinline__ uint32_t fast_index4(uint32_t base, uint32_t i) {
    uint32_t a;
    asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(a) : "r"(i), "r"(base));
    return a;
}
// EXTEND (huffman.rs:256-268) of the `size` (0..16) bits at the top of `top`: first bit 1 -> the bits v as they are,
// 0 -> v - (2^size - 1).  With neg = all ones in the second case, (neg << size | v) is v - 2^size; size 0 gives 0.
__device__ __forceinline__ int32_t fast_extend(uint32_t top, uint32_t size) {
    const uint32_t neg = (uint32_t)((int32_t)~top >> 31);
    return (int32_t)(__funnelshift_l(top, neg, size) - neg);
}

// CHECK = false: the caller guarantees st.p < st.lim (no look at the interval end, no window wrap pending).
template <bool WRITE, bool CHECK, typename LANE>
__device__ __forceinline__ uint32_t fast_step(const FastCtx& cx, FastState& st, LANE& wl) {
    if (CHECK && st.p >= st.lim) {
        if (st.p >= st.wrap_lim) fast_fix_wrap(cx, st);
        if (st.p >= st.seg_lim) {
            const int32_t g_before = st.g;
            const uint32_t ev = fast_interval_end(cx, st);
            if (ev) {
                if constexpr (WRITE) wl.on_interval(ev, g_before, cx, st);
                return ev;
            }
        }
    }
    const uint32_t hi = fast_peek(st);            // the next 32 bits
    const uint32_t z = (uint32_t)st.g & 63u;
    const uint32_t lut = z ? st.lut_ac : st.lut_dc;
    uint32_t e = lds32(fast_index4(lut, hi >> (32 - kLutBits)));
    if ((int32_t)e <= 0) e = fast_long_code(cx, st, lut, e, hi);
    const uint32_t tb = e & 255u, len = __byte_perm(e, 0u, 0x4441), adv = __byte_perm(e, 0u, 0x4442);
    const uint32_t size = tb - len;
    const uint32_t top = hi << len;               // len <= 16
    const int32_t val = fast_extend(top, size);
    const bool is_dc = z == 0u;
    // decoder.rs:208-210: st.dcur += is_dc ? val : 0, as one predicated add
    asm("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q add.s32 %0, %0, %1;\n}" : "+r"(st.dcur) : "r"(val), "r"((uint32_t)is_dc));
    const uint32_t nz = z + adv;
    if constexpr (WRITE) {
        // huffman.rs:183-189.  Symbols without a value (EOB, ZRL) store a zero at a position the block has not reached.
        // A DC predictor past the int16 range is stored saturated (sat_i16); AC values (size <= 15) are unchanged by it.
        const uint32_t off = lds8(cx.sp_addr + nz - 1u);   // nz - 1 <= 126: FastTablesT::sp
        sts16_sat_if(wl.row_swz ^ off, is_dc ? st.dcur : val, wl.store_on != 0u);
    }
    fast_advance(cx, st, st.p + tb);
    if constexpr (WRITE) {
        // Block complete: the lane has no free buffer before the next flush anyway, so everything a block end takes
        // (next block's tables and predictor, buffer bookkeeping) waits for the phase boundary, where all lanes that
        // completed a block do it together (fast_block_end) instead of one or two at a time in every step.
        st.g += (int32_t)adv;                        // z + adv >= 64 carries into the block index
        wl.state = nz >= 64u ? (uint32_t)LANE::kBlockEnd : wl.state;
        return 0u;
    } else {
        if (nz >= 64u) {  // block complete
            st.g = (st.g | 63) + 1;
            st.info_ptr = lds32(st.info_ptr + 8u);
            fast_load_block(cx, st);
            return kEvBlock;
        }
        st.g += (int32_t)adv;
        return 0u;
    }
}
// Write pass, at a phase boundary: what fast_step() left undone for a lane in state kBlockEnd.
template <typename LANE>
__device__ __forceinline__ void fast_block_end(const FastCtx& cx, FastState& st, LANE& wl) {
    st.g &= ~63;
    st.info_ptr = lds32(st.info_ptr + 8u);
    fast_load_block(cx, st);
    wl.close_block((uint32_t)(st.g >> 6) - 1u, st.p, st.g);
}

// Synchronisation pass: one lookup in the multi-symbol tables (jpgpu_core.h) = every symbol whose code lies in the next
// kMultiBitsAc bits, as far as they stay inside the current block.  The caller guarantees that all of them start before
// st.lim and before the bit it decodes to (st.p + 32 <= both: an entry consumes at most 26 bits).
__device__ __forceinline__ void fast_mstep(const FastCtx& cx, FastState& st) {
    const uint32_t hi = fast_peek(st);
    const uint32_t z = (uint32_t)st.g & 63u;
    const bool is_dc = z == 0u;
    const uint32_t e = lds32(fast_index4(is_dc ? st.m_dc : st.m_ac, hi >> (is_dc ? 32 - kMultiBitsDc : 32 - kMultiBitsAc)));
    if (e == 0u) {   // code longer than the window, no such code, oversized DC symbol: the single-symbol step knows
        NoLane nl;
        fast_step<false, false>(cx, st, nl);
        return;
    }
    const uint32_t pre = (e >> 12) & 63u;                  // AC: advance before the entry's last symbol; DC: code length
    const bool ok = z + pre <= 63u;                        // no symbol before the last completes the block
    const uint32_t tb = (ok ? e : e >> 18) & 31u;
    const uint32_t adv = (ok ? e >> 5 : e >> 23) & 127u;
    // DC difference (decoder.rs:208-210): EXTEND of the tb - len bits after the code, as in fast_step
    const uint32_t len = is_dc ? pre : 0u;
    const uint32_t top = hi << len;
    const int32_t val = fast_extend(top, tb - len);
    st.dcur += is_dc ? val : 0;
    fast_advance(cx, st, st.p + tb);
    if (z + adv >= 64u) {  // block complete
        st.g = (st.g | 63) + 1;
        st.info_ptr = lds32(st.info_ptr + 8u);
        fast_load_block(cx, st);
    } else {
        st.g += (int32_t)adv;
    }
}

// Decode every symbol that starts before end_bit (sync pass form: the interval-end test is hoisted out of the loop).
// MULTI: through the multi-symbol tables while that cannot carry past end_bit or st.lim; the last 32 bits before either
// go symbol by symbol, so the state at end_bit is that of the FIRST symbol at or after it however the entries fell -
// what the chain verification and the repair walks (single-symbol) compare.
template <bool MULTI>
__device__ __forceinline__ void fast_run_to(const FastCtx& cx, FastState& st, uint32_t end_bit) {
    NoLane nl;
#pragma unroll 1
    while (true) {
        if (st.p >= st.wrap_lim) fast_fix_wrap(cx, st);
        const uint32_t lim = min(end_bit, st.lim);
        if constexpr (MULTI) {
            if (lim >= 32u) {
                const uint32_t mlim = lim - 32u;
#pragma unroll 1
                while (st.p <= mlim) fast_mstep(cx, st);
            }
            if (st.p >= st.wrap_lim) continue;
        }
#pragma unroll 1
        while (st.p < lim) fast_step<false, false>(cx, st, nl);
        if (st.p >= st.wrap_lim) continue;
        if (st.p >= end_bit) return;
        const uint32_t ev = fast_interval_end(cx, st);
        if (ev & kEvEnd) return;
        if (ev == 0u) fast_step<false, false>(cx, st, nl);
    }
}

template <class SM, class FT>
__device__ __forceinline__ FastCtx make_fast_ctx(const BatchDev& b, const SM& sm, int slot, const ImgDyn& d, const FT& ft) {
    const ImgDev& im = sm.img[slot];
    FastCtx cx;
    cx.words = b.stream + im.stream_off;
    cx.lw = b.lw;
    cx.wmask5 = (((1u << b.lw) - 1u) & ~(kPieceWords - 1u)) << 5;
    cx.gmask_inv = ~((32u << b.lw) - 1u);
    
    cx.seg = b.segtab + im.seg_off;
    cx.nseg = d.nseg;
    cx.stream_bits = d.stream_bits;
    cx.seg_units = im.seg_units;
    cx.info_addr = smem_addr(ft.info[slot]);
    cx.dc_addr = smem_addr(ft.dc) + threadIdx.x * 4u;
    cx.dc_stride = 4u * FT::kThreads;
    cx.sp_addr = smem_addr(ft.sp);
    cx.luts = sm.lut;
    cx.lut0_addr = smem_addr(&sm.lut[0]);
    cx.minfo_addr = 0u;
    // keep the per-symbol operands in registers instead of re-deriving them from the parameter bank every step
    JPGPU_PIN64(cx.words);
    JPGPU_PIN32(cx.wmask5);
    JPGPU_PIN32(cx.dc_addr); JPGPU_PIN32(cx.sp_addr);
    // The shared-memory reads of the fast path are plain (non-volatile) asm: nothing but their address operands
    // orders them.  Making the table addresses opaque here - after the tables were written - keeps the compiler
    // from moving such a read above the code that fills the table (it did, when a loop was put around this).
    JPGPU_PIN32(cx.info_addr); JPGPU_PIN32(cx.lut0_addr);
    return cx;
}

// sync_segment() / sync_subsequence() of jpgpu_core.h on the fast step.
template <bool MULTI>
__device__ __forceinline__ void fast_sync_segment(const FastCtx& cx, FastState& st, uint32_t end_bit, SegRec& r) {
    const int32_t g_base = st.g;
    fast_set_dc(cx, st, 0, 0, 0);
    // standing on the first bit of a restart interval = absolute state, crossing inside the segment or not (see
    // sync_segment() in jpgpu_core.h)
    if (st.p == cx.seg[st.seg] && st.p < cx.stream_bits) st.flags |= kCrossed; else st.flags &= ~kCrossed;
    fast_run_to<MULTI>(cx, st, min(end_bit, cx.stream_bits));
    r.p = st.p;
    r.cz = ((uint32_t)st.g & 63u) | (fast_c(st) << 6) | (st.flags & kCrossed);
    r.n = (st.flags & kCrossed) ? st.g : st.g - g_base;
    fast_get_dc(cx, st, r.dc);
    r.pad[0] = r.pad[1] = 0;
}
__device__ __forceinline__ void store_segrec(SegRec* dst, const SegRec& r) {
    uint4* d = reinterpret_cast<uint4*>(dst);
    d[0] = make_uint4(r.p, r.cz, (uint32_t)r.n, (uint32_t)r.dc[0]);
    d[1] = make_uint4((uint32_t)r.dc[1], (uint32_t)r.dc[2], 0u, 0u);
}
template <bool MULTI>
__device__ __forceinline__ void fast_sync_subsequence(const FastCtx& cx, FastState& st, uint32_t own, uint32_t S, uint32_t C,
                                                      SegRec* segs, bool compare, SubInfo& rec) {
    const uint32_t nsegs = S / C;
    int32_t acc[4] = {0, 0, 0, 0};
    uint32_t crossed = 0, k = 0, last_p = st.p, last_cz = 0;
#pragma unroll 1
    for (; k < nsegs; k++) {
        SegRec r;
        fast_sync_segment<MULTI>(cx, st, own + (k + 1) * C, r);
        bool met = false;
        if (compare) {
            const uint2 old = *reinterpret_cast<const uint2*>(segs + k);
            met = old.x == r.p && ((old.y ^ r.cz) & kCzMask) == 0u;
        }
        store_segrec(segs + k, r);
        fold_advance(acc, crossed, r.cz, r.n, r.dc);
        last_p = r.p; last_cz = r.cz;
        if (met) { k++; break; }
    }
#pragma unroll 1
    for (; k < nsegs; k++) {  // met the recorded decode: the remaining segments stand as they are
        const SegRec r = segs[k];
        fold_advance(acc, crossed, r.cz, r.n, r.dc);
        last_p = r.p; last_cz = r.cz;
    }
    rec.pB = last_p;
    rec.cz = (rec.cz & kCzMask) | ((last_cz & kCzMask) << 10) | crossed;
    rec.n = acc[0]; rec.dc[0] = acc[1]; rec.dc[1] = acc[2]; rec.dc[2] = acc[3];
    rec.pad = 0;
}

// One thread per subsequence j.  It starts cold (block 0 of an MCU, zigzag 0) lookback_bits
// before j*S; by the time it reaches j*S it has, with high probability, fallen into step with
// the true decode (self-synchronisation of Huffman streams).  It records the state there (A),
// decodes its own S bits and records the state at the end (B) with the advance in coefficient
// positions and the DC sums in between, segment by segment.  Whether A was right is checked
// afterwards against the predecessor's B (verify_scan_kernel); thread 0 and threads that
// passed a restart marker are right by construction.  All threads do the same amount of
// work: no rounds, no barriers.
__global__ void __launch_bounds__(kSeqThreads) sync_kernel(BatchDev b) {
    __shared__ EntropySmem sm;
    __shared__ FastTables ft;
    const int warp = threadIdx.x >> 5;
    if (b.seqs[b.job0 + blockIdx.x * kJobsPerCta].img == kNoImage) return;   // a CTA of padding jobs only
    const SeqDesc sd = b.seqs[b.job0 + blockIdx.x * kJobsPerCta + warp];
    const uint32_t S = b.sub_bits;
    load_entropy_img(b, sd.img, sm, 32);
    load_entropy_luts(b, sm, kSeqThreads);
    fast_tables_init(ft, sm, sd.img != kNoImage, 32, kSeqThreads);
    __syncthreads();
    if (sd.img == kNoImage) return;
    const ImgDev& img = sm.img[warp];
    if (img.interval_mode) return;   // its decode threads start at restart-interval boundaries: nothing to synchronise
    const ImgDyn dyn = b.dyn[sd.img];
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    const FastCtx cx = make_fast_ctx(b, sm, warp, dyn, ft);
    const uint32_t j = sd.first_sub + (threadIdx.x & 31u);
    if (j >= nsub) return;

    const uint32_t own = j * S, p0 = own > b.lookback_bits ? own - b.lookback_bits : 0u;
    FastState st;
    fast_init(cx, st, p0, 0, 0u, 0, 0, 0);
    fast_run_to<false>(cx, st, own);
    SubInfo rec;
    rec.pA = st.p;
    rec.cz = ((uint32_t)st.g & 63u) | (fast_c(st) << 6);
    fast_sync_subsequence<false>(cx, st, own, S, b.seg_bits, b.segs + (size_t)(img.sub_off + j) * (S / b.seg_bits), false, rec);
    b.subs[img.sub_off + j] = rec;
}

// Multi-symbol tables of the CTA's slots (those of sm.img[0], as the Huffman tables) into shared memory, and, for the
// warp job in `slot` (its image in sm.img[slot]), which of them each block of an MCU uses: minfo[slot * 12 + block] =
// {DC table address, AC table address}.  The Huffman tables must be loaded (is_dc is read from them).
template <class SM>
__device__ __forceinline__ void load_multi_tables(const BatchDev& b, const SM& sm, uint32_t* mlut, uint2* minfo, int slot, bool valid, int nthreads) {
    const int nslots = sm.img[0].nslots;
    uint32_t moff[kMaxLutSlots], acc = 0;
#pragma unroll
    for (int s2 = 0; s2 < kMaxLutSlots; s2++) {
        moff[s2] = acc;
        if (s2 < nslots) acc += 1u << (sm.lut[s2].is_dc ? kMultiBitsDc : kMultiBitsAc);
    }
    for (int s2 = 0; s2 < nslots; s2++) {
        const uint4* src = reinterpret_cast<const uint4*>(b.mlut + b.mlut_off[sm.img[0].slot_lut[s2]]);
        uint4* dst = reinterpret_cast<uint4*>(mlut + moff[s2]);
        const int nvec = (1 << (sm.lut[s2].is_dc ? kMultiBitsDc : kMultiBitsAc)) / 4;
        for (int i = threadIdx.x; i < nvec; i += nthreads) dst[i] = __ldg(src + i);
    }
    const int t = threadIdx.x & 31;
    if (valid && (int)(threadIdx.x >> 5) == slot && t < kMaxBlocksPerMcu) {
        const int nblk = sm.img[slot].blocks_per_mcu;
        const uint32_t info = sm.img[slot].blk_info[t < nblk ? t : 0];
        const uint32_t base = smem_addr(mlut);
        uint32_t a_dc = base, a_ac = base;
#pragma unroll
        for (int s2 = 0; s2 < kMaxLutSlots; s2++) {
            if ((info & 255u) == (uint32_t)s2) a_dc = base + moff[s2] * 4u;
            if (((info >> 8) & 255u) == (uint32_t)s2) a_ac = base + moff[s2] * 4u;
        }
        minfo[slot * kMaxBlocksPerMcu + t] = make_uint2(a_dc, a_ac);
    }
}

// The same pass through the multi-symbol tables (jpgpu_core.h): 256-thread CTAs (eight warp jobs share one copy of the
// tables), dynamic shared memory = Huffman tables of the slots in use + fast-path tables + multi-symbol tables.
#ifndef JPGPU_SYNC_THREADS
#define JPGPU_SYNC_THREADS 256
#endif
constexpr int kSyncThreads = JPGPU_SYNC_THREADS;
constexpr int kSyncJobs = kSyncThreads / 32;
struct SyncLayout {
    uint32_t ft_off, minfo_off, mlut_off, total;
};
__host__ __device__ inline SyncLayout sync_layout(uint32_t max_slots, uint32_t max_mlut_words) {
    SyncLayout l;
    const uint32_t lut_bytes = (uint32_t)(sizeof(EntropySmemT<kSyncJobs>) - (kMaxLutSlots - max_slots) * sizeof(HuffLut));
    l.ft_off = (lut_bytes + 15u) & ~15u;
    l.minfo_off = (l.ft_off + (uint32_t)sizeof(FastTablesT<kSyncThreads>) + 15u) & ~15u;
    l.mlut_off = l.minfo_off + kSyncJobs * kMaxBlocksPerMcu * 8u;
    l.total = l.mlut_off + max_mlut_words * 4u;
    return l;
}
__global__ void __launch_bounds__(kSyncThreads) sync_multi_kernel(BatchDev b) {
    extern __shared__ __align__(128) uint8_t dyn_smem[];
    using Smem = EntropySmemT<kSyncJobs>;
    using Tables = FastTablesT<kSyncThreads>;
    Smem& sm = *reinterpret_cast<Smem*>(dyn_smem);
    const SyncLayout lay = sync_layout(b.max_slots, b.max_mlut_words);
    Tables& ft = *reinterpret_cast<Tables*>(dyn_smem + lay.ft_off);
    uint2* const minfo = reinterpret_cast<uint2*>(dyn_smem + lay.minfo_off);
    uint32_t* const mlut = reinterpret_cast<uint32_t*>(dyn_smem + lay.mlut_off);
    const int warp = threadIdx.x >> 5;
    if (b.seqs[b.job0 + blockIdx.x * kSyncJobs].img == kNoImage) return;   // a CTA of padding jobs only
    const uint32_t job = blockIdx.x * kSyncJobs + warp;
    const SeqDesc sd = job < b.n_seqs ? b.seqs[b.job0 + job] : SeqDesc{kNoImage, 0u};
    const uint32_t S = b.sub_bits;
    load_entropy_img(b, sd.img, sm, 32);
    load_entropy_luts(b, sm, kSyncThreads);
    fast_tables_init(ft, sm, sd.img != kNoImage, 32, kSyncThreads);
    load_multi_tables(b, sm, mlut, minfo, warp, sd.img != kNoImage, kSyncThreads);
    __syncthreads();
    if (sd.img == kNoImage) return;
    const ImgDev& img = sm.img[warp];
    if (img.interval_mode) return;   // its decode threads start at restart-interval boundaries: nothing to synchronise
    const ImgDyn dyn = b.dyn[sd.img];
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    FastCtx cx = make_fast_ctx(b, sm, warp, dyn, ft);
    cx.minfo_addr = smem_addr(minfo + warp * kMaxBlocksPerMcu);
    JPGPU_PIN32(cx.minfo_addr);
    const uint32_t j = sd.first_sub + (threadIdx.x & 31u);
    if (j >= nsub) return;

    const uint32_t own = j * S, p0 = own > b.lookback_bits ? own - b.lookback_bits : 0u;
    FastState st;
    fast_init(cx, st, p0, 0, 0u, 0, 0, 0);
    fast_run_to<true>(cx, st, own);
    SubInfo rec;
    rec.pA = st.p;
    rec.cz = ((uint32_t)st.g & 63u) | (fast_c(st) << 6);
    fast_sync_subsequence<true>(cx, st, own, S, b.seg_bits, b.segs + (size_t)(img.sub_off + j) * (S / b.seg_bits), false, rec);
    b.subs[img.sub_off + j] = rec;
}

constexpr int kInterThreads = kSeqThreads;
constexpr int kRepairJobs = 2 * kInterThreads;

// One CTA per image. (1) Verification: the chain is right where A(j) == B(j-1).  The broken links
// (look-back too short for that spot) are collected and each is decoded again from B(j-1) by one
// thread, segment by segment, until the walk meets the decode recorded for subsequence j — from
// there on that record was already the true one.  Repeated until the chain holds: the lowest
// broken link always starts from a correct state, so every iteration extends the correct prefix.
// (2) Exclusive prefix scan turning per-subsequence advances into the absolute state at every A
// (segmented where a restart interval began).
// MULTI: the repair walks go through the multi-symbol tables like the synchronisation pass (dynamic shared memory:
// 12 x 8 bytes of per-block table addresses, then the tables); the states they record at segment ends are the same.
template <bool MULTI>
__global__ void __launch_bounds__(kInterThreads) verify_scan_kernel(BatchDev b) {
    extern __shared__ __align__(128) uint8_t dyn_smem[];
    __shared__ EntropySmem sm;
    __shared__ FastTables ft;
    __shared__ int32_t s_agg[kInterThreads][5];
    __shared__ RepairJob s_jobs[kRepairJobs];
    __shared__ uint32_t s_count;

    const uint32_t img = b.img0 + blockIdx.x;
    const uint32_t S = b.sub_bits;
    load_entropy_img(b, threadIdx.x < 32 ? img : kNoImage, sm, 32);
    const ImgDev& im = sm.img[0];
    if (im.interval_mode) return;
    const ImgDyn dyn = b.dyn[img];
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    SubInfo* subs = b.subs + im.sub_off;
    const uint32_t tid = threadIdx.x;

    bool loaded = false;
#pragma unroll 1
    for (uint32_t iter = 0; iter <= nsub; iter++) {
        if (tid == 0) s_count = 0u;
        __syncthreads();
        for (uint32_t j = 1 + tid; j < nsub; j += kInterThreads) {
            const uint32_t start_p = subs[j - 1].pB, start_cz = (subs[j - 1].cz >> 10) & kCzMask;
            if (start_p != subs[j].pA || start_cz != (subs[j].cz & kCzMask)) {
                const uint32_t k = atomicAdd(&s_count, 1u);
                if (k < (uint32_t)kRepairJobs) s_jobs[k] = RepairJob{j, start_p, start_cz};  // the rest waits for the next iteration
            }
        }
        __syncthreads();
        const uint32_t njobs = min(s_count, (uint32_t)kRepairJobs);
        if (njobs == 0u) break;
        if (!loaded) {
            load_entropy_luts(b, sm, kInterThreads);
            fast_tables_init(ft, sm, threadIdx.x < 32, 32, kInterThreads);
            if constexpr (MULTI)
                load_multi_tables(b, sm, reinterpret_cast<uint32_t*>(dyn_smem + 128), reinterpret_cast<uint2*>(dyn_smem), 0, true, kInterThreads);
            __syncthreads();
            loaded = true;
        }
        FastCtx cx = make_fast_ctx(b, sm, 0, dyn, ft);
        if constexpr (MULTI) {
            cx.minfo_addr = smem_addr(dyn_smem);
            JPGPU_PIN32(cx.minfo_addr);
        }
        for (uint32_t i = tid; i < njobs; i += kInterThreads) {
            const RepairJob job = s_jobs[i];
            FastState st;
            fast_init(cx, st, job.p, (int32_t)(job.cz & 63u), job.cz >> 6, 0, 0, 0);
            SubInfo rec;
            rec.pA = st.p;
            rec.cz = job.cz;
            fast_sync_subsequence<MULTI>(cx, st, job.sub * S, S, b.seg_bits, b.segs + (size_t)(im.sub_off + job.sub) * (S / b.seg_bits), true, rec);
            subs[job.sub] = rec;
        }
        __syncthreads();
    }

    // ---- exclusive scan: n/dc become the absolute state at A (segmented by `crossed`)
    const uint32_t chunk = (nsub + kInterThreads - 1) / kInterThreads;
    const uint32_t lo = tid * chunk, hi = min(nsub, lo + chunk);
    int32_t acc[4] = {0, 0, 0, 0};
    uint32_t crossed = 0;
    for (uint32_t jj = lo; jj < hi; jj++) {
        const SubInfo s = subs[jj];
        fold_advance(acc, crossed, s.cz, s.n, s.dc);
    }
    s_agg[tid][0] = acc[0]; s_agg[tid][1] = acc[1]; s_agg[tid][2] = acc[2]; s_agg[tid][3] = acc[3]; s_agg[tid][4] = (int32_t)crossed;
    __syncthreads();
    int32_t run[4] = {0, 0, 0, 0};
    for (uint32_t k = 0; k < tid; k++) {  // exclusive prefix over the preceding chunks
        if (s_agg[k][4]) { run[0] = s_agg[k][0]; run[1] = s_agg[k][1]; run[2] = s_agg[k][2]; run[3] = s_agg[k][3]; }
        else { run[0] = sat_pos((int64_t)run[0] + s_agg[k][0]); run[1] += s_agg[k][1]; run[2] += s_agg[k][2]; run[3] += s_agg[k][3]; }
    }
    for (uint32_t jj = lo; jj < hi; jj++) {
        SubInfo s = subs[jj];
        const int32_t at_a[4] = {run[0], run[1], run[2], run[3]};
        uint32_t dummy = 0;
        fold_advance(run, dummy, s.cz, s.n, s.dc);
        s.n = at_a[0]; s.dc[0] = at_a[1]; s.dc[1] = at_a[2]; s.dc[2] = at_a[3];
        subs[jj] = s;
    }
}

// One thread per subsequence re-decodes it from its now exact start state and produces the
// coefficients.  A lane assembles each 8x8 block in a private, pre-zeroed 128-byte buffer in
// shared memory (kWriteBufs of them, 16-byte pieces XOR-swizzled so that both the scattered
// 2-byte stores and the flush are nearly conflict-free).  Lanes run kPhaseSymbols symbols (or
// until their buffers are full), then the warp flushes every completed block cooperatively:
// 8 lanes store one block as 8 x 16 bytes, so HBM only ever sees whole 128-byte blocks, written
// once — no memset of the arena, no read-modify-write of partial sectors.
// A block belongs to the lane in whose subsequence it STARTS: a lane that begins inside a block
// decodes the rest of it without storing, a lane that ends inside a block runs on until the
// block is complete.
struct WriteLayout {
    uint32_t lut_bytes, ft_off, buf_off, list_off, total;
};
__host__ __device__ inline WriteLayout write_layout(uint32_t max_slots, uint32_t nbuf) {
    WriteLayout l;
    l.lut_bytes = (uint32_t)(sizeof(EntropySmemT<kWriteJobsPerCta>) - (kMaxLutSlots - max_slots) * sizeof(HuffLut));
    l.ft_off = (l.lut_bytes + 15u) & ~15u;
    l.buf_off = (l.ft_off + (uint32_t)sizeof(FastTablesT<kWriteThreads>) + 127u) & ~127u;
    l.list_off = l.buf_off + kWriteThreads * nbuf * 128u;
    l.total = l.list_off + kWriteJobsPerCta * 32u * nbuf * 8u;
    return l;
}

template <int NBUF, int PHASE>
__global__ void __launch_bounds__(kWriteThreads) decode_write_kernel(BatchDev b) {
    extern __shared__ __align__(128) uint8_t dyn_smem[];
    using Smem = EntropySmemT<kWriteJobsPerCta>;
    using Tables = FastTablesT<kWriteThreads>;
    Smem& sm = *reinterpret_cast<Smem*>(dyn_smem);
    const WriteLayout lay = write_layout(b.max_slots, NBUF);
    Tables& ft = *reinterpret_cast<Tables*>(dyn_smem + lay.ft_off);
    int16_t* const bufs = reinterpret_cast<int16_t*>(dyn_smem + lay.buf_off);
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint2* const flist = reinterpret_cast<uint2*>(dyn_smem + lay.list_off) + warp * (32 * NBUF);

    // The write pass works in UNITS of sub_bits >> wp_shift bits (a whole number of checkpoint segments): the
    // synchronisation pass wants long subsequences (less look-back per decoded bit, fewer links to verify), this pass
    // short ones (many short jobs fill the machine better and end closer together).  Warp job q covers the 32 units
    // q*32 .. q*32+31 of sequence q >> wp_shift; unit u of a sequence is part u & (H-1) of its subsequence u >> wp_shift.
    const uint32_t hs = b.wp_shift, H = 1u << hs;
    if (b.seqs[b.job0 + ((blockIdx.x * kWriteJobsPerCta) >> hs)].img == kNoImage) return;   // a CTA of padding jobs only
    const uint32_t job = blockIdx.x * kWriteJobsPerCta + warp;
    const SeqDesc sd = (job >> hs) < b.n_seqs ? b.seqs[b.job0 + (job >> hs)] : SeqDesc{kNoImage, 0u};
    const uint32_t S = b.sub_bits;
    load_entropy_img(b, sd.img, sm, 32);
    load_entropy_luts(b, sm, kWriteThreads);
    fast_tables_init(ft, sm, sd.img != kNoImage, 32, kWriteThreads);
    for (uint32_t i = tid; i < kWriteThreads * NBUF * 8u; i += kWriteThreads)
        reinterpret_cast<uint4*>(bufs)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    if (sd.img == kNoImage) return;
    const ImgDev& img = sm.img[warp];
    const ImgDyn dyn = b.dyn[sd.img];
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    const FastCtx cx = make_fast_ctx(b, sm, warp, dyn, ft);
    const uint32_t unit = ((job & (H - 1u)) << 5) + lane;
    const uint32_t j = sd.first_sub + (unit >> hs), part = unit & (H - 1u);
    const uint32_t unit_bit = j * S + part * (S >> hs), end_bit = unit_bit + (S >> hs);
    bool active = j < nsub && unit_bit < dyn.stream_bits;
    if (!__ballot_sync(0xffffffffu, active)) return;

    const int32_t total = (int32_t)img.total_coefs;
    int16_t* __restrict__ coefs = b.coefs + img.coef_off;
    FastState st;
    bool store_on = true;
    const bool by_interval = img.interval_mode != 0u;
    uint32_t k0 = 0;
    if (active && by_interval) {   // this lane owns the restart intervals that start inside its unit
        k0 = first_interval_from(cx.seg, cx.nseg, unit_bit);
        active = k0 < cx.nseg && cx.seg[k0] < end_bit;
    }
    if (active) {
        if (by_interval) {
            fast_init(cx, st, cx.seg[k0], (int32_t)(k0 * cx.seg_units), 0u, 0, 0, 0);
        } else {
            // state at the start of the unit: that of its subsequence at A (exact after verify_scan_kernel), carried
            // over the checkpoint segments that precede the unit
            const SubInfo me = b.subs[img.sub_off + j];
            uint32_t p0 = me.pA, cz0 = me.cz & kCzMask, crossed = 0u;
            int32_t acc[4] = {me.n, me.dc[0], me.dc[1], me.dc[2]};
            const uint32_t nsegs = S / b.seg_bits, npre = part * (nsegs >> hs);
            const SegRec* sg = b.segs + (size_t)(img.sub_off + j) * nsegs;
#pragma unroll 1
            for (uint32_t k = 0; k < npre; k++) {
                const uint4 lo = __ldg(reinterpret_cast<const uint4*>(sg + k));
                const uint2 hi = __ldg(reinterpret_cast<const uint2*>(sg + k) + 2);
                const int32_t dc[3] = {(int32_t)lo.w, (int32_t)hi.x, (int32_t)hi.y};
                fold_advance(acc, crossed, lo.y, (int32_t)lo.z, dc);
                p0 = lo.x; cz0 = lo.y & kCzMask;
            }
            fast_init(cx, st, p0, acc[0], (cz0 >> 6) & 15u, acc[1], acc[2], acc[3]);
        }
        st.flags &= ~kCrossed;
        store_on = (st.g & 63) == 0;
        if ((uint32_t)st.g >= (uint32_t)total || (st.p >= end_bit && store_on)) active = false;   // past the scan (or a saturated position)
    } else {
        st.p = 0; st.g = 0; st.flags = 0; st.info_ptr = cx.info_addr; st.w0 = st.w1 = st.w2 = 0; st.kp = cx.words;
        st.seg = 0; st.seg_end = st.seg_lim = st.lim = 0; st.wrap_lim = 0xffffffffu; st.dcur = 0; st.dc_off = 0; st.lut_dc = st.lut_ac = cx.lut0_addr;
    }
    const int32_t g_start = st.g;
    WriteLane<NBUF> wl;
    wl.row0 = tid * NBUF;   // this lane's first buffer row (one row = one 128-byte block)
    wl.rows_addr = smem_addr(bufs) + wl.row0 * 128u;
    wl.select(0u);
    wl.ndone = 0;
    wl.dest0 = wl.dest1 = 0u;
    wl.end_bit = end_bit;
    wl.end_bit_blk = by_interval ? 0xffffffffu : end_bit;   // an interval-mode lane only ends where an interval ends
    wl.total = total;
    wl.seg_limit = cx.seg_units ? min(total, (int32_t)((st.seg + 1u) * cx.seg_units)) : total;
    wl.store_on = store_on && st.g < wl.seg_limit ? 1u : 0u;
    wl.state = active ? (uint32_t)WriteLane<NBUF>::kRun : (uint32_t)WriteLane<NBUF>::kFinished;
    wl.coefs = coefs;

#pragma unroll 1
    while (true) {
        // ---- phase A: every lane decodes up to PHASE symbols into its own buffers.  Whether a lane is finished
        // (block boundary at or past the end of its subsequence, or past the last block of the scan) or out of
        // buffers can only change when a block completes or a restart interval ends, so it is only looked at
        // there (WriteLane::close_block / on_interval).
#pragma unroll 1
        for (int k = PHASE; k > 0 && wl.state == WriteLane<NBUF>::kRun; k--) fast_step<true, true>(cx, st, wl);
        if (wl.state == WriteLane<NBUF>::kBlockEnd) fast_block_end(cx, st, wl);
        if (wl.state == WriteLane<NBUF>::kBlocked) wl.state = WriteLane<NBUF>::kRun;
        active = wl.state != WriteLane<NBUF>::kFinished;
        const uint32_t ndone = wl.ndone, cur = wl.cur, row0 = wl.row0;
        // ---- phase B: the warp flushes all completed blocks, 8 lanes per block
        uint32_t offs = 0, count = 0;
#pragma unroll
        for (int i = 0; i < NBUF; i++) {
            const uint32_t m = __ballot_sync(0xffffffffu, ndone > (uint32_t)i);
            offs += __popc(m & ((1u << lane) - 1u));
            count += __popc(m);
        }
        if (count == 0) {
            if (!__ballot_sync(0xffffffffu, active)) break;
            continue;
        }
        {
            uint32_t r = cur + NBUF - ndone;  // oldest completed buffer
#pragma unroll
            for (int i = 0; i < NBUF; i++) {
                if ((uint32_t)i < ndone) {
                    if (r >= (uint32_t)NBUF) r -= NBUF;
                    flist[offs + i] = make_uint2(row0 + r, i == 0 ? wl.dest0 : wl.dest1);
                    r++;
                }
            }
        }
        __syncwarp();
        const uint32_t piece = lane & 7u;
#pragma unroll 1
        for (uint32_t i = lane >> 3; i < count; i += 4) {
            const uint2 e = flist[i];
            uint4* src = reinterpret_cast<uint4*>(bufs + e.x * 64u) + (piece ^ (e.x & 7u));
            const uint4 v = *src;
            *src = make_uint4(0u, 0u, 0u, 0u);
            if (e.y != 0xffffffffu) reinterpret_cast<uint4*>(coefs + (size_t)e.y * 64u)[piece] = v;
        }
        __syncwarp();
        wl.ndone = 0;
    }
    if (j < nsub && unit_bit < dyn.stream_bits) {
        uint32_t bits = st.flags & (kStBadCode | kStDcSize | kStRestart);
        if (g_start < total && st.g >= total) {  // this thread decoded the last block of the scan
            b.dyn[sd.img].bits_consumed = st.p;
            bits |= kStDone;
        }
        if (bits) atomicOr(&b.dyn[sd.img].status, bits);
        // the data ended before the scan was complete: everything from the block this lane stood in is unwritten
        if (g_start < total && st.g < total && st.p >= dyn.stream_bits) atomicMax(&b.dyn[sd.img].coef_end, (uint32_t)st.g & ~63u);
    }
}

// The coefficient arena is reused wave after wave and never cleared (that memset was 6.4 GB per plan).  A complete
// scan stores every one of its blocks; a scan whose data ended early leaves the blocks from ImgDyn::coef_end on
// unwritten - holding an earlier image's coefficients - and this kernel, one CTA per image, zero-fills them.  For an
// image that decoded completely (all but damaged files) it reads one word and returns.
__global__ void __launch_bounds__(256) zero_tail_kernel(BatchDev b) {
    const uint32_t img = b.img0 + blockIdx.x;
    const ImgDyn d = b.dyn[img];
    const ImgDev& im = b.imgs[img];
    const uint32_t limit = coef_block_limit(d);
    const uint32_t nblk = im.total_coefs >> 6;
    if (limit >= nblk) return;
    uint4* dst = reinterpret_cast<uint4*>(b.coefs + im.coef_off) + (size_t)limit * 8;
    const size_t nvec = (size_t)(nblk - limit) * 8;
    for (size_t i = threadIdx.x; i < nvec; i += 256) dst[i] = make_uint4(0u, 0u, 0u, 0u);
}

// Every image's output lies at a 256-byte aligned offset of the RGB arena; the up to 255 bytes (1020 with float output)
// between the end of one and the start of the next are never written by a decode.  jpgpu_batch_download_contiguous and the
// pipeline copy the arena as a whole, so those gaps are given defined contents once per plan / output arena / format.
__global__ void __launch_bounds__(256) zero_output_pads_kernel(BatchDev b) {
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i >= b.n_images) return;
    const ImgDev& im = b.imgs[b.img0 + i];
    const size_t sb = b.out_planar == 2u ? 4u : 1u;
    const size_t n = (size_t)im.out_pixels * 3u, end = (n + 255u) & ~(size_t)255u;
    uint8_t* base = b.rgb + im.rgb_off * sb;
    for (size_t k = n * sb; k < end * sb; k++) base[k] = 0u;
}

// ============================================ stage 2+3: dequant + IDCT + upsample + colour
constexpr int kIdctThreads = 128;
#ifndef JPGPU_IDCT_TMA
#define JPGPU_IDCT_TMA 0     // 1: coefficient tiles through cp.async.bulk + mbarrier (experiment, see DESIGN.md 4.3)
#endif
#ifndef JPGPU_TILES_PER_CTA
#define JPGPU_TILES_PER_CTA 5
#endif
#ifdef JPGPU_IDCT_MIN_CTAS
#define JPGPU_IDCT_BOUNDS __launch_bounds__(kIdctThreads, JPGPU_IDCT_MIN_CTAS)
#else
#define JPGPU_IDCT_BOUNDS __launch_bounds__(kIdctThreads)
#endif
constexpr int kTilesPerCta = JPGPU_TILES_PER_CTA;  // consecutive tiles one CTA walks (amortises set-up, lets loads run ahead)
constexpr int kScrRowPitch = 12;     // floats; 4*odd -> conflict-free 128-bit row reads
constexpr int kScrBlkPitch = 104;    // floats; 8 mod 32 -> conflict-free column writes across the 4 blocks of a warp
constexpr int kOutPitch = 400;       // bytes per staged output row (128 px * 3 = 384, padded)

// decoder.rs:382-390 (clamp to [0,255], truncate) in two steps: truncation to s32 here, the clamp in pack4's
// saturating byte pack (I2IP) - 6 instructions per 4 output bytes.
__device__ __forceinline__ int32_t f32_to_u8_sat(float x) {
    int32_t r;
    asm("cvt.rzi.s32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

// 8 lanes own one 8x8 block; lane t holds column t (16 bytes = 8 coefficients), runs the
// vertical pass, the block is transposed through shared memory, and lane t finishes row t.
// qt points at this lane's multipliers: qt[0..3] = rows 0-3, qt[32..35] = rows 4-7.
__device__ __forceinline__ void block_idct(const uint4 raw, const float4 q0, const float4 q1, int t,
                                           float* scr_w, const float* scr_r, float dc_bias, float out[8]) {
    // scr_w and scr_r alias the same shared scratch tile: no __restrict__ on them.
    float f0 = (float)(int16_t)(raw.x & 0xffffu) * q0.x;
    float f1 = (float)(int16_t)(raw.x >> 16) * q0.y;
    float f2 = (float)(int16_t)(raw.y & 0xffffu) * q0.z;
    float f3 = (float)(int16_t)(raw.y >> 16) * q0.w;
    float f4 = (float)(int16_t)(raw.z & 0xffffu) * q1.x;
    float f5 = (float)(int16_t)(raw.z >> 16) * q1.y;
    float f6 = (float)(int16_t)(raw.w & 0xffffu) * q1.z;
    float f7 = (float)(int16_t)(raw.w >> 16) * q1.w;
    if (t == 0) f0 += dc_bias;  // level shift folded into the DC term
    idct8(f0, f1, f2, f3, f4, f5, f6, f7);  // vertical: f[y] = sample (y, column t) before the horizontal pass
    __syncwarp();                           // previous pass finished reading scr
    scr_w[0 * kScrRowPitch] = f0; scr_w[1 * kScrRowPitch] = f1; scr_w[2 * kScrRowPitch] = f2;
    scr_w[3 * kScrRowPitch] = f3; scr_w[4 * kScrRowPitch] = f4; scr_w[5 * kScrRowPitch] = f5;
    scr_w[6 * kScrRowPitch] = f6; scr_w[7 * kScrRowPitch] = f7;
    __syncwarp();
    const float4 a = *reinterpret_cast<const float4*>(scr_r);
    const float4 c = *reinterpret_cast<const float4*>(scr_r + 4);
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = c.x; out[5] = c.y; out[6] = c.z; out[7] = c.w;
    idct8(out[0], out[1], out[2], out[3], out[4], out[5], out[6], out[7]);  // horizontal: row t
}

__device__ __forceinline__ void block_idct(const uint4 raw, const float* __restrict__ qt, int t,
                                           float* scr_w, const float* scr_r, float dc_bias, float out[8]) {
    block_idct(raw, *reinterpret_cast<const float4*>(qt), *reinterpret_cast<const float4*>(qt + 32), t, scr_w, scr_r,
               dc_bias, out);
}

__device__ __forceinline__ uint32_t pack4(int32_t a, int32_t b, int32_t c, int32_t d) {  // bytes a (lowest) .. d, each clamped
    uint32_t t, r;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(d), "r"(c), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(b), "r"(a), "r"(t));
    return r;
}

// ---- two blocks at a time on the packed FP32 pipe (FADD2 / FMUL2 / FFMA2 of sm_100: one instruction, two lanes of a
// 64-bit register pair).  A thread that has two blocks of the same component to transform (two luma or two chroma
// passes of a tile) runs them as the two halves of f32x2 values: the butterflies cost half the issue slots, and the
// transposition through shared memory moves both blocks with 8-byte stores / 16-byte loads.
#ifndef JPGPU_IDCT_PAIRS
#define JPGPU_IDCT_PAIRS 1
#endif
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// idct8() of jpgpu_core.h on both halves
__device__ __forceinline__ void idct8x2(f32x2 (&x)[8]) {
    const f32x2 c1414 = pk2(1.414213562f, 1.414213562f), c1847 = pk2(1.847759065f, 1.847759065f);
    const f32x2 n1082 = pk2(-1.082392200f, -1.082392200f), n2613 = pk2(-2.613125930f, -2.613125930f);
    const f32x2 t10 = add2(x[0], x[4]), t11 = sub2(x[0], x[4]);
    const f32x2 t13 = add2(x[2], x[6]);
    const f32x2 t12 = sub2(mul2(sub2(x[2], x[6]), c1414), t13);
    const f32x2 e0 = add2(t10, t13), e3 = sub2(t10, t13), e1 = add2(t11, t12), e2 = sub2(t11, t12);
    const f32x2 z13 = add2(x[5], x[3]), z10 = sub2(x[5], x[3]), z11 = add2(x[1], x[7]), z12 = sub2(x[1], x[7]);
    const f32x2 o7 = add2(z11, z13);
    const f32x2 t11o = mul2(sub2(z11, z13), c1414);
    const f32x2 z5 = mul2(add2(z10, z12), c1847);
    const f32x2 t10o = fma2(z12, n1082, z5);
    const f32x2 t12o = fma2(z10, n2613, z5);
    const f32x2 o6 = sub2(t12o, o7);
    const f32x2 o5 = sub2(t11o, o6);
    const f32x2 o4 = sub2(t10o, o5);
    x[0] = add2(e0, o7); x[7] = sub2(e0, o7);
    x[1] = add2(e1, o6); x[6] = sub2(e1, o6);
    x[2] = add2(e2, o5); x[5] = sub2(e2, o5);
    x[3] = add2(e3, o4); x[4] = sub2(e3, o4);
}

constexpr int kScr2RowPitch = 10;    // f32x2 units; 2*odd -> conflict-free 16-byte row reads
constexpr int kScr2BlkPitch = 88;    // f32x2 units; 8 mod 16 -> conflict-free 8-byte column writes across a half warp
// block_idct() for two blocks (raw_a, raw_b: column t of each, same component): out_a / out_b = row t of each.
// scr_w = scratch + bp * kScr2BlkPitch + t, scr_r = scratch + bp * kScr2BlkPitch + t * kScr2RowPitch (f32x2 units).
__device__ __forceinline__ void block_idct2p(const uint4 raw_a, const uint4 raw_b, const float* __restrict__ qt, int t,
                                             f32x2* scr_w, const f32x2* scr_r, float dc_bias, f32x2 (&x)[8]);
__device__ __forceinline__ void block_idct2(const uint4 raw_a, const uint4 raw_b, const float* __restrict__ qt, int t,
                                            f32x2* scr_w, const f32x2* scr_r, float dc_bias, float out_a[8], float out_b[8]) {
    f32x2 x[8];
    block_idct2p(raw_a, raw_b, qt, t, scr_w, scr_r, dc_bias, x);
#pragma unroll
    for (int i = 0; i < 8; i++) upk2(x[i], out_a[i], out_b[i]);
}
// the same, rows left packed: x[i] = (sample i of row t of block a, of block b)
__device__ __forceinline__ void block_idct2p(const uint4 raw_a, const uint4 raw_b, const float* __restrict__ qt, int t,
                                             f32x2* scr_w, const f32x2* scr_r, float dc_bias, f32x2 (&x)[8]) {
    const float4 q0 = *reinterpret_cast<const float4*>(qt), q1 = *reinterpret_cast<const float4*>(qt + 32);
    const float q[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    const uint32_t wa[4] = {raw_a.x, raw_a.y, raw_a.z, raw_a.w}, wb[4] = {raw_b.x, raw_b.y, raw_b.z, raw_b.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t ua = wa[i >> 1], ub = wb[i >> 1];
        float fa = (float)(int16_t)((i & 1) ? (ua >> 16) : (ua & 0xffffu)) * q[i];
        float fb = (float)(int16_t)((i & 1) ? (ub >> 16) : (ub & 0xffffu)) * q[i];
        if (i == 0 && t == 0) { fa += dc_bias; fb += dc_bias; }   // level shift folded into the DC term
        x[i] = pk2(fa, fb);
    }
    idct8x2(x);   // vertical
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 8; r++) scr_w[r * kScr2RowPitch] = x[r];
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(scr_r + 2 * k);
        x[2 * k] = v.x; x[2 * k + 1] = v.y;
    }
    idct8x2(x);   // horizontal
}

// Tile = 128 pixels x (8*VY) rows = 16/HY MCUs.  Phase A: chroma blocks -> shared f32
// planes.  Phase B: luma blocks; each lane ends with 8 horizontally adjacent Y samples,
// fetches the replicated chroma, converts and stages 24 output bytes.  Phase C: the
// staged tile is stored with 16-byte vectors.  A CTA walks kTilesPerCta consecutive
// tiles; the coefficient loads of the next tile are issued before the current one is
// computed.
// PLANAR: the output is three W x H byte planes (R, G, B) instead of interleaved triples (jpgpu_batch_set_output_format).
template <int HY, int VY, bool GRAY, int FORMAT>
__global__ void JPGPU_IDCT_BOUNDS idct_colour_kernel(BatchDev b, const uint32_t* __restrict__ img_list) {
    // FORMAT (jpgpu_batch_set_output_format): 0 interleaved u8 triples, 1 three u8 planes, 2 three f32 planes holding
    // u8 * scale[c] + bias[c] - staged like 1, converted while the tile is copied out
    constexpr bool PLANAR = FORMAT != 0, F32 = FORMAT == 2;
    constexpr int MH = 8 * VY;
    constexpr int NM = 128 / (8 * HY);         // MCUs per tile
    constexpr int NY = HY * VY;                // luma blocks per MCU
    constexpr int NB = GRAY ? 1 : NY + 2;      // blocks per MCU
    constexpr int CW = NM * 8;                 // chroma samples per tile row
    constexpr int CWP = CW + 4;                // padded pitch: rows land on different banks
    constexpr int CH_PASSES = GRAY ? 0 : (2 * NM) / 16;
    constexpr int Y_PASSES = (NM * NY) / 16;
    constexpr int NL = CH_PASSES + Y_PASSES;   // 16-byte loads per thread and tile
#ifndef JPGPU_IDCT_PACKED_COLOUR
#define JPGPU_IDCT_PACKED_COLOUR 1
#endif
    constexpr bool Y_PAIRS = JPGPU_IDCT_PAIRS && Y_PASSES % 2 == 0, CH_PAIRS = JPGPU_IDCT_PAIRS && CH_PASSES > 0 && CH_PASSES % 2 == 0;
    // 4:2:0: a thread's two luma blocks are the horizontal neighbours 2*bp, 2*bp+1 of one MCU row; they share their
    // chroma rows, so the colour conversion runs packed as well (the chroma samples c and c+4 of an MCU are stored
    // next to each other)
    constexpr bool PACKED_COLOUR = Y_PAIRS && !GRAY && HY == 2 && VY == 2 && Y_PASSES == 2 && JPGPU_IDCT_PACKED_COLOUR;
    auto luma_block = [](int p, int bp) { return PACKED_COLOUR ? 2 * bp + p : p * 16 + bp; };   // index in the tile
    constexpr int kScrFloats = (Y_PAIRS || CH_PAIRS) ? 16 * kScr2BlkPitch * 2 : 16 * kScrBlkPitch;
    __shared__ __align__(16) float s_scr[kScrFloats];
    __shared__ __align__(16) float s_chroma[GRAY ? 4 : 2 * 8 * CWP];
    constexpr int kPlanePitch = 144;                      // bytes per staged row of one plane (128 + 16: rows 4 banks apart)
    constexpr int kPlaneSize = MH * kPlanePitch;
    __shared__ __align__(16) uint8_t s_out[PLANAR ? 3 * kPlaneSize : MH * kOutPitch];
    __shared__ __align__(16) float s_qt[3 * 64];

    const ImgDev& im = b.imgs[img_list[blockIdx.y]];
    const uint32_t ntiles = im.tiles_x * im.tiles_y;
    uint32_t tile = blockIdx.x * kTilesPerCta;
    if (tile >= ntiles) return;
    const uint32_t tile_end = min(ntiles, tile + kTilesPerCta);
    const int tid = threadIdx.x, t = tid & 7, bp = tid >> 3;

    // multipliers, re-laid so that lane t's two float4 reads are conflict-free: [comp][half][t][4]
    for (int i = tid; i < (GRAY ? 64 : 192); i += kIdctThreads) {
        const int comp = i >> 6, r = i & 63, tt = r >> 3, v = r & 7;
        s_qt[comp * 64 + (v >> 2) * 32 + tt * 4 + (v & 3)] = b.qt[im.qt_off[comp] + r];
    }

    const uint4* __restrict__ coefs = reinterpret_cast<const uint4*>(b.coefs + im.coef_off);
    uint8_t* __restrict__ rgb = b.rgb + im.rgb_off * (F32 ? 4u : 1u);
    const uint32_t W = im.width, H = im.height, mcux = im.mcux, units = im.units, tiles_x = im.tiles_x;
    float* const scr_w = s_scr + bp * kScrBlkPitch + t;
    const float* const scr_r = s_scr + bp * kScrBlkPitch + t * kScrRowPitch;
    f32x2* const scr2_w = reinterpret_cast<f32x2*>(s_scr) + bp * kScr2BlkPitch + t;
    const f32x2* const scr2_r = reinterpret_cast<const f32x2*>(s_scr) + bp * kScr2BlkPitch + t * kScr2RowPitch;
    const float* const qt_l = s_qt + t * 4;

    // per-thread block assignment inside a tile (in units of blocks, relative to the tile's first MCU)
    int blk_of[NL > 0 ? NL : 1];       // index of the block this thread handles in load l
    int mcu_of[NL > 0 ? NL : 1];
#pragma unroll
    for (int a = 0; a < CH_PASSES; a++) {
        const int cb = a * 16 + bp, m = cb >> 1;
        mcu_of[a] = m; blk_of[a] = m * NB + NY + (cb & 1);
    }
#pragma unroll
    for (int p = 0; p < Y_PASSES; p++) {
        const int yb = luma_block(p, bp), m = yb / NY;
        mcu_of[CH_PASSES + p] = m; blk_of[CH_PASSES + p] = m * NB + yb % NY;
    }

    // copy-out plan of this thread: which 16-byte vectors of the staged tile it stores (tile-invariant)
    constexpr int NV = (MH * 24 + kIdctThreads - 1) / kIdctThreads;
    const bool vec_ok = PLANAR ? (W & 15u) == 0u : ((W * 3u) & 15u) == 0u;
    const uint32_t plane_bytes = W * H;
    uint32_t co_rk[NV], co_s[NV], co_g[NV];
#pragma unroll
    for (int n = 0; n < NV; n++) {
        const uint32_t i = (uint32_t)tid + (uint32_t)n * kIdctThreads;
        if (PLANAR) {   // vector i: plane i / (MH*8), row (i / 8) % MH, 16-byte piece i % 8
            const uint32_t pl = i / (MH * 8u), r = (i >> 3) % MH, k = i & 7u;
            co_rk[n] = i < (uint32_t)MH * 24u ? (r | (k << 8)) : 255u;
            co_s[n] = pl * kPlaneSize + r * kPlanePitch + k * 16u;
            co_g[n] = pl * plane_bytes + r * W + k * 16u;
        } else {
            const uint32_t r = i / 24u, k = i - r * 24u;
            co_rk[n] = i < (uint32_t)MH * 24u ? (r | (k << 8)) : 255u;   // row 255 never passes the bounds test
            co_s[n] = r * kOutPitch + k * 16u;
            co_g[n] = r * W * 3u + k * 16u;
        }
    }

#if JPGPU_IDCT_TMA
    // Experiment (DESIGN.md 4.3): the coefficients of a tile are one contiguous run in HBM (consecutive MCUs of an MCU
    // row), so one elected thread fetches them with a bulk asynchronous copy (cp.async.bulk shared <- global, completion
    // on an mbarrier) into a double-buffered shared tile, and the IDCT passes read their 16-byte columns from there.  No
    // coefficient vector lives in registers across the tile loop.
    constexpr int kTileVecs = NM * NB * 8;
    __shared__ __align__(128) uint4 s_coef[2][kTileVecs];
    __shared__ __align__(8) uint64_t s_bar[2];
    const uint32_t bar0 = smem_addr(&s_bar[0]);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0 + 8u));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    auto tma_issue = [&](uint32_t tx, uint32_t ty, uint32_t buf) {   // thread 0 only
        const uint32_t mcu0 = ty * mcux + tx * NM;
        const uint32_t here = min(min((uint32_t)NM, mcux - tx * NM), units > mcu0 ? units - mcu0 : 0u);
        const uint32_t bytes = here * NB * 128u;
        const uint32_t bar = bar0 + buf * 8u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
        if (bytes)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_addr(&s_coef[buf][0])), "l"(coefs + (size_t)mcu0 * NB * 8), "r"(bytes), "r"(bar) : "memory");
    };
    auto tma_wait = [&](uint32_t buf, uint32_t parity) {
        uint32_t ok = 0;
        const uint32_t bar = bar0 + buf * 8u;
        while (!ok)
            asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                         : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    };
    uint32_t tma_k = 0, here_cur = 0;
    // column t of block l of this thread's assignment in the current tile (zeros past the image's last MCU)
#define JPGPU_COEF(l) ((uint32_t)mcu_of[l] < here_cur ? s_coef[tma_k & 1u][blk_of[l] * 8 + t] : make_uint4(0u, 0u, 0u, 0u))
#else
    uint4 cur[NL], nxt[NL];
#define JPGPU_COEF(l) cur[l]
    auto issue_loads = [&](uint32_t tx, uint32_t ty, uint4 (&dst)[NL]) {
        const uint32_t mcu0 = ty * mcux + tx * NM;
        const uint32_t here = min((uint32_t)NM, mcux - tx * NM);
#pragma unroll
        for (int l = 0; l < NL; l++) {
            const bool valid = (uint32_t)mcu_of[l] < here && mcu0 + mcu_of[l] < units;
            dst[l] = make_uint4(0u, 0u, 0u, 0u);
            if (valid) dst[l] = __ldg(coefs + ((size_t)mcu0 * NB + blk_of[l]) * 8 + t);
        }
    };
#endif
    uint32_t tx = tile % tiles_x, ty = tile / tiles_x;   // tile coordinates, advanced incrementally
#if JPGPU_IDCT_TMA
    __syncthreads();  // s_qt ready, barriers initialised
    if (tid == 0) tma_issue(tx, ty, 0u);
#else
    issue_loads(tx, ty, cur);
    __syncthreads();  // s_qt ready
#endif

#pragma unroll 1
    for (; tile < tile_end; tile++) {
        const uint32_t ntx = tx + 1u == tiles_x ? 0u : tx + 1u, nty = ty + (tx + 1u == tiles_x ? 1u : 0u);
#if JPGPU_IDCT_TMA
        // the other buffer was last read in the previous tile, before that tile's closing barrier: free to refill
        if (tid == 0 && tile + 1 < tile_end) tma_issue(ntx, nty, (tma_k + 1u) & 1u);
        {
            const uint32_t mcu0 = ty * mcux + tx * NM;
            here_cur = min(min((uint32_t)NM, mcux - tx * NM), units > mcu0 ? units - mcu0 : 0u);
        }
        tma_wait(tma_k & 1u, (tma_k >> 1) & 1u);
#else
        if (tile + 1 < tile_end) issue_loads(ntx, nty, nxt);
#endif

        if (!GRAY) {
            auto put_chroma = [&](int a, const float (&o)[8]) {
                const int cb = a * 16 + bp, m = cb >> 1, comp = 1 + (cb & 1);
                float* dst = s_chroma + ((comp - 1) * 8 + t) * CWP + m * 8;
                if constexpr (PACKED_COLOUR) {   // (c0,c4) (c1,c5) (c2,c6) (c3,c7): left / right luma block of the MCU
                    *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[4], o[1], o[5]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(o[2], o[6], o[3], o[7]);
                } else {
                    *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4], o[5], o[6], o[7]);
                }
            };
            if constexpr (CH_PAIRS) {
#pragma unroll
                for (int a = 0; a < CH_PASSES; a += 2) {   // blocks a*16+bp and (a+1)*16+bp: same component (bp & 1)
                    float oa[8], ob[8];
                    block_idct2(JPGPU_COEF(a), JPGPU_COEF(a + 1), qt_l + (1 + (bp & 1)) * 64, t, scr2_w, scr2_r, 0.0f, oa, ob);
                    put_chroma(a, oa);
                    put_chroma(a + 1, ob);
                }
            } else {
#pragma unroll
                for (int a = 0; a < CH_PASSES; a++) {
                    float o[8];
                    block_idct(JPGPU_COEF(a), qt_l + (1 + (bp & 1)) * 64, t, scr_w, scr_r, 0.0f, o);
                    put_chroma(a, o);
                }
            }
            __syncthreads();
        }

        // truncation / clamp (decoder.rs:382-390) and staging of row t of luma block p of this thread
        auto stage_rgb = [&](int p, const float (&rf)[8], const float (&gf)[8], const float (&bf)[8], bool) {
            const int yb = luma_block(p, bp), m = yb / NY, sub = yb % NY, by = sub / HY, bx = sub % HY;
            const int px0 = (m * HY + bx) * 8, row = by * 8 + t;
            int32_t r8[8], g8[8], b8[8];
#pragma unroll
            for (int x = 0; x < 8; x++) { r8[x] = f32_to_u8_sat(rf[x]); g8[x] = f32_to_u8_sat(gf[x]); b8[x] = f32_to_u8_sat(bf[x]); }
            if (PLANAR) {
                uint8_t* dst = s_out + row * kPlanePitch + px0;
                *reinterpret_cast<uint2*>(dst) = make_uint2(pack4(r8[0], r8[1], r8[2], r8[3]), pack4(r8[4], r8[5], r8[6], r8[7]));
                *reinterpret_cast<uint2*>(dst + kPlaneSize) = make_uint2(pack4(g8[0], g8[1], g8[2], g8[3]), pack4(g8[4], g8[5], g8[6], g8[7]));
                *reinterpret_cast<uint2*>(dst + 2 * kPlaneSize) = make_uint2(pack4(b8[0], b8[1], b8[2], b8[3]), pack4(b8[4], b8[5], b8[6], b8[7]));
            } else {
                uint2* dst = reinterpret_cast<uint2*>(s_out + row * kOutPitch + px0 * 3);
                dst[0] = make_uint2(pack4(r8[0], g8[0], b8[0], r8[1]), pack4(g8[1], b8[1], r8[2], g8[2]));
                dst[1] = make_uint2(pack4(b8[2], r8[3], g8[3], b8[3]), pack4(r8[4], g8[4], b8[4], r8[5]));
                dst[2] = make_uint2(pack4(g8[5], b8[5], r8[6], g8[6]), pack4(b8[6], r8[7], g8[7], b8[7]));
            }
        };
        // colour conversion of one transformed luma block (pass p of this thread, not paired): y = row t of the block
        auto finish_luma = [&](int p, const float (&y)[8]) {
            if constexpr (GRAY) {
                stage_rgb(p, y, y, y, true);   // decoder.rs:317-324
            } else {
                const int yb = luma_block(p, bp), m = yb / NY, sub = yb % NY, by = sub / HY, bx = sub % HY;
                const int crow = (by * 8 + t) / VY, cc0 = ((m * HY + bx) * 8) / HY;
                float cbv[8], crv[8];
                const float* pcb = s_chroma + (0 * 8 + crow) * CWP + cc0;
                const float* pcr = s_chroma + (1 * 8 + crow) * CWP + cc0;
                if (HY == 2) {
                    const float4 u = *reinterpret_cast<const float4*>(pcb);
                    const float4 v = *reinterpret_cast<const float4*>(pcr);
                    cbv[0] = cbv[1] = u.x; cbv[2] = cbv[3] = u.y; cbv[4] = cbv[5] = u.z; cbv[6] = cbv[7] = u.w;
                    crv[0] = crv[1] = v.x; crv[2] = crv[3] = v.y; crv[4] = crv[5] = v.z; crv[6] = crv[7] = v.w;
                } else {
                    const float4 u0 = *reinterpret_cast<const float4*>(pcb), u1 = *reinterpret_cast<const float4*>(pcb + 4);
                    const float4 v0 = *reinterpret_cast<const float4*>(pcr), v1 = *reinterpret_cast<const float4*>(pcr + 4);
                    cbv[0] = u0.x; cbv[1] = u0.y; cbv[2] = u0.z; cbv[3] = u0.w; cbv[4] = u1.x; cbv[5] = u1.y; cbv[6] = u1.z; cbv[7] = u1.w;
                    crv[0] = v0.x; crv[1] = v0.y; crv[2] = v0.z; crv[3] = v0.w; crv[4] = v1.x; crv[5] = v1.y; crv[6] = v1.z; crv[7] = v1.w;
                }
                float rr[8], gg[8], bb[8];
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    // decoder.rs:392-401 with the +128 already inside y: r = cr*(2-2*0.299) + y, b = cb*(2-2*0.114) + y,
                    // g = (y - 0.114*b - 0.299*r)/0.587 = y - 0.344136*cb - 0.714136*cr
                    rr[x] = fmaf(crv[x], 1.402f, y[x]);
                    bb[x] = fmaf(cbv[x], 1.772f, y[x]);
                    gg[x] = fmaf(cbv[x], -0.34413629f, fmaf(crv[x], -0.71413629f, y[x]));
                }
                stage_rgb(p, rr, gg, bb, false);
            }
        };
        if constexpr (Y_PAIRS) {
#pragma unroll
            for (int p = 0; p < Y_PASSES; p += 2) {
                f32x2 y2[8];
                block_idct2p(JPGPU_COEF(CH_PASSES + p), JPGPU_COEF(CH_PASSES + p + 1), qt_l, t, scr2_w, scr2_r, 128.0f, y2);
                if constexpr (!PACKED_COLOUR) {
                    float ya[8], yb2[8];
#pragma unroll
                    for (int x = 0; x < 8; x++) upk2(y2[x], ya[x], yb2[x]);
                    finish_luma(p, ya);
                    finish_luma(p + 1, yb2);
                } else {
                    // both blocks of the pair at once: the left block's chroma is the first, the right block's the
                    // second half of the pairs stored by put_chroma
                    const int yb = luma_block(p, bp), m = yb / NY, by = (yb % NY) / HY;
                    const int crow = (by * 8 + t) / VY;
                    const f32x2* pcb = reinterpret_cast<const f32x2*>(s_chroma + (0 * 8 + crow) * CWP) + m * 4;
                    const f32x2* pcr = reinterpret_cast<const f32x2*>(s_chroma + (1 * 8 + crow) * CWP) + m * 4;
                    f32x2 cb2[4], cr2[4];
#pragma unroll
                    for (int k = 0; k < 4; k += 2) {
                        const ulonglong2 u = *reinterpret_cast<const ulonglong2*>(pcb + k), v = *reinterpret_cast<const ulonglong2*>(pcr + k);
                        cb2[k] = u.x; cb2[k + 1] = u.y; cr2[k] = v.x; cr2[k + 1] = v.y;
                    }
                    const f32x2 k1402 = pk2(1.402f, 1.402f), k1772 = pk2(1.772f, 1.772f);
                    const f32x2 kn0344 = pk2(-0.34413629f, -0.34413629f), kn0714 = pk2(-0.71413629f, -0.71413629f);
                    float ra[8], ga[8], ba[8], rb[8], gb[8], bb[8];
#pragma unroll
                    for (int x = 0; x < 8; x++) {   // decoder.rs:392-401, as in finish_luma
                        const f32x2 c_b = cb2[x / 2], c_r = cr2[x / 2];
                        upk2(fma2(c_r, k1402, y2[x]), ra[x], rb[x]);
                        upk2(fma2(c_b, k1772, y2[x]), ba[x], bb[x]);
                        upk2(fma2(c_b, kn0344, fma2(c_r, kn0714, y2[x])), ga[x], gb[x]);
                    }
                    stage_rgb(p, ra, ga, ba, false);
                    stage_rgb(p + 1, rb, gb, bb, false);
                }
            }
        } else {
#pragma unroll
            for (int p = 0; p < Y_PASSES; p++) {
                float y[8];
                block_idct(JPGPU_COEF(CH_PASSES + p), qt_l, t, scr_w, scr_r, 128.0f, y);
                finish_luma(p, y);
            }
        }
        __syncthreads();

        const uint32_t x0 = tx * 128u, y0 = ty * MH;
        const uint32_t wpx = min(128u, W - x0), rows = min((uint32_t)MH, H - y0);
        const uint32_t rowbytes = PLANAR ? wpx : wpx * 3u;
        uint8_t* const tile_out = PLANAR ? rgb + ((size_t)y0 * W + x0) * (F32 ? 4u : 1u) : rgb + ((size_t)y0 * W + x0) * 3u;
        if constexpr (F32) {
            // one float per staged byte: thread i converts 4 bytes of one row of one plane into one 16-byte store
            const uint32_t per_plane = rows * (wpx >> 2);
            const bool vec4 = (W & 3u) == 0u && (wpx & 3u) == 0u;
            for (uint32_t i = tid; vec4 && i < 3u * per_plane; i += kIdctThreads) {
                const uint32_t pl = i / per_plane, q = i - pl * per_plane, r = q / (wpx >> 2), k = q - r * (wpx >> 2);
                const uint32_t v = *reinterpret_cast<const uint32_t*>(s_out + pl * kPlaneSize + r * kPlanePitch + k * 4u);
                const float sc = b.out_scale[pl], bi = b.out_bias[pl];
                float4 f;
                f.x = fmaf((float)(v & 255u), sc, bi); f.y = fmaf((float)((v >> 8) & 255u), sc, bi);
                f.z = fmaf((float)((v >> 16) & 255u), sc, bi); f.w = fmaf((float)(v >> 24), sc, bi);
                *reinterpret_cast<float4*>(tile_out + ((size_t)pl * plane_bytes + (size_t)r * W + k * 4u) * 4u) = f;
            }
            for (uint32_t i = tid; !vec4 && i < 3u * rows * wpx; i += kIdctThreads) {
                const uint32_t pl = i / (rows * wpx), q = i - pl * rows * wpx, r = q / wpx, k = q - r * wpx;
                reinterpret_cast<float*>(tile_out)[(size_t)pl * plane_bytes + (size_t)r * W + k] =
                    fmaf((float)s_out[pl * kPlaneSize + r * kPlanePitch + k], b.out_scale[pl], b.out_bias[pl]);
            }
        } else if (vec_ok && (rowbytes & 15u) == 0u) {
            const uint32_t vpr = rowbytes >> 4;  // <= 24 (planar: <= 8)
#pragma unroll
            for (int n = 0; n < NV; n++) {
                const uint32_t r = co_rk[n] & 255u, k = co_rk[n] >> 8;
                if (r < rows && k < vpr) {
                    const uint4 v = *reinterpret_cast<const uint4*>(s_out + co_s[n]);
                    *reinterpret_cast<uint4*>(tile_out + co_g[n]) = v;
                }
            }
        } else if (PLANAR) {
            for (uint32_t i = tid; i < 3u * rows * rowbytes; i += kIdctThreads) {
                const uint32_t pl = i / (rows * rowbytes), q = i - pl * rows * rowbytes, r = q / rowbytes, k = q - r * rowbytes;
                tile_out[(size_t)pl * plane_bytes + (size_t)r * W + k] = s_out[pl * kPlaneSize + r * kPlanePitch + k];
            }
        } else {
            for (uint32_t i = tid; i < rows * rowbytes; i += kIdctThreads) {
                const uint32_t r = i / rowbytes, k = i - r * rowbytes;
                tile_out[(size_t)r * W * 3u + k] = s_out[r * kOutPitch + k];
            }
        }
        // s_out / s_chroma are rewritten only after the next tile's phase-A barrier (or, for gray,
        // after the barrier below) — every thread has left phase C by then.
        if (GRAY) __syncthreads();
        tx = ntx; ty = nty;
#if JPGPU_IDCT_TMA
        tma_k++;   // (all reads of this tile's buffer lie before the barrier that precedes the copy-out)
#else
#pragma unroll
        for (int l = 0; l < NL; l++) cur[l] = nxt[l];
#endif
    }
#undef JPGPU_COEF
}

// ============================================ gather path: REF placement / generic sampling
// Stage A: dequant + IDCT of every block of the image, f32 samples stored per block in
// arena order ([block][row*8+col]); luma (component 0) carries the +128 level shift.
__global__ void __launch_bounds__(kIdctThreads) block_idct_kernel(BatchDev b, const uint32_t* __restrict__ img_list) {
    __shared__ __align__(16) float s_scr[16 * kScrBlkPitch];
    const ImgDev& im = b.imgs[img_list[blockIdx.y]];
    const uint32_t nblk = im.units * im.blocks_per_mcu;
    const int tid = threadIdx.x, t = tid & 7, bp = tid >> 3;
    const uint32_t blk = blockIdx.x * 16u + bp;
    if (blockIdx.x * 16u >= nblk) return;
    const bool valid = blk < nblk;
    const uint32_t comp = valid ? im.blk_comp[blk % im.blocks_per_mcu] : 0u;
    const float* __restrict__ qt = b.qt + im.qt_off[comp] + t * 8;
    uint4 raw = make_uint4(0u, 0u, 0u, 0u);
    if (valid) raw = __ldg(reinterpret_cast<const uint4*>(b.coefs + im.coef_off) + (size_t)blk * 8 + t);
    float o[8];
    block_idct(raw, __ldg(reinterpret_cast<const float4*>(qt)), __ldg(reinterpret_cast<const float4*>(qt + 4)), t,
               s_scr + bp * kScrBlkPitch + t, s_scr + bp * kScrBlkPitch + t * kScrRowPitch, comp == 0u ? 128.0f : 0.0f, o);
    if (valid) {
        float4* dst = reinterpret_cast<float4*>(b.samples + im.smp_off + (size_t)blk * 64 + t * 8);
        dst[0] = make_float4(o[0], o[1], o[2], o[3]);
        dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
}

// Stage B: four pixels per thread. Per component the placement map names the sample the
// layout's last writer put at this pixel (decoder.rs:290-312, 347-379), or nothing: the
// reference's planes start as 0.0 (decoder.rs:253-256), i.e. 128 after the level shift for luma.
constexpr int kGatherThreads = 256;
__global__ void __launch_bounds__(kGatherThreads) gather_colour_kernel(BatchDev b, const uint32_t* __restrict__ img_list) {
    const ImgDev& im = b.imgs[img_list[blockIdx.y]];
    if (im.frame) return;   // its samples go through compose_colour_kernel
    const uint32_t npix = im.width * im.height;
    const uint32_t q = blockIdx.x * kGatherThreads + threadIdx.x;
    if (q * 4u >= npix) return;
    const uint32_t* __restrict__ map = b.gmap + im.map_off;
    const float* __restrict__ smp = b.samples + im.smp_off;
    const int ncomp = im.ncomp;
    float v[3][4];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const float none = c == 0 ? 128.0f : 0.0f;
        if (c < ncomp) {
            const uint4 m = __ldg(reinterpret_cast<const uint4*>(map + (size_t)c * im.map_plane) + q);
            v[c][0] = m.x == kMapNone ? none : __ldg(smp + m.x);
            v[c][1] = m.y == kMapNone ? none : __ldg(smp + m.y);
            v[c][2] = m.z == kMapNone ? none : __ldg(smp + m.z);
            v[c][3] = m.w == kMapNone ? none : __ldg(smp + m.w);
        } else {
            v[c][0] = v[c][1] = v[c][2] = v[c][3] = none;
        }
    }
    int32_t r8[4], g8[4], b8[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (ncomp == 1) {
            r8[k] = g8[k] = b8[k] = f32_to_u8_sat(v[0][k]);  // decoder.rs:317-324
        } else {
            const float y = v[0][k], cb = v[1][k], cr = v[2][k];  // decoder.rs:392-401, as in idct_colour_kernel
            r8[k] = f32_to_u8_sat(fmaf(cr, 1.402f, y));
            g8[k] = f32_to_u8_sat(fmaf(cb, -0.34413629f, fmaf(cr, -0.71413629f, y)));
            b8[k] = f32_to_u8_sat(fmaf(cb, 1.772f, y));
        }
    }
    if (b.out_planar == 2u) {   // f32 planes: u8 * scale + bias
        float* out = reinterpret_cast<float*>(b.rgb + im.rgb_off * 4u) + (size_t)q * 4u;
        for (uint32_t k = 0; k < 4u && q * 4u + k < npix; k++) {
            out[k] = fmaf((float)min(max(r8[k], 0), 255), b.out_scale[0], b.out_bias[0]);
            out[npix + k] = fmaf((float)min(max(g8[k], 0), 255), b.out_scale[1], b.out_bias[1]);
            out[2 * (size_t)npix + k] = fmaf((float)min(max(b8[k], 0), 255), b.out_scale[2], b.out_bias[2]);
        }
        return;
    }
    if (b.out_planar) {
        uint8_t* out = b.rgb + im.rgb_off + (size_t)q * 4u;
        if (q * 4u + 4u <= npix && (npix & 3u) == 0u) {
            *reinterpret_cast<uint32_t*>(out) = pack4(r8[0], r8[1], r8[2], r8[3]);
            *reinterpret_cast<uint32_t*>(out + npix) = pack4(g8[0], g8[1], g8[2], g8[3]);
            *reinterpret_cast<uint32_t*>(out + 2 * (size_t)npix) = pack4(b8[0], b8[1], b8[2], b8[3]);
        } else {
            for (uint32_t k = 0; k < 4u && q * 4u + k < npix; k++) {
                out[k] = (uint8_t)min(max(r8[k], 0), 255); out[npix + k] = (uint8_t)min(max(g8[k], 0), 255); out[2 * (size_t)npix + k] = (uint8_t)min(max(b8[k], 0), 255);
            }
        }
        return;
    }
    uint8_t* out = b.rgb + im.rgb_off + (size_t)q * 12u;
    if (q * 4u + 4u <= npix) {
        uint32_t* o32 = reinterpret_cast<uint32_t*>(out);
        o32[0] = pack4(r8[0], g8[0], b8[0], r8[1]);
        o32[1] = pack4(g8[1], b8[1], r8[2], g8[2]);
        o32[2] = pack4(b8[2], r8[3], g8[3], b8[3]);
    } else {
        for (uint32_t k = 0; q * 4u + k < npix; k++) {
            out[3 * k] = (uint8_t)min(max(r8[k], 0), 255); out[3 * k + 1] = (uint8_t)min(max(g8[k], 0), 255); out[3 * k + 2] = (uint8_t)min(max(b8[k], 0), 255);
        }
    }
}

// Compose path, stage B: four horizontally adjacent pixels of one frame per thread, put together plane by plane from
// the per-block samples of block_idct_kernel.  Sub-sampled components are either replicated (the reference's
// fill_block_in_array, decoder.rs:347-379) or interpolated with libjpeg's "fancy" triangle filter: 3/4 of the nearer and
// 1/4 of the farther sample per direction (jdsample.c h2v1 / h2v2 fancy up-sampling without its integer rounding), the
// neighbour clamped at the component's edges.  Colour conversion, truncation and clamp as everywhere else
// (decoder.rs:382-402).  Not the tuned path: one scalar load per sample.
__device__ __forceinline__ float plane_sample(const float* __restrict__ smp, const PlaneRef& p, int xs, int ys) {
    xs = min(max(xs, 0), (int)p.wc - 1);
    ys = min(max(ys, 0), (int)p.hc - 1);
    const uint32_t bx = (uint32_t)xs >> 3, by = (uint32_t)ys >> 3;
    const uint32_t blk = ((by / p.v) * p.mcux + bx / p.h) * p.bpm + p.first + (by % p.v) * p.h + bx % p.h;
    return __ldg(smp + p.smp_off + (size_t)blk * 64 + ((uint32_t)ys & 7u) * 8u + ((uint32_t)xs & 7u)) + p.bias;
}
__device__ __forceinline__ float frame_sample(const float* __restrict__ smp, const PlaneRef& p, bool fancy, int x, int y) {
    if (p.fx == 1u && p.fy == 1u) return plane_sample(smp, p, x, y);
    const int xs = p.fx == 2u ? x >> 1 : x, ys = p.fy == 2u ? y >> 1 : y;
    if (!fancy) return plane_sample(smp, p, xs, ys);
    const int xn = p.fx == 2u ? xs + ((x & 1) ? 1 : -1) : xs, yn = p.fy == 2u ? ys + ((y & 1) ? 1 : -1) : ys;
    float a = plane_sample(smp, p, xs, ys), c = plane_sample(smp, p, xn, ys);
    if (p.fy == 2u) {   // vertical first, as libjpeg's h2v2 ("thiscolsum")
        a = 0.75f * a + 0.25f * plane_sample(smp, p, xs, yn);
        c = 0.75f * c + 0.25f * plane_sample(smp, p, xn, yn);
    }
    return p.fx == 2u ? 0.75f * a + 0.25f * c : a;
}
__global__ void __launch_bounds__(kGatherThreads) compose_colour_kernel(BatchDev b, uint32_t frame0) {
    const FrameDev& f = b.frames[frame0 + blockIdx.y];
    for (uint32_t c = 0; c < f.ncomp && c < 3u; c++)
        if (f.pl[c].h == 0u || f.pl[c].wc == 0u) return;   // a scan of the frame failed to plan: no pixels (its status says why)
    const uint32_t W = f.width, npix = W * f.height;
    const uint32_t q = blockIdx.x * kGatherThreads + threadIdx.x;
    if (q * 4u >= npix) return;
    const float* __restrict__ smp = b.samples;
    const size_t sb = b.out_planar == 2u ? 4u : 1u;
    uint8_t* const base = b.rgb + f.rgb_off * sb;
    for (uint32_t k = 0; k < 4u && q * 4u + k < npix; k++) {
        const uint32_t i = q * 4u + k;
        const int x = (int)(i % W), y = (int)(i / W);
        int32_t r8, g8, b8;
        const float yy = frame_sample(smp, f.pl[0], f.fancy != 0u, x, y);
        if (f.ncomp == 1u) {
            r8 = g8 = b8 = f32_to_u8_sat(yy);
        } else {
            const float cb = frame_sample(smp, f.pl[1], f.fancy != 0u, x, y), cr = frame_sample(smp, f.pl[2], f.fancy != 0u, x, y);
            r8 = f32_to_u8_sat(fmaf(cr, 1.402f, yy));
            g8 = f32_to_u8_sat(fmaf(cb, -0.34413629f, fmaf(cr, -0.71413629f, yy)));
            b8 = f32_to_u8_sat(fmaf(cb, 1.772f, yy));
        }
        r8 = min(max(r8, 0), 255); g8 = min(max(g8, 0), 255); b8 = min(max(b8, 0), 255);
        if (b.out_planar == 2u) {
            float* o = reinterpret_cast<float*>(base);
            o[i] = fmaf((float)r8, b.out_scale[0], b.out_bias[0]);
            o[npix + i] = fmaf((float)g8, b.out_scale[1], b.out_bias[1]);
            o[2 * (size_t)npix + i] = fmaf((float)b8, b.out_scale[2], b.out_bias[2]);
        } else if (b.out_planar) {
            base[i] = (uint8_t)r8; base[npix + i] = (uint8_t)g8; base[2 * (size_t)npix + i] = (uint8_t)b8;
        } else {
            base[3 * (size_t)i] = (uint8_t)r8; base[3 * (size_t)i + 1] = (uint8_t)g8; base[3 * (size_t)i + 2] = (uint8_t)b8;
        }
    }
}

// ===================================================================== launchers
// Kernels that take the image from blockIdx.y are launched in slices of at most kMaxGridY images (grid.y <= 65535).
constexpr uint32_t kMaxGridY = 65535;
template <class F>
static void for_image_slices(const BatchDev& b, F&& launch) {
    for (uint32_t i0 = 0; i0 < b.n_images; i0 += kMaxGridY) {
        BatchDev d = b;
        d.img0 = b.img0 + i0;
        d.n_images = min(kMaxGridY, b.n_images - i0);
        launch(d);
    }
}
void launch_prepass_step(const BatchDev& b, cudaStream_t s, int step) {
    if (!b.n_images || !b.max_chunks) return;
    if (step == 1) { prepass_scan_kernel<<<b.n_images, kPreThreads, 0, s>>>(b); return; }
    for_image_slices(b, [&](const BatchDev& d) {
        if (step == 0) prepass_count_kernel<<<dim3((d.max_chunks + kCountChunks - 1) / kCountChunks, d.n_images), kPreThreads, 0, s>>>(d);
        else prepass_write_kernel<<<dim3(d.max_chunks, d.n_images), kPreThreads, 0, s>>>(d);
    });
}
void launch_zero_output_pads(const BatchDev& b, cudaStream_t s) {
    if (b.n_images && b.rgb) zero_output_pads_kernel<<<(b.n_images + 255u) / 256u, 256, 0, s>>>(b);
}
void launch_gather_scans(const BatchDev& b, const void* base, const uint64_t* dev_offs, cudaStream_t s) {
    if (!b.n_images || !b.max_chunks) return;
    for_image_slices(b, [&](const BatchDev& d) {
        gather_scans_kernel<<<dim3(d.max_chunks, d.n_images), kPreThreads, 0, s>>>(d, static_cast<const uint8_t*>(base), dev_offs);
    });
}
void launch_prepass(const BatchDev& b, cudaStream_t s) {
    for (int step = 0; step < 3; step++) launch_prepass_step(b, s, step);
}
// Opt-in dynamic shared memory is a per-device attribute of a kernel: set once per device (contexts of several devices
// launch from several host threads, hence the lock).
template <class K>
static cudaError_t ensure_smem_attr(K kernel, uint32_t bytes, uint64_t& configured, std::mutex& mu) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    if (dev < 0 || dev >= 64 || !(configured >> dev & 1u)) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured |= 1ull << dev;
    }
    return cudaSuccess;
}
cudaError_t launch_sync(const BatchDev& b, cudaStream_t s) {
    if (!b.n_seqs || !b.nsync) return cudaSuccess;
    if (!b.sync_multi) {
        sync_kernel<<<b.n_seqs / kJobsPerCta, kSeqThreads, 0, s>>>(b);
        return cudaSuccess;
    }
    static std::mutex mu;
    static uint64_t configured = 0;
    // the largest layout: every slot an AC table
    const cudaError_t e = ensure_smem_attr(sync_multi_kernel, sync_layout(kMaxLutSlots, kMaxLutSlots << kMultiBitsAc).total, configured, mu);
    if (e != cudaSuccess) return e;
    sync_multi_kernel<<<(b.n_seqs + kSyncJobs - 1) / kSyncJobs, kSyncThreads, sync_layout(b.max_slots, b.max_mlut_words).total, s>>>(b);
    return cudaSuccess;
}
cudaError_t launch_verify_scan(const BatchDev& b, cudaStream_t s) {
    if (!b.n_images || !b.nsync) return cudaSuccess;
    if (!b.verify_multi) {
        verify_scan_kernel<false><<<b.n_images, kInterThreads, 0, s>>>(b);
        return cudaSuccess;
    }
    static std::mutex mu;
    static uint64_t configured = 0;
    const cudaError_t e = ensure_smem_attr(verify_scan_kernel<true>, 128u + ((uint32_t)kMaxLutSlots << kMultiBitsAc) * 4u, configured, mu);
    if (e != cudaSuccess) return e;
    verify_scan_kernel<true><<<b.n_images, kInterThreads, 128u + b.max_mlut_words * 4u, s>>>(b);
    return cudaSuccess;
}
template <int NBUF, int PHASE>
static cudaError_t launch_write_variant(const BatchDev& b, cudaStream_t s) {
    const WriteLayout lay = write_layout(b.max_slots, NBUF);
    static std::mutex mu;
    static uint64_t configured = 0;   // bit d: device d is set up (for the largest layout)
    const cudaError_t e = ensure_smem_attr(decode_write_kernel<NBUF, PHASE>, write_layout(kMaxLutSlots, NBUF).total, configured, mu);
    if (e != cudaSuccess) return e;
    const uint32_t jobs = b.n_seqs << b.wp_shift;   // n_seqs is a multiple of kWriteJobsPerCta (build_plan)
    decode_write_kernel<NBUF, PHASE><<<(jobs + kWriteJobsPerCta - 1) / kWriteJobsPerCta, kWriteThreads, lay.total, s>>>(b);
    return cudaSuccess;
}
cudaError_t launch_decode_write(const BatchDev& b, cudaStream_t s) {
    if (!b.n_seqs) return cudaSuccess;
    // one block buffer per lane and 5-symbol phases measured best on B200 (2 buffers / 8-12 symbols: fewer flushes, but
    // half the resident warps); see DESIGN.md 4.2
    const cudaError_t e = launch_write_variant<kWriteBufs, kPhaseSymbols>(b, s);
    if (e != cudaSuccess) return e;
    if (b.n_images) zero_tail_kernel<<<b.n_images, 256, 0, s>>>(b);   // blocks a damaged scan never reached
    return cudaSuccess;
}

int launch_idct_colour(const BatchDev& b, cudaStream_t s) {
    int launches = 0;
    for (int k = 0; k < kNumKinds; k++) {
        if (!b.kind_count[k] || !b.kind_max_tiles[k]) continue;
        for (uint32_t i0 = 0; i0 < b.kind_count[k]; i0 += kMaxGridY) {
            const dim3 grid((b.kind_max_tiles[k] + kTilesPerCta - 1) / kTilesPerCta, min(kMaxGridY, b.kind_count[k] - i0));
            const uint32_t* list = b.kind_imgs[k] + i0;
#define JPGPU_LAUNCH_IDCT(HY, VY, GRAY)                                                                 \
    do {                                                                                               \
        if (b.out_planar == 2u) idct_colour_kernel<HY, VY, GRAY, 2><<<grid, kIdctThreads, 0, s>>>(b, list);   \
        else if (b.out_planar) idct_colour_kernel<HY, VY, GRAY, 1><<<grid, kIdctThreads, 0, s>>>(b, list);    \
        else idct_colour_kernel<HY, VY, GRAY, 0><<<grid, kIdctThreads, 0, s>>>(b, list);                      \
    } while (0)
            switch (k) {
                case kKindGray: JPGPU_LAUNCH_IDCT(1, 1, true); break;
                case kKind444: JPGPU_LAUNCH_IDCT(1, 1, false); break;
                case kKind422: JPGPU_LAUNCH_IDCT(2, 1, false); break;
                case kKind420: JPGPU_LAUNCH_IDCT(2, 2, false); break;
                case kKind440: JPGPU_LAUNCH_IDCT(1, 2, false); break;
                default: continue;
            }
#undef JPGPU_LAUNCH_IDCT
            launches++;
        }
    }
    if (b.gather_max_blocks) {
        for (uint32_t i0 = 0; i0 < b.kind_count[kKindGeneric]; i0 += kMaxGridY) {
            const uint32_t cnt = min(kMaxGridY, b.kind_count[kKindGeneric] - i0);
            const uint32_t* list = b.kind_imgs[kKindGeneric] + i0;
            block_idct_kernel<<<dim3((b.gather_max_blocks + 15) / 16, cnt), kIdctThreads, 0, s>>>(b, list);
            launches++;
            if (!b.gather_max_quads) continue;   // compose-path images only: their pixels come from compose_colour_kernel
            gather_colour_kernel<<<dim3((b.gather_max_quads + kGatherThreads - 1) / kGatherThreads, cnt), kGatherThreads, 0, s>>>(b, list);
            launches++;
        }
    }
    if (b.n_frames && b.frame_max_quads) {   // compose path (after block_idct_kernel above produced the samples)
        for (uint32_t i0 = 0; i0 < b.n_frames; i0 += kMaxGridY) {
            compose_colour_kernel<<<dim3((b.frame_max_quads + kGatherThreads - 1) / kGatherThreads, min(kMaxGridY, b.n_frames - i0)), kGatherThreads, 0, s>>>(b, i0);
            launches++;
        }
    }
    return launches;
}

}  // namespace jpgpu
