// jpsim.cpp — CPU SIMULATION of the CUDA kernels' algorithm.  TEST INFRASTRUCTURE ONLY.
//
// It executes the same per-thread code (jpgpu_core.h: decode_span, init_state, idct8,
// ...) and the same host planner (jpgpu_host.cpp) as the product, with the kernels'
// thread/round/barrier structure replayed serially.  It lets the not-gpu test suite
// check the self-synchronising decode, the scan, the coefficient layout and the fused
// IDCT/colour arithmetic against the oracle on a box without a GPU.  It is NOT a
// fallback: nothing in jpeg_rust_b200/ or libjpgpu.so can reach it.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../jpeg_rust_b200/csrc/jpgpu_host.h"

using namespace jpgpu;

namespace {

struct SimBatch {
    HostPlan plan;
    std::vector<uint8_t> raw;
    std::vector<uint32_t> stream;
    std::vector<uint32_t> segtab;
    std::vector<SubInfo> subs;
    std::vector<SegRec> segs;
    std::vector<ImgDyn> dyn;
    std::vector<int16_t> coefs;
    std::vector<uint8_t> rgb;
    std::vector<float> samples;    // per-block IDCT samples of the compose-path images
    uint8_t store_pos[64];
    // diagnostics
    uint32_t repair_iters = 0;     // most repair iterations any image needed
    uint64_t repairs = 0;          // subsequences decoded again because the look-back had not synchronised
    uint64_t max_broken = 0;       // most broken links one repair round of one image found
    uint64_t crowded_rounds = 0;   // repair rounds that found more broken links than one round takes (256)
    uint64_t sync_decodes = 0;     // subsequences decoded by the sync pass
    uint64_t flush_phases = 0, flushed_blocks = 0;
    uint64_t sync_digest = 0;      // hash of the records the synchronisation pass wrote (SubInfo + SegRec)
};

// mirrors prepass_kernel's per-byte rule (the warp/CTA scan itself is GPU plumbing)
void sim_prepass(SimBatch& sb, size_t img) {
    const ImgDev& im = sb.plan.imgs[img];
    const uint8_t* in = sb.raw.data() + im.raw_off;
    const uint32_t n = im.raw_len;
    const uint32_t lw = sb.plan.lw;
    uint32_t* out = sb.stream.data() + im.stream_off;
    uint32_t* seg = sb.segtab.data() + im.seg_off;
    const bool dri = im.restart_interval != 0;
    uint32_t emitted = 0, rst_total = 0, status = 0;
    std::vector<uint8_t> bytes;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t cur = in[i], p = i ? in[i - 1] : 0, nxt = i + 1 < n ? in[i + 1] : 0;
        const bool has_next = i + 1 < n;
        bool drop = (cur == 0 && p == 0xff);
        bool r1 = false;
        if (dri) {
            r1 = cur == 0xff && has_next && (nxt & 0xf8) == 0xd0;
            const bool r2 = p == 0xff && (cur & 0xf8) == 0xd0;
            const bool fill = cur == 0xff && has_next && nxt == 0xff;
            drop = drop || r1 || r2 || fill;
        }
        if (r1) {
            if (rst_total + 1 < im.nseg_cap) seg[rst_total + 1] = emitted * 8;
            if ((nxt & 7) != (rst_total & 7)) status |= kStRestart;
            rst_total++;
        }
        if (!drop) { bytes.push_back((uint8_t)cur); emitted++; }
    }
    const uint32_t nwords = (emitted + 3) >> 2;
    for (uint32_t w = 0; w < nwords; w++) {
        uint32_t v = 0;
        for (uint32_t k = 0; k < 4; k++)
            if (w * 4 + k < emitted) v |= (uint32_t)bytes[w * 4 + k] << (24 - 8 * k);
        out[stream_phys(w, lw)] = v;
    }
    for (int i = 0; i < kStreamPadWords; i++) out[stream_phys(nwords + i, lw)] = 0;
    uint32_t nseg = rst_total + 1;
    if (nseg != im.nseg_cap && dri) status |= kStRestart;
    if (nseg > im.nseg_cap) nseg = im.nseg_cap;
    seg[0] = 0;
    seg[nseg] = emitted * 8;
    sb.dyn[img] = ImgDyn{emitted * 8, nseg, status, 0};
}

bool g_sync_multi = true;   // jpsim_set_sync_multi(): the synchronisation pass goes through the multi-symbol tables

DecCtx make_ctx(const SimBatch& sb, size_t img, const HuffLut* slots) {
    const ImgDev& im = sb.plan.imgs[img];
    DecCtx cx;
    cx.words = sb.stream.data() + im.stream_off;
    cx.lw = sb.plan.lw;
    cx.seg = sb.segtab.data() + im.seg_off;
    cx.nseg = sb.dyn[img].nseg;
    cx.stream_bits = sb.dyn[img].stream_bits;
    cx.seg_units = im.seg_units;
    cx.nblk = im.blocks_per_mcu;
    cx.luts = slots;
    cx.blk_info = im.blk_info;
    cx.mluts = nullptr;
    return cx;
}

void load_slots(const SimBatch& sb, size_t img, std::vector<HuffLut>& slots) {
    const ImgDev& im = sb.plan.imgs[img];
    slots.resize(kMaxLutSlots);
    for (int s = 0; s < im.nslots; s++) slots[s] = sb.plan.luts[im.slot_lut[s]];
}

// mirrors sync_kernel: one independent thread per subsequence
void sim_sync(SimBatch& sb, const SeqDesc& sd) {
    if (sd.img == kNoImage) return;
    std::vector<HuffLut> slots;
    load_slots(sb, sd.img, slots);
    const ImgDev& im = sb.plan.imgs[sd.img];
    if (im.interval_mode) return;
    const ImgDyn dyn = sb.dyn[sd.img];
    const uint32_t S = sb.plan.sub_bits, L = sb.plan.lookback_bits;
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    if (sd.first_sub >= nsub) return;
    DecCtx cx = make_ctx(sb, sd.img, slots.data());
    const uint32_t* mslots[kMaxLutSlots] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int s = 0; s < im.nslots; s++) mslots[s] = sb.plan.mluts.data() + sb.plan.mlut_off[im.slot_lut[s]];
    if (g_sync_multi) cx.mluts = mslots;   // sync_multi_kernel
    for (uint32_t tid = 0; tid < 32u; tid++) {  // one warp job
        const uint32_t j = sd.first_sub + tid;
        if (j >= nsub) continue;
        const uint32_t own = j * S, p0 = own > L ? own - L : 0u;
        DecState st;
        init_state(cx, st, p0, 0, 0, 0, 0, 0);
        while (st.p < own) {
            if (cx.mluts && st.p + 32u <= own && st.p + 39u <= st.seg_end) { multi_symbol(cx, st); continue; }
            if (decode_symbol<false>(cx, st, nullptr, 0u, nullptr, false) & kEvEnd) break;
        }
        SubInfo rec;
        rec.pA = st.p;
        rec.cz = pack_cz(st);
        const uint32_t C = sb.plan.seg_bits;
        sync_subsequence(cx, st, own, S, C, sb.segs.data() + (size_t)(im.sub_off + j) * (S / C), false, rec);
        sb.subs[im.sub_off + j] = rec;
        sb.sync_decodes++;
    }
}

// mirrors verify_scan_kernel: a round takes the lowest 256 broken links (kRepairJobs), the sweep starting at the
// previous round's lowest one.  Within a round the order of the repairs does not matter: every repair starts from a
// snapshot of its predecessor taken before any of them writes, and writes only its own subsequence's records.
void sim_verify_scan(SimBatch& sb, size_t img) {
    std::vector<HuffLut> slots;
    load_slots(sb, img, slots);
    const ImgDev& im = sb.plan.imgs[img];
    if (im.interval_mode) return;
    const ImgDyn dyn = sb.dyn[img];
    const uint32_t S = sb.plan.sub_bits, C = sb.plan.seg_bits;
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    DecCtx cx = make_ctx(sb, img, slots.data());
    const uint32_t* mslots[kMaxLutSlots] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int s = 0; s < im.nslots; s++) mslots[s] = sb.plan.mluts.data() + sb.plan.mlut_off[im.slot_lut[s]];
    if (g_sync_multi) cx.mluts = mslots;   // verify_scan_kernel<true>: the repair walks use the multi-symbol tables too
    SubInfo* subs = sb.subs.data() + im.sub_off;
    uint32_t iters = 0, from = 1;
    for (uint32_t iter = 0; iter <= nsub; iter++) {
        std::vector<RepairJob> jobs;
        for (uint32_t j = from; j < nsub; j++) {   // all of them, for the diagnostics; the kernel stops at 256
            const uint32_t start_p = subs[j - 1].pB, start_cz = (subs[j - 1].cz >> 10) & kCzMask;
            if (start_p != subs[j].pA || start_cz != (subs[j].cz & kCzMask)) jobs.push_back(RepairJob{j, start_p, start_cz});
        }
        sb.max_broken = std::max<uint64_t>(sb.max_broken, jobs.size());
        if (jobs.size() > 256) sb.crowded_rounds++;
        if (jobs.size() > 256) jobs.resize(256);  // kRepairJobs
        if (jobs.empty()) break;
        from = jobs[0].sub;
        for (const RepairJob& job : jobs) {
            DecState st;
            init_state(cx, st, job.p, (int32_t)(job.cz & 63u), (int32_t)(job.cz >> 6), 0, 0, 0);
            SubInfo rec;
            rec.pA = st.p;
            rec.cz = job.cz;
            sync_subsequence(cx, st, job.sub * S, S, C, sb.segs.data() + (size_t)(im.sub_off + job.sub) * (S / C), true, rec);
            subs[job.sub] = rec;
            sb.repairs++;
        }
        iters++;
    }
    sb.repair_iters = std::max(sb.repair_iters, iters);
    // exclusive scan (serial form of the chunked scan)
    int32_t run[4] = {0, 0, 0, 0};
    for (uint32_t jj = 0; jj < nsub; jj++) {
        SubInfo& s = subs[jj];
        const int32_t at_a[4] = {run[0], run[1], run[2], run[3]};
        uint32_t dummy = 0;
        fold_advance(run, dummy, s.cz, s.n, s.dc);
        s.n = at_a[0]; s.dc[0] = at_a[1]; s.dc[1] = at_a[2]; s.dc[2] = at_a[3];
    }
}

// mirrors decode_write_kernel: warps in lock-step phases, per-lane swizzled block buffers, cooperative flush
// one warp job of the write kernel: units group*32 .. group*32+31 of sequence sd (a unit = sub_bits >> wp_shift bits)
void sim_decode_write(SimBatch& sb, const SeqDesc& sd, uint32_t group) {
    if (sd.img == kNoImage) return;
    std::vector<HuffLut> slots;
    load_slots(sb, sd.img, slots);
    const ImgDev& im = sb.plan.imgs[sd.img];
    const ImgDyn dyn = sb.dyn[sd.img];
    const uint32_t S = sb.plan.sub_bits;
    const uint32_t nsub = (dyn.stream_bits + S - 1) / S;
    if (sd.first_sub >= nsub) return;
    const uint32_t hs = sb.plan.wp_shift, H = 1u << hs, C = sb.plan.seg_bits, nsegs = S / C;
    const DecCtx cx = make_ctx(sb, sd.img, slots.data());
    const int32_t total = (int32_t)im.total_coefs;
    int16_t* coefs = sb.coefs.data() + im.coef_off;
    std::vector<int16_t> bufs((size_t)32 * kWriteBufs * 64, 0);
    for (uint32_t warp = 0; warp < 1u; warp++) {  // one warp job
        struct Lane { DecState st; bool active, store_on, valid; uint32_t j, unit_bit, end_bit, cur, ndone, dest[kWriteBufs]; int32_t g_start, seg_limit; };
        Lane ln[32];
        bool any_active = false;
        for (uint32_t lane = 0; lane < 32; lane++) {
            Lane& l = ln[lane];
            const uint32_t unit = group * 32 + lane, part = unit & (H - 1u);
            l.j = sd.first_sub + (unit >> hs);
            l.unit_bit = l.j * S + part * (S >> hs);
            l.end_bit = l.unit_bit + (S >> hs);
            l.valid = l.active = l.j < nsub && l.unit_bit < dyn.stream_bits;
            l.cur = l.ndone = 0;
            l.store_on = true;
            l.st.p = 0; l.st.g = 0; l.st.flags = 0;
            uint32_t k0 = 0;
            if (l.active && im.interval_mode) {   // the lane owns the restart intervals that start inside its subsequence
                k0 = first_interval_from(cx.seg, cx.nseg, l.unit_bit);
                l.active = k0 < cx.nseg && cx.seg[k0] < l.end_bit;
            }
            if (l.active) {
                if (im.interval_mode) {
                    init_state(cx, l.st, cx.seg[k0], (int32_t)(k0 * cx.seg_units), 0, 0, 0, 0);
                } else {
                    const SubInfo me = sb.subs[im.sub_off + l.j];   // state at A, carried over the segments before the unit
                    uint32_t p0 = me.pA, cz0 = me.cz & kCzMask, crossed = 0;
                    int32_t acc[4] = {me.n, me.dc[0], me.dc[1], me.dc[2]};
                    const SegRec* sg = sb.segs.data() + (size_t)(im.sub_off + l.j) * nsegs;
                    for (uint32_t k = 0; k < part * (nsegs >> hs); k++) {
                        fold_advance(acc, crossed, sg[k].cz, sg[k].n, sg[k].dc);
                        p0 = sg[k].p; cz0 = sg[k].cz & kCzMask;
                    }
                    init_state(cx, l.st, p0, acc[0], (int32_t)((cz0 >> 6) & 15u), acc[1], acc[2], acc[3]);
                }
                l.st.flags &= ~kCrossed;
                l.seg_limit = cx.seg_units ? std::min(total, (int32_t)((l.st.seg + 1u) * cx.seg_units)) : total;
                l.store_on = (l.st.g & 63) == 0 && l.st.g < l.seg_limit;
                if (l.st.g >= total || (l.st.p >= l.end_bit && (l.st.g & 63) == 0)) l.active = false;
            }
            l.g_start = l.st.g;
            any_active = any_active || l.active;
        }
        if (!any_active) {
            bool any_j = false;
            for (auto& l : ln) any_j = any_j || l.valid;
            if (!any_j) continue;
        }
        while (true) {
            for (uint32_t lane = 0; lane < 32; lane++) {
                Lane& l = ln[lane];
                const uint32_t row0 = (warp * 32 + lane) * kWriteBufs;
                for (int k = 0; k < kPhaseSymbols && l.active && l.ndone < (uint32_t)kWriteBufs; k++) {
                    if ((!im.interval_mode && l.st.p >= l.end_bit && (l.st.g & 63) == 0) || l.st.g >= total) { l.active = false; break; }
                    const uint32_t row = row0 + l.cur;
                    const int32_t g_before = l.st.g;
                    const uint32_t ev = decode_symbol<true>(cx, l.st, bufs.data() + (size_t)row * 64, row & 7u, sb.store_pos, l.store_on);
                    if (ev & kEvBlock) {
                        if (l.store_on) { l.dest[l.ndone++] = (uint32_t)(g_before >> 6); l.cur = l.cur + 1 == (uint32_t)kWriteBufs ? 0u : l.cur + 1; }
                        l.store_on = l.st.g < l.seg_limit;
                    } else if (ev & kEvCross) {
                        const int32_t old_limit = l.seg_limit, gap_from = g_before & ~63;
                        l.seg_limit = std::min(total, l.st.g + (int32_t)cx.seg_units);
                        if (g_before != old_limit) l.st.flags |= kStRestart;
                        if ((g_before & 63) != 0 && l.store_on) { l.dest[l.ndone++] = 0xffffffffu; l.cur = l.cur + 1 == (uint32_t)kWriteBufs ? 0u : l.cur + 1; }
                        for (int32_t g = gap_from; g < old_limit && g < l.st.g; g += 64)
                            for (int e = 0; e < 64; e++) coefs[(size_t)g + e] = 0;
                        l.store_on = true;
                        if (im.interval_mode && l.st.p >= l.end_bit) l.active = false;   // the next interval is another lane's
                    } else if (ev & kEvEnd) {
                        l.active = false;
                    }
                }
            }
            uint32_t count = 0;
            bool act = false;
            for (auto& l : ln) { count += l.ndone; act = act || l.active; }
            if (count == 0) { if (!act) break; continue; }
            for (uint32_t lane = 0; lane < 32; lane++) {
                Lane& l = ln[lane];
                const uint32_t row0 = (warp * 32 + lane) * kWriteBufs;
                uint32_t r = l.cur + kWriteBufs - l.ndone;
                for (uint32_t i = 0; i < l.ndone; i++, r++) {
                    if (r >= (uint32_t)kWriteBufs) r -= kWriteBufs;
                    const uint32_t row = row0 + r;
                    int16_t* src = bufs.data() + (size_t)row * 64;
                    for (uint32_t piece = 0; piece < 8; piece++)
                        for (int e = 0; e < 8; e++) {
                            int16_t& v = src[((piece ^ (row & 7u)) << 3) + e];
                            if (l.dest[i] != 0xffffffffu) coefs[(size_t)l.dest[i] * 64 + piece * 8 + e] = v;
                            v = 0;
                        }
                    sb.flushed_blocks++;
                }
                l.ndone = 0;
            }
            sb.flush_phases++;
        }
        for (auto& l : ln) {
            if (!l.valid) continue;
            uint32_t bits = l.st.flags & (kStBadCode | kStDcSize | kStRestart);
            if (l.g_start < total && l.st.g >= total) { sb.dyn[sd.img].bits_consumed = l.st.p; bits |= kStDone; }
            sb.dyn[sd.img].status |= bits;
            if (l.g_start < total && l.st.g < total && l.st.p >= dyn.stream_bits)
                sb.dyn[sd.img].coef_end = std::max(sb.dyn[sd.img].coef_end, (uint32_t)l.st.g & ~63u);
        }
    }
}

inline uint8_t sat_u8_trunc(float x) {  // cvt.rzi.sat.u8.f32
    if (!(x > 0.0f)) return 0;
    if (x >= 255.0f) return 255;
    return (uint8_t)x;
}

// the arithmetic of block_idct (vertical pass on columns, horizontal pass on rows)
void sim_block_idct(const int16_t* src, bool valid, const float* qt, float dc_bias, float out[64]) {
    float tmp[64];
    for (int t = 0; t < 8; t++) {
        float f[8];
        for (int v = 0; v < 8; v++) f[v] = valid ? (float)src[t * 8 + v] * qt[t * 8 + v] : 0.0f;
        if (t == 0) f[0] += dc_bias;
        idct8(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7]);
        for (int y = 0; y < 8; y++) tmp[y * 8 + t] = f[y];
    }
    for (int t = 0; t < 8; t++) {
        float* r = tmp + t * 8;
        idct8(r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]);
        for (int x = 0; x < 8; x++) out[t * 8 + x] = r[x];
    }
}

// mirrors idct_colour_kernel (any HY, VY in {1,2}; gray)
void sim_idct_colour(SimBatch& sb, size_t img) {
    const ImgDev& im = sb.plan.imgs[img];
    const bool gray = im.kind == kKindGray;
    const int HY = gray ? 1 : im.h[0], VY = gray ? 1 : im.v[0];
    const int NY = HY * VY, NB = gray ? 1 : NY + 2;
    const int16_t* coefs = sb.coefs.data() + im.coef_off;
    uint8_t* rgb = sb.rgb.data() + im.rgb_off;
    const float* qt = sb.plan.qt.data();
    const uint32_t W = im.width, H = im.height;
    const uint32_t blk_limit = coef_block_limit(sb.dyn[img]);
    for (uint32_t my = 0; my < im.mcuy; my++)
        for (uint32_t mx = 0; mx < im.mcux; mx++) {
            const uint32_t mcu = my * im.mcux + mx;
            const bool valid = mcu < im.units;
            auto ok = [&](uint32_t blk) { return valid && blk < blk_limit; };
            float cb[64], cr[64];
            if (!gray) {
                sim_block_idct(coefs + ((size_t)mcu * NB + NY) * 64, ok(mcu * NB + NY), qt + im.qt_off[1], 0.0f, cb);
                sim_block_idct(coefs + ((size_t)mcu * NB + NY + 1) * 64, ok(mcu * NB + NY + 1), qt + im.qt_off[2], 0.0f, cr);
            }
            for (int sub = 0; sub < NY; sub++) {
                const int by = sub / HY, bx = sub % HY;
                float y[64];
                sim_block_idct(coefs + ((size_t)mcu * NB + sub) * 64, ok(mcu * NB + sub), qt + im.qt_off[0], 128.0f, y);
                for (int t = 0; t < 8; t++)
                    for (int x = 0; x < 8; x++) {
                        const uint32_t px = (mx * HY + bx) * 8 + x, py = (my * VY + by) * 8 + t;
                        if (px >= W || py >= H) continue;
                        uint8_t* o = rgb + ((size_t)py * W + px) * 3;
                        if (gray) {
                            o[0] = o[1] = o[2] = sat_u8_trunc(y[t * 8 + x]);
                        } else {
                            const int crow = (by * 8 + t) / VY, ccol = (bx * 8 + x) / HY;
                            const float cbv = cb[crow * 8 + ccol], crv = cr[crow * 8 + ccol], yy = y[t * 8 + x];
                            o[0] = sat_u8_trunc(fmaf(crv, 1.402f, yy));
                            o[1] = sat_u8_trunc(fmaf(cbv, -0.34413629f, fmaf(crv, -0.71413629f, yy)));
                            o[2] = sat_u8_trunc(fmaf(cbv, 1.772f, yy));
                        }
                    }
            }
        }
}

// mirrors block_idct_kernel for an image of the compose path: per-block samples into the shared sample arena
void sim_block_idct_all(SimBatch& sb, size_t img) {
    const ImgDev& im = sb.plan.imgs[img];
    const uint32_t nblk = im.units * im.blocks_per_mcu;
    const int16_t* coefs = sb.coefs.data() + im.coef_off;
    const float* qt = sb.plan.qt.data();
    for (uint32_t blk = 0; blk < nblk; blk++) {
        const int comp = im.blk_comp[blk % im.blocks_per_mcu];
        sim_block_idct(coefs + (size_t)blk * 64, blk < coef_block_limit(sb.dyn[img]), qt + im.qt_off[comp], comp == 0 ? 128.0f : 0.0f,
                       sb.samples.data() + im.smp_off + (size_t)blk * 64);
    }
}

// mirror compose_colour_kernel (plane_sample / frame_sample: same clamping, same weights, same operation order)
float sim_plane_sample(const SimBatch& sb, const PlaneRef& p, int xs, int ys) {
    xs = std::min(std::max(xs, 0), (int)p.wc - 1);
    ys = std::min(std::max(ys, 0), (int)p.hc - 1);
    const uint32_t bx = (uint32_t)xs >> 3, by = (uint32_t)ys >> 3;
    const uint32_t blk = ((by / p.v) * p.mcux + bx / p.h) * p.bpm + p.first + (by % p.v) * p.h + bx % p.h;
    return sb.samples[p.smp_off + (size_t)blk * 64 + ((uint32_t)ys & 7u) * 8u + ((uint32_t)xs & 7u)] + p.bias;
}
float sim_frame_sample(const SimBatch& sb, const PlaneRef& p, bool fancy, int x, int y) {
    if (p.fx == 1u && p.fy == 1u) return sim_plane_sample(sb, p, x, y);
    const int xs = p.fx == 2u ? x >> 1 : x, ys = p.fy == 2u ? y >> 1 : y;
    if (!fancy) return sim_plane_sample(sb, p, xs, ys);
    const int xn = p.fx == 2u ? xs + ((x & 1) ? 1 : -1) : xs, yn = p.fy == 2u ? ys + ((y & 1) ? 1 : -1) : ys;
    float a = sim_plane_sample(sb, p, xs, ys), c = sim_plane_sample(sb, p, xn, ys);
    if (p.fy == 2u) {
        a = 0.75f * a + 0.25f * sim_plane_sample(sb, p, xs, yn);
        c = 0.75f * c + 0.25f * sim_plane_sample(sb, p, xn, yn);
    }
    return p.fx == 2u ? 0.75f * a + 0.25f * c : a;
}
void sim_compose(SimBatch& sb, const FrameDev& f) {
    for (uint32_t c = 0; c < f.ncomp && c < 3u; c++)
        if (f.pl[c].h == 0u || f.pl[c].wc == 0u) return;   // a scan of the frame failed to plan
    uint8_t* rgb = sb.rgb.data() + f.rgb_off;
    for (uint32_t y = 0; y < f.height; y++)
        for (uint32_t x = 0; x < f.width; x++) {
            uint8_t* o = rgb + ((size_t)y * f.width + x) * 3;
            const float yy = sim_frame_sample(sb, f.pl[0], f.fancy != 0u, (int)x, (int)y);
            if (f.ncomp == 1u) { o[0] = o[1] = o[2] = sat_u8_trunc(yy); continue; }
            const float cb = sim_frame_sample(sb, f.pl[1], f.fancy != 0u, (int)x, (int)y), cr = sim_frame_sample(sb, f.pl[2], f.fancy != 0u, (int)x, (int)y);
            o[0] = sat_u8_trunc(fmaf(cr, 1.402f, yy));
            o[1] = sat_u8_trunc(fmaf(cb, -0.34413629f, fmaf(cr, -0.71413629f, yy)));
            o[2] = sat_u8_trunc(fmaf(cb, 1.772f, yy));
        }
}

// mirrors block_idct_kernel + gather_colour_kernel (REF placement / generic sampling)
void sim_gather(SimBatch& sb, size_t img) {
    const ImgDev& im = sb.plan.imgs[img];
    const uint32_t nblk = im.units * im.blocks_per_mcu;
    const int16_t* coefs = sb.coefs.data() + im.coef_off;
    const float* qt = sb.plan.qt.data();
    std::vector<float> smp((size_t)nblk * 64);
    for (uint32_t blk = 0; blk < nblk; blk++) {
        const int comp = im.blk_comp[blk % im.blocks_per_mcu];
        sim_block_idct(coefs + (size_t)blk * 64, blk < coef_block_limit(sb.dyn[img]), qt + im.qt_off[comp], comp == 0 ? 128.0f : 0.0f, smp.data() + (size_t)blk * 64);
    }
    const uint32_t* map = sb.plan.gmap.data() + im.map_off;
    uint8_t* rgb = sb.rgb.data() + im.rgb_off;
    const size_t npix = (size_t)im.width * im.height;
    for (size_t p = 0; p < npix; p++) {
        float v[3];
        for (int c = 0; c < 3; c++) {
            const float none = c == 0 ? 128.0f : 0.0f;
            const uint32_t m = c < im.ncomp ? map[(size_t)c * im.map_plane + p] : kMapNone;
            v[c] = m == kMapNone ? none : smp[m];
        }
        uint8_t* o = rgb + p * 3;
        if (im.ncomp == 1) {
            o[0] = o[1] = o[2] = sat_u8_trunc(v[0]);
        } else {
            o[0] = sat_u8_trunc(fmaf(v[2], 1.402f, v[0]));
            o[1] = sat_u8_trunc(fmaf(v[1], -0.34413629f, fmaf(v[2], -0.71413629f, v[0])));
            o[2] = sat_u8_trunc(fmaf(v[1], 1.772f, v[0]));
        }
    }
}

}  // namespace

extern "C" {

void jpsim_set_sync_multi(int on) { g_sync_multi = on != 0; }

// build_multi_lut for unit tests: writes the 2^kMultiBits entries of one table to out (cap entries); returns their number
int jpsim_build_multi_lut(const uint8_t bits[16], const uint8_t* vals, int is_dc, uint32_t* out, size_t cap) {
    std::vector<uint32_t> v;
    build_multi_lut(bits, vals, is_dc != 0, v);
    if (v.size() > cap) return -1;
    memcpy(out, v.data(), v.size() * sizeof(uint32_t));
    return (int)v.size();
}

// Runs the whole simulated pipeline on a batch of descriptors.
//   rgb_out[i]   : W*H*3 bytes (may be NULL)
//   coef_out[i]  : reference-order coefficients (may be NULL), coef_cap[i] int16 each
//   diag[7]      : max repair iterations, repaired subsequences, sync-pass subsequences, flush phases, digest of the
//                  synchronisation records, most broken links in one repair round, rounds with more than 256 of them
int jpsim_decode_batch(const jpgpu_image_desc* descs, size_t n, uint8_t* const* rgb_out, int16_t* const* coef_out,
                       const size_t* coef_cap, uint32_t* nblocks /* n x 4 */, int32_t* statuses, uint64_t* bytes_read,
                       uint64_t* diag, uint32_t sub_bits) {
    SimBatch sb;
    int st = build_plan(descs, n, sb.plan, sub_bits);
    if (st != JPGPU_OK) return st;
    HostPlan& p = sb.plan;
    sb.raw.assign(p.raw_bytes + 64, 0);
    sb.stream.assign(p.stream_words + 64, 0);
    sb.segtab.assign(p.seg_entries + 8, 0);
    sb.subs.assign(p.sub_entries + 1, SubInfo());
    sb.segs.assign(p.sub_entries * (p.sub_bits / p.seg_bits) + 1, SegRec());
    sb.dyn.assign(n + 1, ImgDyn());
    sb.coefs.assign(p.coef_elems + 64, 0x5555);  // the write pass must produce every coefficient itself
    sb.rgb.assign(p.rgb_bytes + 256, 0);
    sb.samples.assign(p.sample_floats + 64, 0.0f);
    for (int k = 0; k < 64; k++) sb.store_pos[k] = (uint8_t)zigzag_to_colmajor(k, kZigzagNaturalHost);
    for (size_t i = 0; i < n; i++)
        if (p.status[i] == JPGPU_OK) memcpy(sb.raw.data() + p.imgs[i].raw_off, descs[i].scan, p.imgs[i].raw_len);
    for (size_t i = 0; i < n; i++) sim_prepass(sb, i);
    for (const SeqDesc& sd : p.seqs) sim_sync(sb, sd);
    {   // FNV-1a over what the synchronisation pass recorded (before repairs): the multi-symbol and the symbol-by-symbol
        // pass must agree on every state they write down, not just on the final result
        uint64_t h = 1469598103934665603ull;
        auto mix = [&h](const void* ptr, size_t len) { const uint8_t* q = (const uint8_t*)ptr; for (size_t k = 0; k < len; k++) { h ^= q[k]; h *= 1099511628211ull; } };
        for (size_t i = 0; i < n; i++) {
            if (p.status[i] != JPGPU_OK || p.imgs[i].interval_mode) continue;
            const uint32_t nsub = (sb.dyn[i].stream_bits + p.sub_bits - 1) / p.sub_bits;
            mix(sb.subs.data() + p.imgs[i].sub_off, (size_t)nsub * sizeof(SubInfo));
            mix(sb.segs.data() + (size_t)p.imgs[i].sub_off * (p.sub_bits / p.seg_bits), (size_t)nsub * (p.sub_bits / p.seg_bits) * sizeof(SegRec));
        }
        sb.sync_digest = h;
    }
    for (size_t i = 0; i < n; i++) sim_verify_scan(sb, i);
    for (const SeqDesc& sd : p.seqs)
        for (uint32_t group = 0; group < (1u << p.wp_shift); group++) sim_decode_write(sb, sd, group);
    for (size_t i = 0; i < n; i++)
        if (p.status[i] == JPGPU_OK) {
            if (p.imgs[i].frame) sim_block_idct_all(sb, i);   // compose path: samples now, pixels once all planes of the frame are there
            else if (p.imgs[i].kind == kKindGeneric) sim_gather(sb, i);
            else sim_idct_colour(sb, i);
        }
    for (const FrameDev& f : p.frames) sim_compose(sb, f);
    for (size_t i = 0; i < n; i++) {
        int32_t s = p.status[i];
        uint64_t br = 0;
        if (s == JPGPU_OK) {
            const uint32_t f = sb.dyn[i].status;
            if (f & kStDcSize) s = JPGPU_PANIC_READ_BITS_ASSERT;
            else if (f & kStBadCode) s = JPGPU_ERR_BAD_CODE;
            else if (f & kStRestart) s = JPGPU_ERR_RESTART;
            else if (!(f & kStDone)) s = JPGPU_ERR_TRUNCATED;
            br = ((uint64_t)sb.dyn[i].bits_consumed + 7) / 8;
            const ImgDev& im = p.imgs[i];
            if (rgb_out && rgb_out[i]) memcpy(rgb_out[i], sb.rgb.data() + im.rgb_off, (size_t)p.out_w[i] * p.out_h[i] * 3);
            if (coef_out && coef_out[i] && coef_cap[i] >= im.total_coefs)
                export_reference_order(im, sb.coefs.data() + im.coef_off, coef_out[i], nblocks + 4 * i);
        }
        if (statuses) statuses[i] = s;
        if (bytes_read) bytes_read[i] = br;
    }
    if (statuses)   // a frame of several scans is as good as its worst scan (jpgpu_batch_results)
        for (size_t i = 0; i < n; i++) {
            if (p.frame_part[i] != 1) continue;
            for (size_t k = i + 1; k < n && p.frame_part[k] == 2; k++)
                if (statuses[i] == JPGPU_OK && statuses[k] != JPGPU_OK) statuses[i] = statuses[k];
        }
    if (diag) {
        diag[0] = sb.repair_iters; diag[1] = sb.repairs; diag[2] = sb.sync_decodes; diag[3] = sb.flush_phases; diag[4] = sb.sync_digest;
        diag[5] = sb.max_broken; diag[6] = sb.crowded_rounds;
    }
    return JPGPU_OK;
}

// idct8-based 8x8 IDCT of natural-order dequantised coefficients, for unit tests of the math
void jpsim_idct_8x8(const float in_natural[64], float out[64]) {
    uint16_t ones[64];
    for (int k = 0; k < 64; k++) ones[k] = 1;
    float mult[64];
    build_qt_multipliers(ones, mult);  // column-major AAN multipliers for q = 1
    float tmp[64];
    for (int u = 0; u < 8; u++) {
        float f[8];
        for (int v = 0; v < 8; v++) f[v] = in_natural[v * 8 + u] * mult[u * 8 + v];
        idct8(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7]);
        for (int y = 0; y < 8; y++) tmp[y * 8 + u] = f[y];
    }
    for (int t = 0; t < 8; t++) {
        float* r = tmp + t * 8;
        idct8(r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]);
        for (int x = 0; x < 8; x++) out[t * 8 + x] = r[x];
    }
}

}  // extern "C"
