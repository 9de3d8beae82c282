// v5ela_host.h — the fused kernel's launch plan: kernel parameters, work decomposition and instantiation, built once on the host for
// either build of the kernel. Shared by the C ABI (v5ela.cu) and the CPU thread emulator (tests/emu).
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#include "v5ela.h"
#include "v5ela_device.cuh"

namespace v5plan {

// Host side: fills the reciprocal constants of one table (see QuantTab).
inline void make_quant(const uint16_t tab[64], QuantTab &q)
{
    for (int i = 0; i < 64; i++) {
        const uint32_t t = tab[i], d = t << 3;
        const uint32_t b = (8192u + d - 1) / d;                     // b*d >= 8192 >= max |coef|
        q.recip[i] = (uint32_t)(0x100000000ull / d) + 1u;           // exact for x*d < 2^32, x < 2^15
        q.bias[i] = (int32_t)(d / 2 + b * d);
        q.t[i] = (int32_t)t;
        q.unbias[i] = (int32_t)(b * t);
    }
}

// JPEG Annex K.1 / K.2 base tables in natural (row-major) order, scaled like libjpeg's jpeg_set_quality with
// force_baseline — what `Image.save(..., 'JPEG', quality=q)` uses (v5_texture_ela.py:67; SURVEY.md A.1).
inline void quant_tables(int quality, uint16_t luma[64], uint16_t chroma[64])
{
    static const uint8_t base_l[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                       14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                       18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                       49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
    static const uint8_t base_c[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                       24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99};
    const int q = quality < 1 ? 1 : (quality > 100 ? 100 : quality);
    const int scale = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int i = 0; i < 64; i++) {
        const int bl = base_l[i], bc = i < 32 ? base_c[i] : 99;
        int l = (bl * scale + 50) / 100, c = (bc * scale + 50) / 100;
        luma[i] = (uint16_t)(l < 1 ? 1 : (l > 255 ? 255 : l));
        chroma[i] = (uint16_t)(c < 1 ? 1 : (c > 255 ? 255 : c));
    }
}

// The kernel's luma / chroma division constants for a JPEG quality.
inline void fill_quant(QuantTab q[2], int quality)
{
    uint16_t ql[64], qc[64];
    quant_tables(quality, ql, qc);
    make_quant(ql, q[0]);
    make_quant(qc, q[1]);
}

// Longer segments are cheaper — every segment pays two chroma-only halo bands and one flush of its histograms — but the launch
// needs enough work items: the fewest segments per frame that still give `rounds` items per resident CTA (target_items = 2 per
// CTA) when the launch has `columns` strips in all. 256 x 1080p: whole-height strips, 1024 items.
// (Swept on a B200: profiles/r02/variants.txt section 10.)
inline int64_t segments_wanted(int64_t target_items, int64_t columns, int rounds = 2)
{
    const int64_t ctas = (target_items + 1) / 2, segs = (rounds * ctas + columns - 1) / columns;
    return segs < 1 ? 1 : segs;
}

// MCU rows per segment of a frame of mh MCU rows cut into about want_segs segments: down to 4.
inline int segment_rows(int mh, int64_t want_segs)
{
    const int rows = (int)((mh + want_segs - 1) / want_segs);
    return rows < 4 ? 4 : rows;
}

// Still too few items for the GPU (a handful of crops): more, narrower strips shorten every band, and with it the latency of the
// call; the extra halo columns do not matter when most SMs would idle anyway. Scales the strip count by target / items, at least 4
// MCUs per strip.
inline int widen_strips(int n_strips, int mw, int64_t items, int64_t target_items)
{
    const int64_t factor = (target_items + items - 1) / (items > 0 ? items : 1);
    int64_t ns = (int64_t)n_strips * factor;
    const int cap = mw / 4 > 1 ? mw / 4 : 1;
    if (ns > cap) ns = cap;
    return ns < n_strips ? n_strips : (int)ns;
}

// Work decomposition: frames x strips (<= TW_MAX MCUs wide, balanced) x vertical segments of about `seg_rows` MCU rows.
// seg_rows <= 0 picks the default (see below: as few segments as keep the GPU supplied, short segments for the last frames);
// total_work_items(p) is the number of work items of the launch. Returns 0 or -1 on invalid arguments.
inline int fill_params(KParams &p, const uint8_t *rgb, int n, int h, int w, int64_t frame_stride, int64_t row_stride,
                       v5ela_record *records, uint8_t *residual, int quality, int seg_rows, int target_items = 0,
                       const int *tune = nullptr)
{
    if (!rgb || !records || n <= 0 || h <= 0 || w <= 0) return -1;
    if (row_stride < (int64_t)3 * w || (n > 1 && frame_stride < row_stride * (int64_t)h)) return -1;
    if (quality < 1 || quality > 100) return -1;
    if ((int64_t)h > 65536 || (int64_t)w > 65536) return -1;
    if ((int64_t)h * w > 0x7fffffffLL) return -1;             // per-frame histogram counters are 32-bit
    memset(&p, 0, sizeof(p));
    p.rgb = rgb;
    p.frame_stride = frame_stride;
    p.row_stride = row_stride;
    p.records = records;
    p.residual = residual;
    p.n = n;
    p.h = h;
    p.w = w;
    p.mw = (w + 15) / 16;
    p.mh = (h + 15) / 16;
    p.n_strips = (p.mw + TW_MAX - 1) / TW_MAX;
    p.split_frame = n;                                        // one regime unless decided otherwise below
    if (seg_rows <= 0) {
        seg_rows = 17;                                          // (no CTA count known: the emulator's default)
        if (target_items > 0) {
            // tune (development knob, V5ELA_DECOMP): {items per CTA wanted, tail segment rows, tail frames per CTA in 1/8 strips}
            const int t_rounds = tune ? tune[0] : 2, t_seg_b = tune ? tune[1] : 8, t_tail8 = tune ? tune[2] : 4;
            const int64_t ctas = (target_items + 1) / 2, columns = (int64_t)n * p.n_strips;
            seg_rows = segment_rows(p.mh, segments_wanted(target_items, columns, t_rounds));
            const int64_t items = columns * ((p.mh + seg_rows - 1) / seg_rows);
            if (items < target_items) p.n_strips = widen_strips(p.n_strips, p.mw, items, target_items);
            // The tail: CTAs finish their last long item up to one item apart. The last frames — half an item per CTA worth of
            // them — are cut into segments of 8 MCU rows instead, drawn after all the long ones.
            const int seg_b = t_seg_b, segs_b = (p.mh + seg_b - 1) / seg_b;
            const int64_t nb = (ctas * t_tail8 + 8 * p.n_strips - 1) / (8 * p.n_strips);
            if (t_tail8 > 0 && seg_rows >= 2 * seg_b && nb < n) {
                p.split_frame = (int)(n - nb);
                p.n_segs_b = segs_b;
            }
        }
    }
    p.n_segs = (p.mh + seg_rows - 1) / seg_rows;
    if (p.split_frame >= n) p.n_segs_b = p.n_segs;
    if ((long long)n * p.n_strips * (p.n_segs > p.n_segs_b ? p.n_segs : p.n_segs_b) > 0x7fffffffLL) return -1;   // work items are 32-bit
    p.work_split = p.split_frame * p.n_strips * p.n_segs;
    p.vec_ok = ((reinterpret_cast<uintptr_t>(rgb) | (uintptr_t)frame_stride | (uintptr_t)row_stride) & 15) == 0;
    p.resid_vec_ok = residual && ((reinterpret_cast<uintptr_t>(residual) | (uintptr_t)(3 * w)) & 15) == 0;
    fill_quant(p.q, quality);
    return 0;
}

inline long long total_work_items(const KParams &p)
{
    return (long long)p.work_split + (long long)(p.n - p.split_frame) * p.n_strips * p.n_segs_b;
}

// A descriptor of a ragged batch has pixels, a size within 65536 x 65536 and 2^31 - 1 pixels (32-bit histogram counters), and a row
// stride of at least 3 * width.
inline bool frame_desc_ok(const v5ela_frame_desc &f)
{
    return f.rgb && f.height > 0 && f.width > 0 && f.height <= 65536 && f.width <= 65536 && (int64_t)f.height * f.width <= 0x7fffffffLL &&
           f.row_stride_bytes >= (int64_t)3 * f.width;
}

// Ragged batch (v5ela_analyze_ragged): fills tab[0..n) — per frame its geometry, pointers, strips x segments and first work item —
// and *total, the work items of the launch. fill_params' rule without its tail split: segments_wanted over the strips of the whole
// batch (4 segments per frame when no CTA count is known), and narrower strips for every frame when the batch as a whole is short of
// items. Returns 0, -1 (bad pointer, size or stride in a descriptor) or -2 (more than 2^31 - 1 work items).
inline int plan_ragged(FrameDesc *tab, const v5ela_frame_desc *frames, int n, int seg_rows, int target_items, long long *total)
{
    if (!tab || !frames || n <= 0) return -1;
    int64_t columns = 0;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames[i];
        if (!frame_desc_ok(f)) return -1;
        FrameDesc &d = tab[i];
        uint8_t *resid = f.residual ? f.residual : f.enhanced;                // an enhanced map alone: the residual is formed in place
        d.rgb = f.rgb;
        d.resid = resid;
        d.row_stride = f.row_stride_bytes;
        d.h = f.height; d.w = f.width;
        d.mw = (f.width + 15) / 16; d.mh = (f.height + 15) / 16;
        d.n_strips = (d.mw + TW_MAX - 1) / TW_MAX;
        const bool vec = ((reinterpret_cast<uintptr_t>(f.rgb) | (uintptr_t)f.row_stride_bytes) & 15) == 0;
        const bool rvec = resid && ((reinterpret_cast<uintptr_t>(resid) | (uintptr_t)(3 * f.width)) & 15) == 0;
        d.flags = (vec ? 1u : 0u) | (rvec ? 2u : 0u);
        columns += d.n_strips;
    }
    const int64_t want_segs = target_items > 0 ? segments_wanted(target_items, columns) : 4;
    int64_t items = 0;                                          // work items with the default strips
    for (int i = 0; i < n; i++) {
        const int rows = seg_rows > 0 ? seg_rows : segment_rows(tab[i].mh, want_segs);
        tab[i].n_segs = (tab[i].mh + rows - 1) / rows;
        items += (int64_t)tab[i].n_strips * tab[i].n_segs;
    }
    const bool widen = seg_rows <= 0 && target_items > 0 && items < target_items;
    long long sum = 0;
    for (int i = 0; i < n; i++) {
        FrameDesc &d = tab[i];
        if (widen) d.n_strips = widen_strips(d.n_strips, d.mw, items, target_items);
        if (sum > 0x7fffffffLL) return -2;
        d.work_base = (uint32_t)sum;
        sum += (long long)d.n_strips * d.n_segs;
    }
    if (sum > 0x7fffffffLL) return -2;
    *total = sum;
    return 0;
}

// A sweep (v5ela_analyze_sweep): n frames at nq qualities, expanded quality-major into n * nq entries — entry q * n + i is frame i at
// qualities[q] and writes record q * n + i — and cut by plan_ragged's rule over the whole expanded list. Beside the frame table, one
// SweepEntry per entry: its table slot (one per distinct quality, in order of first appearance) and its ghost map, map (q, i) at
// ghost + q * M + sum_{j<i} m_j with m_j = ceil(h_j/16) * ceil(w_j/16), M = sum_j m_j.
struct SweepPlan {
    int status = V5ELA_OK;                      // V5ELA_OK, or why the call is refused ...
    const char *error = "";
    int bad_frame = -1, bad_quality = -1;       // ... and the frame or the quality index it is refused for
    std::vector<FrameDesc> frames;              // n * nq entries
    std::vector<SweepEntry> entries;
    std::vector<QuantTab> quant;                // luma, chroma of each slot
    std::vector<int> slot_quality;
    long long total = 0;                        // work items of the launch
    size_t off_entries = 0, off_quant = 0, table_bytes = 0;   // device table: frames | entries | quant (sweep_entries, sweep_quant)
};

inline void plan_sweep(SweepPlan &P, const v5ela_frame_desc *frames, int n, const int *qualities, int nq, uint32_t *ghost, int seg_rows,
                       int target_items)
{
    auto refuse = [&P](const char *why, int frame, int quality) {
        P.status = V5ELA_ERR_INVALID;
        P.error = why;
        P.bad_frame = frame;
        P.bad_quality = quality;
    };
    if (!frames || !qualities || n < 0) return refuse("null descriptor or quality array, or n < 0", -1, -1);
    if (nq < 1 || nq > 100) return refuse("nq must be in 1..100", -1, -1);
    for (int q = 0; q < nq; q++)
        if (qualities[q] < 1 || qualities[q] > 100) return refuse("quality outside 1..100", -1, q);
    for (int i = 0; i < n; i++) {
        if (!frame_desc_ok(frames[i])) return refuse("bad pointer, size or stride", i, -1);
        if (frames[i].residual || frames[i].enhanced) return refuse("residual and enhanced maps must be NULL in a sweep", i, -1);
    }
    const int64_t m = (int64_t)n * nq;
    if (m > 0x7fffffffLL) return refuse("more than 2^31 - 1 work items", -1, -1);
    std::vector<v5ela_frame_desc> expanded((size_t)m);
    for (int q = 0; q < nq; q++)
        for (int i = 0; i < n; i++) expanded[(size_t)q * n + i] = frames[i];
    P.frames.resize((size_t)m);
    if (m > 0 && plan_ragged(P.frames.data(), expanded.data(), (int)m, seg_rows, target_items, &P.total) != 0)
        return refuse("more than 2^31 - 1 work items", -1, -1);
    std::vector<int64_t> map_off((size_t)n);
    int64_t M = 0;
    for (int i = 0; i < n; i++) {
        map_off[(size_t)i] = M;
        M += (int64_t)P.frames[(size_t)i].mh * P.frames[(size_t)i].mw;
    }
    int slot_of[101];
    for (int &s : slot_of) s = -1;
    P.entries.resize((size_t)m);
    for (int q = 0; q < nq; q++) {
        int &slot = slot_of[qualities[q]];
        if (slot < 0) {
            slot = (int)P.slot_quality.size();
            P.slot_quality.push_back(qualities[q]);
        }
        for (int i = 0; i < n; i++) {
            SweepEntry &e = P.entries[(size_t)q * n + i];
            e.ghost = ghost ? ghost + (int64_t)q * M + map_off[(size_t)i] : nullptr;
            e.slot = slot;
            e.pad = 0;
        }
    }
    P.quant.resize(2 * P.slot_quality.size());
    for (size_t s = 0; s < P.slot_quality.size(); s++) fill_quant(&P.quant[2 * s], P.slot_quality[s]);
    P.off_entries = sizeof(FrameDesc) * P.frames.size();
    P.off_quant = P.off_entries + sizeof(SweepEntry) * P.entries.size();
    P.table_bytes = P.off_quant + sizeof(QuantTab) * P.quant.size();
}

// Which instantiation of the fused kernel a call takes (v5ela_device.cuh, FAST): widths that are a multiple of the MCU
// width (1280, 1920, 3840, ...), 16-byte aligned, without a residual map — the statistics-only keyframe batches the
// benchmark drives.
inline bool fast_path_ok(const KParams &p)
{
#ifdef V5_NO_FAST_PATH
    return false;
#else
    return p.w % 16 == 0 && p.residual == nullptr && p.tex_hist == nullptr && p.vec_ok;
#endif
}

// The general instantiation over a frame table (KParams::frames). Internal to the plan: v5ela_last_instantiation reports a ragged
// launch as V5ELA_INST_GENERAL.
constexpr int INST_RAGGED = V5ELA_INST_TEXHIST + 1;
// The sweep kernel (v5ela_analyze_sweep's frame table, with the sweep's tables behind it). Internal to the plan as well, and not
// reported by v5ela_last_instantiation.
constexpr int INST_SWEEP = INST_RAGGED + 1;

// The instantiation a launch takes: RAGGED for a frame table, TEXHIST if a texture histogram is wanted, else FAST where
// fast_path_ok, else GENERAL.
inline int choose_instantiation(const KParams &p)
{
    if (p.frames) return INST_RAGGED;
    if (p.tex_hist) return V5ELA_INST_TEXHIST;
    return fast_path_ok(p) ? V5ELA_INST_FAST : V5ELA_INST_GENERAL;
}

// ela_sum / ela_sumsq / ela_max follow from the histogram (host mirror of finalize_kernel, used by the emulator).
inline void finalize_record(v5ela_record &r)
{
    for (int c = 0; c < 3; c++) {
        uint64_t s = 0, sq = 0;
        int mx = 0;
        for (int b = 0; b < 256; b++) {
            const uint64_t cnt = r.ela_hist[c][b];
            s += cnt * (uint64_t)b;
            sq += cnt * (uint64_t)(b * b);
            if (cnt) mx = b;
        }
        r.ela_sum[c] = s;
        r.ela_sumsq[c] = sq;
        r.ela_max[c] = (uint8_t)mx;
    }
}

}  // namespace v5plan
