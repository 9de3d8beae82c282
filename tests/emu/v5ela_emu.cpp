// tests/emu/v5ela_emu.cpp — TEST INFRASTRUCTURE: runs the CUDA kernel's device code (csrc/v5ela_device.cuh,
// csrc/v5ela_workitem.cuh, compiled by g++ with the V5_* host shims) with the threads of each CTA emulated sequentially
// between barriers. It exists so the band/halo/edge indexing of the fused kernel can be checked against the oracle in
// the build container, which has no GPU. It is NOT a CPU fallback: nothing under fake-video-detection-engine_b200/ loads it.
//
// Build: g++ -O2 -shared -fPIC -I include -I fake-video-detection-engine_b200/csrc tests/emu/v5ela_emu.cpp -o tests/emu/libv5ela_emu.so
#include <cstdlib>
#include <cstring>
#include <vector>

#include "v5ela_workitem.cuh"
#include "v5ela_host.h"

static int g_last_split = -1, g_last_segs_b = -1, g_last_segs = -1;   // the decomposition of the most recent v5emu_analyze call
extern "C" int v5emu_last_split_frame(void) { return g_last_split; }
extern "C" int v5emu_last_segments(int tail) { return tail ? g_last_segs_b : g_last_segs; }
static int g_target_items = 0;       // v5emu_set_target_items: the host's small-batch decomposition (short segments, narrow strips)
extern "C" void v5emu_set_target_items(int t) { g_target_items = t; }

// Every work item of the plan p, in order, through the instantiation the C ABI launches for it; then the finalize kernel's step.
static int run_plan(v5plan::KParams &p, long long total)
{
    static v5plan::LaneConsts lane_consts[32];
    if (!v5::mma::make_lane_consts(lane_consts)) return -2;
    p.lane_consts = lane_consts;
    memset(p.records, 0, sizeof(v5ela_record) * (size_t)p.n);
    v5::Smem *S = (v5::Smem *)aligned_alloc(16, sizeof(v5::Smem));
    memset(S, 0xA5, sizeof(v5::Smem));                       // poison: uninitialised reads must not matter
    std::vector<v5::ThreadAcc> acc(v5::NT);
    const int inst = v5plan::choose_instantiation(p);
    for (int work = 0; work < (int)total; work++) {
        if (inst == v5plan::INST_RAGGED) v5::process_work_item<false, false, true>(*S, p, work, acc.data());
        else if (inst == V5ELA_INST_TEXHIST) v5::process_work_item<false, true>(*S, p, work, acc.data());
        else if (inst == V5ELA_INST_FAST) v5::process_work_item<true, false>(*S, p, work, acc.data());
        else v5::process_work_item<false, false>(*S, p, work, acc.data());
    }
    for (int i = 0; i < p.n; i++) v5plan::finalize_record(p.records[i]);
    free(S);
    return 0;
}

extern "C" int v5emu_analyze(const uint8_t *rgb, int n, int h, int w, int64_t frame_stride, int64_t row_stride,
                             int quality, v5ela_record *records, uint8_t *residual, int seg_rows, uint32_t *tex_hist)
{
    v5plan::KParams p;
    if (v5plan::fill_params(p, rgb, n, h, w, frame_stride, row_stride, records, residual, quality, seg_rows, g_target_items) != 0) return -1;
    p.tex_hist = tex_hist;
    g_last_split = p.split_frame; g_last_segs = p.n_segs; g_last_segs_b = p.n_segs_b;
    if (tex_hist) memset(tex_hist, 0, sizeof(uint32_t) * 256 * (size_t)n);
    return run_plan(p, v5plan::total_work_items(p));
}

// n frames (h, w) = hw[2i], hw[2i+1], tightly packed one after the other in rgb (and in residual, when given).
static std::vector<v5ela_frame_desc> packed_frames(const uint8_t *rgb, const int *hw, int n, uint8_t *residual)
{
    std::vector<v5ela_frame_desc> f((size_t)n);
    size_t off = 0;
    for (int i = 0; i < n; i++) {
        const int h = hw[2 * i], w = hw[2 * i + 1];
        f[(size_t)i] = v5ela_frame_desc{rgb + off, h, w, 3 * (int64_t)w, residual ? residual + off : nullptr, nullptr};
        off += (size_t)h * w * 3;
    }
    return f;
}

// The RAGGED instantiation over the library's ragged plan (v5plan::plan_ragged with the target of v5emu_set_target_items).
extern "C" int v5emu_analyze_ragged(const uint8_t *rgb, const int *hw, int n, int quality, v5ela_record *records, uint8_t *residual,
                                    int seg_rows)
{
    const std::vector<v5ela_frame_desc> frames = packed_frames(rgb, hw, n, residual);
    std::vector<v5plan::FrameDesc> tab((size_t)n);
    long long total = 0;
    if (v5plan::plan_ragged(tab.data(), frames.data(), n, seg_rows, g_target_items, &total) != 0) return -1;
    v5plan::KParams p;
    memset(&p, 0, sizeof(p));
    p.records = records;
    p.n = n;
    p.frames = tab.data();
    v5plan::fill_quant(p.q, quality);
    return run_plan(p, total);
}

// The ragged plan alone: per frame (n_strips, n_segs, work_base) into plan[3i..3i+2], the launch's work items into *total.
extern "C" int v5emu_plan_ragged(const int *hw, int n, int seg_rows, int target_items, int *plan, long long *total)
{
    static const uint8_t pixels[16] = {};                     // plan_ragged reads no pixel
    const std::vector<v5ela_frame_desc> frames = packed_frames(pixels, hw, n, nullptr);
    std::vector<v5plan::FrameDesc> tab((size_t)n);
    const int rc = v5plan::plan_ragged(tab.data(), frames.data(), n, seg_rows, target_items, total);
    for (int i = 0; rc == 0 && i < n; i++) {
        plan[3 * i] = tab[(size_t)i].n_strips;
        plan[3 * i + 1] = tab[(size_t)i].n_segs;
        plan[3 * i + 2] = (int)tab[(size_t)i].work_base;
    }
    return rc;
}

// The uniform plan of n frames h x w (v5plan::fill_params): n_strips, n_segs, split_frame, n_segs_b into plan[0..3].
extern "C" int v5emu_plan_uniform(int n, int h, int w, int seg_rows, int target_items, int *plan)
{
    static const uint8_t pixels[16] = {};
    v5plan::KParams p;
    const int rc = v5plan::fill_params(p, pixels, n, h, w, 3 * (int64_t)h * w, 3 * (int64_t)w, (v5ela_record *)pixels, nullptr, 90, seg_rows,
                                       target_items);
    if (rc == 0) {
        plan[0] = p.n_strips;
        plan[1] = p.n_segs;
        plan[2] = p.split_frame;
        plan[3] = p.n_segs_b;
    }
    return rc;
}

// 16-bit hand-offs of the block stage (int16 pairs / 8-bit limb pairs) that left their range, since the library was loaded
extern "C" long long v5emu_range_violations(void)
{
    return v5::range_violations();
}

extern "C" int v5emu_quant_selftest(void)
{
    // exhaustive: the reciprocal division equals libjpeg's rounding for every table entry and coefficient
    for (int t = 1; t <= 255; t++) {
        uint16_t tab[64];
        for (int i = 0; i < 64; i++) tab[i] = (uint16_t)t;
        v5plan::QuantTab q;
        v5plan::make_quant(tab, q);
        for (int c = -8192; c <= 8192; c++) {
            const int div = t << 3, a = c < 0 ? -c : c;
            int ref = (a + (div >> 1)) / div;
            if (c < 0) ref = -ref;
            const uint32_t x = (uint32_t)(c + (c >> 31) + q.bias[0]);
            const int got = (int)v5::umulhi32(x, q.recip[0]) * q.t[0] - q.unbias[0];
            if (got != ref * t) return t * 100000 + (c + 8192);
        }
    }
    return 0;
}
