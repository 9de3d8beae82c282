// tests/emu/v5ela_sweep_emu.cpp — TEST INFRASTRUCTURE: the sweep kernel's work items (csrc/v5ela_workitem.cuh, process_work_item with
// SWEEP) run by g++ with the threads of each CTA emulated sequentially between barriers, over the library's own sweep plan
// (csrc/v5ela_host.h plan_sweep). A shim of its own next to tests/emu/v5ela_emu.cpp, built the same way; nothing under
// fake-video-detection-engine_b200/ loads it.
//
// Build: g++ -O2 -shared -fPIC -I include -I fake-video-detection-engine_b200/csrc tests/emu/v5ela_sweep_emu.cpp -o tests/emu/libv5ela_sweep_emu.so
#include <cstdlib>
#include <cstring>
#include <vector>

#include "v5ela_workitem.cuh"
#include "v5ela_host.h"

static int g_target_items = 0;       // v5emu_set_target_items: the host's small-batch decomposition (short segments, narrow strips)
extern "C" void v5emu_set_target_items(int t) { g_target_items = t; }

// n frames (h, w) = hw[2i], hw[2i+1], tightly packed one after the other in rgb.
static std::vector<v5ela_frame_desc> packed_frames(const uint8_t *rgb, const int *hw, int n)
{
    std::vector<v5ela_frame_desc> f((size_t)n);
    size_t off = 0;
    for (int i = 0; i < n; i++) {
        const int h = hw[2 * i], w = hw[2 * i + 1];
        f[(size_t)i] = v5ela_frame_desc{rgb + off, h, w, 3 * (int64_t)w, nullptr, nullptr};
        off += (size_t)h * w * 3;
    }
    return f;
}

// The sweep kernel's work items, in order, over the sweep plan of n frames packed in rgb at nq qualities (v5ela_analyze_sweep's device
// table, laid out as the C ABI uploads it), then the finalize kernel's step: n * nq records, optional ghost maps in plan_sweep's layout.
extern "C" int v5emu_analyze_sweep(const uint8_t *rgb, const int *hw, int n, const int *qualities, int nq, v5ela_record *records,
                                   uint32_t *ghost, int seg_rows)
{
    const std::vector<v5ela_frame_desc> frames = packed_frames(rgb, hw, n);
    v5plan::SweepPlan P;
    v5plan::plan_sweep(P, frames.data(), n, qualities, nq, ghost, seg_rows, g_target_items);
    if (P.status) return -1;
    std::vector<uint64_t> table((P.table_bytes + 7) / 8);
    uint8_t *t = reinterpret_cast<uint8_t *>(table.data());
    memcpy(t, P.frames.data(), sizeof(v5plan::FrameDesc) * P.frames.size());
    memcpy(t + P.off_entries, P.entries.data(), sizeof(v5plan::SweepEntry) * P.entries.size());
    memcpy(t + P.off_quant, P.quant.data(), sizeof(v5plan::QuantTab) * P.quant.size());
    static v5plan::LaneConsts lane_consts[32];
    if (!v5::mma::make_lane_consts(lane_consts)) return -2;
    v5plan::KParams p;
    memset(&p, 0, sizeof(p));
    p.records = records;
    p.n = (int)P.frames.size();
    p.frames = reinterpret_cast<const v5plan::FrameDesc *>(t);
    p.lane_consts = lane_consts;
    memset(records, 0, sizeof(v5ela_record) * (size_t)p.n);
    v5::Smem *S = (v5::Smem *)aligned_alloc(16, sizeof(v5::Smem));
    memset(S, 0xA5, sizeof(v5::Smem));                       // poison: uninitialised reads must not matter
    std::vector<v5::ThreadAcc> acc(v5::NT);
    for (long long work = 0; work < P.total; work++) v5::process_work_item<false, false, true, true>(*S, p, (int)work, acc.data());
    for (int i = 0; i < p.n; i++) v5plan::finalize_record(records[i]);
    free(S);
    return 0;
}

// The sweep plan alone. Per entry e, plan[6e .. 6e+5] = its pixel pointer, quality slot, strips, segments, first work item and ghost-map
// pointer (0: none); slot_quality[s] = the quality of slot s (up to nq slots), *n_slots, *total work items. Returns the plan's status
// and the frame and quality index it names (-1: none).
extern "C" int v5emu_plan_sweep(const v5ela_frame_desc *frames, int n, const int *qualities, int nq, uint32_t *ghost, int seg_rows,
                                int target_items, int64_t *plan, int *slot_quality, int *n_slots, long long *total, int *bad_frame,
                                int *bad_quality)
{
    v5plan::SweepPlan P;
    v5plan::plan_sweep(P, frames, n, qualities, nq, ghost, seg_rows, target_items);
    *bad_frame = P.bad_frame;
    *bad_quality = P.bad_quality;
    if (P.status) return P.status;
    for (size_t e = 0; e < P.frames.size(); e++) {
        int64_t *o = plan + 6 * e;
        o[0] = (int64_t)reinterpret_cast<uintptr_t>(P.frames[e].rgb);
        o[1] = P.entries[e].slot;
        o[2] = P.frames[e].n_strips;
        o[3] = P.frames[e].n_segs;
        o[4] = P.frames[e].work_base;
        o[5] = (int64_t)reinterpret_cast<uintptr_t>(P.entries[e].ghost);
    }
    for (size_t s = 0; s < P.slot_quality.size(); s++) slot_quality[s] = P.slot_quality[s];
    *n_slots = (int)P.slot_quality.size();
    *total = P.total;
    return 0;
}

// The ragged plan of the same frames (v5plan::plan_ragged), which the sweep plan must equal over its expanded list: per frame
// (n_strips, n_segs, work_base) into plan[3i..3i+2], the launch's work items into *total.
extern "C" int v5emu_plan_ragged(const int *hw, int n, int seg_rows, int target_items, int *plan, long long *total)
{
    static const uint8_t pixels[16] = {};                     // plan_ragged reads no pixel
    const std::vector<v5ela_frame_desc> frames = packed_frames(pixels, hw, n);
    std::vector<v5plan::FrameDesc> tab((size_t)n);
    const int rc = v5plan::plan_ragged(tab.data(), frames.data(), n, seg_rows, target_items, total);
    for (int i = 0; rc == 0 && i < n; i++) {
        plan[3 * i] = tab[(size_t)i].n_strips;
        plan[3 * i + 1] = tab[(size_t)i].n_segs;
        plan[3 * i + 2] = (int)tab[(size_t)i].work_base;
    }
    return rc;
}
