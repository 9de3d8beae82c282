// tests/emu/v5ela_spec_emu.cpp — TEST INFRASTRUCTURE: the ragged spectrum plan (csrc/v5ela_spec_plan.h, compiled by g++) behind a
// small extern "C" surface, so that tests/test_spectrum_plan.py can check path choice, CTA coverage, workspace ranges, twiddle
// de-duplication, chunking and refusals without a GPU. NOT a CPU fallback: nothing under fake-video-detection-engine_b200/ loads it.
//
// Build (tests/test_spectrum_plan.py does it): g++ -O2 -shared -fPIC -I include -I <csrc> v5ela_spec_emu.cpp
#include "v5ela_spec_plan.h"

using namespace v5fft;

static SpecPlan plan;                  // the last plan made (one test process plans one call at a time)

// The uniform rule for one height x width image: returns 1 for the FFT path and its columns per CTA in *cc.
extern "C" int v5semu_fft_path(int fft_on, int height, int width, int *cc)
{
    FftPlan pw, ph;
    FftShape s;
    const bool fast = fft_path(fft_on != 0, height, width, pw, ph, s);
    *cc = s.cc;
    return fast ? 1 : 0;
}

// Plans a call; returns its status, and the refused frame in *bad_frame.
extern "C" int v5semu_plan(const v5ela_gray_desc *frames, int n, int fft_on, int64_t chunk_bytes, int *bad_frame)
{
    plan_spectrum_ragged(frames, n, fft_on != 0, (size_t)chunk_bytes, plan);
    *bad_frame = plan.bad_frame;
    return plan.status;
}

extern "C" const char *v5semu_error() { return plan.error; }

// counts[0..4] = frames, sizes, chunks, launches, twiddle entries
extern "C" void v5semu_counts(int64_t *counts)
{
    counts[0] = (int64_t)plan.frames.size();
    counts[1] = (int64_t)plan.sizes.size();
    counts[2] = (int64_t)plan.chunks.size();
    counts[3] = plan.launches;
    counts[4] = (int64_t)plan.tw_elems;
}

// out[0..11] = h, w, wh, cc, g_off, ms_off, sw, sh, mm, gx, bx, by
extern "C" void v5semu_frame(int i, int64_t *out)
{
    const SpecFrame &f = plan.frames[(size_t)i];
    const int64_t v[12] = {f.h, f.w, f.wh, f.cc, f.g_off, f.ms_off, f.sw, f.sh, f.mm, f.gx, f.bx, f.by};
    for (int k = 0; k < 12; k++) out[k] = v[k];
}

// out[0..3] = n, tw, fft
extern "C" void v5semu_size(int k, int64_t *out)
{
    const SpecSize &s = plan.sizes[(size_t)k];
    out[0] = s.n;
    out[1] = s.tw;
    out[2] = s.fft;
}

// out[0..11] = f0, n, g_elems, ms_elems, ctas[5], rows_smem, cols_smem, launches
extern "C" void v5semu_chunk(int c, int64_t *out)
{
    const SpecChunk &C = plan.chunks[(size_t)c];
    out[0] = C.f0;
    out[1] = C.n;
    out[2] = (int64_t)C.g_elems;
    out[3] = (int64_t)C.ms_elems;
    for (int k = 0; k < L_KINDS; k++) out[4 + k] = C.ctas[k];
    out[9] = (int64_t)C.rows_smem;
    out[10] = (int64_t)C.cols_smem;
    out[11] = C.launches;
}

// Every CTA of launch `kind` (L_FFT_ROWS .. L_IMAGE) of chunk c, as the kernels find it: its frame (within the chunk) and local
// index. kind = -1: the call's twiddle launch (frame = size entry).
extern "C" void v5semu_walk(int c, int kind, int32_t *frame_out, int32_t *local_out)
{
    const uint32_t *base;
    int n;
    uint32_t ctas;
    if (kind < 0) {
        base = plan.tw_base.data();
        n = (int)plan.sizes.size();
        ctas = plan.tw_base.back();
    } else {
        const SpecChunk &C = plan.chunks[(size_t)c];
        base = plan.bases.data() + C.off_base + (size_t)kind * (C.n + 1);
        n = C.n;
        ctas = C.ctas[kind];
    }
    for (uint32_t cta = 0; cta < ctas; cta++) {
        const int f = cta_frame(base, n, cta);
        frame_out[cta] = f;
        local_out[cta] = (int32_t)(cta - base[f]);
    }
}
