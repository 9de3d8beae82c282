// v5ela_spec_plan.h — the spectrum path's host plan: the Stockham FFT plan of one size, the rule that picks the FFT or the
// exact-size DFT for a frame, and the launch plan of a ragged call (v5ela_spectrum_ragged): per-frame path, de-duplicated
// twiddle tables, chunks under the workspace cap, workspace offsets, and the CTA prefix table of every ragged launch.
// Host only, no CUDA runtime calls: shared by both spectrum entry points (v5ela.cu), the kernels (v5ela_fft.cuh: the plan
// structs and the CTA lookup) and the CPU tests (tests/emu/v5ela_spec_emu.cpp).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <unordered_map>
#include <vector>

#include "v5ela.h"

#ifdef __CUDACC__
#define V5S_HOSTDEV __host__ __device__ __forceinline__
#else
#define V5S_HOSTDEV inline
#endif

namespace v5fft {

constexpr int TILE = 32;     // DFT path: output tile edge per CTA (16x16 threads, 2x2 outputs each)

// Fast path for sizes whose prime factors are all in {2, 3, 5}: mixed-radix (5, 3, 4, 2) Stockham stages (v5ela_fft.cuh).
struct FftPlan {
    int n;
    int nst;
    int radix[24];
    uint32_t inv_s[24];         // floor(2^32 / s) + 1 for the stride s of every stage: idx / s == umulhi(idx, inv_s) for idx < 2^16
    uint32_t inv_per_seq[24];   // the same for N / radix (butterflies per sequence)
};

// exact unsigned division of a < 2^16 by d in 2..2^16 through its reciprocal (error term a / 2^32 < 1 / d)
V5S_HOSTDEV uint32_t recip_u16(uint32_t d) { return (uint32_t)(0x100000000ull / d) + 1u; }

// Host: factor n into 5s, 3s and 2s; returns false when another prime factor remains.
inline bool make_plan(int n, FftPlan &plan)
{
    plan.n = n;
    plan.nst = 0;
    const int rs[4] = {5, 3, 4, 2};                             // radix 4 before 2: half the stages (barriers, shared-memory passes)
    for (int r : rs)
        while (n % r == 0 && plan.nst < 24) {
            plan.radix[plan.nst++] = r;
            n /= r;
        }
    int s = 1;
    for (int st = 0; st < plan.nst; st++) {
        plan.inv_s[st] = recip_u16((uint32_t)s);
        plan.inv_per_seq[st] = recip_u16((uint32_t)(plan.n / plan.radix[st]));
        s *= plan.radix[st];
    }
    return n == 1 && plan.n <= 65536;
}

constexpr size_t FFT_SMEM_MAX = 200u << 10;                     // dynamic shared memory of the FFT kernels

// The FFT path's shape for one height x width frame, and whether the frame takes it: both sides made of 2, 3 and 5 only, and
// both passes within FFT_SMEM_MAX (rows: two real rows packed in one complex row, ping-pong; columns: cc adjacent columns,
// ping-pong). Otherwise the frame takes the exact-size DFT products. fft_on = false (V5ELA_FFT=0) forces the DFT.
struct FftShape {
    int cc;                     // columns per CTA of the column pass: 1, 2 or 4
    size_t rows_smem, cols_smem;
};
inline bool fft_path(bool fft_on, int height, int width, FftPlan &plan_w, FftPlan &plan_h, FftShape &s)
{
    s.rows_smem = 16 * 2 * (size_t)width;
    int cc = (int)((size_t)(96u << 10) / (16 * 2 * (size_t)height));
    s.cc = cc >= 4 ? 4 : (cc >= 2 ? 2 : cc);                    // (the kernel shifts and masks)
    s.cols_smem = 16 * 2 * (size_t)(s.cc > 0 ? s.cc : 1) * (size_t)height;
    return fft_on && make_plan(width, plan_w) && make_plan(height, plan_h) && s.cc >= 1 && s.rows_smem <= FFT_SMEM_MAX &&
           s.cols_smem <= FFT_SMEM_MAX;
}

// The image kernel's CTAs for one height x width frame: column blocks of 256 pixels, and row blocks such that every CTA walks ~16
// rows, so that the per-thread set-up (the double-precision 255 / (max - min)) is paid once per 16 pixels. Sides of at most 65536
// keep by <= 4096, within a grid's y limit.
struct ImageGrid {
    int bx, by;
};
inline ImageGrid image_grid(int height, int width) { return {(width + 255) / 256, (height + 15) / 16}; }

// ------------------------------------------------------------------------------------------------------------ ragged calls
// One distinct side length of a call: its twiddle table (tw[m] = exp(-2 pi i m / n), m < n) in the call's twiddle arena, and
// its FFT plan (valid when `fft` is set).
struct SpecSize {
    FftPlan plan;
    int64_t tw;                 // first entry in the twiddle arena (double2 units)
    int32_t n;
    int32_t fft;
};

// One frame as the kernels see it. Workspace offsets are relative to the chunk's d_g / d_ms; mm is its min/max pair.
struct SpecFrame {
    const uint8_t *gray;
    uint8_t *out;
    int64_t row_stride;
    int64_t g_off;              // double2 units, h * wh entries
    int64_t ms_off;             // double units, h * wh entries
    int32_t h, w, wh;
    int32_t cc;                 // FFT path: columns per CTA of the column pass; 0: DFT path
    int32_t sw, sh;             // SpecSize entries of the width and the height
    int32_t mm;
    int32_t gx;                 // DFT path: tiles across the half spectrum, ceil(wh / TILE)
    int32_t bx, by;             // image kernel: column blocks and row blocks
};

// The ragged launches, each with a CTA prefix table per chunk: CTA c of the launch belongs to the frame f with
// base[f] <= c < base[f + 1] (frames the launch skips have base[f] == base[f + 1]).
enum { L_FFT_ROWS, L_FFT_COLS, L_DFT_ROWS, L_DFT_COLS, L_IMAGE, L_KINDS };

// Flat CTA index -> the frame it belongs to (the largest f < n with base[f] <= cta); local index = cta - base[f].
V5S_HOSTDEV int cta_frame(const uint32_t *base, int n, uint32_t cta)
{
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (base[mid] <= cta) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

struct SpecChunk {
    int f0 = 0, n = 0;                          // frames [f0, f0 + n) of the call
    size_t g_elems = 0, ms_elems = 0;           // workspace: double2 and double entries
    uint32_t ctas[L_KINDS] = {0, 0, 0, 0, 0};   // CTAs of each launch (0: not launched)
    size_t rows_smem = 0, cols_smem = 0;        // dynamic shared memory of the two FFT launches: the largest frame's
    size_t off_base = 0;                        // the chunk's L_KINDS prefix tables (n + 1 entries each) in the device table
    int launches = 0;                           // counted kernel launches (the twiddle launch is the call's, not a chunk's)
};

struct SpecPlan {
    int status = V5ELA_OK;                      // V5ELA_OK, or why the call is refused ...
    const char *error = "";
    int bad_frame = -1;                         // ... and the frame it is refused for
    std::vector<SpecSize> sizes;
    std::vector<SpecFrame> frames;
    std::vector<SpecChunk> chunks;
    std::vector<uint32_t> tw_base;              // twiddle launch: CTA prefix table over `sizes` (256 entries per CTA)
    std::vector<uint32_t> bases;                // every chunk's prefix tables, back to back
    size_t tw_elems = 0;                        // twiddle arena, double2 entries
    size_t g_max = 0, ms_max = 0;               // workspace the largest chunk needs (entries)
    int mm_max = 0;                             // min/max pairs the largest chunk needs
    // device table: sizes | frames | tw_base | bases, each 16-byte aligned
    size_t off_sizes = 0, off_frames = 0, off_tw_base = 0, off_bases = 0, table_bytes = 0;
    int launches = 0;                           // counted kernel launches of the call
};

// Why a descriptor of a ragged call is refused, or nullptr.
inline const char *gray_desc_error(const v5ela_gray_desc &d)
{
    return !d.gray || !d.out                     ? "null pointer"
           : d.height <= 0 || d.width <= 0       ? "non-positive size"
           : d.height > 65536 || d.width > 65536 ? "side over 65536"
           : d.row_stride_bytes < d.width        ? "row stride smaller than the width"
                                                 : nullptr;
}

inline size_t spec_align(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Plans a ragged call of n frames into P. Nothing is planned past a refusal (P.status). chunk_bytes caps the float64 workspace
// of a chunk (24 bytes per half-spectrum sample, as v5ela_spectrum counts it); a frame over the cap gets a chunk of its own.
inline void plan_spectrum_ragged(const v5ela_gray_desc *frames, int n, bool fft_on, size_t chunk_bytes, SpecPlan &P)
{
    P = SpecPlan();
    if (!frames || n < 0) {
        P.status = V5ELA_ERR_INVALID;
        P.error = "null descriptor array or negative count";
        return;
    }
    for (int i = 0; i < n; i++) {
        if (const char *why = gray_desc_error(frames[i])) {
            P.status = V5ELA_ERR_INVALID;
            P.error = why;
            P.bad_frame = i;
            return;
        }
    }
    // ---- distinct side lengths: one twiddle table (and FFT plan) each, whether a width or a height
    std::unordered_map<int, int> index_of;
    auto size_index = [&](int s) {
        const auto it = index_of.find(s);
        if (it != index_of.end()) return it->second;
        index_of[s] = (int)P.sizes.size();
        SpecSize z;
        z.plan = FftPlan();
        z.fft = make_plan(s, z.plan) ? 1 : 0;
        z.n = s;
        z.tw = (int64_t)P.tw_elems;
        P.tw_elems += (size_t)s;
        P.sizes.push_back(z);
        return (int)P.sizes.size() - 1;
    };
    P.frames.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        const v5ela_gray_desc &d = frames[i];
        SpecFrame &f = P.frames[(size_t)i];
        f.gray = d.gray;
        f.out = d.out;
        f.row_stride = d.row_stride_bytes;
        f.h = d.height;
        f.w = d.width;
        f.wh = d.width / 2 + 1;
        f.sw = size_index(d.width);
        f.sh = size_index(d.height);
        FftPlan pw, ph;
        FftShape s;
        f.cc = fft_path(fft_on, f.h, f.w, pw, ph, s) ? s.cc : 0;
        f.gx = (f.wh + TILE - 1) / TILE;
        const ImageGrid ig = image_grid(f.h, f.w);
        f.bx = ig.bx;
        f.by = ig.by;
    }
    P.tw_base.resize(P.sizes.size() + 1);
    P.tw_base[0] = 0;
    for (size_t k = 0; k < P.sizes.size(); k++) P.tw_base[k + 1] = P.tw_base[k] + (uint32_t)((P.sizes[k].n + 255) / 256);
    // ---- chunks in frame order; workspace ranges 256-byte aligned
    size_t used = 0;
    for (int i = 0; i < n; i++) {
        SpecFrame &f = P.frames[(size_t)i];
        const size_t samples = (size_t)f.h * f.wh, g = spec_align(samples, 16), ms = spec_align(samples, 32);
        const size_t bytes = 16 * g + 8 * ms;
        if (P.chunks.empty() || used + bytes > chunk_bytes) {
            P.chunks.emplace_back();
            P.chunks.back().f0 = i;
            used = 0;
        }
        SpecChunk &C = P.chunks.back();
        f.g_off = (int64_t)C.g_elems;
        f.ms_off = (int64_t)C.ms_elems;
        f.mm = C.n;
        C.g_elems += g;
        C.ms_elems += ms;
        C.n++;
        used += bytes;
    }
    // ---- per chunk: the CTA prefix table of every launch
    P.launches = n > 0 ? 1 : 0;                                // the twiddle launch
    for (SpecChunk &C : P.chunks) {
        C.off_base = P.bases.size();
        P.bases.resize(P.bases.size() + (size_t)L_KINDS * (C.n + 1));
        uint32_t *base = P.bases.data() + C.off_base;
        uint64_t sum[L_KINDS] = {0, 0, 0, 0, 0};
        for (int j = 0; j < C.n; j++) {
            const SpecFrame &f = P.frames[(size_t)(C.f0 + j)];
            uint64_t cnt[L_KINDS] = {0, 0, 0, 0, 0};
            if (f.cc) {
                cnt[L_FFT_ROWS] = (uint64_t)(f.h + 1) / 2;
                cnt[L_FFT_COLS] = (uint64_t)(f.wh + f.cc - 1) / f.cc;
                const size_t rs = 16 * 2 * (size_t)f.w, cs = 16 * 2 * (size_t)f.cc * f.h;
                C.rows_smem = rs > C.rows_smem ? rs : C.rows_smem;
                C.cols_smem = cs > C.cols_smem ? cs : C.cols_smem;
            } else {
                cnt[L_DFT_ROWS] = cnt[L_DFT_COLS] = (uint64_t)f.gx * (uint64_t)((f.h + TILE - 1) / TILE);
            }
            cnt[L_IMAGE] = (uint64_t)f.bx * (uint64_t)f.by;
            for (int k = 0; k < L_KINDS; k++) {
                base[k * (C.n + 1) + j] = (uint32_t)sum[k];
                sum[k] += cnt[k];
            }
        }
        for (int k = 0; k < L_KINDS; k++) {
            if (sum[k] > 0x7fffffffull) {
                P.status = V5ELA_ERR_INVALID;
                P.error = "more than 2^31 - 1 CTAs in one launch";
                return;
            }
            base[k * (C.n + 1) + C.n] = (uint32_t)sum[k];
            C.ctas[k] = (uint32_t)sum[k];
            C.launches += sum[k] > 0 ? 1 : 0;
        }
        P.launches += C.launches;
        P.g_max = C.g_elems > P.g_max ? C.g_elems : P.g_max;
        P.ms_max = C.ms_elems > P.ms_max ? C.ms_elems : P.ms_max;
        P.mm_max = C.n > P.mm_max ? C.n : P.mm_max;
    }
    P.off_sizes = 0;
    P.off_frames = spec_align(sizeof(SpecSize) * P.sizes.size(), 16);
    P.off_tw_base = P.off_frames + spec_align(sizeof(SpecFrame) * P.frames.size(), 16);
    P.off_bases = P.off_tw_base + spec_align(sizeof(uint32_t) * P.tw_base.size(), 16);
    P.table_bytes = P.off_bases + spec_align(sizeof(uint32_t) * P.bases.size(), 16);
}

}  // namespace v5fft
