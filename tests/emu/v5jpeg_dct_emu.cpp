// tests/emu/v5jpeg_dct_emu.cpp — TEST INFRASTRUCTURE: runs the host/device-shared logic of the DCT-statistics kernels
// (csrc/v5jpeg_dct.cuh compiled by g++) over a file's quantised coefficients, with the CTAs, warps and lanes of dct_hist_kernel,
// dct_lut_kernel and dct_map_kernel emulated sequentially, so that block geometry, the coefficient layout, the period decision
// and the map can be checked against NumPy in a container without a GPU. The warp sums are plain loops here; the CUDA versions
// are covered by the -m gpu tests. NOT a CPU fallback: nothing under fake-video-detection-engine_b200/ loads it.
//
// Build (tests/test_dct_stats_emu.py does it): g++ -O2 -shared -fPIC -ffp-contract=off -I include -I <csrc> ...
#include <cstdlib>
#include <cstring>
#include <vector>

#include "v5jpeg_dct.cuh"

using namespace v5j;

// dct_lut_kernel's warp for one frequency: histogram h (129 bins) -> period, table row (DQ_LUT entries)
static int emu_lut_warp(const uint32_t *h, double *row)
{
    DqLane L[32];
    int n = 0, abs2r = 0, R[DQ_TWIDDLES];
    for (int lane = 0; lane < 32; lane++) {
        dq_lane(h, lane, L[lane]);
        n += L[lane].n;
        abs2r += L[lane].abs2r;
    }
    for (int p = 2; p <= DQ_PMAX; p++)
        for (int j = 0; j < p; j++) {
            int sum = 0;
            for (int lane = 0; lane < 32; lane++) sum += dq_lane_residue(L[lane], p, j);
            R[dq_twiddle_base(p) + j] = sum;
        }
    const int p = dq_choose_period(R, abs2r, n);
    for (int b = 0; b < DQ_LUT; b++) row[b] = dq_lut_entry(h, p, b);
    return p;
}

extern "C" int v5jdct_emu_period(const uint32_t *h, double *row) { return emu_lut_warp(h, row); }

extern "C" void v5jdct_emu_twiddles(double *cos_out, double *sin_out)
{
    for (int i = 0; i < DQ_TWIDDLES; i++) {
        cos_out[i] = dq_cos(i);
        sin_out[i] = dq_sin(i);
    }
}

// One file. coef: every block of the scan (dummy blocks included) in scan order, zigzag order inside the block, DC values at
// position 0 — what the oracle decoder exports. They are laid out the way the GPU decoder leaves them (AC coefficients at
// their zigzag index, position 0 zero, DC values in a dense array of their own) before the kernels' logic runs.
// Outputs: hist [DQ_HIST], qtab [3][64], period [DQ_FREQS], lut [DQ_FREQS][DQ_LUT], map [ceil(H/8)][ceil(W/8)].
// Returns 0, or the parse error.
extern "C" int v5jdct_emu_stats(const uint8_t *data, int64_t len, const int16_t *coef, uint32_t *hist, uint16_t *qtab, int32_t *period,
                                double *lut, float *map)
{
    FileInfo *F = new FileInfo();
    const int rc = parse_file(data, (size_t)len, *F);
    if (rc) {
        delete F;
        return rc;
    }
    DecImage im;
    memset(&im, 0, sizeof(im));
    dec_geometry(im, F->h, F->w, F->ncomp, F->hs, F->vs);
    std::vector<int16_t> dcoef((size_t)im.blocks * 64), dcv((size_t)im.blocks);
    for (int g = 0; g < im.blocks; g++) {
        memcpy(&dcoef[(size_t)g * 64], coef + (size_t)g * 64, 128);
        dcoef[(size_t)g * 64] = 0;
        dcv[(size_t)g] = coef[(size_t)g * 64];
    }
    // ---- dct_hist_kernel: CTAs of DQ_CHUNK blocks, DQ_HIST_NT / 32 warps striding over them, shared counters, flush
    memset(hist, 0, sizeof(uint32_t) * DQ_HIST);
    std::vector<uint32_t> counts(DQ_HIST);
    for (int g0 = 0; g0 < im.blocks; g0 += DQ_CHUNK) {
        std::fill(counts.begin(), counts.end(), 0xA5A5A5A5u);                // poison: the kernel zeroes what it uses
        const int used = im.ncomp * 64 * DQ_BINS;
        for (int i = 0; i < used; i++) counts[(size_t)i] = 0;
        const int g_end = im.blocks - g0 < DQ_CHUNK ? im.blocks : g0 + DQ_CHUNK;
        for (int w = DQ_HIST_NT / 32; w-- > 0;)                              // any order: warps are independent
            for (int g = g0 + w; g < g_end; g += DQ_HIST_NT / 32) {
                int bx, by;
                const int comp = dq_block_pos(im, g, bx, by);
                if (!dq_block_real(im, comp, bx, by)) continue;
                for (int lane = 0; lane < 32; lane++) {
                    const int16_t *b = &dcoef[(size_t)g * 64 + 2 * lane];
                    const uint32_t pair = (uint32_t)(uint16_t)b[0] | ((uint32_t)(uint16_t)b[1] << 16);
                    int bins[2];
                    dq_lane_bins(comp, lane, pair, lane == 0 ? dcv[(size_t)g] : 0, kZigzag, bins);
                    counts[(size_t)bins[0]]++;
                    counts[(size_t)bins[1]]++;
                }
            }
        for (int i = 0; i < used; i++) hist[i] += counts[(size_t)i];
    }
    for (int c = 0; c < 3; c++)
        for (int k = 0; k < 64; k++) qtab[c * 64 + k] = c < im.ncomp ? F->qt[c ? 1 : 0][k] : 0;
    // ---- dct_lut_kernel: one warp per luma frequency at zigzag positions 1 .. DQ_FREQS
    for (int f = 0; f < DQ_FREQS; f++) period[f] = emu_lut_warp(hist + kZigzag[f + 1] * DQ_BINS, lut + f * DQ_LUT);
    // ---- dct_map_kernel: one thread per real luma block
    const int bw = (im.w + 7) / 8, bh = (im.h + 7) / 8;
    for (int i = 0; i < bw * bh; i++) {
        const int by = i / bw, bx = i - by * bw;
        map[i] = dq_map_block(&dcoef[(size_t)dq_luma_block(im, bx, by) * 64], lut, period);
    }
    delete F;
    return 0;
}
