// v5jpeg_dct.cuh — DCT-domain statistics of JPEG files (v5ela_jpeg_dct_stats, DESIGN.md §4.8): per-frequency histograms of the
// quantised coefficients the decoder leaves in its workspace, and a per-block map of aligned double JPEG compression after
// Lin, He, Tang & Tang (2009). The decode plan runs up to dc_kernel (coefficients only: no IDCT, no colour, no planes), then
//
//   dct_hist_kernel  one CTA per (chunk of DQ_CHUNK blocks, file): a warp per block, lane l takes zigzag positions 2l, 2l+1
//                    (the DC VALUE from the dense DC array in place of position 0), shared-memory counters for the three
//                    components, flushed with one global atomic per non-zero counter; CTA 0 of a file writes its DQT tables
//   dct_lut_kernel   one warp per (file, luma AC frequency at zigzag position 1..15): the period p_k of the frequency's
//                    histogram and the 129-entry table log P_u(v), plus log P_t = -log p_k
//   dct_map_kernel   one thread per real luma block: 1 / (1 + exp(sum_k log P_u(v_k) - log P_t)) over the frequencies with p_k > 1
//
// The coefficient layout is the decoder's: block g of a file (scan order, MCU-interleaved) at coef[(coef_off + g) * 64 + z] with
// z the ZIGZAG index (z = 0 is never written), its DC value at dc[coef_off + g] once dc_kernel (or huffman_rst_kernel) has run.
// The per-block and per-warp arithmetic is __host__ __device__ so that tests/emu/v5jpeg_dct_emu.cpp runs it on the CPU; the
// estimator is restated in NumPy as v5ela.records.dq_periods / dq_map.
#pragma once
#include <math.h>
#include <stdint.h>

#include "v5ela_device.cuh"
#include "v5jpeg_dec.cuh"

namespace v5j {

constexpr int DQ_BINS = 129;                       // quantised values -64 .. 64, the end bins saturating
constexpr int DQ_HIST = 3 * 64 * DQ_BINS;          // one file: [component][natural-order frequency][value + 64]
constexpr int DQ_FREQS = 15;                       // luma AC frequencies of the map: zigzag positions 1 .. 15
constexpr int DQ_LUT = DQ_BINS + 1;                // one frequency's table: log P_u of every bin, then log P_t
constexpr int DQ_PMAX = 12;                        // candidate periods 2 .. DQ_PMAX
constexpr int DQ_TWIDDLES = (DQ_PMAX + 1) * DQ_PMAX / 2 - 1;   // sum of p over the candidates: 77
constexpr int DQ_CHUNK = 4096;                     // blocks per CTA of dct_hist_kernel
constexpr int DQ_HIST_NT = 512;
constexpr int DQ_MIN_COUNT = 64;                   // fewer folded AC values than this: p_k = 1
constexpr double DQ_TAU = 0.5;                     // S(p*) must reach this ...
constexpr double DQ_RHO = 0.05;                    // ... and sum |r| must reach DQ_RHO * N (DESIGN.md §4.8: how they were chosen)

// cos / sin (2 pi j / p) for p = 2 .. 12, j = 0 .. p-1, p-major (candidate p starts at dq_twiddle_base(p)); the same literals
// as v5ela.records, so that the GPU and the NumPy restatement multiply the same doubles.
V5_HOSTDEV int dq_twiddle_base(int p) { return p * (p - 1) / 2 - 1; }
#define V5J_DQ_COS \
    1.0, -1.0, \
    1.0, -0.5, -0.5, \
    1.0, 0.0, -1.0, 0.0, \
    1.0, 0.30901699437494745, -0.8090169943749475, -0.8090169943749475, 0.30901699437494745, \
    1.0, 0.5, -0.5, -1.0, -0.5, 0.5, \
    1.0, 0.6234898018587335, -0.2225209339563144, -0.9009688679024191, -0.9009688679024191, -0.2225209339563144, 0.6234898018587335, \
    1.0, 0.7071067811865476, 0.0, -0.7071067811865476, -1.0, -0.7071067811865476, 0.0, 0.7071067811865476, \
    1.0, 0.766044443118978, 0.17364817766693036, -0.5, -0.9396926207859084, -0.9396926207859084, -0.5, 0.17364817766693036, 0.766044443118978, \
    1.0, 0.8090169943749475, 0.30901699437494745, -0.30901699437494745, -0.8090169943749475, -1.0, -0.8090169943749475, -0.30901699437494745, \
    0.30901699437494745, 0.8090169943749475, \
    1.0, 0.8412535328311812, 0.41541501300188644, -0.14231483827328514, -0.6548607339452851, -0.9594929736144974, -0.9594929736144974, \
    -0.6548607339452851, -0.14231483827328514, 0.41541501300188644, 0.8412535328311812, \
    1.0, 0.8660254037844386, 0.5, 0.0, -0.5, -0.8660254037844386, -1.0, -0.8660254037844386, -0.5, 0.0, 0.5, 0.8660254037844386
#define V5J_DQ_SIN \
    0.0, 0.0, \
    0.0, 0.8660254037844386, -0.8660254037844386, \
    0.0, 1.0, 0.0, -1.0, \
    0.0, 0.9510565162951535, 0.5877852522924731, -0.5877852522924731, -0.9510565162951535, \
    0.0, 0.8660254037844386, 0.8660254037844386, 0.0, -0.8660254037844386, -0.8660254037844386, \
    0.0, 0.7818314824680298, 0.9749279121818236, 0.4338837391175581, -0.4338837391175581, -0.9749279121818236, -0.7818314824680298, \
    0.0, 0.7071067811865476, 1.0, 0.7071067811865476, 0.0, -0.7071067811865476, -1.0, -0.7071067811865476, \
    0.0, 0.6427876096865394, 0.984807753012208, 0.8660254037844386, 0.3420201433256687, -0.3420201433256687, -0.8660254037844386, \
    -0.984807753012208, -0.6427876096865394, \
    0.0, 0.5877852522924731, 0.9510565162951535, 0.9510565162951535, 0.5877852522924731, 0.0, -0.5877852522924731, -0.9510565162951535, \
    -0.9510565162951535, -0.5877852522924731, \
    0.0, 0.5406408174555976, 0.9096319953545183, 0.9898214418809327, 0.7557495743542583, 0.28173255684142967, -0.28173255684142967, \
    -0.7557495743542583, -0.9898214418809327, -0.9096319953545183, -0.5406408174555976, \
    0.0, 0.5, 0.8660254037844386, 1.0, 0.8660254037844386, 0.5, 0.0, -0.5, -0.8660254037844386, -1.0, -0.8660254037844386, -0.5
static const double kDqCos[DQ_TWIDDLES] = {V5J_DQ_COS}, kDqSin[DQ_TWIDDLES] = {V5J_DQ_SIN};
#ifdef __CUDACC__
__constant__ double kDqCosDev[DQ_TWIDDLES] = {V5J_DQ_COS}, kDqSinDev[DQ_TWIDDLES] = {V5J_DQ_SIN};
#endif
V5_HOSTDEV double dq_cos(int i)
{
#ifdef __CUDA_ARCH__
    return kDqCosDev[i];
#else
    return kDqCos[i];
#endif
}
V5_HOSTDEV double dq_sin(int i)
{
#ifdef __CUDA_ARCH__
    return kDqSinDev[i];
#else
    return kDqSin[i];
#endif
}

// Rounded double operations that the compiler may not fuse into an FMA: the period decision must come out the same on the GPU
// and in NumPy (which never fuses).
V5_HOSTDEV double dq_mul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
V5_HOSTDEV double dq_add(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// ---------------------------------------------------------------------------------------------------- block geometry
// Block g (scan order) of a file: its component (0 luma, 1 Cb, 2 Cr) and its column / row in that component's block grid.
V5_HOSTDEV int dq_block_pos(const DecImage &im, int g, int &bx, int &by)
{
    if (im.bpm == 1) {
        by = g / im.mcux;
        bx = g - by * im.mcux;
        return 0;
    }
    const int m = g / im.bpm, i = g - im.bpm * m, ny = im.bpm - 2;
    const int my = m / im.mcux, mx = m - my * im.mcux;
    if (i < ny) {                                                         // luma blocks of an MCU: row-major, hs across
        bx = im.hs * mx + (im.hs == 2 ? (i & 1) : 0);
        by = im.vs * my + (im.hs == 2 ? (i >> 1) : i);                   // (vs == 2 implies hs == 2)
        return 0;
    }
    bx = mx;
    by = my;
    return i - ny + 1;
}

// A real block covers samples of the component: bx < ceil(ceil(W h_c / h_max) / 8), likewise down. The others pad the MCU grid.
V5_HOSTDEV bool dq_block_real(const DecImage &im, int comp, int bx, int by)
{
    const int cw = comp ? (im.w + im.hs - 1) / im.hs : im.w, ch = comp ? (im.h + im.vs - 1) / im.vs : im.h;
    return bx < (cw + 7) / 8 && by < (ch + 7) / 8;
}

// The scan-order index of real luma block (bx, by).
V5_HOSTDEV int dq_luma_block(const DecImage &im, int bx, int by)
{
    if (im.bpm == 1) return by * im.mcux + bx;
    const int mx = bx / im.hs, my = by / im.vs, i = (by - im.vs * my) * im.hs + (bx - im.hs * mx);
    return (my * im.mcux + mx) * im.bpm + i;
}

V5_HOSTDEV int dq_bin(int v) { return (v < -64 ? -64 : (v > 64 ? 64 : v)) + 64; }

// dct_hist_kernel, lane `lane` of the warp that takes a block of component `comp`: the counters (inside a file's histogram)
// of zigzag positions 2 lane and 2 lane + 1. `pair` is the block's 32-bit coefficient word `lane` (position 2 lane in the low
// half), `dcv` the block's DC value, which stands in for position 0. z2n: zigzag -> natural order.
V5_HOSTDEV void dq_lane_bins(int comp, int lane, uint32_t pair, int dcv, const uint8_t *z2n, int bins[2])
{
    const int v0 = lane == 0 ? dcv : (int)(int16_t)(pair & 0xffffu), v1 = (int)(int16_t)(pair >> 16);
    bins[0] = (comp * 64 + z2n[2 * lane]) * DQ_BINS + dq_bin(v0);
    bins[1] = (comp * 64 + z2n[2 * lane + 1]) * DQ_BINS + dq_bin(v1);
}

// ------------------------------------------------------------------------------------------- period of one frequency
// h: the frequency's 129 bins (value v at h[v + 64]). Folded g(v) = h(v) + h(-v), v = 1..63; 2r(v) = 2 g(v) - g(v-1) - g(v+1),
// v = 2..62 (twice the residual, so that everything stays integer: sums of up to 4 N, N < 2^27 for any baseline file).
V5_HOSTDEV int dq_fold(const uint32_t *h, int v) { return (int)(h[64 + v] + h[64 - v]); }

struct DqLane {                  // what lane l of dct_lut_kernel's warp contributes before the warp sums
    int n;                       // g(v) over v = l + 1, l + 33 (<= 63)
    int abs2r;                   // |2r(v)| over v = l + 2, l + 34 (<= 62)
    int va, ra, vb, rb;          // those two v and their 2r (rb = 0 when vb > 62)
};

V5_HOSTDEV void dq_lane(const uint32_t *h, int lane, DqLane &L)
{
    L.n = dq_fold(h, lane + 1) + (lane + 33 <= 63 ? dq_fold(h, lane + 33) : 0);
    L.va = lane + 2;
    L.vb = lane + 34;
    L.ra = 2 * dq_fold(h, L.va) - dq_fold(h, L.va - 1) - dq_fold(h, L.va + 1);
    L.rb = L.vb <= 62 ? 2 * dq_fold(h, L.vb) - dq_fold(h, L.vb - 1) - dq_fold(h, L.vb + 1) : 0;
    L.abs2r = (L.ra < 0 ? -L.ra : L.ra) + (L.rb < 0 ? -L.rb : L.rb);
}

// the lane's share of R_j(p) = sum of 2r(v) over v = j (mod p)
V5_HOSTDEV int dq_lane_residue(const DqLane &L, int p, int j) { return (L.va % p == j ? L.ra : 0) + (L.vb % p == j ? L.rb : 0); }

// S(p) = |sum_v 2r(v) e^{-2 pi i v / p}| / max(sum |2r|, 2) from the residue sums R[dq_twiddle_base(p) + j] (= |sum r e^..| /
// max(sum |r|, 1)). Real and imaginary parts are summed over j = 0 .. p-1 in that order.
V5_HOSTDEV double dq_score(const int *R, int p, int abs2r)
{
    const int b = dq_twiddle_base(p);
    double re = 0.0, im = 0.0;
    for (int j = 0; j < p; j++) {
        re = dq_add(re, dq_mul((double)R[b + j], dq_cos(b + j)));
        im = dq_add(im, dq_mul((double)R[b + j], dq_sin(b + j)));
    }
    const double mag = sqrt(dq_add(dq_mul(re, re), dq_mul(im, im)));
    return mag / (double)(abs2r > 2 ? abs2r : 2);
}

// p_k from the warp's sums: N, sum |2r| and the 77 residue sums
V5_HOSTDEV int dq_choose_period(const int *R, int abs2r, int n)
{
    if (n < DQ_MIN_COUNT) return 1;
    int best = 2;
    double s_best = dq_score(R, 2, abs2r);
    for (int p = 3; p <= DQ_PMAX; p++) {
        const double s = dq_score(R, p, abs2r);
        if (s > s_best) {                                                 // the smaller p wins ties
            s_best = s;
            best = p;
        }
    }
    return s_best >= DQ_TAU && dq_mul(0.5, (double)abs2r) >= dq_mul(DQ_RHO, (double)n) ? best : 1;
}

// Table entry b (v = b - 64) for period p: log(h(v) / sum of h over the p bins from p floor(v / p) on, clipped to -63 .. 63),
// log(1 / p) when that group is empty; the saturating end bins v = +-64 take the entries of v = +-63. Entry DQ_BINS: log P_t.
V5_HOSTDEV double dq_lut_entry(const uint32_t *h, int p, int b)
{
    if (b == DQ_BINS) return -log((double)p);
    int v = b - 64;
    v = v > 63 ? 63 : (v < -63 ? -63 : v);
    const int s = v >= 0 ? (v / p) * p : -((-v + p - 1) / p) * p;
    uint32_t mass = 0;
    for (int u = s; u < s + p; u++)
        if (u >= -63 && u <= 63) mass += h[64 + u];
    if (mass == 0) return -log((double)p);
    return log((double)h[64 + v] / (double)mass);
}

// dct_map_kernel, one luma block: blk = its 64 coefficients in zigzag order (position 0 is not read); lut / period: the file's
// DQ_FREQS tables and periods. The posterior that the block was NOT aligned-double-compressed; 0.5 when no frequency has p > 1.
V5_HOSTDEV float dq_map_block(const int16_t *blk, const double *lut, const int32_t *period)
{
    double s = 0.0;
    bool any = false;
    for (int f = 0; f < DQ_FREQS; f++) {
        if (period[f] <= 1) continue;
        const double *t = lut + f * DQ_LUT;
        s += t[dq_bin(blk[f + 1])] - t[DQ_BINS];
        any = true;
    }
    return any ? (float)(1.0 / (1.0 + exp(s))) : 0.5f;
}

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------------- kernels
// grid = (ceil(max blocks / DQ_CHUNK), files of the chunk). hist: the chunk's first file's histogram (zeroed by the caller).
// qtab_out (optional): [file][component][64] natural order, the components a file does not have left zero.
__global__ void __launch_bounds__(DQ_HIST_NT) dct_hist_kernel(const DecImage *images, const uint16_t *qtabs, const int16_t *coef,
                                                              const int16_t *dc, uint32_t *hist, uint16_t *qtab_out)
{
    extern __shared__ __align__(16) uint32_t dq_counts[];                 // DQ_HIST counters
    __shared__ uint8_t z2n[64];
    const DecImage im = images[blockIdx.y];
    const int t = (int)threadIdx.x;
    if (qtab_out && blockIdx.x == 0 && t < 3 * 64) {
        const int c = t >> 6, k = t & 63;
        qtab_out[(int64_t)blockIdx.y * 3 * 64 + t] = c < im.ncomp ? qtabs[(int64_t)im.qt * 128 + (c ? 64 : 0) + k] : (uint16_t)0;
    }
    const int g0 = (int)blockIdx.x * DQ_CHUNK;
    if (g0 >= im.blocks) return;
    const int used = im.ncomp * 64 * DQ_BINS;                             // counters of the components the file has
    for (int i = t; i < used; i += DQ_HIST_NT) dq_counts[i] = 0u;
    if (t < 64) z2n[t] = kZigzagToNaturalDev[t];
    __syncthreads();
    const int lane = t & 31, g_end = im.blocks - g0 < DQ_CHUNK ? im.blocks : g0 + DQ_CHUNK;
    const uint32_t *words = reinterpret_cast<const uint32_t *>(coef + im.coef_off * 64);
    for (int g = g0 + (t >> 5); g < g_end; g += DQ_HIST_NT / 32) {
        int bx, by;
        const int comp = dq_block_pos(im, g, bx, by);
        if (!dq_block_real(im, comp, bx, by)) continue;                  // warp-uniform
        const uint32_t pair = __ldg(words + (int64_t)g * 32 + lane);
        const int dcv = lane == 0 ? (int)dc[im.coef_off + g] : 0;
        int bins[2];
        dq_lane_bins(comp, lane, pair, dcv, z2n, bins);
        atomicAdd(&dq_counts[bins[0]], 1u);
        atomicAdd(&dq_counts[bins[1]], 1u);
    }
    __syncthreads();
    uint32_t *dst = hist + (int64_t)blockIdx.y * DQ_HIST;
    for (int i = t; i < used; i += DQ_HIST_NT) {
        const uint32_t v = dq_counts[i];
        if (v) atomicAdd(dst + i, v);
    }
}

// grid = files of the chunk, DQ_FREQS warps: warp f estimates the period of the luma frequency at zigzag position f + 1 and
// writes its table. lut: [file][DQ_FREQS][DQ_LUT], period: [file][DQ_FREQS].
__global__ void __launch_bounds__(DQ_FREQS * 32) dct_lut_kernel(const uint32_t *hist, double *lut, int32_t *period)
{
    const int f = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
    const uint32_t *h = hist + (int64_t)blockIdx.x * DQ_HIST + kZigzagToNaturalDev[f + 1] * DQ_BINS;
    DqLane L;
    dq_lane(h, lane, L);
    const int n = __reduce_add_sync(0xffffffffu, L.n), abs2r = __reduce_add_sync(0xffffffffu, L.abs2r);
    int R[DQ_TWIDDLES];
#pragma unroll
    for (int p = 2; p <= DQ_PMAX; p++)
#pragma unroll
        for (int j = 0; j < p; j++) R[dq_twiddle_base(p) + j] = __reduce_add_sync(0xffffffffu, dq_lane_residue(L, p, j));
    const int p = dq_choose_period(R, abs2r, n);
    double *row = lut + ((int64_t)blockIdx.x * DQ_FREQS + f) * DQ_LUT;
    for (int b = lane; b < DQ_LUT; b += 32) row[b] = dq_lut_entry(h, p, b);
    if (lane == 0) period[blockIdx.x * DQ_FREQS + f] = p;
}

// grid = (ceil(max luma blocks / 256), files of the chunk). map_offs: element offset of every file's map.
__global__ void __launch_bounds__(256) dct_map_kernel(const DecImage *images, const int64_t *map_offs, const int16_t *coef,
                                                      const double *lut, const int32_t *period, float *map)
{
    const DecImage im = images[blockIdx.y];
    const int bw = (im.w + 7) >> 3, bh = (im.h + 7) >> 3;
    const int i = (int)blockIdx.x * 256 + (int)threadIdx.x;
    if (i >= bw * bh) return;
    const int by = i / bw, bx = i - by * bw;
    const int16_t *blk = coef + (im.coef_off + dq_luma_block(im, bx, by)) * 64;
    map[map_offs[blockIdx.y] + i] = dq_map_block(blk, lut + (int64_t)blockIdx.y * DQ_FREQS * DQ_LUT, period + blockIdx.y * DQ_FREQS);
}
#endif  // __CUDACC__

}  // namespace v5j
