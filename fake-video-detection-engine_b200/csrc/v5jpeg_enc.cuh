// v5jpeg_enc.cuh — baseline JPEG encoder on the GPU (SURVEY.md §8f-3): the artefact files the reference writes with
// PIL / OpenCV (v5_texture_ela.py:66-67 temp_ela_i.jpg q90, :80-81 ela_i.jpg q75, :90-91 fft_i.jpg q95 one component),
// byte-identical to libjpeg's output. Five launches per batch of equally sized images:
//
//   coef_kernel     colour convert + h2v2 downsample (SURVEY App. A.2/A.3) + ISLOW fDCT + quantise (A.4/A.5), one CTA per
//                   strip of 16 MCUs -> int16 coefficients, scan (MCU-interleaved) block order, zigzag order in the block
//   count_kernel    one thread per block: Huffman-coded length in bits (T.81 F.1.2, Annex K.3 tables)
//   scan_kernel     one CTA per image: exclusive prefix sum of the lengths -> bit offset of every block, total bits
//   write_kernel    one thread per block: codes -> 32-bit big-endian words of the unstuffed bit stream (only the two words a
//                   block shares with its neighbours need atomics)
//   stuff_kernel    one CTA per image: header + byte stuffing (FF -> FF 00) + one-bit padding + EOI -> the file
//
// The per-block logic is __host__ __device__ so that tests/emu can run it on the CPU (a debugging aid, not a fallback).
#pragma once
#include <stdint.h>

#include "v5ela_device.cuh"
#include "v5jpeg_common.h"

namespace v5j {

using v5::U2;
using v5::U4;

constexpr int ENC_NT = 384;            // coef_kernel: 96 blocks x 4 threads
constexpr int ENC_TM = 16;             // MCUs (colour) per CTA strip; 96 blocks per strip in either mode
constexpr int ENC_BLOCKS = 96;

struct EncQuant {                      // exact division by 8T, see v5plan::make_quant: q = umulhi(c + (c>>31) + bias, recip) - b
    uint32_t recip[64];
    int32_t bias[64];
    int32_t b[64];
};

struct EncGeo {
    int h, w, ncomp;
    int mcux, mcuy;                    // MCU grid: 16x16 px (colour) or 8x8 px (one component)
    int bpm;                           // blocks per MCU: 6 or 1
    int ybw, ybh;                      // real luma blocks per row / column
    int blocks;                        // blocks per image = mcux * mcuy * bpm
};

inline EncGeo enc_geo(int h, int w, int ncomp)
{
    EncGeo g;
    g.h = h; g.w = w; g.ncomp = ncomp;
    const int m = ncomp == 3 ? 16 : 8;
    g.mcux = (w + m - 1) / m; g.mcuy = (h + m - 1) / m;
    g.bpm = ncomp == 3 ? 6 : 1;
    g.ybw = (w + 7) / 8; g.ybh = (h + 7) / 8;
    g.blocks = g.mcux * g.mcuy * g.bpm;
    return g;
}

inline void make_enc_quant(const uint16_t tab[64], EncQuant &q)
{
    for (int i = 0; i < 64; i++) {
        const uint32_t d = (uint32_t)tab[i] << 3, b = (8192u + d - 1) / d;
        q.recip[i] = (uint32_t)(0x100000000ull / d) + 1u;
        q.bias[i] = (int32_t)(d / 2 + b * d);
        q.b[i] = (int32_t)b;
    }
}

struct CoefParams {
    const uint8_t *img;
    int64_t frame_stride, row_stride;
    int16_t *coef;                     // [n][blocks][64]
    EncGeo g;
    EncQuant q[2];
};

// --------------------------------------------------------------------------------------------------- coef_kernel
struct alignas(16) CoefSmem {
    // sample planes of the strip. colour: Y 16 x 256 at [0], Cb and Cr 8 x 128 each at [4096]; one component: 8 x 768 at [0]
    uint8_t px[16 * ENC_TM * 16 + 2 * 8 * ENC_TM * 8];
    V5_HOSTDEV uint8_t *y(int row) { return px + row * (ENC_TM * 16); }
    V5_HOSTDEV uint8_t *c(int comp, int row) { return px + 16 * ENC_TM * 16 + (comp * 8 + row) * (ENC_TM * 8); }
    V5_HOSTDEV const uint8_t *y(int row) const { return px + row * (ENC_TM * 16); }
    V5_HOSTDEV const uint8_t *c(int comp, int row) const { return px + 16 * ENC_TM * 16 + (comp * 8 + row) * (ENC_TM * 8); }
    alignas(16) int16_t ws[ENC_BLOCKS][64 + 8];    // per block workspace, natural order (row stride 16 B, block stride 144 B)
    uint8_t zz[64];
    alignas(16) uint8_t rgb[16][3 * 16 * ENC_TM];   // colour only: the strip's pixels, edges replicated
    // exact-division constants {recip, bias, b, -} per coefficient, [0] luma [1] chroma: one 128-bit shared load each
    // (read straight from the kernel parameters they would be divergent constant-bank loads, which throttle the MIO queue)
    alignas(16) uint32_t q[2][64][4];
};
static_assert(8 * 8 * ENC_BLOCKS <= 16 * ENC_TM * 16 + 2 * 8 * ENC_TM * 8, "the one-component strip must fit the plane area");

// Luma block i of an MCU that lies outside the component's real block grid is a libjpeg "dummy" block: all zero except a
// DC copied from the block before it in the MCU (jccoefct.c). Returns the real block that DC finally comes from.
V5_HOSTDEV int dummy_source(const EncGeo &g, int mx, int my, int i)
{
    for (;;) {
        const int gy = 2 * my + (i >> 1), gx = 2 * mx + (i & 1);
        if ((gy < g.ybh && gx < g.ybw) || i == 0) return i;
        i--;
    }
}

// Stage the strip's RGB (16 lines x up to 256 px) in shared memory — 32-bit loads when the frame allows it — with the
// right / bottom edges replicated (A.3), then convert 2x2 quads from there.
V5_DEV void coef_stage_rgb(int tid, CoefSmem &S, const CoefParams &p, const uint8_t *frame, int tile_x, int my)
{
    const EncGeo &g = p.g;
    const int x_begin = 16 * ENC_TM * tile_x;                            // first pixel column of the strip
    int npx = g.w - x_begin;                                             // real pixels in the strip
    npx = npx > 16 * ENC_TM ? 16 * ENC_TM : npx;
    const int nbytes = 3 * npx;
    const bool vec = ((reinterpret_cast<uintptr_t>(frame) | (uintptr_t)p.row_stride) & 3) == 0;   // 3 * x_begin is a multiple of 4
    const int nw = vec ? nbytes >> 2 : 0;                                // 32-bit words per line
    const int pad3 = 3 * (16 * ((npx + 15) / 16) - npx);                 // replicate pixel W-1 up to the next MCU boundary
    const int64_t col0 = 3 * (int64_t)x_begin;
    for (int e = tid; e < 16 * nw; e += ENC_NT) {
        const int l = e / nw, i = e - l * nw;
        int y = 16 * my + l;
        y = y < g.h - 1 ? y : g.h - 1;
        reinterpret_cast<uint32_t *>(S.rgb[l])[i] = reinterpret_cast<const uint32_t *>(frame + (int64_t)y * p.row_stride + col0)[i];
    }
    const int rest = nbytes - 4 * nw + pad3;                             // bytes per line not covered by the word copies
    for (int e = tid; e < 16 * rest; e += ENC_NT) {
        const int l = e / rest, i = 4 * nw + (e - l * rest);
        int y = 16 * my + l;
        y = y < g.h - 1 ? y : g.h - 1;
        const uint8_t *src = frame + (int64_t)y * p.row_stride + col0;
        S.rgb[l][i] = i < nbytes ? src[i] : src[nbytes - 3 + ((i - nbytes) % 3)];
    }
}

// units of 2 lines x 8 px through the fused kernel's packed-byte conversion (v5::convert8x2: dp2a colour conversion,
// h2v2 box filter with the 1,2,1,2 bias)
V5_DEV void coef_load_colour(int tid, CoefSmem &S, const CoefParams &p, int tile_x, int my)
{
    const EncGeo &g = p.g;
    const int hc1 = ((g.h + 1) >> 1) - 1;
    const int mcus = g.mcux - tile_x * ENC_TM < ENC_TM ? g.mcux - tile_x * ENC_TM : ENC_TM;
    for (int u = tid; u < 8 * 2 * ENC_TM; u += ENC_NT) {
        const int li = u / (2 * ENC_TM), ox = u - li * (2 * ENC_TM);
        if (ox >= 2 * mcus) continue;
        U2 y0, y1;
        uint32_t cb, cr;
        v5::convert8x2<true, true>(&S.rgb[2 * li][24 * ox], &S.rgb[2 * li + 1][24 * ox], y0, y1, cb, cr);
        // staged lines already replicate row H-1; below the image the chroma rule differs: it replicates the DOWNSAMPLED last
        // row, i.e. averages rows (2 jc, min(2 jc + 1, H-1)) with jc = min(j, Hc-1) — both inside this MCU row's 16 lines
        const int j = 8 * my + li, jc = j < hc1 ? j : hc1;
        const int l0 = 2 * jc - 16 * my, l1 = (2 * jc + 1 < g.h - 1 ? 2 * jc + 1 : g.h - 1) - 16 * my;
        if (l0 != 2 * li || l1 != 2 * li + 1) {
            U2 d0, d1;
            v5::convert8x2<false, true>(&S.rgb[l0][24 * ox], &S.rgb[l1][24 * ox], d0, d1, cb, cr);
        }
        *reinterpret_cast<U2 *>(S.y(2 * li) + 8 * ox) = y0;
        *reinterpret_cast<U2 *>(S.y(2 * li + 1) + 8 * ox) = y1;
        *reinterpret_cast<uint32_t *>(S.c(0, li) + 4 * ox) = cb;
        *reinterpret_cast<uint32_t *>(S.c(1, li) + 4 * ox) = cr;
    }
}

V5_DEV void coef_load_gray(int tid, CoefSmem &S, const CoefParams &p, const uint8_t *frame, int tile_x, int my)
{
    const EncGeo &g = p.g;
    uint8_t *plane = S.px;                                               // 8 x 768
    const int blocks = g.mcux - tile_x * ENC_BLOCKS < ENC_BLOCKS ? g.mcux - tile_x * ENC_BLOCKS : ENC_BLOCKS;
    for (int e = tid; e < 8 * 8 * ENC_BLOCKS; e += ENC_NT) {
        const int y = e / (8 * ENC_BLOCKS), x = e - y * (8 * ENC_BLOCKS);
        if (x >= 8 * blocks) continue;
        const int gx = 8 * ENC_BLOCKS * tile_x + x, gy = 8 * my + y;
        plane[y * (8 * ENC_BLOCKS) + x] = frame[(int64_t)(gy < g.h - 1 ? gy : g.h - 1) * p.row_stride + (gx < g.w - 1 ? gx : g.w - 1)];
    }
}

V5_DEV void coef_load_quant(int tid, CoefSmem &S, const CoefParams &p)
{
    if (tid < 128) {
        const int t = tid >> 6, i = tid & 63;
        S.q[t][i][0] = p.q[t].recip[i];
        S.q[t][i][1] = (uint32_t)p.q[t].bias[i];
        S.q[t][i][2] = (uint32_t)p.q[t].b[i];
        S.q[t][i][3] = 0;
    }
}

// where block b of the strip reads its samples
V5_DEV const uint8_t *coef_block_src(const CoefSmem &S, int ncomp, int b, int &pitch)
{
    if (ncomp == 1) {
        pitch = 8 * ENC_BLOCKS;
        return S.px + 8 * b;
    }
    const int m = b / 6, i = b - 6 * m;
    if (i < 4) {
        pitch = ENC_TM * 16;
        return S.y(8 * (i >> 1)) + 16 * m + 8 * (i & 1);
    }
    pitch = ENC_TM * 8;
    return S.c(i - 4, 0) + 8 * m;
}

// thread (b, j): rows 2j, 2j+1 of block b -> ws (row pass of the forward DCT); 64-bit loads, 128-bit stores
V5_DEV void coef_rows(int tid, CoefSmem &S, int ncomp, int nblocks)
{
    const int b = tid >> 2, j = tid & 3;
    if (b >= nblocks) return;
    int pitch;
    const uint8_t *src = coef_block_src(S, ncomp, b, pitch);
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int r = 2 * j + rr;
        const U2 w = *reinterpret_cast<const U2 *>(src + r * pitch);
        int v[8];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            v[k] = (int)v5::byte_of(w.x, k);
            v[4 + k] = (int)v5::byte_of(w.y, k);
        }
        v5::fdct8<1, true>(v);
        *reinterpret_cast<U4 *>(&S.ws[b][8 * r]) = U4{v5::pack_s16(v[0], v[1]), v5::pack_s16(v[2], v[3]), v5::pack_s16(v[4], v[5]), v5::pack_s16(v[6], v[7])};
    }
}

// thread (b, j): columns 2j, 2j+1 (one 32-bit word per row) -> column pass, exact quantisation, back into ws
V5_DEV void coef_cols(int tid, CoefSmem &S, const CoefParams &p, int nblocks)
{
    const int b = tid >> 2, j = tid & 3;
    if (b >= nblocks) return;
    const uint32_t(*q)[4] = S.q[(p.g.ncomp == 3 && (b % 6) >= 4) ? 1 : 0];
    uint32_t *wsw = reinterpret_cast<uint32_t *>(S.ws[b]);               // row k = words 4k .. 4k+3
    int a[8], c[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t w = wsw[4 * k + j];
        a[k] = v5::s16_lo(w);
        c[k] = v5::s16_hi(w);
    }
    v5::fdct8<1, false>(a);
    v5::fdct8<1, false>(c);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int i = 8 * k + 2 * j;
        const U4 qa = *reinterpret_cast<const U4 *>(q[i]), qc = *reinterpret_cast<const U4 *>(q[i + 1]);
        const uint32_t xa = (uint32_t)(a[k] + (a[k] >> 31) + (int)qa.y), xc = (uint32_t)(c[k] + (c[k] >> 31) + (int)qc.y);
        wsw[4 * k + j] = v5::pack_s16((int)v5::umulhi32(xa, qa.x) - (int)qa.z, (int)v5::umulhi32(xc, qc.x) - (int)qc.z);
    }
}

// all threads: ws -> global, zigzag order, dummy luma blocks replaced by their definition
V5_DEV void coef_store(int tid, const CoefSmem &S, const CoefParams &p, int16_t *dst, int mx0, int my, int nblocks)
{
    for (int e = tid; e < nblocks * 32; e += ENC_NT) {                   // two coefficients per step
        const int b = e >> 5, k = (e & 31) * 2;
        int v0 = S.ws[b][S.zz[k]], v1 = S.ws[b][S.zz[k + 1]];
        if (p.g.ncomp == 3) {
            const int m = b / 6, i = b - 6 * m;
            if (i > 0 && i < 4) {
                const int src = dummy_source(p.g, mx0 + m, my, i);
                if (src != i) {
                    v0 = k == 0 ? S.ws[6 * m + src][0] : 0;
                    v1 = 0;
                }
            }
        }
        reinterpret_cast<uint32_t *>(dst)[e] = ((uint32_t)v0 & 0xffffu) | ((uint32_t)v1 << 16);
    }
}

// --------------------------------------------------------------------------------- per-block entropy coding (F.1.2)
// Scan-order predecessor of block g for the DC prediction: the previous block of the same component, or -1.
V5_HOSTDEV int dc_predecessor(int g, int bpm)
{
    if (bpm == 1) return g - 1;
    const int m = g / 6, i = g - 6 * m;
    if (i >= 1 && i <= 3) return g - 1;
    if (m == 0) return -1;
    return i == 0 ? 6 * (m - 1) + 3 : g - 6;
}

V5_HOSTDEV int bit_length(uint32_t v)
{
#ifdef __CUDA_ARCH__
    return 32 - __clz((int)v);
#else
    int n = 0;
    while (v) { n++; v >>= 1; }
    return n;
#endif
}

struct BitCounter {
    uint32_t total = 0;
    V5_HOSTDEV void put(uint32_t, int len) { total += (uint32_t)len; }
};

// Appends to a stream of 32-bit words holding the bit stream most-significant-bit first. Words fully owned by this block
// are stored; the first and the last word may be shared with the neighbouring blocks and are OR-ed atomically into a
// zero-initialised buffer.
struct BitSink {
    uint32_t *raw;
    uint32_t wi;
    uint64_t acc;
    int nacc;
    bool first;
    V5_HOSTDEV void init(uint32_t *raw_, uint64_t bitoff)
    {
        raw = raw_;
        wi = (uint32_t)(bitoff >> 5);
        acc = 0;
        nacc = (int)(bitoff & 31);
        first = true;
    }
    V5_HOSTDEV void or_word(uint32_t word)
    {
#ifdef __CUDA_ARCH__
        if (word) atomicOr(&raw[wi], word);
#else
        raw[wi] |= word;
#endif
    }
    V5_HOSTDEV void put(uint32_t bits, int len)
    {
        acc = (acc << len) | bits;
        nacc += len;
        if (nacc >= 32) {
            const uint32_t word = (uint32_t)(acc >> (nacc - 32));
            if (first) or_word(word); else raw[wi] = word;
            first = false;
            wi++;
            nacc -= 32;
        }
    }
    V5_HOSTDEV void finish()
    {
        if (nacc > 0) or_word((uint32_t)(acc << (32 - nacc)));
    }
};

// Bit k set <=> coefficient k (zigzag order) of the block is non-zero. The block is 128 aligned bytes.
V5_HOSTDEV uint64_t nonzero_mask(const int16_t *coef)
{
    uint64_t m = 0;
#ifdef __CUDA_ARCH__
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(coef) + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t b = ((w[k] & 0xffffu) ? 1u : 0u) | ((w[k] >> 16) ? 2u : 0u);
            m |= (uint64_t)b << (8 * i + 2 * k);
        }
    }
#else
    for (int k = 0; k < 64; k++) m |= (uint64_t)(coef[k] != 0) << k;
#endif
    return m;
}

V5_HOSTDEV int lowest_bit(uint64_t m)
{
#ifdef __CUDA_ARCH__
    return __ffsll((long long)m) - 1;
#else
    return __builtin_ctzll(m);
#endif
}

// coef: the block's 64 coefficients in zigzag order; pred: DC of the predecessor block (0 at the start of the scan).
// Only the non-zero coefficients are visited (T.81 F.1.2.2: run lengths are the gaps between them).
template <class Sink>
V5_HOSTDEV void encode_block(const int16_t *coef, int pred, const uint32_t *dc_tab, const uint32_t *ac_tab, Sink &sink)
{
    {
        int t = (int)coef[0] - pred, t2 = t;
        if (t < 0) { t = -t; t2--; }
        const int nb = bit_length((uint32_t)t);
        const uint32_t e = dc_tab[nb];
        sink.put(((e & 0xffffu) << nb) | ((uint32_t)t2 & ((1u << nb) - 1u)), (int)(e >> 16) + nb);
    }
    uint64_t mask = nonzero_mask(coef) & ~(uint64_t)1;
    int prev = 0;
    while (mask) {
        const int k = lowest_bit(mask);
        mask &= mask - 1;
        int run = k - prev - 1;
        prev = k;
        while (run > 15) {
            const uint32_t z = ac_tab[0xF0];
            sink.put(z & 0xffffu, (int)(z >> 16));
            run -= 16;
        }
        int t = coef[k], t2 = t;
        if (t < 0) { t = -t; t2--; }
        const int nb = bit_length((uint32_t)t);
        const uint32_t e = ac_tab[(run << 4) + nb];
        sink.put(((e & 0xffffu) << nb) | ((uint32_t)t2 & ((1u << nb) - 1u)), (int)(e >> 16) + nb);
    }
    if (prev < 63) {
        const uint32_t e = ac_tab[0];
        sink.put(e & 0xffffu, (int)(e >> 16));
    }
}

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------------- kernels
__constant__ uint8_t kZigzagDev[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                       41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                       30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

__global__ void __launch_bounds__(ENC_NT) coef_kernel(const __grid_constant__ CoefParams p)
{
    __shared__ CoefSmem S;
    const int tid = (int)threadIdx.x, tile_x = (int)blockIdx.x, my = (int)blockIdx.y, img = (int)blockIdx.z;
    const EncGeo &g = p.g;
    const uint8_t *frame = p.img + (int64_t)img * p.frame_stride;
    if (tid < 64) S.zz[tid] = kZigzagDev[tid];
    coef_load_quant(tid, S, p);
    const int per = g.ncomp == 3 ? ENC_TM : ENC_BLOCKS;                  // MCUs per strip
    const int mx0 = tile_x * per;
    const int mcus = g.mcux - mx0 < per ? g.mcux - mx0 : per;
    const int nblocks = mcus * g.bpm;
    if (g.ncomp == 3) {
        coef_stage_rgb(tid, S, p, frame, tile_x, my);
        __syncthreads();
        coef_load_colour(tid, S, p, tile_x, my);
    } else {
        coef_load_gray(tid, S, p, frame, tile_x, my);
    }
    __syncthreads();
    coef_rows(tid, S, g.ncomp, nblocks);
    __syncthreads();
    coef_cols(tid, S, p, nblocks);
    __syncthreads();
    int16_t *dst = p.coef + ((int64_t)img * g.blocks + ((int64_t)my * g.mcux + mx0) * g.bpm) * 64;
    coef_store(tid, S, p, dst, mx0, my, nblocks);
}

struct EntropyParams {
    const int16_t *coef;               // [n][blocks][64]
    uint32_t *bitoff;                  // [n][blocks]: lengths after count_kernel, exclusive offsets after scan_kernel
    uint32_t *total_bits;              // [n]
    uint32_t *raw;                     // [n][raw_words] zero-initialised
    int64_t raw_words;
    int blocks, bpm, n;
};

template <bool WRITE>
__global__ void __launch_bounds__(128) entropy_kernel(const EntropyParams p, const EncTables *tabs)
{
    __shared__ uint32_t s_dc[2][16], s_ac[2][256];
    for (int i = threadIdx.x; i < 32; i += blockDim.x) (&s_dc[0][0])[i] = (&tabs->dc[0][0])[i];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) (&s_ac[0][0])[i] = (&tabs->ac[0][0])[i];
    __syncthreads();
    const int img = (int)blockIdx.y;
    const int g = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (g >= p.blocks) return;
    const int16_t *base = p.coef + (int64_t)img * p.blocks * 64;
    const int16_t *c = base + (int64_t)g * 64;       // 128 bytes = one cache line per thread, walked through L1
    const int prev = dc_predecessor(g, p.bpm);
    const int pred = prev >= 0 ? base[(int64_t)prev * 64] : 0;
    const int t = (p.bpm == 6 && (g % 6) >= 4) ? 1 : 0;
    if (!WRITE) {
        BitCounter cnt;
        encode_block(c, pred, s_dc[t], s_ac[t], cnt);
        p.bitoff[(int64_t)img * p.blocks + g] = cnt.total;
    } else {
        const uint32_t off = p.bitoff[(int64_t)img * p.blocks + g];
        const uint32_t end = g + 1 < p.blocks ? p.bitoff[(int64_t)img * p.blocks + g + 1] : p.total_bits[img];
        if (end < off || (uint64_t)end > (uint64_t)p.raw_words * 32) return;       // does not fit: reported by stuff_kernel
        BitSink sink;
        sink.init(p.raw + (int64_t)img * p.raw_words, off);
        encode_block(c, pred, s_dc[t], s_ac[t], sink);
        sink.finish();
    }
}

// CTA-wide exclusive scan of one value per thread (1024 threads); returns the exclusive prefix, total in *sum.
__device__ __forceinline__ uint32_t cta_exclusive_scan(uint32_t v, uint32_t *warp_sums, uint32_t *sum)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_sums[lane] = wi - w;                                         // exclusive over warps
        if (lane == 31) warp_sums[32] = wi;
    }
    __syncthreads();
    const uint32_t excl = incl - v + warp_sums[warp];
    *sum = warp_sums[32];
    __syncthreads();
    return excl;
}

__global__ void __launch_bounds__(1024) scan_kernel(const EntropyParams p)
{
    __shared__ uint32_t warp_sums[33];
    const int img = (int)blockIdx.x;
    uint32_t *a = p.bitoff + (int64_t)img * p.blocks;
    uint32_t running = 0;
    for (int base = 0; base < p.blocks; base += 1024) {
        const int i = base + (int)threadIdx.x;
        const uint32_t v = i < p.blocks ? a[i] : 0u;
        uint32_t sum;
        const uint32_t ex = cta_exclusive_scan(v, warp_sums, &sum);
        if (i < p.blocks) a[i] = running + ex;
        running += sum;
    }
    if (threadIdx.x == 0) p.total_bits[img] = running;
}

struct StuffParams {
    const uint32_t *raw;
    int64_t raw_words;
    const uint32_t *total_bits;
    const uint8_t *header;
    int header_len;
    uint8_t *out;                      // [n][out_stride]
    int64_t out_stride;
    int32_t *sizes;                    // [n] file size; > out_stride when the file did not fit (contents then undefined)
};

__global__ void __launch_bounds__(1024) stuff_kernel(const StuffParams p)
{
    __shared__ uint32_t warp_sums[33];
    const int img = (int)blockIdx.x;
    const uint32_t *raw = p.raw + (int64_t)img * p.raw_words;
    uint8_t *out = p.out + (int64_t)img * p.out_stride;
    const uint32_t bits = p.total_bits[img];
    const uint32_t nbytes = (bits + 7) >> 3;
    const bool fits_raw = (uint64_t)nbytes <= (uint64_t)p.raw_words * 4;
    for (int i = threadIdx.x; i < p.header_len && i < p.out_stride; i += blockDim.x) out[i] = p.header[i];
    uint32_t running = (uint32_t)p.header_len;
    const uint32_t nwords = (nbytes + 3) >> 2;
    for (uint32_t base = 0; base < nwords; base += 1024) {
        const uint32_t wi = base + threadIdx.x;
        uint32_t word = 0, nb = 0, nff = 0;
        if (wi < nwords) {
            word = fits_raw ? raw[wi] : 0u;
            nb = nbytes - 4 * wi < 4 ? nbytes - 4 * wi : 4;
            if (wi == nwords - 1 && (bits & 7)) word |= (0xffu >> (bits & 7)) << (8 * (3 - ((nbytes - 1) & 3)));   // pad with ones
            for (uint32_t k = 0; k < nb; k++) nff += ((word >> (24 - 8 * k)) & 0xffu) == 0xffu;
        }
        uint32_t sum;
        uint32_t o = running + cta_exclusive_scan(nb + nff, warp_sums, &sum);
        for (uint32_t k = 0; k < nb; k++) {
            const uint8_t v = (uint8_t)(word >> (24 - 8 * k));
            if ((int64_t)o < p.out_stride) out[o] = v;
            o++;
            if (v == 0xff) {
                if ((int64_t)o < p.out_stride) out[o] = 0;
                o++;
            }
        }
        running += sum;
    }
    if (threadIdx.x == 0) {
        if ((int64_t)running + 2 <= p.out_stride) {
            out[running] = 0xFF;
            out[running + 1] = 0xD9;
        }
        p.sizes[img] = fits_raw ? (int32_t)(running + 2) : 0x7fffffff;
    }
}
#endif  // __CUDACC__

}  // namespace v5j
