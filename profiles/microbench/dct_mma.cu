// profiles/microbench/dct_mma.cu — round-2 experiment (VERDICT r01 task 2): the four ISLOW passes of the 8x8 JPEG round trip
// (SURVEY.md A.4-A.6) as int8 limb-split tensor-core contractions, bit-exact.
//
// Every 1-D ISLOW pass is an exact integer map  out = (M . in + rnd) >> n  (the butterflies only factor M). M's entries are
// < 2^14, the data is < 2^16, so both are split into 8-bit limbs and the product is rebuilt from three int32 accumulator
// groups:  M = 256 Mh + Ml (Ml in -128..127),  in + OFF = 256 hu + lu (unsigned limbs; the offset's contribution and the
// rounding term ride in the MMA's C operand):   M.in = G0 + 256 G1 + 65536 G2,  G0 = Ml.lu, G1 = Mh.lu + Ml.hu, G2 = Mh.hu.
// mma.sync.m16n8k16 (SASS IMMA.16816.U8.S8) has a fragment layout in which the accumulator fragment of one pass IS the
// operand fragment of the next (thread (g,q) holds D[row g][cols 2q,2q+1]; an A fragment wants A[row g][k 4q..4q+3] and a
// B fragment B[k 4q..4q+3][col g]; with k = 2 j + limb the two 16-bit results are exactly those four bytes):
//   F1 (rows)   constant-as-A: D1[(G,u), r]   = sum_x  A[(G,u), x]        . X[r][x]          (B fragment = 4 pixels of row g)
//   F2 (cols)   data-as-A:     D2[u, (G,v)]   = sum_r  W1[u][(r,limb)]    . B_G[(r,limb), v]
//   quantise / dequantise in registers (thread holds coefficients (v = 2q,2q+1; u = g))
//   I1 (cols)   constant-as-A: D3[(G,y), u]   = sum_v  A[(G,y), (v,limb)] . W2[(v,limb)][u]
//   I2 (rows)   data-as-A:     D4[y, (G,x)]   = sum_u  W3[y][(u,limb)]    . B_G[(u,limb), x]
// so a warp takes two horizontally adjacent blocks through the whole round trip in registers: 12 IMMA, no shared-memory
// transposes, no __syncwarp. This file (1) checks that against a scalar restatement of libjpeg's arithmetic — on the host
// through a lane-by-lane emulation of the fragment layout (`--cpu`, runs without a GPU) and on the device — and (2) times
// it against the shipped 4-threads-per-block shared-memory-transpose implementation (v5ela_device.cuh) in the same harness,
// plus the raw IMMA issue rate.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -I../../include -I../../fake-video-detection-engine_b200/csrc
//             -o dct_mma dct_mma.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>

#define V5_MMA_BLOCKS 0          // the shipped-until-round-1 block stage (4 threads per block) is the comparison partner here
#include "v5ela_host.h"
#include "v5ela_device.cuh"

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e_ = (x);                                                                   \
        if (e_ != cudaSuccess) {                                                                \
            printf("CUDA error %s at line %d\n", cudaGetErrorString(e_), __LINE__);             \
            return 1;                                                                           \
        }                                                                                       \
    } while (0)

// ------------------------------------------------------------------------------------------------ scalar restatement
#define HD __host__ __device__ inline
namespace ref {
constexpr int C0_298 = 2446, C0_390 = 3196, C0_541 = 4433, C0_765 = 6270, C0_899 = 7373, C1_175 = 9633, C1_501 = 12299,
              C1_847 = 15137, C1_961 = 16069, C2_053 = 16819, C2_562 = 20995, C3_072 = 25172;

// pre-descale sums of the forward / inverse 8-point pass (exact, linear); DC rows carry the factor 8192 so that one descale
// amount serves all eight outputs
template <class T>
HD void fdct_lin(const T *d, T *o)
{
    const T t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    const T t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    const T t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    o[0] = (t10 + t11) * 8192;
    o[4] = (t10 - t11) * 8192;
    T z1 = (t12 + t13) * C0_541;
    o[2] = z1 + t13 * C0_765;
    o[6] = z1 - t12 * C1_847;
    z1 = t4 + t7;
    T z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const T z5 = (z3 + z4) * C1_175;
    const T a4 = t4 * C0_298, a5 = t5 * C2_053, a6 = t6 * C3_072, a7 = t7 * C1_501;
    z1 = z1 * -C0_899;
    z2 = z2 * -C2_562;
    z3 = z3 * -C1_961 + z5;
    z4 = z4 * -C0_390 + z5;
    o[7] = a4 + z1 + z3;
    o[5] = a5 + z2 + z4;
    o[3] = a6 + z2 + z3;
    o[1] = a7 + z1 + z4;
}
template <class T>
HD void idct_lin(const T *i, T *o)
{
    T z1 = (i[2] + i[6]) * C0_541;
    const T t2 = z1 - i[6] * C1_847, t3 = z1 + i[2] * C0_765;
    const T t0 = (i[0] + i[4]) * 8192, t1 = (i[0] - i[4]) * 8192;
    const T t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    T u0 = i[7], u1 = i[5], u2 = i[3], u3 = i[1];
    z1 = u0 + u3;
    T z2 = u1 + u2, z3 = u0 + u2, z4 = u1 + u3;
    const T z5 = (z3 + z4) * C1_175;
    u0 = u0 * C0_298; u1 = u1 * C2_053; u2 = u2 * C3_072; u3 = u3 * C1_501;
    z1 = z1 * -C0_899; z2 = z2 * -C2_562;
    z3 = z3 * -C1_961 + z5; z4 = z4 * -C0_390 + z5;
    u0 += z1 + z3; u1 += z2 + z4; u2 += z2 + z3; u3 += z1 + z4;
    o[0] = t10 + u3; o[7] = t10 - u3; o[1] = t11 + u2; o[6] = t11 - u2;
    o[2] = t12 + u1; o[5] = t12 - u1; o[3] = t13 + u0; o[4] = t13 - u0;
}

// libjpeg's round trip of one 8x8 block (natural order quantisation table `tab`): SURVEY.md A.4, A.5, A.6
HD void roundtrip(const uint8_t *in, int pitch, const uint16_t *tab, uint8_t *out, int opitch)
{
    int ws[64];
    for (int r = 0; r < 8; r++) {                               // forward rows, descale 11 (DC rows: << 2)
        int d[8], o[8];
        for (int x = 0; x < 8; x++) d[x] = (int)in[r * pitch + x] - 128;
        fdct_lin<int>(d, o);
        for (int u = 0; u < 8; u++) ws[r * 8 + u] = (o[u] + 1024) >> 11;
    }
    for (int u = 0; u < 8; u++) {                               // forward columns, descale 15 (DC rows: 2)
        int d[8], o[8];
        for (int r = 0; r < 8; r++) d[r] = ws[r * 8 + u];
        fdct_lin<int>(d, o);
        for (int v = 0; v < 8; v++) ws[v * 8 + u] = (o[v] + 16384) >> 15;
    }
    for (int i = 0; i < 64; i++) {                              // quantise (round half away from zero), dequantise
        const int c = ws[i], dv = (int)tab[i] << 3;
        const int a = c < 0 ? -c : c, qv = (a + (dv >> 1)) / dv;
        ws[i] = (c < 0 ? -qv : qv) * (int)tab[i];
    }
    for (int u = 0; u < 8; u++) {                               // inverse columns, descale 11
        int d[8], o[8];
        for (int v = 0; v < 8; v++) d[v] = ws[v * 8 + u];
        idct_lin<int>(d, o);
        for (int y = 0; y < 8; y++) ws[y * 8 + u] = (o[y] + 1024) >> 11;
    }
    for (int y = 0; y < 8; y++) {                               // inverse rows, descale 18, +128, clamp
        int o[8];
        idct_lin<int>(&ws[y * 8], o);
        for (int x = 0; x < 8; x++) {
            const int s = ((o[x] + (1 << 17)) >> 18) + 128;
            out[y * opitch + x] = (uint8_t)(s < 0 ? 0 : (s > 255 ? 255 : s));
        }
    }
}
}  // namespace ref

// ------------------------------------------------------------------------------------------- constants of the MMA form
constexpr int OFF1 = 8192;      // F1 output + OFF1 in 0..65535 (|F1 out| <= 4096 + rounding)
constexpr int OFF2 = 32768;     // dequantised coefficient + OFF2
constexpr int OFF3 = 32768;     // I1 output + OFF3 (|I1 out| <= 21047, DESIGN.md 4.1)

struct LaneConsts {             // per lane (g = lane >> 2, q = lane & 3); 19 registers
    uint32_t f1a[2][2];         // F1: A fragments (a0: rows G0, a1: rows G1) for the left / right block of a pair
    uint32_t f2b[3];            // F2: B fragment per accumulator group
    uint32_t i1a[3];            // I1: A fragments: MMA 1 (a0 = G0 rows, a1 = G1 rows), MMA 2 (a0 = G2 rows; a1 = 0)
    uint32_t i2b[3];            // I2: B fragment per group
    int32_t kf1, kf2[2], ki1, ki2[2];   // C-operand constants (rounding, offsets) of group 0
};

struct Matrices {
    int f[8][8], i[8][8];       // M of the forward / inverse pass: out[o] = sum_k M[o][k] in[k]
};

static Matrices make_matrices()
{
    Matrices m;
    for (int k = 0; k < 8; k++) {
        long long e[8] = {0, 0, 0, 0, 0, 0, 0, 0}, o[8];
        e[k] = 1;
        ref::fdct_lin<long long>(e, o);
        for (int r = 0; r < 8; r++) m.f[r][k] = (int)o[r];
        ref::idct_lin<long long>(e, o);
        for (int r = 0; r < 8; r++) m.i[r][k] = (int)o[r];
    }
    return m;
}
static inline int limb_hi(int m) { return (m + 128) >> 8; }
static inline int limb_lo(int m) { return m - 256 * limb_hi(m); }                 // -128..127

// value of group G's constant for matrix entry m against data limb `limb` (0 = low, 1 = high)
static inline int group_entry(int m, int G, int limb)
{
    if (G == 0) return limb == 0 ? limb_lo(m) : 0;
    if (G == 1) return limb == 0 ? limb_hi(m) : limb_lo(m);
    return limb == 0 ? 0 : limb_hi(m);
}
static inline uint32_t pack4(const int b[4])
{
    return (uint32_t)(b[0] & 255) | ((uint32_t)(b[1] & 255) << 8) | ((uint32_t)(b[2] & 255) << 16) | ((uint32_t)(b[3] & 255) << 24);
}

static void make_lane_consts(LaneConsts lc[32])
{
    const Matrices m = make_matrices();
    for (int e = 0; e < 64; e++) {
        if (limb_hi(m.f[e >> 3][e & 7]) < -128 || limb_hi(m.f[e >> 3][e & 7]) > 127 || limb_hi(m.i[e >> 3][e & 7]) < -128 ||
            limb_hi(m.i[e >> 3][e & 7]) > 127) {
            printf("matrix entry does not fit two signed limbs\n");
            exit(1);
        }
    }
    long long rs_f[8], rs_i[8];
    for (int o = 0; o < 8; o++) {
        rs_f[o] = rs_i[o] = 0;
        for (int k = 0; k < 8; k++) { rs_f[o] += m.f[o][k]; rs_i[o] += m.i[o][k]; }
    }
    for (int lane = 0; lane < 32; lane++) {
        const int g = lane >> 2, q = lane & 3;
        LaneConsts &L = lc[lane];
        int b[4];
        // F1, constant-as-A, one data limb (pixels, u8): A[(G,u)][k = x (+8 for the right block)], G0 = Ml, G1 = Mh
        for (int blk = 0; blk < 2; blk++)
            for (int G = 0; G < 2; G++) {
                for (int i = 0; i < 4; i++) {
                    const int k = 4 * q + i, x = k - 8 * blk;
                    b[i] = (x >= 0 && x < 8) ? (G == 0 ? limb_lo(m.f[g][x]) : limb_hi(m.f[g][x])) : 0;
                }
                L.f1a[blk][G] = pack4(b);
            }
        // F2, data-as-A: B_G[k = 2 r + limb][n = v]; thread holds k = 4q + i, n = g
        for (int G = 0; G < 3; G++) {
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(m.f[g][k >> 1], G, k & 1); }
            L.f2b[G] = pack4(b);
        }
        // I1, constant-as-A: A[(G,y)][k = 2 v + limb]; a-fragment rows g (and g + 8), k = 4q + i
        for (int G = 0; G < 3; G++) {
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(m.i[g][k >> 1], G, k & 1); }
            L.i1a[G] = pack4(b);
        }
        // I2, data-as-A: B_G[k = 2 u + limb][n = x]
        for (int G = 0; G < 3; G++) {
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(m.i[g][k >> 1], G, k & 1); }
            L.i2b[G] = pack4(b);
        }
        // C operands (mod 2^32). F1: input is the raw pixel (level shift = -128 rowsum); output carries +OFF1.
        L.kf1 = (int32_t)(uint32_t)(1024 - 128 * rs_f[g] + ((long long)OFF1 << 11));
        for (int j = 0; j < 2; j++) {
            L.kf2[j] = (int32_t)(uint32_t)(16384 - (long long)OFF1 * rs_f[2 * q + j]);
            L.ki2[j] = (int32_t)(uint32_t)((1ll << 17) + (128ll << 18) - (long long)OFF3 * rs_i[2 * q + j]);
        }
        L.ki1 = (int32_t)(uint32_t)(1024 - (long long)OFF2 * rs_i[g] + ((long long)OFF3 << 11));
    }
}

// quantisation constants in the order the MMA form reads them: entry (u, v) [u = horizontal, v = vertical frequency] at
// position (8 u + v) ^ (u & 1) — two LDS.128 per thread, bank-conflict free; unbias absorbs -OFF2
static void make_qswz(const uint16_t tab[64], v5::QEntry out[64])
{
    v5plan::QuantTab qt;
    v5plan::make_quant(tab, qt);
    for (int u = 0; u < 8; u++)
        for (int v = 0; v < 8; v++) {
            const int nat = 8 * v + u;
            out[(8 * u + v) ^ (u & 1)] = v5::QEntry{qt.recip[nat], qt.bias[nat], qt.t[nat], qt.unbias[nat] - OFF2};
        }
}

// ------------------------------------------------------------------------------------- the warp routine (device + emu)
// One m16n8k16 MMA: D = A(u8 or s8) . B(s8 or u8) + C. `A_DATA`: the A operand is the data (u8), B the constants (s8);
// otherwise A holds constants (s8) and B data (u8).
#ifdef __CUDA_ARCH__
template <bool A_DATA>
__device__ __forceinline__ void imma(int d[4], uint32_t a0, uint32_t a1, uint32_t b0, int c0, int c1, int c2, int c3)
{
    if (A_DATA)
        asm("mma.sync.aligned.m16n8k16.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%8,%9,%10};"
            : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
            : "r"(a0), "r"(a1), "r"(b0), "r"(c0), "r"(c1), "r"(c2), "r"(c3));
    else
        asm("mma.sync.aligned.m16n8k16.row.col.s32.s8.u8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%8,%9,%10};"
            : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
            : "r"(a0), "r"(a1), "r"(b0), "r"(c0), "r"(c1), "r"(c2), "r"(c3));
}
#endif

// accumulator groups -> the pass's sum (mod 2^32; the true value fits int32)
__host__ __device__ inline int comb2(int g1, int g0) { return (int)(((uint32_t)g1 << 8) + (uint32_t)g0); }
__host__ __device__ inline int comb3(int g2, int g1, int g0) { return (int)(((uint32_t)g2 << 16) + ((uint32_t)g1 << 8) + (uint32_t)g0); }

// The round trip of two horizontally adjacent 8x8 blocks by one warp. in/out: the pair's top-left pixel, pitches in bytes.
#ifdef __CUDACC__
// NP pairs (each 16 pixels to the right of the previous one) go through the passes stage by stage, so NP independent
// dependency chains are in flight per warp.
template <int NP>
__device__ __forceinline__ void dct_pairs_mma(const uint8_t *in, int ipitch, uint8_t *out, int opitch, const v5::QEntry *qs,
                                              const LaneConsts &K, int lane)
{
#ifdef __CUDA_ARCH__
    const int g = lane >> 2, q = lane & 3;
    uint32_t px[NP], a0[NP], a1[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) px[p] = *reinterpret_cast<const uint32_t *>(in + 16 * p + g * ipitch + 4 * q);   // pixels 4q..4q+3 of pair row g
#pragma unroll
    for (int p = 0; p < NP; p++) {
        int d[4], e[4];
        imma<false>(d, K.f1a[0][0], K.f1a[0][1], px[p], K.kf1, K.kf1, 0, 0);        // left block:  rows u = g, cols r = 2q, 2q+1
        imma<false>(e, K.f1a[1][0], K.f1a[1][1], px[p], K.kf1, K.kf1, 0, 0);        // right block
        const uint32_t w0 = (uint32_t)(comb2(d[2], d[0]) >> 11), w1 = (uint32_t)(comb2(d[3], d[1]) >> 11);
        const uint32_t w2 = (uint32_t)(comb2(e[2], e[0]) >> 11), w3 = (uint32_t)(comb2(e[3], e[1]) >> 11);
        a0[p] = v5::prmt(w0, w1, 0x5410u);
        a1[p] = v5::prmt(w2, w3, 0x5410u);
    }
    // F2: rows u = g (left block) / g + 8 (right block), cols v = 2q, 2q+1; quantise, dequantise
    const int e0i = (8 * g + 2 * q) ^ (g & 1);
    const v5::QEntry qe[2] = {qs[e0i], qs[e0i ^ 1]};
    uint32_t bl[NP], br[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) {
        int g0[4], g1[4], g2[4];
        imma<true>(g0, a0[p], a1[p], K.f2b[0], K.kf2[0], K.kf2[1], K.kf2[0], K.kf2[1]);
        imma<true>(g1, a0[p], a1[p], K.f2b[1], 0, 0, 0, 0);
        imma<true>(g2, a0[p], a1[p], K.f2b[2], 0, 0, 0, 0);
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int c = comb3(g2[i], g1[i], g0[i]) >> 15;
            const v5::QEntry &t = qe[i & 1];
            w[i] = (uint32_t)((int)__umulhi((uint32_t)(c + (c >> 31) + t.bias), t.recip) * t.t - t.unbias);   // + OFF2
        }
        bl[p] = v5::prmt(w[0], w[1], 0x5410u);
        br[p] = v5::prmt(w[2], w[3], 0x5410u);
    }
    // I1 per block: rows y = g, cols u = 2q, 2q+1
#pragma unroll
    for (int p = 0; p < NP; p++) {
#pragma unroll
        for (int blk = 0; blk < 2; blk++) {
            int h0[4], h1[4];
            const uint32_t bb = blk ? br[p] : bl[p];
            imma<false>(h0, K.i1a[0], K.i1a[1], bb, K.ki1, K.ki1, 0, 0);
            imma<false>(h1, K.i1a[2], 0u, bb, 0, 0, 0, 0);
            const uint32_t v0 = (uint32_t)(comb3(h1[0], h0[2], h0[0]) >> 11);
            const uint32_t v1 = (uint32_t)(comb3(h1[1], h0[3], h0[1]) >> 11);
            (blk ? a1[p] : a0[p]) = v5::prmt(v0, v1, 0x5410u);
        }
    }
    // I2: rows y = g (left) / g + 8 (right), cols x = 2q, 2q+1
#pragma unroll
    for (int p = 0; p < NP; p++) {
        int g0[4], g1[4], g2[4], s[4];
        imma<true>(g0, a0[p], a1[p], K.i2b[0], K.ki2[0], K.ki2[1], K.ki2[0], K.ki2[1]);
        imma<true>(g1, a0[p], a1[p], K.i2b[1], 0, 0, 0, 0);
        imma<true>(g2, a0[p], a1[p], K.i2b[2], 0, 0, 0, 0);
#pragma unroll
        for (int i = 0; i < 4; i++) s[i] = comb3(g2[i], g1[i], g0[i]) >> 18;
        *reinterpret_cast<uint16_t *>(out + 16 * p + g * opitch + 2 * q) = (uint16_t)v5::packsat2(s[1], s[0], 0u);
        *reinterpret_cast<uint16_t *>(out + 16 * p + g * opitch + 8 + 2 * q) = (uint16_t)v5::packsat2(s[3], s[2], 0u);
    }
#endif
}
#endif

// Host emulation of the same routine: fragments as arrays over the 32 lanes, mma by definition of the m16n8k16 layout
// (PTX ISA "Matrix Fragments for mma.m16n8k16" with 8-bit types: A row = g (+8 for the second register), k = 4q + i;
// B k = 4q + i, n = g; C/D row = g (+8 for c2,c3), col = 2q + (i & 1)).
namespace emu {
static void imma(bool a_data, int d[32][4], const uint32_t a0[32], const uint32_t a1[32], const uint32_t b0[32], const int c[32][4])
{
    int A[16][16], B[16][8];
    for (int lane = 0; lane < 32; lane++) {
        const int g = lane >> 2, q = lane & 3;
        for (int i = 0; i < 4; i++) {
            const uint32_t x0 = (a0[lane] >> (8 * i)) & 255, x1 = (a1[lane] >> (8 * i)) & 255, y = (b0[lane] >> (8 * i)) & 255;
            A[g][4 * q + i] = a_data ? (int)x0 : (int)(int8_t)x0;
            A[g + 8][4 * q + i] = a_data ? (int)x1 : (int)(int8_t)x1;
            B[4 * q + i][g] = a_data ? (int)(int8_t)y : (int)y;
        }
    }
    for (int lane = 0; lane < 32; lane++) {
        const int g = lane >> 2, q = lane & 3;
        for (int i = 0; i < 4; i++) {
            const int row = g + (i >= 2 ? 8 : 0), col = 2 * q + (i & 1);
            uint32_t acc = (uint32_t)c[lane][i];
            for (int k = 0; k < 16; k++) acc += (uint32_t)(A[row][k] * B[k][col]);
            d[lane][i] = (int32_t)acc;
        }
    }
}
static inline uint32_t prmt5410(uint32_t a, uint32_t b) { return (a & 0xffffu) | (b << 16); }
static inline int sra(int v, int n) { return v >> n; }
static inline int u2i(uint32_t v) { return (int32_t)v; }

static void dct_pair(const uint8_t *in, int ipitch, uint8_t *out, int opitch, const v5::QEntry *qs, const LaneConsts K[32])
{
    uint32_t px[32], a0[32], a1[32], f0[32], f1[32], zero[32] = {0};
    int c[32][4], d[32][4], e[32][4], g0[32][4], g1[32][4], g2[32][4], cz[32][4];
    memset(cz, 0, sizeof(cz));
    for (int l = 0; l < 32; l++) {
        const int g = l >> 2, q = l & 3;
        memcpy(&px[l], in + g * ipitch + 4 * q, 4);
        c[l][0] = c[l][1] = K[l].kf1; c[l][2] = c[l][3] = 0;
        f0[l] = K[l].f1a[0][0]; f1[l] = K[l].f1a[0][1];
    }
    imma(false, d, f0, f1, px, c);
    for (int l = 0; l < 32; l++) { f0[l] = K[l].f1a[1][0]; f1[l] = K[l].f1a[1][1]; }
    imma(false, e, f0, f1, px, c);
    for (int l = 0; l < 32; l++) {
        const uint32_t w0 = (uint32_t)sra(u2i(((uint32_t)d[l][2] << 8) + (uint32_t)d[l][0]), 11), w1 = (uint32_t)sra(u2i(((uint32_t)d[l][3] << 8) + (uint32_t)d[l][1]), 11);
        const uint32_t w2 = (uint32_t)sra(u2i(((uint32_t)e[l][2] << 8) + (uint32_t)e[l][0]), 11), w3 = (uint32_t)sra(u2i(((uint32_t)e[l][3] << 8) + (uint32_t)e[l][1]), 11);
        if (w0 > 65535u || w1 > 65535u || w2 > 65535u || w3 > 65535u) { printf("emu: F1 output leaves 16 bits\n"); exit(1); }
        a0[l] = prmt5410(w0, w1);
        a1[l] = prmt5410(w2, w3);
    }
    for (int G = 0; G < 3; G++) {
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].f2b[G];
            c[l][0] = c[l][2] = G == 0 ? K[l].kf2[0] : 0;
            c[l][1] = c[l][3] = G == 0 ? K[l].kf2[1] : 0;
        }
        imma(true, G == 0 ? g0 : (G == 1 ? g1 : g2), a0, a1, f0, c);
    }
    uint32_t bl[32], br[32], pa[2][32];
    for (int l = 0; l < 32; l++) {
        const int g = l >> 2, q = l & 3;
        const int e0i = (8 * g + 2 * q) ^ (g & 1);
        const v5::QEntry qe[2] = {qs[e0i], qs[e0i ^ 1]};
        uint32_t w[4];
        for (int i = 0; i < 4; i++) {
            const int cc = sra(u2i(((uint32_t)g2[l][i] << 16) + ((uint32_t)g1[l][i] << 8) + (uint32_t)g0[l][i]), 15);
            const v5::QEntry &t = qe[i & 1];
            const uint32_t x = (uint32_t)(cc + (cc >> 31) + t.bias);
            w[i] = (uint32_t)((int)(uint32_t)(((uint64_t)x * t.recip) >> 32) * t.t - t.unbias);
            if (w[i] > 65535u) { printf("emu: dequantised coefficient leaves 16 bits\n"); exit(1); }
        }
        bl[l] = prmt5410(w[0], w[1]);
        br[l] = prmt5410(w[2], w[3]);
    }
    for (int blk = 0; blk < 2; blk++) {
        int h0[32][4], h1[32][4];
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].i1a[0]; f1[l] = K[l].i1a[1];
            c[l][0] = c[l][1] = K[l].ki1; c[l][2] = c[l][3] = 0;
        }
        imma(false, h0, f0, f1, blk ? br : bl, c);
        for (int l = 0; l < 32; l++) f0[l] = K[l].i1a[2];
        imma(false, h1, f0, zero, blk ? br : bl, cz);
        for (int l = 0; l < 32; l++) {
            const uint32_t v0 = (uint32_t)sra(u2i(((uint32_t)h1[l][0] << 16) + ((uint32_t)h0[l][2] << 8) + (uint32_t)h0[l][0]), 11);
            const uint32_t v1 = (uint32_t)sra(u2i(((uint32_t)h1[l][1] << 16) + ((uint32_t)h0[l][3] << 8) + (uint32_t)h0[l][1]), 11);
            if (v0 > 65535u || v1 > 65535u) { printf("emu: I1 output leaves 16 bits\n"); exit(1); }
            pa[blk][l] = prmt5410(v0, v1);
        }
    }
    for (int G = 0; G < 3; G++) {
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].i2b[G];
            c[l][0] = c[l][2] = G == 0 ? K[l].ki2[0] : 0;
            c[l][1] = c[l][3] = G == 0 ? K[l].ki2[1] : 0;
        }
        imma(true, G == 0 ? g0 : (G == 1 ? g1 : g2), pa[0], pa[1], f0, c);
    }
    for (int l = 0; l < 32; l++) {
        const int g = l >> 2, q = l & 3;
        for (int i = 0; i < 4; i++) {
            int s = sra(u2i(((uint32_t)g2[l][i] << 16) + ((uint32_t)g1[l][i] << 8) + (uint32_t)g0[l][i]), 18);
            s = s < 0 ? 0 : (s > 255 ? 255 : s);
            out[g * opitch + (i >= 2 ? 8 : 0) + 2 * q + (i & 1)] = (uint8_t)s;
        }
    }
}
}  // namespace emu

// ------------------------------------------------------------------------------------------------------- test content
static uint32_t rng_state = 12345;
static inline uint32_t rnd() { rng_state = rng_state * 1664525u + 1013904223u; return rng_state >> 8; }

// tile = 8 rows x 512 pixels = 64 blocks; kinds cycle per tile
static void fill_tile(uint8_t *t, int kind)
{
    for (int y = 0; y < 8; y++)
        for (int x = 0; x < 512; x++) {
            int v;
            switch (kind % 8) {
                case 0: v = rnd() & 255; break;                                               // uniform noise
                case 1: v = (x * 3 + y * 17 + (int)(rnd() % 13)) & 255; break;                  // ramps + small noise
                case 2: v = ((x ^ y) & 1) ? 255 : 0; break;                                     // checkerboard
                case 3: v = (rnd() & 1) ? 255 : 0; break;                                       // binary noise
                case 4: v = 128 + (int)(rnd() % 7) - 3; break;                                  // flat
                case 5: v = ((x >> 2) + (y >> 1)) & 1 ? 255 : 0; break;                         // coarse checker
                case 6: v = (x & 8) ? 255 : 0; break;                                           // block edges
                default: {                                                                      // sign pattern of a random basis function
                    const int u = (x >> 3) % 8, vv = (x >> 6) % 8;
                    static const int sgn[8][8] = {{1, 1, 1, 1, 1, 1, 1, 1},     {1, 1, 1, 1, -1, -1, -1, -1}, {1, 1, -1, -1, -1, -1, 1, 1},
                                                  {1, 1, -1, -1, 1, 1, -1, -1}, {1, -1, -1, 1, 1, -1, -1, 1}, {1, -1, -1, 1, -1, 1, 1, -1},
                                                  {1, -1, 1, 1, -1, -1, 1, -1}, {1, -1, 1, -1, 1, -1, 1, -1}};
                    v = sgn[u][x & 7] * sgn[vv][y] > 0 ? 255 : 0;
                }
            }
            t[y * 512 + x] = (uint8_t)v;
        }
}

// ------------------------------------------------------------------------------------------------------------ kernels
constexpr int TILE_BYTES = 8 * 512;

struct alignas(16) HarnessSmem {
    uint8_t in[8][512];
    uint8_t out[8][512];
    v5::QEntry qs[64];
};

// `reps`: the tile in shared memory is processed that many times (compute-only throughput: the harness's global load/store
// latency is amortised); UNROLL pairs are in flight per warp (the compiler interleaves their dependency chains).
template <int UNROLL>
__global__ void __launch_bounds__(256, 2) k_mma(const uint8_t *src, uint8_t *dst, int ntiles, const LaneConsts *lc, const v5::QEntry *qsw, int reps)
{
    __shared__ HarnessSmem H;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const LaneConsts K = lc[lane];
    if (tid < 64) H.qs[tid] = qsw[tid];
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        __syncthreads();
        reinterpret_cast<uint4 *>(&H.in[0][0])[tid] = reinterpret_cast<const uint4 *>(src + (size_t)t * TILE_BYTES)[tid];
        __syncthreads();
#pragma unroll 1
        for (int rep = 0; rep < reps; rep++) {
#pragma unroll 1
            for (int p = 0; p < 4; p += UNROLL) {
                const int x0 = 16 * (4 * warp + p);
                dct_pairs_mma<UNROLL>(&H.in[0][x0], 512, &H.out[0][x0], 512, H.qs, K, lane);
            }
        }
        __syncthreads();
        reinterpret_cast<uint4 *>(dst + (size_t)t * TILE_BYTES)[tid] = reinterpret_cast<const uint4 *>(&H.out[0][0])[tid];
    }
}

// the shipped implementation (4 threads per block, two shared-memory transposes) in the same harness
__global__ void __launch_bounds__(256, 2) k_smem(const uint8_t *src, uint8_t *dst, int ntiles, const v5::QEntry *qnat, int reps)
{
    extern __shared__ __align__(16) uint8_t raw[];
    v5::Smem &S = *reinterpret_cast<v5::Smem *>(raw);
    uint8_t(*in)[512] = S.yorig;                                  // 8 rows used
    uint8_t(*out)[512] = S.ydec;
    const int tid = threadIdx.x;
    if (tid < 64) S.qtab[0][tid] = qnat[tid];
    int col[16];
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        __syncthreads();
        reinterpret_cast<uint4 *>(&in[0][0])[tid] = reinterpret_cast<const uint4 *>(src + (size_t)t * TILE_BYTES)[tid];
        __syncthreads();
        v5::BlockTask task;
        const int blk = (tid >> 5) * 8 + ((tid & 31) >> 2);
        task.q = S.qtab[0];
        task.in = &in[0][8 * blk];
        task.out = &out[0][8 * blk];
        task.pitch = 512;
        task.active = true;
#pragma unroll 1
        for (int rep = 0; rep < reps; rep++) {
            v5::blocks_rows_fwd(tid, S, task);
            __syncwarp();
            v5::blocks_cols(tid, S, task, col);
            __syncwarp();
            v5::blocks_cols_store(tid, S, task, col);
            __syncwarp();
            v5::blocks_rows_inv(tid, S, task);
            __syncwarp();
        }
        __syncthreads();
        reinterpret_cast<uint4 *>(dst + (size_t)t * TILE_BYTES)[tid] = reinterpret_cast<const uint4 *>(&out[0][0])[tid];
    }
}

__global__ void k_ref(const uint8_t *src, uint8_t *dst, int ntiles, const uint16_t *tab)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= (long long)ntiles * 64) return;
    const long long t = b >> 6;
    const int blk = (int)(b & 63);
    ref::roundtrip(src + t * TILE_BYTES + 8 * blk, 512, tab, dst + t * TILE_BYTES + 8 * blk, 512);
}

// raw IMMA issue rate: ILP independent accumulator chains per warp
template <int ILP>
__global__ void __launch_bounds__(256, 2) k_imma_rate(int *out, int iters, long long *cycles)
{
    int acc[ILP][4];
#pragma unroll
    for (int i = 0; i < ILP; i++) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = i;
    const uint32_t a0 = threadIdx.x * 0x01010101u, a1 = ~a0, b0 = 0x01020304u + threadIdx.x;
    __syncthreads();
    const long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < ILP; i++)
            asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                         : "+r"(acc[i][0]), "+r"(acc[i][1]), "+r"(acc[i][2]), "+r"(acc[i][3])
                         : "r"(a0), "r"(a1), "r"(b0));
    }
    const long long t1 = clock64();
    int s = 0;
#pragma unroll
    for (int i = 0; i < ILP; i++) s += acc[i][0] + acc[i][1] + acc[i][2] + acc[i][3];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}


// Does an IMMA only occupy the tensor pipe, or also the issue port? MODE 0: IMMA only (4 independent chains); 1: ALU only
// (per iteration 4 x (3 IMAD + 3 LOP3), independent chains); 2: both interleaved.
template <int MODE>
__global__ void __launch_bounds__(256, 2) k_mix(int *out, int iters, long long *cycles)
{
    int acc[4][4], v[12], w[12];
#pragma unroll
    for (int i = 0; i < 4; i++) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = i;
#pragma unroll
    for (int i = 0; i < 12; i++) { v[i] = threadIdx.x * 7 + i; w[i] = threadIdx.x * 3 + i + 1; }
    const uint32_t a0 = threadIdx.x * 0x01010101u, a1 = ~a0, b0 = 0x01020304u + threadIdx.x;
    __syncthreads();
    const long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (MODE != 1)
                asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                             : "+r"(acc[i][0]), "+r"(acc[i][1]), "+r"(acc[i][2]), "+r"(acc[i][3])
                             : "r"(a0), "r"(a1), "r"(b0));
            if (MODE != 0) {
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    v[3 * i + j] = v[3 * i + j] * w[3 * i + j] + 12345;           // IMAD (FMA pipe)
                    w[3 * i + j] = (w[3 * i + j] ^ it) & 0x7fffffff;              // LOP3 (ALU pipe)
                }
            }
        }
    }
    const long long t1 = clock64();
    int s = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) s += acc[i][0] + acc[i][1] + acc[i][2] + acc[i][3];
#pragma unroll
    for (int i = 0; i < 12; i++) s += v[i] ^ w[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

template <int MODE>
static int run_mix(const char *name, int sms)
{
    const int grid = sms * 2, iters = 4096;
    int *out;
    long long *cyc;
    CK(cudaMalloc(&out, grid * 256 * sizeof(int)));
    CK(cudaMalloc(&cyc, grid * sizeof(long long)));
    for (int r = 0; r < 2; r++) {
        k_mix<MODE><<<grid, 256>>>(out, iters, cyc);
        CK(cudaDeviceSynchronize());
    }
    std::vector<long long> h(grid);
    CK(cudaMemcpy(h.data(), cyc, grid * sizeof(long long), cudaMemcpyDeviceToHost));
    double avg = 0;
    for (long long c : h) avg += (double)c;
    avg /= grid;
    printf("%-44s %.1f cycles per iteration per SM-resident warp set (16 warps x [4 IMMA | 12 IMAD + 12 LOP3])\n", name, avg / iters);
    cudaFree(out);
    cudaFree(cyc);
    return 0;
}

template <int ILP>
static int run_rate(const char *name, int sms)
{
    const int grid = sms * 2, iters = 4096;
    int *out;
    long long *cyc;
    CK(cudaMalloc(&out, grid * 256 * sizeof(int)));
    CK(cudaMalloc(&cyc, grid * sizeof(long long)));
    k_imma_rate<ILP><<<grid, 256>>>(out, iters, cyc);
    CK(cudaDeviceSynchronize());
    k_imma_rate<ILP><<<grid, 256>>>(out, iters, cyc);
    CK(cudaDeviceSynchronize());
    std::vector<long long> h(grid);
    CK(cudaMemcpy(h.data(), cyc, grid * sizeof(long long), cudaMemcpyDeviceToHost));
    double avg = 0;
    for (long long c : h) avg += (double)c;
    avg /= grid;
    // per SM: 2 CTAs x 8 warps x iters x ILP instructions in `avg` cycles
    printf("%-28s IMMA.16816 warp-inst/clk/SM %.3f  (int8 MAC/clk/SM %.0f)\n", name, 16.0 * iters * ILP / avg, 16.0 * iters * ILP / avg * 2048);
    cudaFree(out);
    cudaFree(cyc);
    return 0;
}

int main(int argc, char **argv)
{
    const bool cpu_only = argc > 1 && !strcmp(argv[1], "--cpu");
    LaneConsts lc[32];
    make_lane_consts(lc);

    // ---------------------------------------------------------------- host check: emulated fragments vs the scalar restatement
    {
        long long bad = 0, total = 0;
        for (int quality : {1, 10, 50, 75, 90, 95, 100}) {
            uint16_t luma[64], chroma[64];
            v5plan::quant_tables(quality, luma, chroma);
            for (int comp = 0; comp < 2; comp++) {
                const uint16_t *tab = comp ? chroma : luma;
                v5::QEntry qs[64];
                make_qswz(tab, qs);
                std::vector<uint8_t> tile(TILE_BYTES), a(TILE_BYTES), b(TILE_BYTES);
                for (int kind = 0; kind < (cpu_only ? 24 : 8); kind++) {
                    fill_tile(tile.data(), kind);
                    for (int pr = 0; pr < 32; pr++) {
                        emu::dct_pair(&tile[16 * pr], 512, &a[16 * pr], 512, qs, lc);
                        ref::roundtrip(&tile[16 * pr], 512, tab, &b[16 * pr], 512);
                        ref::roundtrip(&tile[16 * pr + 8], 512, tab, &b[16 * pr + 8], 512);
                    }
                    for (int i = 0; i < TILE_BYTES; i++) bad += a[i] != b[i];
                    total += TILE_BYTES;
                }
            }
        }
        printf("host emulation of the MMA form vs scalar restatement: %lld mismatching samples of %lld\n", bad, total);
        if (bad) return 2;
    }
    if (cpu_only) return 0;

    // ---------------------------------------------------------------------------------------------------------- device
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("device %s  SMs %d\n", prop.name, prop.multiProcessorCount);
    run_rate<1>("dependent chain (ILP 1)", prop.multiProcessorCount);
    run_rate<2>("ILP 2", prop.multiProcessorCount);
    run_rate<4>("ILP 4", prop.multiProcessorCount);
    run_rate<8>("ILP 8", prop.multiProcessorCount);
    run_mix<0>("mix probe: IMMA only", prop.multiProcessorCount);
    run_mix<1>("mix probe: IMAD + LOP3 only", prop.multiProcessorCount);
    run_mix<2>("mix probe: IMMA and IMAD + LOP3 interleaved", prop.multiProcessorCount);

    const int ntiles = argc > 1 ? atoi(argv[1]) : 194400;          // 12.4 M blocks = the luma+chroma blocks of 256 x 1080p
    std::vector<uint8_t> h_src((size_t)ntiles * TILE_BYTES);
    for (int t = 0; t < ntiles; t++) {
        if (t < 4096) fill_tile(&h_src[(size_t)t * TILE_BYTES], t);
        else memcpy(&h_src[(size_t)t * TILE_BYTES], &h_src[(size_t)(t % 4096) * TILE_BYTES], TILE_BYTES);
    }
    uint8_t *d_src, *d_a, *d_b, *d_c;
    CK(cudaMalloc(&d_src, h_src.size()));
    CK(cudaMalloc(&d_a, h_src.size()));
    CK(cudaMalloc(&d_b, h_src.size()));
    CK(cudaMalloc(&d_c, h_src.size()));
    CK(cudaMemcpy(d_src, h_src.data(), h_src.size(), cudaMemcpyHostToDevice));
    LaneConsts *d_lc;
    CK(cudaMalloc(&d_lc, sizeof(lc)));
    CK(cudaMemcpy(d_lc, lc, sizeof(lc), cudaMemcpyHostToDevice));
    v5::QEntry *d_qs, *d_qn;
    uint16_t *d_tab;
    CK(cudaMalloc(&d_qs, sizeof(v5::QEntry) * 64));
    CK(cudaMalloc(&d_qn, sizeof(v5::QEntry) * 64));
    CK(cudaMalloc(&d_tab, sizeof(uint16_t) * 64));
    CK(cudaFuncSetAttribute(k_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5::Smem)));
    const int grid = prop.multiProcessorCount * 2;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    int rc = 0;
    for (int quality : {90, 1, 100, 50}) {
        for (int comp = 0; comp < 2; comp++) {
            uint16_t luma[64], chroma[64];
            v5plan::quant_tables(quality, luma, chroma);
            const uint16_t *tab = comp ? chroma : luma;
            v5::QEntry qs[64], qn[64];
            make_qswz(tab, qs);
            v5plan::QuantTab qt;
            v5plan::make_quant(tab, qt);
            for (int i = 0; i < 64; i++) qn[i] = v5::QEntry{qt.recip[i], qt.bias[i], qt.t[i], qt.unbias[i]};
            CK(cudaMemcpy(d_qs, qs, sizeof(qs), cudaMemcpyHostToDevice));
            CK(cudaMemcpy(d_qn, qn, sizeof(qn), cudaMemcpyHostToDevice));
            CK(cudaMemcpy(d_tab, tab, sizeof(uint16_t) * 64, cudaMemcpyHostToDevice));
            const int nt_check = quality == 90 ? ntiles : 8192;
            float ms_mma = 0, ms_smem = 0;
            if (quality == 90 && comp == 0) {
                // compute-only throughput: 16 passes over every tile while it sits in shared memory
                const int reps = 16, nt = ntiles / 8;
                for (int v = 0; v < 4; v++) {
                    float ms = 0;
                    for (int rep = 0; rep < 3; rep++) {
                        CK(cudaEventRecord(e0));
                        if (v == 0) k_mma<1><<<grid, 256>>>(d_src, d_a, nt, d_lc, d_qs, reps);
                        if (v == 1) k_mma<2><<<grid, 256>>>(d_src, d_a, nt, d_lc, d_qs, reps);
                        if (v == 2) k_mma<4><<<grid, 256>>>(d_src, d_a, nt, d_lc, d_qs, reps);
                        if (v == 3) k_smem<<<grid, 256, sizeof(v5::Smem)>>>(d_src, d_b, nt, d_qn, reps);
                        CK(cudaEventRecord(e1));
                        CK(cudaDeviceSynchronize());
                        CK(cudaEventElapsedTime(&ms, e0, e1));
                    }
                    const double blocks = (double)nt * 64 * reps;
                    printf("compute-only (%d passes per staged tile)  %-22s %.3f ms  %.1f Mblocks/s  %.2f clk/block/SM at 1.9 GHz\n", reps,
                           v == 0 ? "mma, 1 pair in flight" : (v == 1 ? "mma, 2 pairs in flight" : (v == 2 ? "mma, 4 pairs in flight" : "smem-transpose")),
                           ms, blocks / ms * 1e-3, ms * 1e-3 * 1.9e9 * prop.multiProcessorCount / blocks);
                }
            }
            for (int rep = 0; rep < 3; rep++) {
                CK(cudaEventRecord(e0));
                k_mma<2><<<grid, 256>>>(d_src, d_a, nt_check, d_lc, d_qs, 1);
                CK(cudaEventRecord(e1));
                CK(cudaDeviceSynchronize());
                CK(cudaEventElapsedTime(&ms_mma, e0, e1));
                CK(cudaEventRecord(e0));
                k_smem<<<grid, 256, sizeof(v5::Smem)>>>(d_src, d_b, nt_check, d_qn, 1);
                CK(cudaEventRecord(e1));
                CK(cudaDeviceSynchronize());
                CK(cudaEventElapsedTime(&ms_smem, e0, e1));
            }
            k_ref<<<(nt_check * 64 + 127) / 128, 128>>>(d_src, d_c, nt_check, d_tab);
            CK(cudaDeviceSynchronize());
            std::vector<uint8_t> a((size_t)nt_check * TILE_BYTES), b(a.size()), c(a.size());
            CK(cudaMemcpy(a.data(), d_a, a.size(), cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(b.data(), d_b, a.size(), cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(c.data(), d_c, a.size(), cudaMemcpyDeviceToHost));
            long long bad_mma = 0, bad_smem = 0;
            for (size_t i = 0; i < a.size(); i++) { bad_mma += a[i] != c[i]; bad_smem += b[i] != c[i]; }
            // the device's scalar kernel against the host's (first 64 tiles)
            long long bad_ref = 0;
            std::vector<uint8_t> hr(64 * TILE_BYTES);
            for (int t = 0; t < 64; t++)
                for (int blk = 0; blk < 64; blk++)
                    ref::roundtrip(&h_src[(size_t)t * TILE_BYTES + 8 * blk], 512, tab, &hr[(size_t)t * TILE_BYTES + 8 * blk], 512);
            for (size_t i = 0; i < hr.size(); i++) bad_ref += hr[i] != c[i];
            printf("q=%3d %s  blocks %9lld  mma %.3f ms (%.1f Mblocks/s)  smem-transpose %.3f ms (%.1f Mblocks/s)  speed-up %.2fx  "
                   "mismatches vs scalar: mma %lld  smem %lld  (scalar device vs host: %lld)\n",
                   quality, comp ? "chroma" : "luma  ", (long long)nt_check * 64, ms_mma, nt_check * 64 / ms_mma * 1e-3, ms_smem,
                   nt_check * 64 / ms_smem * 1e-3, ms_smem / ms_mma, bad_mma, bad_smem, bad_ref);
            if (bad_mma || bad_smem || bad_ref) rc = 3;
        }
    }
    return rc;
}
