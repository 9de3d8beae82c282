// v5ela_dctmma.cuh — the 8x8 block round trip (ISLOW fDCT -> quantise -> dequantise -> ISLOW IDCT, SURVEY.md A.4-A.6) as int8
// limb-split tensor-core contractions, bit-exact. Included by v5ela_device.cuh (needs its shims and QEntry).
//
// Every 1-D ISLOW pass is an exact integer map  out = (M . in + rnd) >> n : the butterflies only factor the 8x8 integer matrix
// M (DC rows carry a factor 8192 so that one descale amount serves all eight outputs). |M| < 2^14 and the data is < 2^16, so both
// are cut into 8-bit limbs and the product is rebuilt from three int32 accumulator groups:
//     M = 256 Mh + Ml (Ml in -128..127),   in + OFF = 256 hu + lu (unsigned limbs),
//     M . (in + OFF) = G0 + 256 G1 + 65536 G2,   G0 = Ml.lu,  G1 = Mh.lu + Ml.hu,  G2 = Mh.hu      (mod 2^32; the true sum fits int32)
// and  -OFF . rowsum(M) + rnd (+ the next pass's offset << n)  rides in the MMA's C operand of group 0.
// mma.sync.m16n8k16 on 8-bit operands (SASS IMMA.16816.U8.S8 / .S8.U8) has a fragment layout in which the accumulator fragment of
// one pass IS the operand fragment of the next: lane (g = lane >> 2, q = lane & 3) holds D[row g][cols 2q, 2q+1] (and row g + 8);
// an A fragment wants A[row g][k = 4q .. 4q+3], a B fragment B[k = 4q .. 4q+3][col g]; with k = 2 j + limb the two 16-bit results
// of a lane are exactly those four bytes (one PRMT). The four passes alternate "constants as A" (rows come out as the new index,
// the old rows become columns) and "data as A" (rows stay, columns become the new index), each contracting the current columns:
//     F1 rows     consts-as-A : D1[(G,u)][r]  = sum_x  A[(G,u)][x]        . X[x][r]         B fragment = 4 pixels of row g
//     F2 columns  data-as-A   : D2[u][(G,v)]  = sum_r  W1[u][(r,limb)]    . B_G[(r,limb)][v]
//     quantise / dequantise in registers: lane holds coefficients (u = g; v = 2q, 2q+1)
//     I1 columns  consts-as-A : D3[(G,y)][u]  = sum_v  A[(G,y)][(v,limb)] . W2[(v,limb)][u]
//     I2 rows     data-as-A   : D4[y][(G,x)]  = sum_u  W3[y][(u,limb)]    . B_G[(u,limb)][x]
// A warp takes two horizontally adjacent blocks ("a pair", 16 x 8 pixels) through the whole round trip in registers with 12 IMMA:
// no shared-memory transposes and no __syncwarp. Measured against the 4-threads-per-block shared-memory-transpose form it replaces
// in profiles/microbench/dct_mma.cu (profiles/r02/dct_mma.txt): 101 instead of 146 warp instructions per pair.
//
// The g++ build (tests/emu) runs the same algorithm with the fragment layout emulated lane by lane (mma_emu); the asm is only
// reachable on the device. Nothing here is a fallback for anything else.
#pragma once

namespace v5plan {

// Per-lane constants, laid out as eight 128-bit words: a lane loads them with eight LDS.128 and every MMA operand that needs
// consecutive registers — the A pair (a0, a1) of a constants-as-A pass, the C quad of group 0 — is an aligned part of one of those
// words, so no register moves are needed in front of the IMMAs. One layout for both builds: KParams::lane_consts points to them.
struct alignas(16) LaneConsts {
    uint32_t f1a[2][2];         // F1: A pair (rows G0, rows G1) for the left / right block of a pair
    uint32_t i1a[4];            // I1: A pair of MMA 1 (rows G0, rows G1), A pair of MMA 2 (rows G2, zero)
    uint32_t f2b[4];            // F2: B fragment per accumulator group (+ pad)
    uint32_t i2b[4];            // I2: B fragment per group (+ pad)
    int32_t cf1[4];             // C quads of group 0: rounding, level shift, limb offsets.  F1: k, k, 0, 0 (rows G0 | rows G1)
    int32_t cf2[4];             // F2: k[2q], k[2q+1], k[2q], k[2q+1] (left | right block)
    int32_t ci1[4];             // I1: k, k, 0, 0
    int32_t ci2[4];             // I2: like F2
};
static_assert(sizeof(LaneConsts) == 128, "LaneConsts layout");

}  // namespace v5plan

namespace V5_NS {
namespace mma {

using v5plan::LaneConsts;

constexpr int OFF1 = 8192;      // F1 output + OFF1 in 0..65535 (|F1 output| <= 4096)
constexpr int OFF2 = 32768;     // dequantised coefficient + OFF2
constexpr int OFF3 = 32768;     // I1 output + OFF3 (|I1 output| <= 21047, DESIGN.md 4.1)
// The descale of I1 is 11 bits; with the matrix doubled and the dequantised coefficients handed over x 16 the MMA accumulates
// 32 x the sum, the descale becomes 16 bits and the two 16-bit results of a lane are bytes 2..3 of its accumulators — one PRMT, no
// shifts. (|2 M| < 2^15 still fits two signed limbs; |16 c'| <= 16 * 1151 fits the 16-bit limb pair.) The other descales (11 after
// one-limb pixels, 15 in front of the quantiser, 18 in front of the saturating pack) need their integer anyway.
constexpr int I1_MSCALE = 2, I1_DSCALE = 16;

// ---- host side: the pass matrices and the per-lane constants ---------------------------------------------------------------------
#define V5M_C0_298 2446
#define V5M_C0_390 3196
#define V5M_C0_541 4433
#define V5M_C0_765 6270
#define V5M_C0_899 7373
#define V5M_C1_175 9633
#define V5M_C1_501 12299
#define V5M_C1_847 15137
#define V5M_C1_961 16069
#define V5M_C2_053 16819
#define V5M_C2_562 20995
#define V5M_C3_072 25172

// pre-descale sums of libjpeg's forward / inverse 8-point pass (jfdctint.c / jidctint.c, SURVEY.md A.4 / A.6): exact and linear
inline void fdct_lin(const long long *d, long long *o)
{
    const long long t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    const long long t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    const long long t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    o[0] = (t10 + t11) * 8192;
    o[4] = (t10 - t11) * 8192;
    long long z1 = (t12 + t13) * V5M_C0_541;
    o[2] = z1 + t13 * V5M_C0_765;
    o[6] = z1 - t12 * V5M_C1_847;
    z1 = t4 + t7;
    long long z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const long long z5 = (z3 + z4) * V5M_C1_175;
    z1 *= -V5M_C0_899;
    z2 *= -V5M_C2_562;
    z3 = z3 * -V5M_C1_961 + z5;
    z4 = z4 * -V5M_C0_390 + z5;
    o[7] = t4 * V5M_C0_298 + z1 + z3;
    o[5] = t5 * V5M_C2_053 + z2 + z4;
    o[3] = t6 * V5M_C3_072 + z2 + z3;
    o[1] = t7 * V5M_C1_501 + z1 + z4;
}
inline void idct_lin(const long long *i, long long *o)
{
    long long z1 = (i[2] + i[6]) * V5M_C0_541;
    const long long t2 = z1 - i[6] * V5M_C1_847, t3 = z1 + i[2] * V5M_C0_765;
    const long long t0 = (i[0] + i[4]) * 8192, t1 = (i[0] - i[4]) * 8192;
    const long long t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    long long u0 = i[7], u1 = i[5], u2 = i[3], u3 = i[1];
    z1 = u0 + u3;
    long long z2 = u1 + u2, z3 = u0 + u2, z4 = u1 + u3;
    const long long z5 = (z3 + z4) * V5M_C1_175;
    u0 *= V5M_C0_298; u1 *= V5M_C2_053; u2 *= V5M_C3_072; u3 *= V5M_C1_501;
    z1 *= -V5M_C0_899; z2 *= -V5M_C2_562;
    z3 = z3 * -V5M_C1_961 + z5; z4 = z4 * -V5M_C0_390 + z5;
    u0 += z1 + z3; u1 += z2 + z4; u2 += z2 + z3; u3 += z1 + z4;
    o[0] = t10 + u3; o[7] = t10 - u3; o[1] = t11 + u2; o[6] = t11 - u2;
    o[2] = t12 + u1; o[5] = t12 - u1; o[3] = t13 + u0; o[4] = t13 - u0;
}

inline int limb_hi(int m) { return (m + 128) >> 8; }
inline int limb_lo(int m) { return m - 256 * limb_hi(m); }                      // -128..127
// group G's constant for matrix entry m against data limb `limb` (0 = low byte, 1 = high byte)
inline int group_entry(int m, int G, int limb)
{
    if (G == 0) return limb == 0 ? limb_lo(m) : 0;
    if (G == 1) return limb == 0 ? limb_hi(m) : limb_lo(m);
    return limb == 0 ? 0 : limb_hi(m);
}
inline uint32_t pack_bytes(const int b[4])
{
    return (uint32_t)(b[0] & 255) | ((uint32_t)(b[1] & 255) << 8) | ((uint32_t)(b[2] & 255) << 16) | ((uint32_t)(b[3] & 255) << 24);
}

// Fills lc[32]; returns false if a matrix entry does not fit two signed limbs (cannot happen with libjpeg's constants).
inline bool make_lane_consts(LaneConsts lc[32])
{
    int mf[8][8], mi[8][8];
    long long rs_f[8], rs_i[8];
    for (int k = 0; k < 8; k++) {
        long long e[8] = {0, 0, 0, 0, 0, 0, 0, 0}, o[8];
        e[k] = 1;
        fdct_lin(e, o);
        for (int r = 0; r < 8; r++) mf[r][k] = (int)o[r];
        idct_lin(e, o);
        for (int r = 0; r < 8; r++) mi[r][k] = (int)o[r];
    }
    for (int o = 0; o < 8; o++) {
        rs_f[o] = rs_i[o] = 0;
        for (int k = 0; k < 8; k++) {
            rs_f[o] += mf[o][k];
            rs_i[o] += mi[o][k];
            if (limb_hi(mf[o][k]) < -128 || limb_hi(mf[o][k]) > 127 || limb_hi(I1_MSCALE * mi[o][k]) < -128 || limb_hi(I1_MSCALE * mi[o][k]) > 127)
                return false;
        }
    }
    for (int lane = 0; lane < 32; lane++) {
        const int g = lane >> 2, q = lane & 3;
        LaneConsts &L = lc[lane];
        memset(&L, 0, sizeof(L));
        int b[4];
        for (int blk = 0; blk < 2; blk++)                       // F1: A[(G,u)][k = x (+ 8 for the right block)], one data limb (pixels)
            for (int G = 0; G < 2; G++) {
                for (int i = 0; i < 4; i++) {
                    const int x = 4 * q + i - 8 * blk;
                    b[i] = (x >= 0 && x < 8) ? (G == 0 ? limb_lo(mf[g][x]) : limb_hi(mf[g][x])) : 0;
                }
                L.f1a[blk][G] = pack_bytes(b);
            }
        for (int G = 0; G < 3; G++) {
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(mf[g][k >> 1], G, k & 1); }
            L.f2b[G] = pack_bytes(b);                           // F2: B_G[k = 2 r + limb][n = v = g]
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(I1_MSCALE * mi[g][k >> 1], G, k & 1); }
            L.i1a[G] = pack_bytes(b);                           // I1: A[(G, y = g)][k = 2 v + limb], matrix x 2 (see I1_MSCALE)
            for (int i = 0; i < 4; i++) { const int k = 4 * q + i; b[i] = group_entry(mi[g][k >> 1], G, k & 1); }
            L.i2b[G] = pack_bytes(b);                           // I2: B_G[k = 2 u + limb][n = x = g]
        }
        // C operands (mod 2^32). F1: the input is the raw pixel (level shift = -128 rowsum); its output carries + OFF1.
        L.cf1[0] = L.cf1[1] = (int32_t)(uint32_t)(1024 - 128 * rs_f[g] + ((long long)OFF1 << 11));
        // I1 works on 32 x the sum (matrix x 2, coefficients x 16): bits 16..31 of it are the output + OFF3.
        L.ci1[0] = L.ci1[1] = (int32_t)(uint32_t)(32 * 1024 - (long long)I1_MSCALE * OFF2 * rs_i[g] + ((long long)OFF3 << 16));
        for (int j = 0; j < 4; j++) {
            L.cf2[j] = (int32_t)(uint32_t)(16384 - (long long)OFF1 * rs_f[2 * q + (j & 1)]);
            L.ci2[j] = (int32_t)(uint32_t)((1ll << 17) + (128ll << 18) - (long long)OFF3 * rs_i[2 * q + (j & 1)]);
        }
    }
    return true;
}

// Quantisation constants in the order the MMA form reads them: entry (u = horizontal, v = vertical frequency) of the natural-order
// table sits at position (8 u + v) ^ (u & 1) — a lane's two entries (v = 2q, 2q+1) are two 128-bit loads without bank conflicts —
// t and unbias carry the factor 16 of I1_DSCALE and unbias absorbs the limb offset: the dequantised value comes out as 16 c' + OFF2.
V5_HOSTDEV QEntry qswz_entry(uint32_t recip, int32_t bias, int32_t t, int32_t unbias)
{
    return QEntry{recip, bias, I1_DSCALE * t, I1_DSCALE * unbias - OFF2};
}
V5_HOSTDEV int qswz_pos(int natural_index)
{
    const int v = natural_index >> 3, u = natural_index & 7;
    return (8 * u + v) ^ (u & 1);
}

// accumulator groups -> the pass's sum (mod 2^32)
V5_HOSTDEV int comb2(int g1, int g0) { return (int)(((uint32_t)g1 << 8) + (uint32_t)g0); }
V5_HOSTDEV int comb3(int g2, int g1, int g0) { return (int)(((uint32_t)g2 << 16) + ((uint32_t)g1 << 8) + (uint32_t)g0); }

// One pair's geometry: top-left pixel of the 16 x 8 input / output, pitches in bytes, which of the two blocks are stored.
struct PairTask {
    const uint8_t *in;
    uint8_t *out;
    const QEntry *q;            // swizzled table (qswz_pos)
    int ipitch, opitch;
    bool left, right;           // store the left / right block (a pair with neither is skipped)
};

#ifdef __CUDA_ARCH__
// D = A . B + C, m16n8k16. A_DATA: A is the data (u8) and B the constants (s8); otherwise A constants (s8), B data (u8).
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

// NP pairs go through the passes stage by stage: NP independent dependency chains per warp. All 32 lanes must call it together
// (inactive pairs are computed on whatever their pointers hold — t[p].in must be readable — and not stored).
template <int NP>
__device__ __forceinline__ void dct_pairs(const PairTask *t, const LaneConsts &K, int lane)
{
    const int g = lane >> 2, q = lane & 3;
    uint32_t a0[NP], a1[NP], bl[NP], br[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) {
        const uint32_t px = *reinterpret_cast<const uint32_t *>(t[p].in + g * t[p].ipitch + 4 * q);   // pixels 4q..4q+3 of pair row g
        int d[4], e[4];
        imma<false>(d, K.f1a[0][0], K.f1a[0][1], px, K.cf1[0], K.cf1[1], K.cf1[2], K.cf1[3]);   // left block: rows u = g, cols r = 2q, 2q+1
        imma<false>(e, K.f1a[1][0], K.f1a[1][1], px, K.cf1[0], K.cf1[1], K.cf1[2], K.cf1[3]);   // right block
        a0[p] = prmt((uint32_t)(comb2(d[2], d[0]) >> 11), (uint32_t)(comb2(d[3], d[1]) >> 11), 0x5410u);
        a1[p] = prmt((uint32_t)(comb2(e[2], e[0]) >> 11), (uint32_t)(comb2(e[3], e[1]) >> 11), 0x5410u);
    }
    const int e0i = (8 * g + 2 * q) ^ (g & 1);
#pragma unroll
    for (int p = 0; p < NP; p++) {                              // F2: rows u = g (left) / g + 8 (right), cols v = 2q, 2q+1
        int g0[4], g1[4], g2[4];
        imma<true>(g0, a0[p], a1[p], K.f2b[0], K.cf2[0], K.cf2[1], K.cf2[2], K.cf2[3]);
        imma<true>(g1, a0[p], a1[p], K.f2b[1], 0, 0, 0, 0);
        imma<true>(g2, a0[p], a1[p], K.f2b[2], 0, 0, 0, 0);
        const QEntry qe[2] = {t[p].q[e0i], t[p].q[e0i ^ 1]};
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {                           // A.5: exact division; dequantised x 16 + OFF2 (inside t / unbias)
            const int c = comb3(g2[i], g1[i], g0[i]) >> 15;
            const QEntry &e = qe[i & 1];
            w[i] = (uint32_t)((int)umulhi32((uint32_t)(c + (c >> 31) + e.bias), e.recip) * e.t - e.unbias);
        }
        bl[p] = prmt(w[0], w[1], 0x5410u);
        br[p] = prmt(w[2], w[3], 0x5410u);
    }
#pragma unroll
    for (int p = 0; p < NP; p++) {                              // I1 per block: rows y = g, cols u = 2q, 2q+1; 32 x the sum
#pragma unroll
        for (int blk = 0; blk < 2; blk++) {
            int h0[4], h1[4];
            const uint32_t bb = blk ? br[p] : bl[p];
            imma<false>(h0, K.i1a[0], K.i1a[1], bb, K.ci1[0], K.ci1[1], K.ci1[2], K.ci1[3]);
            imma<false>(h1, K.i1a[2], K.i1a[3], bb, 0, 0, 0, 0);
            const uint32_t v = prmt((uint32_t)comb3(h1[0], h0[2], h0[0]), (uint32_t)comb3(h1[1], h0[3], h0[1]), 0x7632u);   // bits 16..31
            if (blk) a1[p] = v;
            else a0[p] = v;
        }
    }
#pragma unroll
    for (int p = 0; p < NP; p++) {                              // I2: rows y = g (left) / g + 8 (right), cols x = 2q, 2q+1
        int g0[4], g1[4], g2[4], s[4];
        imma<true>(g0, a0[p], a1[p], K.i2b[0], K.ci2[0], K.ci2[1], K.ci2[2], K.ci2[3]);
        imma<true>(g1, a0[p], a1[p], K.i2b[1], 0, 0, 0, 0);
        imma<true>(g2, a0[p], a1[p], K.i2b[2], 0, 0, 0, 0);
#pragma unroll
        for (int i = 0; i < 4; i++) s[i] = comb3(g2[i], g1[i], g0[i]) >> 18;         // + 128 is in ci2; the pack saturates to 0..255
        uint8_t *o = t[p].out + g * t[p].opitch + 2 * q;
        if (t[p].left) *reinterpret_cast<uint16_t *>(o) = (uint16_t)packsat2(s[1], s[0], 0u);
        if (t[p].right) *reinterpret_cast<uint16_t *>(o + 8) = (uint16_t)packsat2(s[3], s[2], 0u);
    }
}
#else
// ---- g++ build: the m16n8k16 fragment layout lane by lane (PTX ISA, "Matrix Fragments for mma.m16n8k16", 8-bit types) -----------
inline void mma_emu(bool a_data, int d[32][4], const uint32_t a0[32], const uint32_t a1[32], const uint32_t b0[32], const int c[32][4])
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

// the intermediate of every pass must fit the 16 bits the limb split assumes; the emulator counts violations (tests assert 0)
inline uint32_t limbs16(int v)
{
    if (v < 0 || v > 65535) range_violations()++;
    return (uint32_t)v;
}

// One pair for the whole warp at once (K: the 32 lanes' constants).
inline void dct_pair_emu(const PairTask &t, const LaneConsts *K)
{
    uint32_t px[32], a0[32], a1[32], f0[32], f1[32];
    int c[32][4], cz[32][4], d[32][4], e[32][4], g0[32][4], g1[32][4], g2[32][4];
    memset(cz, 0, sizeof(cz));
    for (int l = 0; l < 32; l++) {
        memcpy(&px[l], t.in + (l >> 2) * t.ipitch + 4 * (l & 3), 4);
        memcpy(c[l], K[l].cf1, sizeof(c[l]));
        f0[l] = K[l].f1a[0][0];
        f1[l] = K[l].f1a[0][1];
    }
    mma_emu(false, d, f0, f1, px, c);
    for (int l = 0; l < 32; l++) { f0[l] = K[l].f1a[1][0]; f1[l] = K[l].f1a[1][1]; }
    mma_emu(false, e, f0, f1, px, c);
    for (int l = 0; l < 32; l++) {
        a0[l] = limbs16(comb2(d[l][2], d[l][0]) >> 11) | (limbs16(comb2(d[l][3], d[l][1]) >> 11) << 16);
        a1[l] = limbs16(comb2(e[l][2], e[l][0]) >> 11) | (limbs16(comb2(e[l][3], e[l][1]) >> 11) << 16);
    }
    for (int G = 0; G < 3; G++) {
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].f2b[G];
            memcpy(c[l], G == 0 ? K[l].cf2 : cz[l], sizeof(c[l]));
        }
        mma_emu(true, G == 0 ? g0 : (G == 1 ? g1 : g2), a0, a1, f0, c);
    }
    uint32_t bl[32], br[32];
    for (int l = 0; l < 32; l++) {
        const int g = l >> 2, q = l & 3, e0i = (8 * g + 2 * q) ^ (g & 1);
        uint32_t w[4];
        for (int i = 0; i < 4; i++) {
            const int cc = comb3(g2[l][i], g1[l][i], g0[l][i]) >> 15;
            if (cc < -8192 || cc > 8192) range_violations()++;          // the exact division's domain (make_quant)
            const QEntry &qe = t.q[e0i ^ (i & 1)];
            w[i] = limbs16((int)umulhi32((uint32_t)(cc + (cc >> 31) + qe.bias), qe.recip) * qe.t - qe.unbias);
        }
        bl[l] = w[0] | (w[1] << 16);
        br[l] = w[2] | (w[3] << 16);
    }
    for (int blk = 0; blk < 2; blk++) {
        int h0[32][4], h1[32][4];
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].i1a[0];
            f1[l] = K[l].i1a[1];
            memcpy(c[l], K[l].ci1, sizeof(c[l]));
        }
        mma_emu(false, h0, f0, f1, blk ? br : bl, c);
        for (int l = 0; l < 32; l++) { f0[l] = K[l].i1a[2]; f1[l] = K[l].i1a[3]; }
        mma_emu(false, h1, f0, f1, blk ? br : bl, cz);
        for (int l = 0; l < 32; l++) {                                   // 32 x the sum: bits 16..31 are the output + OFF3
            const uint32_t x0 = (uint32_t)comb3(h1[l][0], h0[l][2], h0[l][0]), x1 = (uint32_t)comb3(h1[l][1], h0[l][3], h0[l][1]);
            const int v0 = (int)(x0 >> 16) - OFF3, v1 = (int)(x1 >> 16) - OFF3;
            if (v0 < -21047 || v0 > 21047 || v1 < -21047 || v1 > 21047) range_violations()++;   // the bound DESIGN.md 4.1 derives
            (blk ? a1 : a0)[l] = (x0 >> 16) | (x1 & 0xffff0000u);
        }
    }
    for (int G = 0; G < 3; G++) {
        for (int l = 0; l < 32; l++) {
            f0[l] = K[l].i2b[G];
            memcpy(c[l], G == 0 ? K[l].ci2 : cz[l], sizeof(c[l]));
        }
        mma_emu(true, G == 0 ? g0 : (G == 1 ? g1 : g2), a0, a1, f0, c);
    }
    for (int l = 0; l < 32; l++) {
        const int g = l >> 2, q = l & 3;
        for (int i = 0; i < 4; i++) {
            if (!(i >= 2 ? t.right : t.left)) continue;
            t.out[g * t.opitch + (i >= 2 ? 8 : 0) + 2 * q + (i & 1)] = (uint8_t)clamp255(comb3(g2[l][i], g1[l][i], g0[l][i]) >> 18);
        }
    }
}
#endif

}  // namespace mma
}  // namespace V5_NS
