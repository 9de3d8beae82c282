// v5ela_device.cuh — device code of the fused V5 ELA + texture kernel (sm_100a).
//
// One CTA walks DOWN a vertical strip of a frame (<= TW_MAX MCUs = 480 px wide, plus one halo MCU column each side),
// one 16-pixel-tall MCU row ("band") per iteration, and for every band does, entirely in shared memory/registers:
//
//   load      : RGB band (16 lines x up to 512 px) global -> smem, edge-replicated            (SURVEY.md A.3)
//   convert   : RGB -> Y, Cb, Cr (16-bit fixed point), h2v2 chroma box downsample            (A.2, A.3)
//   blocks    : per 8x8 block, one thread: ISLOW fDCT -> quantise -> dequantise -> ISLOW IDCT (A.4, A.5, A.6)
//   residual  : h2v2 fancy upsample, YCbCr -> RGB, |orig - recon|, histogram; luma Laplacian  (A.7, A.8, A.9, §8a)
//
// The decoder's fancy upsampling needs one chroma sample beyond every 8x8 chroma block: horizontally that is what the
// halo MCU columns are for (their chroma is recomputed, (TW+2)/TW extra chroma work); vertically the strip walk keeps the
// previous band's decoded chroma in a two-band ring, and the residual stage of iteration r covers pixel rows
// 16r-1 .. 16r+14 — the last row of a band is finished one iteration later, when the chroma row below it exists.
// Each frame byte is read from HBM once (halo columns come from L2).
//
// The file is also compiled by g++ for tests/emu (a thread-emulating CPU harness used to debug indexing without a GPU);
// every CUDA-specific construct therefore goes through the small V5_* shims below. The product never runs that build.
#pragma once
#include <stdint.h>
#include <string.h>

#include "v5ela.h"

#ifdef __CUDACC__
#define V5_DEV __device__ __forceinline__
#define V5_HOSTDEV __host__ __device__ __forceinline__
#else
#define V5_DEV inline
#define V5_HOSTDEV inline
#endif

// The library carries the device code twice, as two translation units with different block stages (V5_MMA_BLOCKS): v5ela.cu builds
// it in namespace v5 (shared-memory transposes, also what the codec kernels take their DCT passes from), v5ela_mma.cu in namespace
// v5m (tensor-core form). V5_NS names the namespace of the current build.
#ifndef V5_NS
#define V5_NS v5
#endif

// The kernel's parameter block and the work decomposition it carries are the same in both builds: namespace v5plan holds them
// once, for the two builds, the C ABI and the emulator (v5ela_host.h fills them).
namespace v5plan {

// ----------------------------------------------------------------------------------------------- geometry constants
#ifndef V5_NT
#define V5_NT 256
#endif
#ifndef V5_TW_MAX
#define V5_TW_MAX 30
#endif
#ifndef V5_MIN_CTAS
#define V5_MIN_CTAS 2
#endif
constexpr int NT = V5_NT;                   // threads per CTA
constexpr int TW_MAX = V5_TW_MAX;           // strip width, MCUs (16 px)
constexpr int MIN_CTAS = V5_MIN_CTAS;       // resident CTAs per SM the kernel is built for

// Exact division constants for one quantisation table entry T (divisor d = 8T), see make_quant():
//   q_biased = umulhi(c + (c >> 31) + bias, recip);  dequantised = q_biased * t - unbias
struct QuantTab {
    uint32_t recip[64];
    int32_t bias[64];
    int32_t t[64];
    int32_t unbias[64];
};

struct LaneConsts;              // v5ela_dctmma.cuh

// One frame of a ragged batch (v5ela_analyze_ragged): its own geometry, pointers and work decomposition. Built on the host,
// read by the RAGGED instantiation's make_geo; uniform batches keep everything in KParams (the kernel-parameter constant bank).
struct FrameDesc {
    const uint8_t *rgb;
    uint8_t *resid;             // optional
    int64_t row_stride;
    int32_t h, w, mw, mh;
    int32_t n_strips, n_segs;
    uint32_t work_base;         // first work item of this frame; items = n_strips * n_segs
    uint32_t flags;             // bit 0: vec_ok, bit 1: resid_vec_ok
};

// One entry of a sweep (v5ela_analyze_sweep) beside its FrameDesc: the entry's quantisation tables and its JPEG-ghost map. Read by
// the sweep kernel only (process_work_item's SWEEP).
struct SweepEntry {
    uint32_t *ghost;            // optional: ceil(h/16) x ceil(w/16) per-MCU sums of the squared residual
    int32_t slot;               // tables sweep_quant(..)[2 * slot] (luma), [2 * slot + 1] (chroma)
    int32_t pad;
};

// A sweep's device table (plan_sweep): its n entries' FrameDesc, then their SweepEntry, then two QuantTab per slot. The sweep kernel
// finds the two tables behind KParams::frames, so that KParams, and with it every other kernel's parameter layout, stays as it is.
V5_HOSTDEV const SweepEntry *sweep_entries(const FrameDesc *frames, int n) { return reinterpret_cast<const SweepEntry *>(frames + n); }
V5_HOSTDEV const QuantTab *sweep_quant(const FrameDesc *frames, int n) { return reinterpret_cast<const QuantTab *>(sweep_entries(frames, n) + n); }
static_assert(sizeof(FrameDesc) % 8 == 0 && sizeof(SweepEntry) % 8 == 0, "sweep table alignment");

struct KParams {
    const uint8_t *rgb;
    int64_t frame_stride;
    int64_t row_stride;
    v5ela_record *records;
    uint8_t *residual;          // optional
    uint32_t *tex_hist;         // optional: n x 256 counters of min(|Laplacian|, 255)
    int n, h, w;
    int mw, mh;                 // MCU columns / rows of the padded frame
    int n_strips, n_segs;       // work decomposition: strips x vertical segments per frame
    int split_frame, n_segs_b;  // frames >= split_frame are cut into n_segs_b (shorter) segments: the tail of the launch (fill_params)
    int work_split;             // first work item of the frames >= split_frame
    unsigned int *ticket;       // work-item counter (zeroed before every launch): CTAs draw items dynamically
    const LaneConsts *lane_consts;        // 32 entries (v5ela_dctmma.cuh), device memory owned by the handle
    const FrameDesc *frames;    // ragged batches only: n descriptors in device memory (then h, w, ... above are unused)
    int vec_ok;                 // 1: every band line start is 16-byte aligned in global memory (128-bit loads)
    int resid_vec_ok;           // 1: residual rows are 16-byte aligned (3*W % 16 == 0 and base aligned): 128-bit stores
    QuantTab q[2];              // [0] luma, [1] chroma — lives in the kernel parameter constant bank
};

}  // namespace v5plan

namespace V5_NS {

using namespace v5plan;                     // the device code, and callers that name the plan through a build (v5::fill_params, ...)

// Block stage (8x8 round trip): 1 = int8 limb-split tensor-core form (v5ela_dctmma.cuh, kernel v11), 0 = the v2..v10 form
// (4 threads per block, two shared-memory transposes) kept as a compile-time variant for A/B runs.
#ifndef V5_MMA_BLOCKS
#define V5_MMA_BLOCKS 0
#endif
#ifndef V5_MMA_NP
#define V5_MMA_NP 1                         // pairs of blocks in flight per warp (1, 2, 4 measured: profiles/r02/variants.txt)
#endif
constexpr int BAND_MCUS = TW_MAX + 2;       // + halo MCU column each side
constexpr int BAND_PX = BAND_MCUS * 16;     // 512
constexpr int RGB_PITCH = BAND_PX * 3;      // 1536 bytes per band line
// Plane pitches. The tensor-core block stage reads 4 pixels of 8 consecutive lines per quarter warp: 16 bytes of padding per line
// put those lines into different banks (pitch / 4 = 4 mod 32) — conflict-free 32-bit loads and 16-bit stores.
constexpr int PLANE_PAD = V5_MMA_BLOCKS ? 16 : 0;
constexpr int Y_PITCH = BAND_PX + PLANE_PAD;        // 512 (+16)
constexpr int C_PITCH = BAND_PX / 2 + PLANE_PAD;    // 256 (+16)

// ------------------------------------------------------------------------------------------------------- shims
struct alignas(16) U4 { uint32_t x, y, z, w; };
struct alignas(8) U2 { uint32_t x, y; };

#ifdef __CUDA_ARCH__
V5_DEV uint32_t umulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
V5_DEV int clamp255(int v) { return __vimin_s32_relu(v, 255); }
V5_DEV void smem_inc(uint32_t *p) { atomicAdd(p, 1u); }
V5_DEV void smem_add(uint32_t *p, uint32_t v) { atomicAdd(p, v); }
V5_DEV uint32_t absdiff4(uint32_t a, uint32_t b) { return __vabsdiffu4(a, b); }
// PTX prmt (default mode): result byte i = byte sel[4i+2:4i] of {b,a}; selector bit 3 replicates that byte's sign bit.
V5_DEV uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
#else
inline uint32_t umulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
inline int clamp255(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }
inline void smem_inc(uint32_t *p) { *p += 1u; }
inline void smem_add(uint32_t *p, uint32_t v) { *p += v; }
inline uint32_t absdiff4(uint32_t a, uint32_t b)
{
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) {
        const int x = (a >> (8 * i)) & 0xff, y = (b >> (8 * i)) & 0xff;
        r |= (uint32_t)(x > y ? x - y : y - x) << (8 * i);
    }
    return r;
}
inline uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    const uint64_t v = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) {
        const uint32_t n = (sel >> (4 * i)) & 0xf;
        uint32_t byte = (uint32_t)(v >> (8 * (n & 7))) & 0xff;
        if (n & 8) byte = (byte & 0x80) ? 0xff : 0x00;
        r |= byte << (8 * i);
    }
    return r;
}
#endif

// Byte-lane selector constants of the residual stage. As literals ptxas rematerialises each one with a UMOV in front of
// (almost) every use — 3 % of the kernel's issue slots; as a table in constant memory four of them arrive with one
// uniform 128-bit load (LDCU.128). Index = 4 * family + byte lane.
enum { SEL_ONE = 0, SEL_THREE = 4, SEL_FOUR = 8, SEL_HALF = 12, SEL_LAP = 16, SEL_TRI = 20 };   // SEL_HALF: 0x8000 (rounding of the colour
                                                                                     // conversion); SEL_TRI: the two triangle kernels
#ifndef V5_CONST_SEL
#define V5_CONST_SEL 1
#endif
#if defined(__CUDACC__) && V5_CONST_SEL
static __constant__ uint32_t kSelTab[24] = {1u,       1u << 8,    1u << 16,    1u << 24,  3u,     3u << 8, 3u << 16, 3u << 24, 4u, 4u << 8,
                                            4u << 16, 4u << 24,   0x8000u,     0u,        0u,      0u,
                                            0x01fc01u, 0x01fc0100u, 0xfc010000u, 0x000001fcu,
                                            0x03090103u, 0x01030309u, 0x09030301u, 0x03010903u};
#endif
#if defined(__CUDA_ARCH__) && V5_CONST_SEL
V5_DEV uint32_t sel_const(int i) { return kSelTab[i]; }
#else
V5_HOSTDEV constexpr uint32_t sel_const(int i)
{
    return i < 12 ? (i < 4 ? 1u : (i < 8 ? 3u : 4u)) << (8 * (i & 3))
                  : (i < 16 ? (i == 12 ? 0x8000u : 0u)
                            : (i == 16 ? 0x01fc01u
                                       : (i == 17 ? 0x01fc0100u
                                                  : (i == 18 ? 0xfc010000u
                                                             : (i == 19 ? 0x000001fcu
                                                                        : (i == 20 ? 0x03090103u
                                                                                   : (i == 21 ? 0x01030309u : (i == 22 ? 0x09030301u : 0x03010903u))))))));
}
#endif

// Integer dot products on packed bytes (IDP on the FMA pipe): they replace byte extraction (PRMT on the ALU pipe).
//   dp4a_us(a, b, c) = c + sum_i u8(a.byte[i]) * s8(b.byte[i])
//   dp2a_lo/hi_su(a, b, c) = c + s16(a.lo) * u8(b.byte[0|2]) + s16(a.hi) * u8(b.byte[1|3]);  _uu: a halves unsigned
#ifdef __CUDA_ARCH__
V5_DEV int dp4a_us(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// dp4a_uu(a, b, c) = c + sum_i u8(a.byte[i]) * u8(b.byte[i])
V5_DEV uint32_t dp4a_uu(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
V5_DEV int dp2a_lo_su(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
V5_DEV int dp2a_hi_su(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
V5_DEV int dp2a_lo_uu(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
V5_DEV int dp2a_hi_uu(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// histogram update: bin = byte k of word; the bin's shared address comes out of one dp4a (base + 4 * byte)
V5_DEV void hist_add(uint32_t *hist_c, uint32_t word, int k)
{
    const uint32_t addr = (uint32_t)dp4a_us(word, sel_const(SEL_FOUR + k), (int)(uint32_t)__cvta_generic_to_shared(hist_c));
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u) : "memory");
}
#else
inline int dp4a_us(uint32_t a, uint32_t b, int c)
{
    for (int i = 0; i < 4; i++) c += (int)((a >> (8 * i)) & 0xff) * (int)(int8_t)((b >> (8 * i)) & 0xff);
    return c;
}
inline uint32_t dp4a_uu(uint32_t a, uint32_t b, uint32_t c)
{
    for (int i = 0; i < 4; i++) c += ((a >> (8 * i)) & 0xff) * ((b >> (8 * i)) & 0xff);
    return c;
}
inline int dp2a_su_(uint32_t a, uint32_t b, int c, int hi, bool sgn)
{
    const int a0 = sgn ? (int)(int16_t)(a & 0xffff) : (int)(a & 0xffff), a1 = sgn ? (int)(int16_t)(a >> 16) : (int)(a >> 16);
    return c + a0 * (int)((b >> (16 * hi)) & 0xff) + a1 * (int)((b >> (16 * hi + 8)) & 0xff);
}
inline int dp2a_lo_su(uint32_t a, uint32_t b, int c) { return dp2a_su_(a, b, c, 0, true); }
inline int dp2a_hi_su(uint32_t a, uint32_t b, int c) { return dp2a_su_(a, b, c, 1, true); }
inline int dp2a_lo_uu(uint32_t a, uint32_t b, int c) { return dp2a_su_(a, b, c, 0, false); }
inline int dp2a_hi_uu(uint32_t a, uint32_t b, int c) { return dp2a_su_(a, b, c, 1, false); }
inline void hist_add(uint32_t *hist_c, uint32_t word, int k) { hist_c[(word >> (8 * k)) & 0xff] += 1u; }
#endif

// Bulk asynchronous copy (TMA, non-tensor form) global -> shared, completion counted in bytes on an mbarrier.
#ifdef __CUDA_ARCH__
V5_DEV uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
V5_DEV void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
V5_DEV void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
V5_DEV void async_proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
V5_DEV void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
V5_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
V5_DEV void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
V5_DEV void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "V5_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra V5_DONE_%=;\n\t"
        "bra V5_WAIT_%=;\n\t"
        "V5_DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
#else
inline void mbar_init(uint64_t *, uint32_t) {}
inline void mbar_init_fence() {}
inline void async_proxy_fence() {}
inline void mbar_expect_tx(uint64_t *, uint32_t) {}
inline void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *) { memcpy(dst, src, bytes); }
inline void mbar_arrive(uint64_t *) {}
inline void mbar_wait(uint64_t *, uint32_t) {}
#endif

// cvt.pack.sat.u8.s32 (SASS I2IP): d = (c.lo16 << 16) | (sat_u8(a) << 8) | sat_u8(b) — clamp to 0..255 and pack in one go
#ifdef __CUDA_ARCH__
V5_DEV uint32_t packsat2(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
#else
inline uint32_t packsat2(int a, int b, uint32_t c)
{
    return ((c & 0xffffu) << 16) | ((uint32_t)clamp255(a) << 8) | (uint32_t)clamp255(b);
}
#endif
// four ints -> bytes [v0, v1, v2, v3], each clamped to 0..255: two I2IP
V5_DEV uint32_t pack4sat(int v0, int v1, int v2, int v3) { return packsat2(v1, v0, packsat2(v3, v2, 0u)); }

// byte k (compile-time) of w, zero-extended: one PRMT
V5_DEV uint32_t byte_of(uint32_t w, int k) { return prmt(w, 0u, 0x4440u + (uint32_t)k); }
// four values 0..255 held in ints -> one word: three PRMTs
V5_DEV uint32_t pack4(int a, int b, int c, int d)
{
    return prmt(prmt((uint32_t)a, (uint32_t)b, 0x0040u), prmt((uint32_t)c, (uint32_t)d, 0x0040u), 0x5410u);
}

// ------------------------------------------------------------------------------------------------- shared memory
struct alignas(16) QEntry { uint32_t recip; int32_t bias, t, unbias; };   // one LDS.128 per coefficient

#ifndef __CUDA_ARCH__
// host compilations only (used by the g++ build, tests/emu): 16-bit hand-offs of the block stage that did not fit 16 bits, counted (tests assert 0)
inline long long &range_violations()
{
    static long long n = 0;
    return n;
}
#endif
}  // namespace V5_NS
#include "v5ela_dctmma.cuh"
namespace V5_NS {

// Two shared-memory layouts, chosen by the number of resident CTAs the kernel is built for:
//   RGB_BUFS == 2 (2 CTAs/SM): double-buffered RGB band (TMA runs a whole iteration ahead), original pixels for the
//                  residual stage come from shared memory, 32-line luma ring.
//   RGB_BUFS == 1 (3 CTAs/SM): one RGB staging buffer (the TMA copy of band r+1 is issued as soon as band r has been
//                  converted and lands during the block and residual stages), the residual stage re-reads the original
//                  pixels from global memory (L2 hits: the band went through L2 moments ago), 24-line luma ring.
#ifndef V5_RGB_BUFS
#define V5_RGB_BUFS (MIN_CTAS >= 3 ? 1 : 2)
#endif
constexpr int RGB_BUFS = V5_RGB_BUFS;       // (a compile-time knob of its own for the CTA-shape experiments, profiles/r02/variants.txt)
constexpr int RING = RGB_BUFS == 2 ? 32 : 24;   // yorig ring lines: 16 of the current band + 2 carried
#ifndef V5_RINGD
#define V5_RINGD (RGB_BUFS == 2 ? 32 : 24)
#endif
constexpr int RINGD = V5_RINGD;         // ydec ring lines (16 + 1 carried); a power of two where shared memory allows: the
                                        // ring index is computed per 8-pixel unit

// Two-phase band loop for the width-multiple-of-16 instantiations (v5ela_workitem.cuh): the residual stage of band r-1 and the
// conversion of band r share one barrier-delimited phase, the block stage of band r is the other — two CTA barriers per band
// instead of three. What the conversion of band r overwrites while the residual stage of band r-1 still reads it is kept aside
// during the block stage before: luma lines 14, 15 of band r-2 (ycarry), and RGB line 15 is carried then as well.
// Measured 2.3-2.7 % SLOWER than three phases with either block stage (profiles/r02/variants.txt section 12: the request for band r+1
// can only be issued one block stage ahead instead of a whole band, and the long mixed phase schedules worse) and therefore off: a
// compile-time variant like the split barrier, kept bit-exact by the emulator tests.
#ifndef V5_FUSE2
#define V5_FUSE2 0
#endif
#ifndef V5_PAIR_ROWS
#define V5_PAIR_ROWS 1
#endif
constexpr bool FUSE2_OK = V5_FUSE2 && RGB_BUFS == 2 && V5_PAIR_ROWS && RING == 32;

struct alignas(16) Smem {
    QEntry qtab[2][64];                 // [0] luma, [1] chroma: copied from the kernel parameters once per work item (tensor-core
                                        // block stage: in mma::qswz_pos order, unbias minus the limb offset)
#if V5_MMA_BLOCKS
#ifdef __CUDA_ARCH__
    U4 lane[8][32];                     // per-lane operand fragments of the four passes (mma::LaneConsts), 128-bit word j of lane l
                                        // at [j][l]: a warp's load of one word is 512 contiguous bytes, conflict-free
#else
    mma::LaneConsts lane[32];
#endif
#endif
    uint8_t rgb[RGB_BUFS][16][RGB_PITCH];   // band r in rgb[rb(r)]; with two buffers the other one receives band r+1
    uint8_t rgb_carry[RGB_BUFS == 2 ? 2 : 1][RGB_BUFS == 2 ? RGB_PITCH : 16];   // line 15 of band r (two-buffer layout only)
#if !V5_MMA_BLOCKS
    uint32_t tscratch[NT / 32][8 * 36]; // block stage: per warp, 8 blocks x (64 int16 + pad): both transpositions;
                                        // 36-word block stride = conflict-free scattered stores and 128-bit loads
#endif
    uint8_t yorig[RING][Y_PITCH];       // luma of the original; band r line l at [(16r + l) mod RING]
    uint8_t ycarry[FUSE2_OK ? 2 : 1][FUSE2_OK ? Y_PITCH : 16];   // two-phase band loop only: lines 14 and 15 of the band before the one the residual stage works on
    uint8_t ydec[RINGD][Y_PITCH];       // luma after the JPEG round trip; band r line l at [(16r + l) mod RINGD]
    uint8_t cenc[2][8][C_PITCH];        // downsampled Cb/Cr of the current band (input of the block stage)
    uint8_t cdec[2][16][C_PITCH];       // decoded Cb/Cr; band r chroma line j at [8*(r&1) + j]
    uint32_t hist[3][256];
    union {
        uint32_t tex_hist[256];         // histogram of min(|Laplacian|, 255); only the TEXHIST instantiation touches it
        uint32_t ghost[2][TW_MAX];      // sweep kernel: the JPEG-ghost cells of the strip's MCUs, MCU row R in ghost[R & 1]
    };
    unsigned long long tex_sumabs, tex_sumsq;
    unsigned long long full_bar[2];     // mbarriers: "band has landed in rgb[b]"
    unsigned long long done_bar;        // mbarrier (count NT): "every thread has finished the residual stage of the band before"
    unsigned long long pad2_;
    uint32_t tex_maxabs;
    uint32_t next_work;                 // ticket drawn by thread 0 for the CTA's next work item
    uint32_t pad_[2];
};
static_assert(2 * TW_MAX <= 256, "the sweep kernel's ghost cells live in tex_hist's shared memory");

// Per work item geometry (uniform across the CTA).
struct Geo {
    const uint8_t *frame;       // first byte of this frame
    uint8_t *resid;             // first byte of this frame's residual map, or null
    int64_t row_stride;         // the frame's geometry: copies of KParams' fields for a uniform batch (the compiler folds them
    int h, w, mw, mh;           // back into constant-bank operands), the frame's own descriptor for a ragged one
    int vec_ok, resid_vec_ok;
    int m0, m1;                 // strip MCU columns [m0, m1)
    int r0, r1;                 // segment MCU rows [r0, r1)
    int xb0;                    // pixel column of band smem column 0 (= 16*(m0-1), may be -16)
    int band_mcus;              // m1 - m0 + 2
};

struct ThreadAcc {              // per-thread state that lives across barriers (registers on the device)
    unsigned long long tex_sumsq;
    uint32_t tex_sumabs;
    uint32_t tex_maxabs;
    uint32_t phase;             // bit b: parity of the next wait on full_bar[b], bit 2: on done_bar (persist across work items)
#if !V5_MMA_BLOCKS
    int col[16];                // block stage: two columns between the two halves of the column sub-stage
#endif
};

V5_DEV int rb(int r) { return RGB_BUFS == 2 ? (r & 1) : 0; }           // RGB buffer / mbarrier of band r
V5_DEV int ring16(int r, int l)                                        // yorig line; l in [-2, 15]
{
    if (RING == 32) return (16 * (r & 1) + l) & 31;
    int i = 16 * (r % 3) + l;                                           // 16r mod 24 cycles 0,16,8
    i = i >= RING ? i - RING : i;
    i = i >= RING ? i - RING : i;
    return i < 0 ? i + RING : i;
}
V5_DEV int ringd(int r, int l)                                         // ydec line; l in [-1, 15]
{
    if (RINGD == 32) return (16 * (r & 1) + l) & 31;
    int i = 16 * (r % 3) + l;                                           // 16r mod 24 cycles 0,16,8
    i = i >= RINGD ? i - RINGD : i;
    i = i >= RINGD ? i - RINGD : i;
    return i < 0 ? i + RINGD : i;
}
V5_DEV int ring8(int r, int j) { return (8 * (r & 1) + j) & 15; }     // j in [-1, 7]

// ------------------------------------------------------------------------------------------------ stage: load band
// Band r, lines 0..15 <- frame rows min(16r + l, H-1), pixel columns [xb0, xb0 + 16*band_mcus) clipped to [0, W);
// columns W .. Wm-1 replicate pixel W-1 (A.3: edges are replicated in full-resolution colour space).
// With 16-byte aligned frames the 16-byte-multiple prefix of every line is fetched by one bulk asynchronous copy per
// line (issued by one thread one whole iteration ahead, completion on full_bar[r & 1]); the few remaining bytes of a
// ragged right edge, the padding columns, and unaligned inputs use ordinary loads.
struct LoadGeo { int xs, nbytes, dst0, npad3, nbulk; };

V5_DEV LoadGeo load_geo(const KParams &p, const Geo &g)
{
    LoadGeo L;
    L.xs = g.xb0 < 0 ? 0 : g.xb0;
    int xe = g.xb0 + 16 * g.band_mcus;
    const int xpad_end = xe > 16 * g.mw ? 16 * g.mw : xe;       // last padded column (exclusive) inside this band
    if (xe > g.w) xe = g.w;
    L.nbytes = 3 * (xe - L.xs);
    L.dst0 = 3 * (L.xs - g.xb0);
    L.npad3 = 3 * (xpad_end - g.w);                             // > 0 only in the strip that holds the right edge
    L.nbulk = g.vec_ok ? (L.nbytes & ~15) : 0;
    return L;
}

V5_DEV bool use_bulk(const KParams &p, const Geo &g) { return load_geo(p, g).nbulk > 0; }

// Threads 0..15 (one per band line): thread 0 arms the barrier with the byte count, every thread issues the bulk copy of
// its line. The barrier phase cannot complete before thread 0's arrive, whatever order the copies land in.
V5_DEV void stage_prefetch(int tid, Smem &S, const KParams &p, const Geo &g, int r)
{
    if (tid >= 16) return;
    const LoadGeo L = load_geo(p, g);
    unsigned long long *bar = &S.full_bar[rb(r)];
    async_proxy_fence();                                        // earlier generic accesses to this buffer are done
    if (tid == 0) mbar_expect_tx(reinterpret_cast<uint64_t *>(bar), 16u * (uint32_t)L.nbulk);
    int y = 16 * r + tid;
    if (y > g.h - 1) y = g.h - 1;
    bulk_g2s(&S.rgb[rb(r)][tid][L.dst0], g.frame + (int64_t)y * g.row_stride + 3 * L.xs, (uint32_t)L.nbulk,
             reinterpret_cast<uint64_t *>(bar));
}

V5_DEV bool load_rest_needed(const KParams &p, const Geo &g, bool bulk)
{
    const LoadGeo L = load_geo(p, g);
    return (bulk ? L.nbulk : 0) != L.nbytes || L.npad3 > 0;
}

// all threads: whatever the bulk copy does not cover (everything when bulk == false)
V5_DEV void stage_load_rest(int tid, Smem &S, const KParams &p, const Geo &g, int r, bool bulk)
{
    const LoadGeo L = load_geo(p, g);
    uint8_t(*dst)[RGB_PITCH] = S.rgb[rb(r)];
    const int warp = tid >> 5, lane = tid & 31;
    int done = bulk ? L.nbulk : 0;
    if (done == L.nbytes && L.npad3 <= 0) return;
    for (int l = warp; l < 16; l += NT / 32) {                  // one warp per band line
        int y = 16 * r + l;
        if (y > g.h - 1) y = g.h - 1;
        const uint8_t *src = g.frame + (int64_t)y * g.row_stride + 3 * L.xs;
        for (int b = done + lane; b < L.nbytes; b += 32) dst[l][L.dst0 + b] = src[b];
        for (int b = lane; b < L.npad3; b += 32)
            dst[l][3 * (g.w - g.xb0) + b] = g.frame[(int64_t)y * g.row_stride + 3 * (g.w - 1) + (b % 3)];
    }
}

// ------------------------------------------------------------------------------------- stage: colour convert (A.2/A.3)
// Colour conversion straight from the packed RGBRGB... words with dp2a (16-bit coefficient pairs x 2 pixel bytes):
// pixel k starts at byte 3k; depending on 3k mod 4 its (R,G)(B) or (R)(G,B) byte pairs sit in the low/high half of one or two
// words. pair() = coefficient pair {first byte, second byte}.
V5_DEV constexpr uint32_t pair(int first, int second) { return ((uint32_t)first & 0xffffu) | ((uint32_t)second << 16); }

// c + cR*R + cG*G + cB*B for pixel k (compile time) of the packed words w[]; UNS: coefficients are unsigned 16-bit
template <bool UNS, int CR, int CG, int CB>
V5_DEV int rgb_dot(const uint32_t *w, int k, int c)
{
    const int o = 3 * k, wi = o >> 2, bp = o & 3;
    const uint32_t rg = pair(CR, CG), b0 = pair(CB, 0), r1 = pair(0, CR), gb = pair(CG, CB);
    if (UNS) {
        if (bp == 0) return dp2a_hi_uu(b0, w[wi], dp2a_lo_uu(rg, w[wi], c));
        if (bp == 3) return dp2a_lo_uu(gb, w[wi + 1], dp2a_hi_uu(r1, w[wi], c));
        if (bp == 2) return dp2a_lo_uu(b0, w[wi + 1], dp2a_hi_uu(rg, w[wi], c));
        return dp2a_hi_uu(gb, w[wi], dp2a_lo_uu(r1, w[wi], c));
    } else {
        if (bp == 0) return dp2a_hi_su(b0, w[wi], dp2a_lo_su(rg, w[wi], c));
        if (bp == 3) return dp2a_lo_su(gb, w[wi + 1], dp2a_hi_su(r1, w[wi], c));
        if (bp == 2) return dp2a_lo_su(b0, w[wi + 1], dp2a_hi_su(rg, w[wi], c));
        return dp2a_hi_su(gb, w[wi], dp2a_lo_su(r1, w[wi], c));
    }
}

// A.2. Cb and Cr have one coefficient equal to 32768, which does not fit a signed 16-bit half, so they are evaluated
// negated: -Cb = (N - K + 65535) >> 16 with N = 11059 R + 21709 G - 32768 B, K = (128 << 16) + 32767 (floor(-x) = -ceil(x)).
V5_DEV int y_of(const uint32_t *w, int k) { return rgb_dot<true, 19595, 38470, 7471>(w, k, 32768) >> 16; }
V5_DEV int neg_cb_of(const uint32_t *w, int k)
{
    return rgb_dot<false, 11059, 21709, -32768>(w, k, 65535 - ((128 << 16) + 32767)) >> 16;
}
V5_DEV int neg_cr_of(const uint32_t *w, int k)
{
    return rgb_dot<false, -32768, 27439, 5329>(w, k, 65535 - ((128 << 16) + 32767)) >> 16;
}

// 8 pixels of two band lines: optional luma (8 bytes per line) and the 4 downsampled Cb/Cr samples.
template <bool WANT_Y, bool WANT_C>
V5_DEV void convert8x2(const uint8_t *la, const uint8_t *lb, U2 &y0, U2 &y1, uint32_t &cbo, uint32_t &cro)
{
    uint32_t a[6], b[6];
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const U2 ta = reinterpret_cast<const U2 *>(la)[i], tb = reinterpret_cast<const U2 *>(lb)[i];
        a[2 * i] = ta.x; a[2 * i + 1] = ta.y;
        b[2 * i] = tb.x; b[2 * i + 1] = tb.y;
    }
    if (WANT_Y) {
        int ya[8], yb[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            ya[k] = y_of(a, k);
            yb[k] = y_of(b, k);
        }
        y0 = U2{pack4sat(ya[0], ya[1], ya[2], ya[3]), pack4sat(ya[4], ya[5], ya[6], ya[7])};
        y1 = U2{pack4sat(yb[0], yb[1], yb[2], yb[3]), pack4sat(yb[4], yb[5], yb[6], yb[7])};
    }
    if (WANT_C) {                                               // h2v2 box filter, bias 1,2,1,2 along x
        int c[4], d[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int bias = 1 + (j & 1);
            c[j] = (bias - (neg_cb_of(a, 2 * j) + neg_cb_of(a, 2 * j + 1) + neg_cb_of(b, 2 * j) + neg_cb_of(b, 2 * j + 1))) >> 2;
            d[j] = (bias - (neg_cr_of(a, 2 * j) + neg_cr_of(a, 2 * j + 1) + neg_cr_of(b, 2 * j) + neg_cr_of(b, 2 * j + 1))) >> 2;
        }
        cbo = pack4sat(c[0], c[1], c[2], c[3]);
        cro = pack4sat(d[0], d[1], d[2], d[3]);
    }
}

// `defer`: the residual stage of band r-1 ended with an arrive on done_bar instead of a CTA barrier (split barrier: a thread
// that is done early starts converting while others still read the shared buffers this stage overwrites — the luma ring lines
// of band r-2, the carried RGB line, and, through the bulk copy of band r+1, the other RGB buffer). Everything up to a
// unit's stores only reads band r and computes, so the wait for the stragglers sits in front of the first store.
V5_DEV void convert_wait_done(int tid, Smem &S, const KParams &p, const Geo &g, int r, ThreadAcc &acc, bool prefetch_next)
{
    mbar_wait(reinterpret_cast<uint64_t *>(&S.done_bar), (acc.phase >> 2) & 1u);
    acc.phase ^= 4u;
    if (prefetch_next) stage_prefetch(tid, S, p, g, r + 1);
}

V5_DEV void stage_convert(int tid, Smem &S, const KParams &p, const Geo &g, int r, ThreadAcc &acc, bool defer, bool prefetch_next, bool copy_carry = true)
{
    // Chroma line j of this band averages frame rows (2jc, min(2jc+1, H-1)) with jc = min(8r+j, He/2-1): below the
    // image the DOWNSAMPLED last row is replicated, which differs from the luma rule (replicate row H-1) when H is even.
    const int last_cline = ((g.h + 1) >> 1) - 1 - 8 * r;        // local index of the last real chroma line
    const int last_line = g.h - 1 - 16 * r;                     // local index of the last real pixel line
    const uint8_t(*src)[RGB_PITCH] = S.rgb[rb(r)];
    bool waiting = defer;
    if (RGB_BUFS == 2 && !waiting && copy_carry)
        for (int i = tid; i < RGB_PITCH / 16; i += NT)          // keep line 15 for the next iteration's residual stage
            reinterpret_cast<U4 *>(S.rgb_carry[r & 1])[i] = reinterpret_cast<const U4 *>(src[15])[i];
#if defined(V5_CONVERT_UNROLL) && V5_CONVERT_UNROLL
#pragma unroll 2
#endif
    for (int u = tid; u < 8 * 2 * BAND_MCUS; u += NT) {          // unit = 2 lines x 8 px
        const int li = u / (2 * BAND_MCUS), ox = u - li * (2 * BAND_MCUS);
        const int mcu = g.m0 - 1 + (ox >> 1);
        if (ox >= 2 * g.band_mcus || mcu < 0 || mcu >= g.mw) continue;
        U2 y0, y1;
        uint32_t cb, cr;
        convert8x2<true, true>(&src[2 * li][24 * ox], &src[2 * li + 1][24 * ox], y0, y1, cb, cr);
        const int jc = li < last_cline ? li : last_cline;
        int lb = 2 * jc + 1;
        if (lb > last_line) lb = last_line;
        if (jc != li || lb != 2 * li + 1) {                     // only in the band that holds the bottom image edge
            U2 d0, d1;
            convert8x2<false, true>(&src[2 * jc][24 * ox], &src[lb][24 * ox], d0, d1, cb, cr);   // rare path
        }
        if (waiting) {
            convert_wait_done(tid, S, p, g, r, acc, prefetch_next);
            waiting = false;
            if (RGB_BUFS == 2)
                for (int i = tid; i < RGB_PITCH / 16; i += NT)
                    reinterpret_cast<U4 *>(S.rgb_carry[r & 1])[i] = reinterpret_cast<const U4 *>(src[15])[i];
        }
        *reinterpret_cast<U2 *>(&S.yorig[ring16(r, 2 * li)][8 * ox]) = y0;
        *reinterpret_cast<U2 *>(&S.yorig[ring16(r, 2 * li + 1)][8 * ox]) = y1;
        *reinterpret_cast<uint32_t *>(&S.cenc[0][li][4 * ox]) = cb;
        *reinterpret_cast<uint32_t *>(&S.cenc[1][li][4 * ox]) = cr;
    }
    if (waiting) {                                              // a thread without any unit to store still owes the wait
        convert_wait_done(tid, S, p, g, r, acc, prefetch_next);
        if (RGB_BUFS == 2)
            for (int i = tid; i < RGB_PITCH / 16; i += NT)
                reinterpret_cast<U4 *>(S.rgb_carry[r & 1])[i] = reinterpret_cast<const U4 *>(src[15])[i];
    }
}

// Two-phase band loop, during the block stage of band r: RGB line 15 of band r (if it exists) for the residual stage of band r+1,
// luma lines 14, 15 of band r-1 for the residual stage of band r — which runs while band r+1 is converted over them.
V5_DEV void stage_carries(int tid, Smem &S, int r, bool has_band)
{
    constexpr int NRGB = RGB_PITCH / 16, NY = Y_PITCH / 16;
    if (tid < NRGB) {
        if (has_band) reinterpret_cast<U4 *>(S.rgb_carry[r & 1])[tid] = reinterpret_cast<const U4 *>(S.rgb[rb(r)][15])[tid];
    } else if (FUSE2_OK && tid < NRGB + 2 * NY) {
        const int k = tid - NRGB, line = k >= NY ? 1 : 0, i = k - line * NY;
        reinterpret_cast<U4 *>(S.ycarry[FUSE2_OK ? line : 0])[FUSE2_OK ? i : 0] = reinterpret_cast<const U4 *>(S.yorig[ring16(r - 1, 14 + line)])[i];
    }
}

// --------------------------------------------------------------------------------- stage: 8x8 block round trip (A.4-A.6)
#define V5_C0_298 2446
#define V5_C0_390 3196
#define V5_C0_541 4433
#define V5_C0_765 6270
#define V5_C0_899 7373
#define V5_C1_175 9633
#define V5_C1_501 12299
#define V5_C1_847 15137
#define V5_C1_961 16069
#define V5_C2_053 16819
#define V5_C2_562 20995
#define V5_C3_072 25172

// Forward 8-point pass over v[0], v[S], ... v[7S]. PASS1: row pass on UNSIGNED samples (the -128 level shift only
// moves the DC term: -8*128 before the << 2), descale 11. Otherwise: column pass, descale 15, DC descale 2.
template <int S, bool PASS1>
V5_DEV void fdct8(int *v)
{
    const int n = PASS1 ? 11 : 15, rnd = 1 << (n - 1);
    const int t0 = v[0] + v[7 * S], t7 = v[0] - v[7 * S], t1 = v[S] + v[6 * S], t6 = v[S] - v[6 * S];
    const int t2 = v[2 * S] + v[5 * S], t5 = v[2 * S] - v[5 * S], t3 = v[3 * S] + v[4 * S], t4 = v[3 * S] - v[4 * S];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    if (PASS1) {
        v[0] = (t10 + t11 - 1024) * 4;
        v[4 * S] = (t10 - t11) * 4;
    } else {
        v[0] = (t10 + t11 + 2) >> 2;
        v[4 * S] = (t10 - t11 + 2) >> 2;
    }
    v[2 * S] = (t12 * V5_C0_541 + t13 * (V5_C0_541 + V5_C0_765) + rnd) >> n;
    v[6 * S] = (t13 * V5_C0_541 + t12 * (V5_C0_541 - V5_C1_847) + rnd) >> n;
    const int z1 = (t4 + t7) * -V5_C0_899, z2 = (t5 + t6) * -V5_C2_562;
    const int z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * V5_C1_175 + rnd;
    const int z3b = z3 * -V5_C1_961 + z5, z4b = z4 * -V5_C0_390 + z5;
    v[7 * S] = (t4 * V5_C0_298 + z1 + z3b) >> n;
    v[5 * S] = (t5 * V5_C2_053 + z2 + z4b) >> n;
    v[3 * S] = (t6 * V5_C3_072 + z2 + z3b) >> n;
    v[S] = (t7 * V5_C1_501 + z1 + z4b) >> n;
}

// Inverse 8-point pass. FINAL: row pass, descale 18, +128 (the clamp to 0..255 happens in the saturating pack that
// follows); otherwise column pass, descale 11.
template <int S, bool FINAL>
V5_DEV void idct8(int *v)
{
    const int n = FINAL ? 18 : 11;
    const int rnd = (1 << (n - 1)) + (FINAL ? (128 << 18) : 0);
    const int i2 = v[2 * S], i6 = v[6 * S];
    const int t2 = i2 * V5_C0_541 + i6 * (V5_C0_541 - V5_C1_847);
    const int t3 = i6 * V5_C0_541 + i2 * (V5_C0_541 + V5_C0_765);
    const int t0 = (v[0] + v[4 * S]) * 8192 + rnd, t1 = (v[0] - v[4 * S]) * 8192 + rnd;
    int u0 = v[7 * S], u1 = v[5 * S], u2 = v[3 * S], u3 = v[S];
    const int z1 = (u0 + u3) * -V5_C0_899, z2 = (u1 + u2) * -V5_C2_562;
    const int z3 = u0 + u2, z4 = u1 + u3;
    const int z5 = (z3 + z4) * V5_C1_175;
    const int z3b = z3 * -V5_C1_961 + z5, z4b = z4 * -V5_C0_390 + z5;
    u0 = u0 * V5_C0_298 + z1 + z3b;
    u1 = u1 * V5_C2_053 + z2 + z4b;
    u2 = u2 * V5_C3_072 + z2 + z3b;
    u3 = u3 * V5_C1_501 + z1 + z4b;
    // three-input sums (t0 +- t3 +- u): one IADD3 each instead of forming t10..t13 first
    v[0] = (t0 + t3 + u3) >> n;
    v[7 * S] = (t0 + t3 - u3) >> n;
    v[S] = (t1 + t2 + u2) >> n;
    v[6 * S] = (t1 + t2 - u2) >> n;
    v[2 * S] = (t1 - t2 + u1) >> n;
    v[5 * S] = (t1 - t2 - u1) >> n;
    v[3 * S] = (t0 - t3 + u0) >> n;
    v[4 * S] = (t0 - t3 - u0) >> n;
}

// int16 pairs in a word (also used by the codec kernels, v5jpeg_*.cuh)
V5_DEV uint32_t pack_s16(int lo, int hi)
{
#ifndef __CUDACC__
    if (lo < -32768 || lo > 32767 || hi < -32768 || hi > 32767) range_violations()++;
#endif
    return prmt((uint32_t)lo, (uint32_t)hi, 0x5410u);
}
V5_DEV int s16_lo(uint32_t w) { return (int)prmt(w, 0u, 0x9910u); }         // sign-extend the low half: one PRMT
V5_DEV int s16_hi(uint32_t w) { return (int)w >> 16; }

#if !V5_MMA_BLOCKS
// The block stage. Four threads share one 8x8 block; thread j owns rows 2j,2j+1 in the row passes and columns 2j,2j+1
// in the column passes. The two transpositions go through a per-warp shared-memory scratch as int16 pairs (ranges:
// |fDCT row output| <= 4096, |IDCT column output| <= 21047 by Parseval + quantisation error, see DESIGN.md), laid out so
// that both the scattered 32-bit stores and the 128-bit loads are bank-conflict free. Only __syncwarp() is needed between
// the three sub-stages, and the code is ~600 instructions instead of ~1900 for a block-per-thread unrolling (the
// instruction cache, not the ALUs, was the first version's limit).
struct BlockTask {
    const QEntry *q;
    const uint8_t *in;
    uint8_t *out;
    int pitch;
    bool active;
};

// FAST (here and below): the width is a multiple of 16, the frames are 16-byte aligned and no residual map is wanted — every
// 8-pixel unit and every block of a strip lies inside the image horizontally and every band arrives by bulk copy alone, so
// the per-unit edge predicates, the residual store and the fall-back loads compile away. The host picks the instantiation
// (fast_path_ok); both are the same arithmetic.
template <bool FAST>
V5_DEV BlockTask block_task(int blk, Smem &S, const KParams &p, const Geo &g, int r, bool want_y)
{
    BlockTask t;
    t.active = false;
    t.q = S.qtab[0];
    t.in = nullptr;
    t.out = nullptr;
    t.pitch = 0;
    const int tw = g.m1 - g.m0;
    const int nl = want_y ? 4 * tw : 0;
    if (blk < nl) {
        const int br = blk >= 2 * tw ? 1 : 0, bc = blk - br * 2 * tw;
        // blocks entirely below / right of the image are libjpeg "dummy" data: never visible, skip them
        if (16 * r + 8 * br >= g.h || (!FAST && 16 * g.m0 + 8 * bc >= g.w)) return t;
        const int row = ring16(r, 8 * br), col = 16 + 8 * bc;
        t.in = &S.yorig[row][col];
        t.out = &S.ydec[ringd(r, 8 * br)][col];
        t.pitch = Y_PITCH;
        t.active = true;
    } else {
        const int c = blk - nl;
        if (c >= 2 * g.band_mcus) return t;
        const int comp = c >= g.band_mcus ? 1 : 0, cbk = c - comp * g.band_mcus;
        const int mcu = g.m0 - 1 + cbk;
        if (mcu < 0 || mcu >= g.mw) return t;
        t.q = S.qtab[1];
        t.in = &S.cenc[comp][0][8 * cbk];
        t.out = &S.cdec[comp][ring8(r, 0)][8 * cbk];
        t.pitch = C_PITCH;
        t.active = true;
    }
    return t;
}

template <bool FAST>
V5_DEV BlockTask block_task_of(int tid, Smem &S, const KParams &p, const Geo &g, int r, bool want_y, int round)
{
    return block_task<FAST>(round * (NT / 4) + (tid >> 5) * 8 + ((tid & 31) >> 2), S, p, g, r, want_y);
}

V5_DEV int blocks_in_band(const Geo &g, bool want_y) { return (want_y ? 4 * (g.m1 - g.m0) : 0) + 2 * g.band_mcus; }


// sub-stage 1: forward row pass of rows 2j, 2j+1 -> tscratch (column-major pairs)
V5_DEV void blocks_rows_fwd(int tid, Smem &S, const BlockTask &t)
{
    const int warp = tid >> 5, lane = tid & 31, j = lane & 3, bw = lane >> 2;
    if (!t.active) return;
    int a[8], b[8];
    const U2 wa = *reinterpret_cast<const U2 *>(t.in + (2 * j) * t.pitch);
    const U2 wb = *reinterpret_cast<const U2 *>(t.in + (2 * j + 1) * t.pitch);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        a[k] = (int)byte_of(wa.x, k); a[4 + k] = (int)byte_of(wa.y, k);
        b[k] = (int)byte_of(wb.x, k); b[4 + k] = (int)byte_of(wb.y, k);
    }
    fdct8<1, true>(a);
    fdct8<1, true>(b);
    uint32_t *ts = &S.tscratch[warp][36 * bw];
#pragma unroll
    for (int c = 0; c < 8; c++) ts[4 * c + j] = pack_s16(a[c], b[c]);
}

// sub-stage 2a: columns 2j, 2j+1: forward column pass, quantise + dequantise (A.5), inverse column pass -> registers
V5_DEV void blocks_cols(int tid, Smem &S, const BlockTask &t, int *col)
{
    const int warp = tid >> 5, lane = tid & 31, j = lane & 3, bw = lane >> 2;
    if (!t.active) return;
    const uint32_t *ts = &S.tscratch[warp][36 * bw];
    const U4 w0 = *reinterpret_cast<const U4 *>(ts + 8 * j), w1 = *reinterpret_cast<const U4 *>(ts + 8 * j + 4);
    int a[8] = {s16_lo(w0.x), s16_hi(w0.x), s16_lo(w0.y), s16_hi(w0.y), s16_lo(w0.z), s16_hi(w0.z), s16_lo(w0.w), s16_hi(w0.w)};
    int b[8] = {s16_lo(w1.x), s16_hi(w1.x), s16_lo(w1.y), s16_hi(w1.y), s16_lo(w1.z), s16_hi(w1.z), s16_lo(w1.w), s16_hi(w1.w)};
    fdct8<1, false>(a);
    fdct8<1, false>(b);
    const QEntry *qj = t.q + 2 * j;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const QEntry ea = qj[8 * k], eb = qj[8 * k + 1];
        const uint32_t xa = (uint32_t)(a[k] + (a[k] >> 31) + ea.bias), xb = (uint32_t)(b[k] + (b[k] >> 31) + eb.bias);
        a[k] = (int)umulhi32(xa, ea.recip) * ea.t - ea.unbias;
        b[k] = (int)umulhi32(xb, eb.recip) * eb.t - eb.unbias;
    }
    idct8<1, false>(a);
    idct8<1, false>(b);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        col[k] = a[k];
        col[8 + k] = b[k];
    }
}

// sub-stage 2b (after every thread of the warp has read its columns): scatter them back row-major into the scratch
V5_DEV void blocks_cols_store(int tid, Smem &S, const BlockTask &t, const int *col)
{
    const int warp = tid >> 5, lane = tid & 31, j = lane & 3, bw = lane >> 2;
    if (!t.active) return;
    uint32_t *rs = &S.tscratch[warp][36 * bw];
#pragma unroll
    for (int k = 0; k < 8; k++) rs[4 * k + j] = pack_s16(col[k], col[8 + k]);
}

// sub-stage 3: final inverse row pass of rows 2j, 2j+1, +128, clamp, store bytes
V5_DEV void blocks_rows_inv(int tid, Smem &S, const BlockTask &t)
{
    const int warp = tid >> 5, lane = tid & 31, j = lane & 3, bw = lane >> 2;
    if (!t.active) return;
    const uint32_t *rs = &S.tscratch[warp][36 * bw];
    const U4 w0 = *reinterpret_cast<const U4 *>(rs + 8 * j), w1 = *reinterpret_cast<const U4 *>(rs + 8 * j + 4);
    int a[8] = {s16_lo(w0.x), s16_hi(w0.x), s16_lo(w0.y), s16_hi(w0.y), s16_lo(w0.z), s16_hi(w0.z), s16_lo(w0.w), s16_hi(w0.w)};
    int b[8] = {s16_lo(w1.x), s16_hi(w1.x), s16_lo(w1.y), s16_hi(w1.y), s16_lo(w1.z), s16_hi(w1.z), s16_lo(w1.w), s16_hi(w1.w)};
    idct8<1, true>(a);
    idct8<1, true>(b);
    *reinterpret_cast<U2 *>(t.out + (2 * j) * t.pitch) = U2{pack4sat(a[0], a[1], a[2], a[3]), pack4sat(a[4], a[5], a[6], a[7])};
    *reinterpret_cast<U2 *>(t.out + (2 * j + 1) * t.pitch) = U2{pack4sat(b[0], b[1], b[2], b[3]), pack4sat(b[4], b[5], b[6], b[7])};
}

#else   // V5_MMA_BLOCKS
// The block stage, tensor-core form (v5ela_dctmma.cuh): a warp takes NP pairs of horizontally adjacent blocks through the four
// passes in registers. A band's blocks come in four sections — luma block rows 0 and 1 (strip width / 16 pairs each), Cb and Cr
// (ceil(band MCUs / 2) pairs each, the halo columns included) — and a section's pairs are dealt to the warps NP at a time, so the
// per-pair set-up is one add. Blocks [act_lo, act_hi) of a section are stored; the others (libjpeg's dummy blocks right of the
// image, chroma halo columns outside it, the odd block of the last chroma pair) are computed on whatever the plane holds and
// dropped. FAST: the width is a multiple of 16, so every luma block of a strip is inside the image.
constexpr int MMA_NP = V5_MMA_NP;

template <int PITCH, bool ALL_ACTIVE>
V5_DEV void blocks_section(int tid, const mma::LaneConsts *K, const uint8_t *in, uint8_t *out, const QEntry *q, int npairs, int act_lo,
                           int act_hi)
{
    const int warp = tid >> 5;
    for (int k0 = warp * MMA_NP; k0 < npairs; k0 += (NT / 32) * MMA_NP) {
        mma::PairTask t[MMA_NP];
#pragma unroll
        for (int j = 0; j < MMA_NP; j++) {
            const int k = k0 + j < npairs ? k0 + j : npairs - 1;        // a group's tail repeats the last pair without storing it
            t[j].in = in + 16 * k;
            t[j].out = out + 16 * k;
            t[j].q = q;
            t[j].ipitch = t[j].opitch = PITCH;
            t[j].left = k0 + j < npairs && (ALL_ACTIVE || (2 * k >= act_lo && 2 * k < act_hi));
            t[j].right = k0 + j < npairs && (ALL_ACTIVE || (2 * k + 1 >= act_lo && 2 * k + 1 < act_hi));
        }
#ifdef __CUDA_ARCH__
        mma::dct_pairs<MMA_NP>(t, *K, tid & 31);
#else
        for (int j = 0; j < MMA_NP; j++)
            if (t[j].left || t[j].right) mma::dct_pair_emu(t[j], K);
#endif
    }
}

// every warp calls it once per band (emulator: once per warp, tid = 32 * warp)
template <bool FAST>
V5_DEV void stage_blocks_mma(int tid, Smem &S, const KParams &p, const Geo &g, int r, bool want_y)
{
    const int tw = g.m1 - g.m0;
#ifdef __CUDA_ARCH__
    mma::LaneConsts Kreg;                                               // eight LDS.128, once per band
#pragma unroll
    for (int j = 0; j < 8; j++) reinterpret_cast<U4 *>(&Kreg)[j] = S.lane[j][tid & 31];
    const mma::LaneConsts *K = &Kreg;
#else
    const mma::LaneConsts *K = S.lane;                                 // the emulator works on all 32 lanes at once
#endif
    if (want_y) {
        int hi = 2 * tw;
        if (!FAST) {
            const int inside = (g.w - 16 * g.m0 + 7) >> 3;             // luma blocks of this strip that hold image columns
            hi = inside < hi ? inside : hi;
        }
#pragma unroll 1
        for (int br = 0; br < 2; br++) {
            if (16 * r + 8 * br >= g.h) break;                         // block rows below the image: dummy data, never visible
            blocks_section<Y_PITCH, FAST>(tid, K, &S.yorig[ring16(r, 8 * br)][16], &S.ydec[ringd(r, 8 * br)][16], S.qtab[0], tw, 0, hi);
        }
    }
    const int lo = g.m0 == 0 ? 1 : 0;                                  // halo MCU columns outside the image are not real blocks
    const int hi = g.band_mcus < g.mw - g.m0 + 1 ? g.band_mcus : g.mw - g.m0 + 1;
#pragma unroll 1
    for (int comp = 0; comp < 2; comp++)
        blocks_section<C_PITCH, false>(tid, K, &S.cenc[comp][0][0], &S.cdec[comp][ring8(r, 0)][0], S.qtab[1], (g.band_mcus + 1) >> 1, lo, hi);
}
#endif  // V5_MMA_BLOCKS

// ------------------------------------------------------------------- stage: upsample, reconstruct, residual, Laplacian
// Horizontal+vertical fancy upsample (A.7) of one chroma component for 8 output pixels of one line.
// lc / ln: decoded chroma lines (current row, neighbour row), pointing at this unit's first chroma column (4-aligned);
// columns -1 and 4 are the horizontal neighbours. gcx0 = global chroma column of lc[0]; wc1 = Wc - 1.
// Outputs are the upsampled samples MINUS 128 (what the colour conversion wants).
V5_DEV void upsample8(const uint8_t *lc, const uint8_t *ln, int gcx0, int wc1, bool fancy, int out[8])
{
    const uint32_t c0 = *reinterpret_cast<const uint32_t *>(lc - 4), n0 = *reinterpret_cast<const uint32_t *>(ln - 4);
    const uint32_t c1 = *reinterpret_cast<const uint32_t *>(lc), n1 = *reinterpret_cast<const uint32_t *>(ln);
    const uint32_t c2 = *reinterpret_cast<const uint32_t *>(lc + 4), n2 = *reinterpret_cast<const uint32_t *>(ln + 4);
    if (!fancy) {                                               // Wc <= 2: libjpeg uses plain replication
#pragma unroll
        for (int j = 0; j < 4; j++) out[2 * j] = out[2 * j + 1] = (int)byte_of(c1, j) - 128;
        return;
    }
    int cs[6];                                                  // cs[j+1] = 3*c[r][j] + c[nb][j], j = -1..4
    cs[0] = dp4a_us(c0, sel_const(SEL_THREE + 3), dp4a_us(n0, sel_const(SEL_ONE + 3), 0));
#pragma unroll
    for (int j = 0; j < 4; j++) cs[1 + j] = dp4a_us(c1, sel_const(SEL_THREE + j), dp4a_us(n1, sel_const(SEL_ONE + j), 0));
    cs[5] = dp4a_us(c2, sel_const(SEL_THREE), dp4a_us(n2, sel_const(SEL_ONE), 0));
    if (gcx0 == 0) cs[0] = cs[1];                               // left image edge: neighbour clamps to column 0
    if (gcx0 + 4 > wc1) {                                       // right image edge inside / just after this unit
#pragma unroll
        for (int j = 1; j < 6; j++)
            if (gcx0 + j - 1 > wc1) cs[j] = cs[j - 1];
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int t3 = 3 * cs[j + 1] + (8 - 2048);
        out[2 * j] = (t3 + cs[j]) >> 4;
        out[2 * j + 1] = (t3 + cs[j + 2] - 1) >> 4;
    }
}

// The same filter for the width-multiple-of-16 instantiation (Wc is a multiple of 8 and >= 8: always "fancy", the right image
// edge can only fall right after a unit). Both filter steps are folded into ONE dot product per output sample: with
// W = bytes [c_j, n_j, c_j+1, n_j+1] (c: nearer chroma row, n: further one),
//   out[2j]   = (3 (3 c_j + n_j) + (3 c_j-1 + n_j-1) + 8) >> 4 = (W_j-1 . [3, 1, 9, 3] + 8) >> 4
//   out[2j+1] = (3 (3 c_j + n_j) + (3 c_j+1 + n_j+1) + 7) >> 4 = (W_j   . [9, 3, 3, 1] + 7) >> 4
// i.e. 9 PRMT + 8 dp4a + 8 shifts per component instead of 12 dp4a + 8 multiply-adds + 8 adds + 8 shifts.
V5_DEV void upsample8_fast(const uint8_t *lc, const uint8_t *ln, bool left_edge, bool right_edge, int out[8])
{
    const uint32_t c0 = *reinterpret_cast<const uint32_t *>(lc - 4), n0 = *reinterpret_cast<const uint32_t *>(ln - 4);
    const uint32_t c1 = *reinterpret_cast<const uint32_t *>(lc), n1 = *reinterpret_cast<const uint32_t *>(ln);
    const uint32_t c2 = *reinterpret_cast<const uint32_t *>(lc + 4), n2 = *reinterpret_cast<const uint32_t *>(ln + 4);
    // columns -1 .. 2 and 1 .. 4 as words; at an image edge the missing neighbour is the edge column itself
    const uint32_t cs = left_edge ? prmt(c1, 0u, 0x2100u) : prmt(c0, c1, 0x6543u), ns = left_edge ? prmt(n1, 0u, 0x2100u) : prmt(n0, n1, 0x6543u);
    const uint32_t ce = right_edge ? prmt(c1, 0u, 0x3321u) : prmt(c1, c2, 0x4321u), ne = right_edge ? prmt(n1, 0u, 0x3321u) : prmt(n1, n2, 0x4321u);
    uint32_t w[5];
    w[0] = prmt(cs, ns, 0x5140u);                               // columns -1, 0
    w[1] = prmt(c1, n1, 0x5140u);                               // 0, 1
    w[2] = prmt(c1, n1, 0x6251u);                               // 1, 2
    w[3] = prmt(c1, n1, 0x7362u);                               // 2, 3
    w[4] = prmt(ce, ne, 0x7362u);                               // 3, 4
    const uint32_t ke = sel_const(SEL_TRI), ko = sel_const(SEL_TRI + 1);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        out[2 * j] = dp4a_us(w[j], ke, 8 - 2048) >> 4;
        out[2 * j + 1] = dp4a_us(w[j + 1], ko, 7 - 2048) >> 4;
    }
}

// TEXHIST: the optional tex_hist[256] output of the record table (SURVEY.md §8a) is wanted — one more shared-memory
// increment per pixel; an instantiation of its own so that calls without it pay nothing.
// Second half of a unit: given the upsampled chroma (minus 128) of its 8 pixels, reconstruct, residual, histogram, Laplacian.
// SWEEP (the sweep kernel) with `ghost` set: the unit's sum of squared residuals goes into its MCU's ghost cell as well.
template <bool FAST, bool TEXHIST, bool SWEEP = false>
V5_DEV void residual_row(Smem &S, const KParams &p, const Geo &g, ThreadAcc &acc, int r, int l, int ox, const int *cb, const int *cr,
                         bool ghost = false)
{
    const int y = 16 * r + l;                                   // global pixel row
    const int gx0 = 16 * g.m0 + 8 * ox;                         // global pixel column of this unit
    const int col = 16 + 8 * ox;                                // band smem column
    const int nvalid = g.w - gx0;                               // pixels k < nvalid are inside the image (may be > 8; FAST: >= 8)

    // ---- reconstruct (A.8), residual (A.9), histogram
    // R = clamp(Y + ((91881 cr' + 32768) >> 16)) == clamp(((Y << 16) + 32768 + 91881 cr') >> 16): one PRMT builds
    // (Y << 16) + 32768 straight from the packed luma word, the multiply-adds do the rest.
    const U2 yd = *reinterpret_cast<const U2 *>(&S.ydec[ringd(r, l)][col]);
    const uint32_t ydw[2] = {yd.x, yd.y};
    uint32_t ow[6], dw[6];
    if (RGB_BUFS == 2) {
        const uint8_t *orig = l < 0 ? &S.rgb_carry[(r - 1) & 1][3 * col] : &S.rgb[r & 1][l][3 * col];
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const U2 t = reinterpret_cast<const U2 *>(orig)[i];
            ow[2 * i] = t.x; ow[2 * i + 1] = t.y;
        }
    } else {
        // single-buffer layout: the band's RGB is gone from shared memory by now; these 24 bytes were fetched through L2
        // one iteration ago. A unit cut by the image edge (or an unaligned frame) must not read past its row.
        const uint8_t *orig = g.frame + (int64_t)y * g.row_stride + 3 * gx0;
        if (g.vec_ok && nvalid >= 8) {
#pragma unroll
            for (int i = 0; i < 3; i++) {
                const U2 t = reinterpret_cast<const U2 *>(orig)[i];
                ow[2 * i] = t.x; ow[2 * i + 1] = t.y;
            }
        } else {
            const int nb = nvalid >= 8 ? 24 : 3 * nvalid;
#pragma unroll
            for (int i = 0; i < 6; i++) {
                uint32_t w = 0;
#pragma unroll
                for (int b = 0; b < 4; b++)
                    if (4 * i + b < nb) w |= (uint32_t)orig[4 * i + b] << (8 * b);
                ow[i] = w;
            }
        }
    }
    int rec[24];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int ykr = (int)prmt(ydw[k >> 2], sel_const(SEL_HALF), 0x4054u + ((uint32_t)(k & 3) << 8));   // bytes: 00 80 Y 00
        const int cbv = cb[k], crv = cr[k];
        rec[3 * k] = (91881 * crv + ykr) >> 16;                // clamped to 0..255 by the saturating pack below
        rec[3 * k + 1] = (-22554 * cbv + (-46802 * crv + ykr)) >> 16;
        rec[3 * k + 2] = (116130 * cbv + ykr) >> 16;
    }
#pragma unroll
    for (int i = 0; i < 6; i++)
        dw[i] = absdiff4(ow[i], pack4sat(rec[4 * i], rec[4 * i + 1], rec[4 * i + 2], rec[4 * i + 3]));
    if (!FAST && g.resid) {
        uint8_t *dst = g.resid + ((int64_t)y * g.w + gx0) * 3;
        if (nvalid >= 8 && g.resid_vec_ok) {
#pragma unroll
            for (int i = 0; i < 3; i++) reinterpret_cast<U2 *>(dst)[i] = U2{dw[2 * i], dw[2 * i + 1]};
        } else {
#pragma unroll
            for (int b = 0; b < 24; b++)
                if (b < 3 * nvalid) dst[b] = (uint8_t)byte_of(dw[b >> 2], b & 3);
        }
    }
    // Histogram: every unit adds all 24 bytes unconditionally; a unit cut by the right image edge first zeroes the bytes
    // of its outside pixels and takes them out of bin 0 again (rare, keeps the common path free of per-byte predicates).
    if (!FAST && nvalid < 8) {
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const int vb = 3 * nvalid - 4 * i;                  // valid bytes in word i
            dw[i] &= vb >= 4 ? 0xffffffffu : (vb <= 0 ? 0u : (1u << (8 * vb)) - 1u);
        }
#ifdef __CUDA_ARCH__
        atomicSub(&S.hist[0][0], (uint32_t)(8 - nvalid));
        atomicSub(&S.hist[1][0], (uint32_t)(8 - nvalid));
        atomicSub(&S.hist[2][0], (uint32_t)(8 - nvalid));
#else
        S.hist[0][0] -= (uint32_t)(8 - nvalid);
        S.hist[1][0] -= (uint32_t)(8 - nvalid);
        S.hist[2][0] -= (uint32_t)(8 - nvalid);
#endif
    }
#pragma unroll
    for (int b = 0; b < 24; b++) hist_add(S.hist[b % 3], dw[b >> 2], b & 3);
    if (SWEEP && ghost) {                                       // outside pixels are zero by now
        uint32_t sq = 0;
#pragma unroll
        for (int i = 0; i < 6; i++) sq = dp4a_uu(dw[i], dw[i], sq);
        smem_add(&S.ghost[(y >> 4) & 1][ox >> 1], sq);
    }

    // ---- texture: Laplacian of the original luma, BORDER_REFLECT_101 (§8a)
    int lu = l - 1, ld = l + 1;
    if (y == 0) lu = g.h > 1 ? l + 1 : l;
    if (y == g.h - 1) ld = g.h > 1 ? l - 1 : l;
    // (two-phase band loop: lines -2 and -1, the last two of the band before, were kept aside — the ring half they lived in is being
    // converted over)
    constexpr bool CARRY = FAST && FUSE2_OK;
    const uint8_t *yc = CARRY && l < 0 ? &S.ycarry[CARRY ? l + 2 : 0][CARRY ? col : 0] : &S.yorig[ring16(r, l)][col];
    const uint8_t *yu = CARRY && lu < 0 ? &S.ycarry[CARRY ? lu + 2 : 0][CARRY ? col : 0] : &S.yorig[ring16(r, lu)][col];
    const uint8_t *yd2 = CARRY && ld < 0 ? &S.ycarry[CARRY ? ld + 2 : 0][CARRY ? col : 0] : &S.yorig[ring16(r, ld)][col];
    const int wide = FAST || g.w > 1;
    uint32_t sabs = 0, ssq = 0, mx = acc.tex_maxabs;
    {
        // e[0..9] = left neighbour, the 8 pixels, right neighbour, as three words; l + r - 4c is one or two dp4a per
        // pixel, up + down two more. Mirroring (REFLECT_101) goes through the neighbour loads: column -1 reads column 1, and
        // when the unit ends exactly at the image edge (every width that is a multiple of 8) column W reads column W-2. Only
        // a unit cut by the edge (ragged widths) leaves its last pixel to the scalar code below.
        const U2 cw = *reinterpret_cast<const U2 *>(yc);
        const U2 uw = *reinterpret_cast<const U2 *>(yu);
        const U2 lw = *reinterpret_cast<const U2 *>(yd2);
        const int edge = !FAST && nvalid < 8 ? nvalid - 1 : -1;
        const int nacc = edge >= 0 ? edge : 8;
        const uint32_t hl = gx0 == 0 ? yc[wide] : yc[-1], hr = nvalid == 8 ? yc[6] : yc[8];
        const uint32_t x[3] = {prmt(hl, cw.x, 0x6540u), prmt(cw.x, cw.y, 0x6543u), prmt(cw.y, hr, 0x7743u)};
        const uint32_t ud[2][2] = {{uw.x, lw.x}, {uw.y, lw.y}};
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int w0 = k >> 2, s0 = k & 3;                  // window e[k..k+2] starts at byte s0 of x[w0]
            int lap = dp4a_us(ud[w0][0], sel_const(SEL_ONE + s0), dp4a_us(ud[w0][1], sel_const(SEL_ONE + s0), 0));   // up + down
            if (s0 <= 1) {
                lap = dp4a_us(x[w0], sel_const(SEL_LAP + s0), lap);                                   // 01 fc 01 << 8 s0
            } else if (s0 == 2) {
                lap = dp4a_us(x[w0 + 1], sel_const(SEL_ONE), dp4a_us(x[w0], sel_const(SEL_LAP + 2), lap));
            } else {
                lap = dp4a_us(x[w0 + 1], sel_const(SEL_LAP + 3), dp4a_us(x[w0], sel_const(SEL_ONE + 3), lap));
            }
            lap = lap < 0 ? -lap : lap;
            if (FAST || k < nacc) {
                sabs += (uint32_t)lap;
                ssq += (uint32_t)(lap * lap);
                mx = (uint32_t)lap > mx ? (uint32_t)lap : mx;
                if (TEXHIST) smem_inc(&S.tex_hist[lap < 255 ? lap : 255]);
            }
        }
        if (!FAST && edge >= 0) {
            const int ctr = yc[edge];
            const int side = wide ? (edge == 0 && gx0 == 0 ? ctr : (int)yc[edge - 1]) : ctr;
            int lap = 2 * side + (int)yu[edge] + (int)yd2[edge] - 4 * ctr;
            lap = lap < 0 ? -lap : lap;
            sabs += (uint32_t)lap;
            ssq += (uint32_t)(lap * lap);
            mx = (uint32_t)lap > mx ? (uint32_t)lap : mx;
            if (TEXHIST) smem_inc(&S.tex_hist[lap < 255 ? lap : 255]);
        }
    }
    acc.tex_sumabs += sabs;
    acc.tex_sumsq += ssq;
    acc.tex_maxabs = mx;
}

// 8 pixels of one output row: ox = 8-pixel column index inside the strip, l = band-relative line in [-1, 14].
template <bool FAST, bool TEXHIST, bool SWEEP = false>
V5_DEV void residual_unit(Smem &S, const KParams &p, const Geo &g, ThreadAcc &acc, int r, int l, int ox, bool ghost = false)
{
    const int y = 16 * r + l;                                   // global pixel row
    const int gx0 = 16 * g.m0 + 8 * ox;                         // global pixel column of this unit
    const int col = 16 + 8 * ox;                                // band smem column

    // ---- chroma upsample (A.7)
    const int hc1 = ((g.h + 1) >> 1) - 1, wc1 = ((g.w + 1) >> 1) - 1;
    const int crow = y >> 1;
    int nrow = (y & 1) ? crow + 1 : crow - 1;
    nrow = nrow < 0 ? 0 : (nrow > hc1 ? hc1 : nrow);
    const int lcur = ring8(r, crow - 8 * r), lnb = ring8(r, nrow - 8 * r);
    const int ccol = col >> 1, gcx0 = gx0 >> 1;
    const bool fancy = wc1 > 1;
    int cb[8], cr[8];
    if (FAST) {
        upsample8_fast(&S.cdec[0][lcur][ccol], &S.cdec[0][lnb][ccol], gcx0 == 0, gcx0 + 4 > wc1, cb);
        upsample8_fast(&S.cdec[1][lcur][ccol], &S.cdec[1][lnb][ccol], gcx0 == 0, gcx0 + 4 > wc1, cr);
    } else {
        upsample8(&S.cdec[0][lcur][ccol], &S.cdec[0][lnb][ccol], gcx0, wc1, fancy, cb);
        upsample8(&S.cdec[1][lcur][ccol], &S.cdec[1][lnb][ccol], gcx0, wc1, fancy, cr);
    }

    residual_row<FAST, TEXHIST, SWEEP>(S, p, g, acc, r, l, ox, cb, cr, ghost);
}

// Two rows per unit (width-multiple-of-16 instantiation, -DV5_PAIR_ROWS=1). Band iteration r finishes rows 16r-1 .. 16r+14:
// eight pairs (2i+1, 2i+2) of an odd row and the even row below it. Both rows of a pair filter the SAME two decoded chroma
// rows a = i and b = i+1 — the odd row with a nearer, the even row with b nearer — so the interleaved byte pairs
// W = [a_j, b_j, a_j+1, b_j+1] are built once and only the dot-product coefficients swap ([3,1,9,3] / [9,3,3,1] for the odd
// row, [1,3,3,9] / [3,9,1,3] for the even one); the column arithmetic is shared as well.
// pi = pair index 0..7 (lines l = 2pi-1 and 2pi); v0 / v1: the row lies inside the segment and the image.
V5_DEV void chroma_pairs(const uint8_t *la, const uint8_t *lb, bool left_edge, bool right_edge, uint32_t w[5])
{
    const uint32_t a0 = *reinterpret_cast<const uint32_t *>(la - 4), b0 = *reinterpret_cast<const uint32_t *>(lb - 4);
    const uint32_t a1 = *reinterpret_cast<const uint32_t *>(la), b1 = *reinterpret_cast<const uint32_t *>(lb);
    const uint32_t a2 = *reinterpret_cast<const uint32_t *>(la + 4), b2 = *reinterpret_cast<const uint32_t *>(lb + 4);
    const uint32_t as = left_edge ? prmt(a1, 0u, 0x2100u) : prmt(a0, a1, 0x6543u), bs = left_edge ? prmt(b1, 0u, 0x2100u) : prmt(b0, b1, 0x6543u);
    const uint32_t ae = right_edge ? prmt(a1, 0u, 0x3321u) : prmt(a1, a2, 0x4321u), be = right_edge ? prmt(b1, 0u, 0x3321u) : prmt(b1, b2, 0x4321u);
    w[0] = prmt(as, bs, 0x5140u);
    w[1] = prmt(a1, b1, 0x5140u);
    w[2] = prmt(a1, b1, 0x6251u);
    w[3] = prmt(a1, b1, 0x7362u);
    w[4] = prmt(ae, be, 0x7362u);
}

template <bool TEXHIST>
V5_DEV void residual_pair(Smem &S, const KParams &p, const Geo &g, ThreadAcc &acc, int r, int pi, int ox, bool v0, bool v1)
{
    const int col = 16 + 8 * ox, ccol = col >> 1, gcx0 = (16 * g.m0 + 8 * ox) >> 1;
    const int hc1 = ((g.h + 1) >> 1) - 1, wc1 = (g.w >> 1) - 1;
    int ja = pi - 1, jb = pi;                                   // chroma lines of this band: a nearer for the odd row, b for the even one
    if (8 * r + ja < 0) ja = jb;                                // row 0: the line above does not exist, libjpeg repeats line 0
    if (8 * r + jb > hc1) jb = ja;                              // last row of an even-height image: the line below repeats the last
    const bool le = gcx0 == 0, re = gcx0 + 4 > wc1;
    uint32_t wb[5], wr[5];
    chroma_pairs(&S.cdec[0][ring8(r, ja)][ccol], &S.cdec[0][ring8(r, jb)][ccol], le, re, wb);
    chroma_pairs(&S.cdec[1][ring8(r, ja)][ccol], &S.cdec[1][ring8(r, jb)][ccol], le, re, wr);
    // unrolled: the two rows interleave (+1.8 % measured against the rolled loop, -DV5_PAIR_UNROLL=0, which is 200 instructions shorter)
#if !defined(V5_PAIR_UNROLL) || V5_PAIR_UNROLL
#pragma unroll
#else
#pragma unroll 1
#endif
    for (int h = 0; h < 2; h++) {
        if (!(h ? v1 : v0)) continue;
        const uint32_t ke = sel_const(SEL_TRI + 2 * h), ko = sel_const(SEL_TRI + 2 * h + 1);
        int cb[8], cr[8];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            cb[2 * j] = dp4a_us(wb[j], ke, 8 - 2048) >> 4;
            cb[2 * j + 1] = dp4a_us(wb[j + 1], ko, 7 - 2048) >> 4;
            cr[2 * j] = dp4a_us(wr[j], ke, 8 - 2048) >> 4;
            cr[2 * j + 1] = dp4a_us(wr[j + 1], ko, 7 - 2048) >> 4;
        }
        residual_row<true, TEXHIST>(S, p, g, acc, r, 2 * pi - 1 + h, ox, cb, cr);
    }
}

template <bool TEXHIST>
V5_DEV void stage_residual_pairs(int tid, Smem &S, const KParams &p, const Geo &g, ThreadAcc &acc, int r)
{
    const int n8 = 2 * (g.m1 - g.m0);                           // 8-pixel units per line (<= 60)
    const uint32_t inv = 65536u / (uint32_t)n8 + 1u;            // exact u / n8 for u < 8 * 60
    const int ylo = 16 * g.r0, yhi = 16 * g.r1 < g.h ? 16 * g.r1 : g.h;
    for (int u = tid; u < 8 * n8; u += NT) {
        const int pi = (int)(((uint32_t)u * inv) >> 16), ox = u - pi * n8;
        const int y0 = 16 * r + 2 * pi - 1;
        const bool v0 = y0 >= ylo && y0 < yhi, v1 = y0 + 1 >= ylo && y0 + 1 < yhi;
        if (!v0 && !v1) continue;
        residual_pair<TEXHIST>(S, p, g, acc, r, pi, ox, v0, v1);
    }
}

// Iteration r finishes pixel rows 16r-1 .. 16r+14 (clipped to the segment and the image).
template <bool FAST, bool TEXHIST, bool SWEEP = false>
V5_DEV void stage_residual(int tid, Smem &S, const KParams &p, const Geo &g, ThreadAcc &acc, int r, bool ghost = false)
{
    const int n8 = 2 * (g.m1 - g.m0);                           // 8-pixel units per line (<= 60)
    const uint32_t inv = 65536u / (uint32_t)n8 + 1u;            // exact u / n8 for u < 16 * 60
    const int ylo = 16 * g.r0, yhi = 16 * g.r1 < g.h ? 16 * g.r1 : g.h;
    for (int u = tid; u < 16 * n8; u += NT) {
        const int wl = (int)(((uint32_t)u * inv) >> 16), ox = u - wl * n8;
        const int l = wl - 1, y = 16 * r + l;
        if (y < ylo || y >= yhi || (!FAST && 16 * g.m0 + 8 * ox >= g.w)) continue;
        residual_unit<FAST, TEXHIST, SWEEP>(S, p, g, acc, r, l, ox, ghost);
    }
}

// ------------------------------------------------------------------------------------------------ work item set-up
template <bool RAGGED>
V5_DEV void make_geo(const KParams &p, int work, Geo &g, int &frame)
{
    uint32_t rem, n_strips, n_segs;
    if (RAGGED) {
        int lo = 0, hi = p.n - 1;                               // last frame whose work_base <= work
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (p.frames[mid].work_base <= (uint32_t)work) lo = mid;
            else hi = mid - 1;
        }
        frame = lo;
        const FrameDesc &d = p.frames[lo];
        rem = (uint32_t)work - d.work_base;
        n_strips = (uint32_t)d.n_strips;
        n_segs = (uint32_t)d.n_segs;
        g.h = d.h; g.w = d.w; g.mw = d.mw; g.mh = d.mh;
        g.row_stride = d.row_stride;
        g.vec_ok = (int)(d.flags & 1u);
        g.resid_vec_ok = (int)((d.flags >> 1) & 1u);
        g.frame = d.rgb;
        g.resid = d.resid;
    } else {
        n_strips = (uint32_t)p.n_strips;
        if (work < p.work_split) {                              // long segments first ...
            n_segs = (uint32_t)p.n_segs;
            const uint32_t per_frame = n_strips * n_segs;
            frame = (int)((uint32_t)work / per_frame);
            rem = (uint32_t)work - (uint32_t)frame * per_frame;
        } else {                                                // ... the last frames in short ones: the CTAs run dry close together
            n_segs = (uint32_t)p.n_segs_b;
            const uint32_t per_frame = n_strips * n_segs, w2 = (uint32_t)(work - p.work_split);
            const uint32_t f2 = w2 / per_frame;
            frame = p.split_frame + (int)f2;
            rem = w2 - f2 * per_frame;
        }
        g.h = p.h; g.w = p.w; g.mw = p.mw; g.mh = p.mh;
        g.row_stride = p.row_stride;
        g.vec_ok = p.vec_ok;
        g.resid_vec_ok = p.resid_vec_ok;
        g.frame = p.rgb + (int64_t)frame * p.frame_stride;
        g.resid = p.residual ? p.residual + (int64_t)frame * p.h * p.w * 3 : nullptr;
    }
    const uint32_t seg = rem / n_strips, strip = rem - seg * n_strips;
    g.m0 = (int)((strip * (uint32_t)g.mw) / n_strips);          // mw, mh <= 4096: no overflow
    g.m1 = (int)(((strip + 1) * (uint32_t)g.mw) / n_strips);
    g.r0 = (int)((seg * (uint32_t)g.mh) / n_segs);
    g.r1 = (int)(((seg + 1) * (uint32_t)g.mh) / n_segs);
    g.xb0 = 16 * (g.m0 - 1);
    g.band_mcus = g.m1 - g.m0 + 2;
}


}  // namespace V5_NS
