// v5jpeg_dec.cuh — baseline JPEG decoder on the GPU (SURVEY.md §8f-2): what the reference does with
// Image.open(crop).convert('RGB') (v5_texture_ela.py:64) and cv2.imread(crop, IMREAD_GRAYSCALE) (:83) on the crop files V1
// wrote with cv2.imwrite (v1_keyframes_facetrack.py:166) — libjpeg's defaults: ISLOW inverse DCT, fancy upsampling (h2v2 for
// the 4:2:0 files both writers produce by default; h2v1 for 4:2:2 and none for 4:4:4, the layouts their sampling options add).
// Pixel-identical to both libraries. Per batch of files (any mix of sizes):
//
//   unstuff_kernel  one CTA per file: entropy-coded segment with FF 00 -> FF (and RSTn markers dropped, their positions
//                   recorded), as a flat bit stream
//   huffman_kernel  one CTA per file: Huffman decoding in parallel by SELF-SYNCHRONISATION. The stream is cut into
//                   1024-bit subsequences, one per thread. Only the first thread knows its decoder state (bit position,
//                   block-in-MCU, zigzag index); the others start blind at their subsequence's first bit, and because
//                   Huffman codes resynchronise after a few symbols, almost all of them are in the right state when they
//                   leave their subsequence. Every thread then keeps decoding into the following subsequences until its
//                   exit state equals the one recorded there, overwriting the record otherwise; when nobody moves, every
//                   recorded state is the true one. A prefix sum of the blocks completed per subsequence gives every thread
//                   its output position and a last pass decodes again, this time writing coefficients (the head of every
//                   block assembled in shared memory and stored as one full sector, BlockHead). Windows of 1024
//                   subsequences are processed in order by the same CTA, carrying the exact state from one to the next.
//   huffman_rst_kernel  files with restart intervals only: every interval starts in a known state, one thread each
//   dc_kernel       one CTA per file: DC differences -> DC values (prefix sum per component, T.81 F.2.2.1) on a dense
//                   int16-per-block array
//   idct_kernel     dequantise + ISLOW inverse DCT (SURVEY App. A.6), 4 threads per block -> sample planes
//   colour_kernel   fancy upsample (A.7) + YCbCr -> RGB (A.8), and/or the luma plane alone
//
// The symbol-level logic is __host__ __device__ so that tests/emu can run it on the CPU (a debugging aid, not a fallback).
#pragma once
#include <stdint.h>

#include "v5ela_device.cuh"
#include "v5jpeg_common.h"

namespace v5j {
using v5::U4;

#ifndef V5J_HUFF_NT
#define V5J_HUFF_NT 1024
#endif
#ifndef V5J_SUB_BITS
#define V5J_SUB_BITS 1024
#endif
#ifndef V5J_HUFF_CTAS
#define V5J_HUFF_CTAS 1
#endif
constexpr int HUFF_NT = V5J_HUFF_NT;       // subsequences per window = threads of the decoding CTA
constexpr int HUFF_CTAS = V5J_HUFF_CTAS;   // resident CTAs per SM the kernel is built for
constexpr uint32_t SUB_BITS = V5J_SUB_BITS;   // bits per subsequence (> 31: a symbol never skips a whole subsequence)

struct DecTabSet {                         // Huffman tables of one file: [0] luma, [1] chroma
    DecTable dc[2], ac[2];
};
struct HuffSpecSet {                       // the same as the files' DHT segments give them (FileInfo): what calls are de-duplicated on
    HuffSpec dc[2], ac[2];
};
inline bool make_tabset(const HuffSpecSet &h, DecTabSet &T)
{
    bool ok = true;
    for (int c = 0; c < 2; c++) ok = make_dec_table(h.dc[c], T.dc[c]) && make_dec_table(h.ac[c], T.ac[c]) && ok;
    return ok;
}

struct DecImage {
    int32_t h, w, ncomp;
    int32_t hs, vs;                        // luma blocks per MCU across / down: 2x2 (4:2:0), 2x1 (4:2:2), 1x1 (4:4:4, one component)
    int32_t mcux, mcuy, bpm, blocks;
    int32_t restart;                       // restart interval in MCUs, 0 = none: the file is decoded interval by interval
    int32_t rst_off;                       // first entry of this file in the interval-start array (restart > 0)
    int32_t tabset;                        // index into the table-set array
    int32_t qt;                            // index into the quantisation-table array (2 x 64 uint16 per entry)
    int32_t yw, yh, cw, ch;                // padded plane sizes
    int64_t scan_off, scan_len;            // entropy-coded segment inside the uploaded file bytes
    int64_t stream_off;                    // unstuffed stream inside the stream buffer (16-byte aligned)
    int64_t coef_off;                      // first block inside the coefficient buffer
    int64_t sub_off;                       // first subsequence inside the per-subsequence arrays (sub_info, sub_block0)
    int64_t plane_off;                     // Y plane inside the plane buffer; Cb follows, then Cr
    int64_t rgb_off, gray_off;             // output positions (bytes), -1 = not wanted
};

// Geometry of a file: MCU grid, blocks per MCU (luma blocks, then Cb, Cr), padded plane sizes.
V5_HOSTDEV void dec_geometry(DecImage &im, int h, int w, int ncomp, int hs, int vs)
{
    im.h = h; im.w = w; im.ncomp = ncomp;
    im.hs = ncomp == 3 ? hs : 1;
    im.vs = ncomp == 3 ? vs : 1;
    im.mcux = (w + 8 * im.hs - 1) / (8 * im.hs);
    im.mcuy = (h + 8 * im.vs - 1) / (8 * im.vs);
    im.bpm = ncomp == 3 ? im.hs * im.vs + 2 : 1;
    im.blocks = im.mcux * im.mcuy * im.bpm;
    im.yw = im.mcux * 8 * im.hs;
    im.yh = im.mcuy * 8 * im.vs;
    im.cw = ncomp == 3 ? im.mcux * 8 : 0;
    im.ch = ncomp == 3 ? im.mcuy * 8 : 0;
}

struct SubState {                          // decoder state between two symbols
    uint32_t p;                            // bit position in the unstuffed stream
    uint16_t c;                            // block inside the MCU (0..bpm-1)
    uint16_t z;                            // next zigzag index (0 = a DC symbol comes next)
};
struct SubInfo {
    SubState s;                            // state on leaving the subsequence
    uint32_t n;                            // blocks completed inside it
    uint32_t pad;
};

V5_HOSTDEV bool same_state(const SubState &a, const SubState &b) { return a.p == b.p && a.c == b.c && a.z == b.z; }

V5_HOSTDEV uint32_t window_of(uint32_t hi, uint32_t lo, uint32_t sh)           // the 32 bits that start sh bits into hi:lo
{
#ifdef __CUDA_ARCH__
    return __funnelshift_l(lo, hi, sh);
#else
    return sh ? (hi << sh) | (lo >> (32 - sh)) : hi;
#endif
}

// Where the decoder reads the stream from: 32-bit words, most significant bit first. word(w) = stream bits 32w .. 32w+31;
// a decoder walks the words in order with a cursor (open at word w, then next() = the word after the one handed out last).
// The stream buffer is padded with zero bytes, so reading a little past the end is harmless.
struct ByteStream {                        // plain bytes in (global) memory
    const uint8_t *data;
    V5_HOSTDEV uint32_t word(uint32_t w) const
    {
#ifdef __CUDA_ARCH__
        return __byte_perm(__ldg(reinterpret_cast<const uint32_t *>(data) + w), 0, 0x0123);
#else
        const uint8_t *b = data + 4 * (size_t)w;
        return ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
#endif
    }
    V5_HOSTDEV uint32_t window(uint32_t p) const { return window_of(word(p >> 5), word((p >> 5) + 1), p & 31u); }   // 32 bits from bit p
    struct Cursor { uint32_t w; };
    V5_HOSTDEV uint32_t open(Cursor &c, uint32_t w) const { c.w = w; return word(w); }
    V5_HOSTDEV uint32_t next(Cursor &c) const { return word(++c.w); }
};

// One window of the stream staged in shared memory as big-endian 32-bit words. Thread t works on words 32t .. 32t+31 (its
// subsequence, then the ones after it) and the threads of a warp tend to sit at similar offsets inside their subsequences.
// Word c of subsequence r is stored at c * STAGE_PITCH + r with STAGE_PITCH = HUFF_NT + 1 = 1 (mod 32): its bank is
// (c + r) mod 32, so equal offsets in 32 consecutive subsequences fall into 32 different banks, and so do the 32 consecutive
// words of one subsequence when the window is staged. A cursor is the slot of the word handed out last: the next word is
// STAGE_PITCH further on, or at the top of the next column when the subsequence ends — no index arithmetic per symbol.
constexpr int SUB_WORDS = (int)(SUB_BITS / 32);
constexpr int WINDOW_WORDS = HUFF_NT * SUB_WORDS;
constexpr int STAGE_PITCH = HUFF_NT + 1;                                   // + one subsequence: a symbol may end just past the window
constexpr int STAGE_WORDS = STAGE_PITCH * SUB_WORDS;
static_assert((SUB_WORDS & (SUB_WORDS - 1)) == 0, "stage_slot: SUB_WORDS must be a power of two");   // (banks: HUFF_NT a multiple of 32)
V5_HOSTDEV int stage_slot(uint32_t w)      // w: word index inside the window, < STAGE_WORDS
{
    return (int)((w & (uint32_t)(SUB_WORDS - 1)) * (uint32_t)STAGE_PITCH + w / (uint32_t)SUB_WORDS);
}
struct StagedStream {
    const uint32_t *words;                 // STAGE_WORDS entries
    uint32_t base_word;                    // stream word index of words[stage_slot(0)], a multiple of SUB_WORDS
    V5_HOSTDEV uint32_t word(uint32_t w) const { return words[stage_slot(w - base_word)]; }
    struct Cursor { const uint32_t *q; };  // the word handed out last
    V5_HOSTDEV uint32_t open(Cursor &c, uint32_t w) const
    {
        c.q = words + stage_slot(w - base_word);
        return *c.q;
    }
    V5_HOSTDEV uint32_t next(Cursor &c) const
    {
        // the last word of a subsequence sits in the last row of the layout: its successor is the first word of the next column
        c.q += c.q >= words + (SUB_WORDS - 1) * STAGE_PITCH ? 1 - (SUB_WORDS - 1) * STAGE_PITCH : STAGE_PITCH;
        return *c.q;
    }
};
// thread t of nt: copies the window that starts at stream word base_word (stream: bytes, padded with zeros up to pad_bytes)
V5_HOSTDEV void stage_window(int t, int nt, uint32_t *words, const uint8_t *stream, uint32_t base_word, uint32_t stream_words)
{
    for (int i = t; i < STAGE_WORDS; i += nt) {
        const uint32_t gw = base_word + (uint32_t)i;
        uint32_t v = 0;
        if (gw < stream_words) {
#ifdef __CUDA_ARCH__
            v = __byte_perm(__ldg(reinterpret_cast<const uint32_t *>(stream) + gw), 0, 0x0123);
#else
            const uint8_t *b = stream + 4 * (size_t)gw;
            v = ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
#endif
        }
        words[stage_slot((uint32_t)i)] = v;
    }
}

// One Huffman symbol from the window, as the packed action word of v5jpeg_common.h (pack_symbol): codes of up to 9 bits from
// the first table, longer ones from the second (one more load), tables whose long codes span too many windows by the walk.
V5_HOSTDEV uint32_t huff_action(const DecTable &t, uint32_t win)
{
    const uint32_t look = t.look[win >> (32 - DEC_LOOK_BITS)];
    if (look) return look;
    const uint32_t k = (win >> 16) - t.long_base;                       // look == 0 implies window16 >= the first long code
    if (k < (uint32_t)DEC_LONG_ENTRIES) return t.lng[k];
    return dec_long_action(t, win);
}

// Decodes from state `s` until the bit position reaches `limit`; returns the number of blocks completed. WRITE: stores
// every non-zero AC coefficient of block (block0 + completed) at coef[block * 64 + zigzag index] and its DC difference at dc[block];
// blocks >= max_blocks (trailing padding bits decoded as symbols) are dropped.
// The write pass assembles the head of every block — zigzag positions 0..BLK_HEAD-1, where most non-zero coefficients are — on
// chip and stores it as ONE full 32-byte sector when the block ends, instead of one 2-byte store per coefficient: each of
// those is a 32-byte request to the memory system (a partial write to a line the zero fill left long ago: fetched again,
// merged, written back), and at quality 95 a block has 18 of them. The L1 -> crossbar request port was what bounded the write
// pass (75 % busy, 48 % of the kernel's time). Thread t owns BLK_HEAD int16 in shared memory as two 128-bit words,
// BlockHead::q[0][t] and q[1][t]. A block that starts or ends in another subsequence is shared with that subsequence's
// thread, so only blocks that lie wholly inside the span are assembled; the two partial ones use plain stores.
constexpr int BLK_HEAD = 16;
struct BlockHead {
    U4 q[2][HUFF_NT];
};

template <bool WRITE, class Src, bool HEADS = false>
V5_HOSTDEV uint32_t decode_span(const Src &stream, SubState &s, uint32_t limit, const DecTabSet &T, int bpm, int16_t *coef,
                                int16_t *dc, int64_t block0, int64_t max_blocks, BlockHead *heads = nullptr, int t = 0)
{
    // One loop body for DC and AC symbols, selects instead of branches: the threads of a warp sit at unrelated places of
    // their blocks, and every divergent path would be paid for by all of them.
    // The table hands back what to do (pack_symbol): value bits to read, how far the zigzag index moves (end of block: 64).
    // The stream words under the bit position travel in registers (a symbol moves the position by less than 32 bits, so at
    // most one new word is needed per symbol), and the word after them is fetched one crossing ahead.
    uint32_t p = s.p, done = 0;
    int c = s.c, z = s.z;
    if (p >= limit) return 0;
    typename Src::Cursor cur;
    uint32_t hi = stream.open(cur, p >> 5), lo = stream.next(cur), ahead = stream.next(cur);
    uint32_t sh = p & 31u;                                             // bit offset of p inside hi
    const int first_chroma = bpm > 1 ? bpm - 2 : bpm;                  // an MCU ends with its Cb and Cr block
    // &T.ac[k] - &T.dc[k] is the same for both k: one pointer (the DC table of the block's component) is kept, it changes at
    // block ends only
    const char *tdc = reinterpret_cast<const char *>(&T.dc[c >= first_chroma ? 1 : 0]);
    constexpr int AC_FWD = (int)(2 * sizeof(DecTable)), CHROMA_FWD = (int)sizeof(DecTable);
    // write pass: `room` blocks from block0 on may be stored (trailing pad bits can decode into phantom blocks past the image);
    // cblk / cdc follow the current block
    const uint32_t room = WRITE ? (uint32_t)(max_blocks > block0 ? max_blocks - block0 : 0) : 1u;
    int16_t *cblk = WRITE ? coef + block0 * 64 : nullptr, *cdc = WRITE ? dc + block0 : nullptr;
    bool whole = HEADS && z == 0;                                       // the current block began inside this span
    int16_t *head = HEADS ? reinterpret_cast<int16_t *>(&heads->q[0][t]) : nullptr;
    constexpr int HEAD_Q1 = (int)(sizeof(U4) / 2) * HUFF_NT;            // int16 distance from q[0][t] to q[1][t]
    do {
        const DecTable &tab = *reinterpret_cast<const DecTable *>(tdc + (z ? AC_FWD : 0));
        const uint32_t win = window_of(hi, lo, sh);
        const uint32_t act = huff_action(tab, win);
        const int zinc = (int)((act >> 16) & 127u), total = (int)(act >> 24);
        if (WRITE) {
            const int len = (int)(act & 31u), sz = (int)((act >> 8) & 15u);
            const int pos = z + zinc - 1;                                // where a value lands: DC 0, AC z + run
            if (sz && pos < 64 && done < room) {
                int v = (int)((win << len) >> (32 - sz));
                v = v < (1 << (sz - 1)) ? v - (1 << sz) + 1 : v;
                // DC differences go to their own dense array (one int16 per block): the prefix sums that turn them into values
                // then touch 2 bytes per block instead of one 128-byte line
                if (z == 0) *cdc = (int16_t)v;
                else if (HEADS && whole && pos < BLK_HEAD) head[(pos & 7) + (pos >> 3) * HEAD_Q1] = (int16_t)v;
                else cblk[pos] = (int16_t)v;
            }
        }
        z += zinc;
        p += (uint32_t)total;
        sh += (uint32_t)total;
        // end of block — as selects: some lane of the warp is at one in almost every step
        const bool eob = z >= 64;
        if (HEADS && eob) {
            if (whole && done < room) {
                U4 *dst = reinterpret_cast<U4 *>(cblk);
                dst[0] = heads->q[0][t];
                dst[1] = heads->q[1][t];
                heads->q[0][t] = U4{0u, 0u, 0u, 0u};
                heads->q[1][t] = U4{0u, 0u, 0u, 0u};
            }
            whole = true;
        }
        if (WRITE) {
            cblk += eob ? 64 : 0;
            cdc += eob ? 1 : 0;
        }
        z = eob ? 0 : z;
        done += eob ? 1u : 0u;
        c += eob ? 1 : 0;
        c = c == bpm ? 0 : c;
        tdc = reinterpret_cast<const char *>(&T.dc[0]) + (c >= first_chroma ? CHROMA_FWD : 0);
        if (sh >= 32u) {
            hi = lo;
            lo = ahead;
            ahead = stream.next(cur);
        }
        sh &= 31u;
    } while (p < limit);
    if (HEADS && whole && z != 0) {
        // the span ends inside a block: the next subsequence's thread writes the rest of it, so what has been assembled goes
        // out coefficient by coefficient
        if (done < room)
            for (int k = 1; k < BLK_HEAD; k++) {
                const int16_t v = head[(k & 7) + (k >> 3) * HEAD_Q1];
                if (v) cblk[k] = v;
            }
        heads->q[0][t] = U4{0u, 0u, 0u, 0u};
        heads->q[1][t] = U4{0u, 0u, 0u, 0u};
    }
    s.p = p;
    s.c = (uint16_t)c;
    s.z = (uint16_t)z;
    return done;
}

// Files with restart intervals (DRI): every interval starts byte-aligned, right after its RSTn marker, with the DC predictors
// at zero — its decoder state is known without any synchronisation, so one thread decodes one interval from start to end
// (huffman_rst_kernel). `nblocks` blocks from bit position p; coef / dc point at the interval's first block and receive the
// AC coefficients and the DC VALUES (predictions undone on the fly). Returns the blocks decoded before `limit` was reached
// (== nblocks for a well-formed interval).
template <class Src>
V5_HOSTDEV int decode_interval(const Src &stream, uint32_t p, uint32_t limit, const DecTabSet &T, int bpm, int nblocks, int16_t *coef, int16_t *dc)
{
    int pred[3] = {0, 0, 0};
    int c = 0;
    for (int b = 0; b < nblocks; b++) {
        const int ci = (bpm > 1 && c >= bpm - 2) ? c - (bpm - 2) + 1 : 0, comp = ci ? 1 : 0;
        int z = 0;
        while (z < 64) {
            if (p >= limit) return b;
            const bool is_dc = z == 0;
            const uint32_t win = stream.window(p);
            const uint32_t act = huff_action(is_dc ? T.dc[comp] : T.ac[comp], win);
            const int len = (int)(act & 31u), sz = (int)((act >> 8) & 15u), zinc = (int)((act >> 16) & 127u), total = (int)(act >> 24);
            const int pos = z + zinc - 1;
            int v = 0;
            if (sz) {
                v = (int)((win << len) >> (32 - sz));
                v = v < (1 << (sz - 1)) ? v - (1 << sz) + 1 : v;
            }
            if (is_dc) {
                pred[ci] += v;
                dc[b] = (int16_t)pred[ci];
            } else if (sz && pos < 64) {
                coef[(int64_t)b * 64 + pos] = (int16_t)v;
            }
            z += zinc;
            p += (uint32_t)total;
        }
        c = c + 1 == bpm ? 0 : c + 1;
    }
    return nblocks;
}

// ------------------------------------------------------------------------------------ window logic of huffman_kernel
// Shared by the kernel and the CPU emulation: every function is one barrier-delimited phase of thread t.
struct HuffWindow {
    SubInfo info[HUFF_NT];                 // info[t]: exit state of subsequence w0 + t, blocks completed inside it
    SubState cur[HUFF_NT];                 // travelling state of thread t
    uint8_t done[HUFF_NT];
    SubState carry;                        // state at the start of the window (exact, or a part's blind start)
    uint32_t base_blocks;                  // huffman_kernel: blocks completed before the window
};

struct HuffJob {
    const uint8_t *stream;                 // unstuffed stream (global memory), zero padded
    StagedStream staged;                   // the current window of it (shared memory)
    uint32_t stream_words;                 // 32-bit words that may be read from `stream`
    uint32_t total_bits, nsub;
    int bpm;
    int64_t max_blocks;
    int16_t *coef;
    int16_t *dc;                           // DC differences (later values), one per block
    BlockHead *heads;                      // write pass: per-thread block heads (shared memory, all zero between passes), or null
};

V5_HOSTDEV uint32_t sub_limit(const HuffJob &J, uint32_t j)
{
    const uint64_t e = (uint64_t)(j + 1) * SUB_BITS;
    return e < J.total_bits ? (uint32_t)e : J.total_bits;
}

V5_HOSTDEV void huff_phase_first(int t, HuffWindow &W, const HuffJob &J, const DecTabSet &T, uint32_t w0)
{
    const uint32_t j = w0 + (uint32_t)t;
    if (j >= J.nsub) {
        W.done[t] = 1;
        return;
    }
    SubState st;
    if (t == 0) st = W.carry;
    else { st.p = j * SUB_BITS; st.c = 0; st.z = 0; }
    W.info[t].n = decode_span<false>(J.staged, st, sub_limit(J, j), T, J.bpm, nullptr, nullptr, 0, 0);
    W.info[t].s = st;
    W.cur[t] = st;
    W.done[t] = 0;
}

// round r >= 1: thread t decodes subsequence w0 + t + r from where it stands
V5_HOSTDEV void huff_phase_round(int t, int r, HuffWindow &W, const HuffJob &J, const DecTabSet &T, uint32_t w0)
{
    if (W.done[t]) return;
    const int k = t + r;
    if (k >= HUFF_NT || w0 + (uint32_t)k >= J.nsub) {
        W.done[t] = 1;
        return;
    }
    SubState st = W.cur[t];
    const uint32_t n = decode_span<false>(J.staged, st, sub_limit(J, w0 + (uint32_t)k), T, J.bpm, nullptr, nullptr, 0, 0);
    if (same_state(st, W.info[k].s)) W.done[t] = 1;                     // synchronised: the rest of the walk is already recorded
    W.info[k].s = st;                                                    // this thread entered k in a state at least as good
    W.info[k].n = n;                                                     // as the recorded one: its block count is the one to keep
    W.cur[t] = st;
}

// write pass: block0 = blocks completed before subsequence w0 + t
V5_HOSTDEV void huff_phase_write(int t, HuffWindow &W, const HuffJob &J, const DecTabSet &T, uint32_t w0, uint32_t block0)
{
    const uint32_t j = w0 + (uint32_t)t;
    if (j >= J.nsub) return;
    SubState st = t == 0 ? W.carry : W.info[t - 1].s;
    decode_span<true, StagedStream, true>(J.staged, st, sub_limit(J, j), T, J.bpm, J.coef, J.dc, (int64_t)block0, J.max_blocks, J.heads, t);
}

// ---- small batches: a file's windows spread over several CTAs -------------------------------------------------------------
// A file's windows are shared out among `parts` CTAs (huffman_sync_kernel); part q owns windows part_first(q) .. part_first(q+1)-1.
V5_HOSTDEV uint32_t window_count(uint32_t nsub) { return (nsub + (uint32_t)HUFF_NT - 1) / (uint32_t)HUFF_NT; }
V5_HOSTDEV uint32_t part_count(uint32_t nsub, uint32_t max_parts)
{
    const uint32_t w = window_count(nsub);
    return w < max_parts ? (w ? w : 1u) : (max_parts ? max_parts : 1u);
}
V5_HOSTDEV uint32_t part_first(uint32_t q, uint32_t parts, uint32_t windows) { return (uint32_t)(((uint64_t)q * windows) / parts); }

// Boundary fix-up between two parts: every part but the first began blind, so its records are only true from the point where
// its own chain fell into step. The walker enters subsequence j0 (the first of a part) in the TRUE state — the exit state of
// the subsequence before it — and re-records subsequences until it leaves one in the recorded state. One thread, reading the
// stream in place. Returns the number of subsequences it had to re-record. A walker that reaches the end of its part without
// meeting a recorded state has changed the next part's entry state; the caller notices and redoes that boundary.
V5_HOSTDEV uint32_t fixup_walk(const uint8_t *stream, uint32_t total_bits, const DecTabSet &T, int bpm, SubInfo *sub_info,
                               uint32_t j0, uint32_t j_end /* first subsequence of the next part: a walker stays inside its part */)
{
    ByteStream bs;
    bs.data = stream;
    SubState st = sub_info[j0 - 1].s;
    uint32_t rewritten = 0;
    for (uint32_t j = j0; j < j_end; j++) {
        const uint64_t e = (uint64_t)(j + 1) * SUB_BITS;
        const uint32_t n = decode_span<false>(bs, st, e < total_bits ? (uint32_t)e : total_bits, T, bpm, nullptr, nullptr, 0, 0);
        const bool met = same_state(st, sub_info[j].s);
        sub_info[j].s = st;
        sub_info[j].n = n;                                               // counted from the true entry state
        if (met) break;
        rewritten++;
    }
    return rewritten;
}

// write pass of one window (huffman_write_kernel): entry state and first block index come from the per-subsequence records
V5_HOSTDEV void huff_write_sub(int t, const HuffJob &J, const DecTabSet &T, uint32_t w0, const SubInfo *sub_info, const uint32_t *sub_block0)
{
    const uint32_t j = w0 + (uint32_t)t;
    if (j >= J.nsub) return;
    SubState st;
    if (j == 0) { st.p = 0; st.c = 0; st.z = 0; }
    else st = sub_info[j - 1].s;
    decode_span<true, StagedStream, true>(J.staged, st, sub_limit(J, j), T, J.bpm, J.coef, J.dc, (int64_t)sub_block0[j], J.max_blocks, J.heads, t);
}

// ------------------------------------------------------------------------------------------------- DC prediction
// diff -> value for the blocks of one MCU (dense DC array: its bpm entries) given the running predictors; in place.
V5_HOSTDEV void dc_apply_mcu(int16_t *mcu_dc, int bpm, int &py, int &pcb, int &pcr)
{
    if (bpm == 1) {
        py += mcu_dc[0];
        mcu_dc[0] = (int16_t)py;
        return;
    }
    const int ny = bpm - 2;
    for (int i = 0; i < ny; i++) {
        py += mcu_dc[i];
        mcu_dc[i] = (int16_t)py;
    }
    pcb += mcu_dc[ny];
    mcu_dc[ny] = (int16_t)pcb;
    pcr += mcu_dc[ny + 1];
    mcu_dc[ny + 1] = (int16_t)pcr;
}

// ------------------------------------------------------------------------------------------- inverse DCT of a block
// The arithmetic of libjpeg-turbo's x86 SIMD ISLOW code (SSE2 / AVX2), which is what Pillow and OpenCV decode with on x86-64:
// 16-bit lanes throughout. Dequantisation keeps the low 16 bits of coefficient x table entry; in0 +- in4, in3 + in7 and
// in1 + in5 wrap to int16 (idct8<.., WRAP16>); the column-pass outputs saturate to int16 and the row-pass outputs to int8
// before the +128. A block whose AC rows 1..7 are all zero takes a shortcut in the column pass: every output is the
// dequantised DC of its column << 2, wrapping in 16 bits. Files written from pixels never leave int16 anywhere here
// (DESIGN.md 4.1), so for them this is T.81 A.6 in wide integers; libjpeg-turbo's C path gives other samples than this on
// blocks that do (DESIGN.md 4.6).

// two ints -> an int16 pair, each saturated (PTX cvt.pack.sat.s16.s32 puts its first source in the high half)
#ifdef __CUDA_ARCH__
V5_DEV uint32_t pack_sat_s16(int lo, int hi)
{
    uint32_t d;
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(d) : "r"(hi), "r"(lo));
    return d;
}
// cvt.pack.sat.s8.s32: d = (c.lo16 << 16) | (sat_s8(a) << 8) | sat_s8(b)
V5_DEV uint32_t packsat2_s8(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
#else
inline uint32_t pack_sat_s16(int lo, int hi)
{
    const auto sat = [](int v) { return (uint32_t)(uint16_t)(v < -32768 ? -32768 : (v > 32767 ? 32767 : v)); };
    return sat(lo) | (sat(hi) << 16);
}
inline uint32_t packsat2_s8(int a, int b, uint32_t c)
{
    const auto sat = [](int v) { return (uint32_t)(uint8_t)(v < -128 ? -128 : (v > 127 ? 127 : v)); };
    return ((c & 0xffffu) << 16) | (sat(a) << 8) | sat(b);
}
#endif
// four row-pass outputs -> samples [v0, v1, v2, v3]: each saturated to -128..127, then + 128 (flipping the top bit of a byte)
V5_DEV uint32_t pack4_samples(int v0, int v1, int v2, int v3) { return packsat2_s8(v1, v0, packsat2_s8(v3, v2, 0u)) ^ 0x80808080u; }

// `nat`: the block's 64 coefficients in NATURAL order (8 rows of 8 int16, 16-byte rows), `qt` likewise. Thread j of 4 takes
// columns 2j, 2j+1 — one 32-bit word per row — dequantises, runs the column pass and leaves int16 pairs in ws; then rows
// 2j, 2j+1 (one 128-bit load each) -> 8 clamped samples each.
V5_DEV void idct_cols(const int16_t *nat, const uint16_t *qt, int j, int16_t *ws)
{
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(nat), *qw = reinterpret_cast<const uint32_t *>(qt);
    uint32_t *ww = reinterpret_cast<uint32_t *>(ws);
    const v5::U4 *rows = reinterpret_cast<const v5::U4 *>(nat);
    uint32_t ac = 0;                                                       // any AC coefficient in rows 1..7, all 8 columns
#pragma unroll
    for (int k = 1; k < 8; k++) {
        const v5::U4 r = rows[k];
        ac |= r.x | r.y | r.z | r.w;
    }
    int a[8], b[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t c = cw[4 * k + j], q = qw[4 * k + j];
        a[k] = (int)(int16_t)(v5::s16_lo(c) * (int)(q & 0xffffu));
        b[k] = (int)(int16_t)(v5::s16_hi(c) * (int)(q >> 16));
    }
    if (!ac) {
        const uint32_t w = v5::prmt((uint32_t)a[0] << 2, (uint32_t)b[0] << 2, 0x5410u);
#pragma unroll
        for (int k = 0; k < 8; k++) ww[4 * k + j] = w;
        return;
    }
    v5::idct8<1, false, true>(a);
    v5::idct8<1, false, true>(b);
#pragma unroll
    for (int k = 0; k < 8; k++) ww[4 * k + j] = pack_sat_s16(a[k], b[k]);
}

V5_DEV void idct_rows(const int16_t *ws, int j, uint8_t *dst, int pitch)
{
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int r = 2 * j + rr;
        const v5::U4 w = *reinterpret_cast<const v5::U4 *>(ws + 8 * r);
        int v[8] = {v5::s16_lo(w.x), v5::s16_hi(w.x), v5::s16_lo(w.y), v5::s16_hi(w.y), v5::s16_lo(w.z), v5::s16_hi(w.z), v5::s16_lo(w.w), v5::s16_hi(w.w)};
        v5::idct8<1, true, true>(v);
        // plane rows are 8-byte aligned (plane offsets are multiples of 16, pitches multiples of 8)
        *reinterpret_cast<v5::U2 *>(dst + r * pitch) = v5::U2{pack4_samples(v[0], v[1], v[2], v[3]), pack4_samples(v[4], v[5], v[6], v[7])};
    }
}

// where block g (scan order) of an image lands: plane pointer offset and pitch
V5_HOSTDEV int64_t block_dest(const DecImage &im, int g, int &pitch, int &comp)
{
    if (im.bpm == 1) {
        pitch = im.yw;
        comp = 0;
        const int my = g / im.mcux, mx = g - my * im.mcux;
        return (int64_t)(8 * my) * im.yw + 8 * mx;
    }
    const int m = g / im.bpm, i = g - im.bpm * m, ny = im.bpm - 2;
    const int my = m / im.mcux, mx = m - my * im.mcux;
    if (i < ny) {                                                         // luma blocks of an MCU: row-major, hs across
        const int br = im.hs == 2 ? i >> 1 : i, bc = im.hs == 2 ? i & 1 : 0;       // (vs == 2 implies hs == 2 here)
        pitch = im.yw;
        comp = 0;
        return (int64_t)(8 * (im.vs * my + br)) * im.yw + 8 * (im.hs * mx + bc);
    }
    pitch = im.cw;
    comp = i - ny + 1;
    return (int64_t)im.yw * im.yh + (int64_t)(i - ny) * im.cw * im.ch + (int64_t)(8 * my) * im.cw + 8 * mx;
}

// ------------------------------------------------------------------------------------------ upsample + colour (A.7/A.8)
// Chroma for a pixel, as libjpeg's upsamplers produce it with do_fancy_upsampling (jdsample.c):
//   4:2:0  h2v2 "triangle" filter: 3/4 nearer + 1/4 further row, then the same along the row, biases 8 / 7, >> 4   (A.7)
//   4:2:2  h2v1: 3/4 nearer + 1/4 further sample along the row, biases 1 / 2, >> 2; rows map one to one
//   4:4:4  the sample itself
// At the first / last column the missing neighbour is the sample itself (libjpeg's special cases reduce to exactly that), and
// planes no wider than two samples are replicated without any filtering.
V5_HOSTDEV void pixel_rgb(const DecImage &im, const uint8_t *planes, int x, int y, uint8_t out[3])
{
    const uint8_t *yp = planes, *cbp = planes + (int64_t)im.yw * im.yh, *crp = cbp + (int64_t)im.cw * im.ch;
    const int yy = yp[(int64_t)y * im.yw + x];
    if (im.ncomp == 1) {
        out[0] = out[1] = out[2] = (uint8_t)yy;
        return;
    }
    const int hs = im.hs, vs = im.vs;
    const int hc = (im.h + vs - 1) / vs, wc = (im.w + hs - 1) / hs, cw = im.cw;
    const int r = vs == 2 ? y >> 1 : y, cx = hs == 2 ? x >> 1 : x;
    int cb, cr;
    if (hs == 1 || wc <= 2) {
        cb = cbp[(int64_t)r * cw + cx];
        cr = crp[(int64_t)r * cw + cx];
    } else {
        int nx = (x & 1) ? cx + 1 : cx - 1;
        nx = nx < 0 ? 0 : (nx > wc - 1 ? wc - 1 : nx);
        if (vs == 2) {
            int nb = (y & 1) ? r + 1 : r - 1;
            nb = nb < 0 ? 0 : (nb > hc - 1 ? hc - 1 : nb);
            const int bias = (x & 1) ? 7 : 8;
            int s0 = 3 * cbp[(int64_t)r * cw + cx] + cbp[(int64_t)nb * cw + cx];
            int s1 = 3 * cbp[(int64_t)r * cw + nx] + cbp[(int64_t)nb * cw + nx];
            cb = (3 * s0 + s1 + bias) >> 4;
            s0 = 3 * crp[(int64_t)r * cw + cx] + crp[(int64_t)nb * cw + cx];
            s1 = 3 * crp[(int64_t)r * cw + nx] + crp[(int64_t)nb * cw + nx];
            cr = (3 * s0 + s1 + bias) >> 4;
        } else {
            const int bias = (x & 1) ? 2 : 1;
            cb = (3 * cbp[(int64_t)r * cw + cx] + cbp[(int64_t)r * cw + nx] + bias) >> 2;
            cr = (3 * crp[(int64_t)r * cw + cx] + crp[(int64_t)r * cw + nx] + bias) >> 2;
        }
    }
    const int cbd = cb - 128, crd = cr - 128;
    out[0] = (uint8_t)v5::clamp255(yy + ((91881 * crd + 32768) >> 16));
    out[1] = (uint8_t)v5::clamp255(yy + ((-22554 * cbd - 46802 * crd + 32768) >> 16));
    out[2] = (uint8_t)v5::clamp255(yy + ((116130 * cbd + 32768) >> 16));
}

// Eight consecutive pixels x0 .. x0+7 (x0 a multiple of 8) of row y: same arithmetic as pixel_rgb with the loads shared —
// two 32-bit words of luma and, per chroma component and row, one aligned word plus the two neighbours beside it (two words
// and no neighbours for 4:4:4). out: 24 bytes R G B R G B ...; pixels at or beyond the image width are left untouched.
V5_HOSTDEV uint32_t load_u32(const uint8_t *p)
{
#ifdef __CUDA_ARCH__
    return *reinterpret_cast<const uint32_t *>(p);
#else
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
#endif
}

V5_HOSTDEV void pixels8_rgb(const DecImage &im, const uint8_t *planes, int x0, int y, uint8_t out[24])
{
    const uint8_t *yrow = planes + (int64_t)y * im.yw + x0;
    const uint32_t yw[2] = {load_u32(yrow), load_u32(yrow + 4)};
    const int nvalid = im.w - x0 < 8 ? im.w - x0 : 8;
    if (im.ncomp == 1) {
        for (int k = 0; k < nvalid; k++) out[3 * k] = out[3 * k + 1] = out[3 * k + 2] = (uint8_t)(yw[k >> 2] >> (8 * (k & 3)));
        return;
    }
    const uint8_t *cbp = planes + (int64_t)im.yw * im.yh, *crp = cbp + (int64_t)im.cw * im.ch;
    const int hs = im.hs, vs = im.vs, cw = im.cw;
    const int hc = (im.h + vs - 1) / vs, wc = (im.w + hs - 1) / hs;
    const int r = vs == 2 ? y >> 1 : y;
    int cbv[8], crv[8];                                                  // chroma of the eight pixels
    if (hs == 1) {                                                        // 4:4:4: plane rows are padded to a multiple of 8
        const uint8_t *pb = cbp + (int64_t)r * cw + x0, *pr = crp + (int64_t)r * cw + x0;
        const uint32_t b[2] = {load_u32(pb), load_u32(pb + 4)}, c[2] = {load_u32(pr), load_u32(pr + 4)};
#pragma unroll
        for (int k = 0; k < 8; k++) {
            cbv[k] = (int)((b[k >> 2] >> (8 * (k & 3))) & 0xffu);
            crv[k] = (int)((c[k >> 2] >> (8 * (k & 3))) & 0xffu);
        }
    } else {
        const int cx0 = x0 >> 1;                                          // a multiple of 4
        int nb = r;
        if (vs == 2) {
            nb = (y & 1) ? r + 1 : r - 1;
            nb = nb < 0 ? 0 : (nb > hc - 1 ? hc - 1 : nb);
        }
        const uint8_t *rows[4] = {cbp + (int64_t)r * cw, cbp + (int64_t)nb * cw, crp + (int64_t)r * cw, crp + (int64_t)nb * cw};
        if (wc <= 2) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                cbv[k] = rows[0][cx0 + (k >> 1)];
                crv[k] = rows[2][cx0 + (k >> 1)];
            }
        } else {
            const int cl = cx0 > 0 ? cx0 - 1 : 0, cr_ = cx0 + 4 < wc ? cx0 + 4 : wc - 1;   // neighbours beside the word, clamped
            // s: chroma columns cx0-1 .. cx0+4 after the vertical step — 3 * nearer + further row (4:2:0), or the row itself (4:2:2)
            const int wn = vs == 2 ? 1 : 0, wcur = vs == 2 ? 3 : 1;
            int s[2][6];
#pragma unroll
            for (int c = 0; c < 2; c++) {
                const uint32_t wr = load_u32(rows[2 * c] + cx0), wnb = load_u32(rows[2 * c + 1] + cx0);
                s[c][0] = wcur * rows[2 * c][cl] + wn * rows[2 * c + 1][cl];
                s[c][5] = wcur * rows[2 * c][cr_] + wn * rows[2 * c + 1][cr_];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    int col = cx0 + j < wc ? j : wc - 1 - cx0;            // columns past the last one repeat it (col >= 0: cx0 < wc)
                    s[c][1 + j] = wcur * (int)((wr >> (8 * col)) & 0xffu) + wn * (int)((wnb >> (8 * col)) & 0xffu);
                }
            }
            const int sh = vs == 2 ? 4 : 2;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int j = 1 + (k >> 1), jn = (k & 1) ? j + 1 : j - 1;
                const int bias = vs == 2 ? ((k & 1) ? 7 : 8) : ((k & 1) ? 2 : 1);
                cbv[k] = (3 * s[0][j] + s[0][jn] + bias) >> sh;
                crv[k] = (3 * s[1][j] + s[1][jn] + bias) >> sh;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (k >= nvalid) break;
        const int yy = (int)((yw[k >> 2] >> (8 * (k & 3))) & 0xffu), cbd = cbv[k] - 128, crd = crv[k] - 128;
        out[3 * k] = (uint8_t)v5::clamp255(yy + ((91881 * crd + 32768) >> 16));
        out[3 * k + 1] = (uint8_t)v5::clamp255(yy + ((-22554 * cbd - 46802 * crd + 32768) >> 16));
        out[3 * k + 2] = (uint8_t)v5::clamp255(yy + ((116130 * cbd + 32768) >> 16));
    }
}

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------------- kernels
__constant__ uint8_t kZigzagToNaturalDev[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                                41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                                30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
__device__ __forceinline__ uint32_t dec_cta_scan(uint32_t v, uint32_t *warp_sums, uint32_t *sum)
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
        const uint32_t w = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_sums[lane] = wi - w;
        if (lane == 31) warp_sums[32] = wi;
    }
    __syncthreads();
    const uint32_t excl = incl - v + warp_sums[warp];
    *sum = warp_sums[32];
    __syncthreads();
    return excl;
}

// FF 00 -> FF. stream_bits[img] = 8 x kept bytes. The stream buffer is zero-initialised and padded by the host side.
// Files with restart intervals: the RSTn markers (FF D0..D7) are dropped as well, and the position where interval k begins
// in the unstuffed stream goes to rst_starts[im.rst_off + k] (entry 0 stays 0).
__global__ void __launch_bounds__(1024) unstuff_kernel(const DecImage *images, const uint8_t *files, uint8_t *streams,
                                                       uint32_t *stream_bits, uint32_t *rst_starts)
{
    __shared__ uint32_t warp_sums[33];
    const DecImage im = images[blockIdx.x];
    const uint8_t *src = files + im.scan_off;
    uint8_t *dst = streams + im.stream_off;
    const int mcus = im.mcux * im.mcuy;
    const uint32_t n_int = im.restart > 0 ? (uint32_t)((mcus + im.restart - 1) / im.restart) : 0u;
    uint32_t running = 0, markers = 0;
    for (int64_t base = 0; base < im.scan_len; base += 4 * 1024) {
        const int64_t i0 = base + 4 * (int64_t)threadIdx.x;
        uint8_t b[6];                                                     // the byte before this thread's four, and the one after
        uint32_t keep = 0, cnt = 0, mark = 0, nmark = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const int64_t i = i0 - 1 + k;
            b[k] = (i >= 0 && i < im.scan_len) ? src[i] : 0;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (i0 + k >= im.scan_len) continue;
            const bool stuffed = b[k + 1] == 0x00 && b[k] == 0xFF;
            const bool rst_ff = n_int && b[k + 1] == 0xFF && b[k + 2] >= 0xD0 && b[k + 2] <= 0xD7;       // first byte of a marker
            const bool rst_dn = n_int && b[k] == 0xFF && b[k + 1] >= 0xD0 && b[k + 1] <= 0xD7;           // its second byte
            if (!stuffed && !rst_ff && !rst_dn) {
                keep |= 1u << k;
                cnt++;
            }
            if (rst_dn) {
                mark |= 1u << k;
                nmark++;
            }
        }
        uint32_t sum;
        uint32_t o = running + dec_cta_scan(cnt, warp_sums, &sum);
        uint32_t msum = 0, m = 0;
        if (n_int) m = markers + dec_cta_scan(nmark, warp_sums, &msum);   // uniform branch: n_int is per file
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (keep & (1u << k)) dst[o++] = b[k + 1];
            if (mark & (1u << k)) {                                       // the interval after this marker starts at output byte o
                if (++m < n_int) rst_starts[im.rst_off + m] = o;
            }
        }
        running += sum;
        markers += msum;
    }
    if (threadIdx.x == 0) stream_bits[blockIdx.x] = running * 8u;
}

struct HuffSmem {
    uint32_t words[STAGE_WORDS];           // the window's share of the stream (128 KB + one subsequence)
    DecTabSet T;
    HuffWindow W;
    uint32_t warp_sums[33];
    uint32_t n_live;
    uint16_t live[HUFF_NT];                // subsequences still walking (rounds >= 2)
    BlockHead heads;                       // write pass: the head of the block every thread is assembling (zero when idle)
};

// Large batches (at least one file per SM): the whole job in one launch, one CTA per file — synchronise a window, scan, write
// its coefficients, carry the exact state into the next window.
__global__ void __launch_bounds__(HUFF_NT, HUFF_CTAS) huffman_kernel(const DecImage *images, const DecTabSet *tabsets, const uint8_t *streams,
                                                          const uint32_t *stream_bits, int16_t *coef, int16_t *dc, int32_t *status)
{
    extern __shared__ __align__(16) uint8_t huff_smem_raw[];
    HuffSmem &S = *reinterpret_cast<HuffSmem *>(huff_smem_raw);
    const int t = (int)threadIdx.x;
    const DecImage im = images[blockIdx.x];
    if (im.restart > 0) {                                                 // decoded interval by interval (huffman_rst_kernel)
        if (t == 0) status[blockIdx.x] = 0;
        return;
    }
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&tabsets[im.tabset]);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&S.T);
        for (int i = t; i < (int)(sizeof(DecTabSet) / 4); i += HUFF_NT) dst[i] = src[i];
    }
    S.heads.q[0][t] = U4{0u, 0u, 0u, 0u};
    S.heads.q[1][t] = U4{0u, 0u, 0u, 0u};
    HuffJob J;
    J.stream = streams + im.stream_off;
    J.staged.words = S.words;
    J.staged.base_word = 0;
    J.stream_words = (uint32_t)((im.scan_len + 32) >> 2);               // the host reserves scan_len + 32 zeroed bytes
    J.total_bits = stream_bits[blockIdx.x];
    J.nsub = (J.total_bits + SUB_BITS - 1) / SUB_BITS;
    J.bpm = im.bpm;
    J.max_blocks = im.blocks;
    J.coef = coef + im.coef_off * 64;
    J.dc = dc + im.coef_off;
    J.heads = &S.heads;
    if (t == 0) {
        S.W.carry.p = 0;
        S.W.carry.c = 0;
        S.W.carry.z = 0;
        S.W.base_blocks = 0;
    }
    __syncthreads();
    for (uint32_t w0 = 0; w0 < J.nsub; w0 += HUFF_NT) {
        J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
        stage_window(t, HUFF_NT, S.words, J.stream, J.staged.base_word, J.stream_words);
        __syncthreads();
        huff_phase_first(t, S.W, J, S.T, w0);
        __syncthreads();
        // Round 1: almost every thread still walks. From round 2 on only the few subsequences that have not met a recorded
        // state keep going: their indices are compacted into a list so that they share a few warps instead of keeping
        // one lane busy in many.
        huff_phase_round(t, 1, S.W, J, S.T, w0);
        __syncthreads();
        for (int r = 2; r < HUFF_NT; r++) {
            if (t == 0) S.n_live = 0;
            __syncthreads();
            if (!S.W.done[t]) S.live[atomicAdd(&S.n_live, 1u)] = (uint16_t)t;
            __syncthreads();
            const uint32_t n_live = S.n_live;
            if (n_live == 0) break;
            if ((uint32_t)t < n_live) huff_phase_round((int)S.live[t], r, S.W, J, S.T, w0);
            __syncthreads();
        }
        const bool active = w0 + (uint32_t)t < J.nsub;
        uint32_t sum;
        const uint32_t ex = dec_cta_scan(active ? S.W.info[t].n : 0u, S.warp_sums, &sum);
        huff_phase_write(t, S.W, J, S.T, w0, S.W.base_blocks + ex);
        __syncthreads();
        if (t == 0) {
            const uint32_t last = J.nsub - w0 < (uint32_t)HUFF_NT ? J.nsub - w0 - 1 : HUFF_NT - 1;
            S.W.carry = S.W.info[last].s;
            S.W.base_blocks += sum;
        }
        __syncthreads();
    }
    // a well-formed stream holds exactly `blocks` blocks (trailing pad bits may decode into at most a few phantom ones)
    if (t == 0) status[blockIdx.x] = S.W.base_blocks >= (uint32_t)im.blocks ? 0 : -1;
}

// Small batches: three launches, so that a handful of files still fill the GPU.
// Pass 1: synchronisation. grid = (max parts, files); CTA (q, f) walks the windows of part q of file f in order and leaves the
// exit state and block count of every subsequence in sub_info. Part 0 starts in the true state, the others blind.
__global__ void __launch_bounds__(HUFF_NT, HUFF_CTAS) huffman_sync_kernel(const DecImage *images, const DecTabSet *tabsets, const uint8_t *streams,
                                                               const uint32_t *stream_bits, SubInfo *sub_info_all)
{
    extern __shared__ __align__(16) uint8_t huff_smem_raw[];
    HuffSmem &S = *reinterpret_cast<HuffSmem *>(huff_smem_raw);
    const int t = (int)threadIdx.x;
    const DecImage im = images[blockIdx.y];
    HuffJob J;
    J.stream = streams + im.stream_off;
    J.staged.words = S.words;
    J.staged.base_word = 0;
    J.stream_words = (uint32_t)((im.scan_len + 32) >> 2);               // the host reserves scan_len + 32 zeroed bytes
    J.total_bits = stream_bits[blockIdx.y];
    J.nsub = (J.total_bits + SUB_BITS - 1) / SUB_BITS;
    J.bpm = im.bpm;
    J.max_blocks = im.blocks;
    J.coef = nullptr;
    J.dc = nullptr;
    J.heads = nullptr;
    const uint32_t windows = window_count(J.nsub), parts = part_count(J.nsub, gridDim.x);
    if (blockIdx.x >= parts || windows == 0 || im.restart > 0) return;
    const uint32_t w_first = part_first(blockIdx.x, parts, windows), w_end = part_first(blockIdx.x + 1, parts, windows);
    SubInfo *sub_info = sub_info_all + im.sub_off;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&tabsets[im.tabset]);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&S.T);
        for (int i = t; i < (int)(sizeof(DecTabSet) / 4); i += HUFF_NT) dst[i] = src[i];
    }
    if (t == 0) {
        S.W.carry.p = w_first * (uint32_t)HUFF_NT * SUB_BITS;          // true for part 0; a blind guess otherwise
        S.W.carry.c = 0;
        S.W.carry.z = 0;
    }
    __syncthreads();
    for (uint32_t w = w_first; w < w_end; w++) {
        const uint32_t w0 = w * (uint32_t)HUFF_NT;
        J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
        stage_window(t, HUFF_NT, S.words, J.stream, J.staged.base_word, J.stream_words);
        __syncthreads();
        huff_phase_first(t, S.W, J, S.T, w0);
        __syncthreads();
        // Round 1: almost every thread still walks. From round 2 on only the few subsequences that have not met a recorded
        // state keep going: their indices are compacted into a list so that they share a few warps instead of keeping
        // one lane busy in many.
        huff_phase_round(t, 1, S.W, J, S.T, w0);
        __syncthreads();
        for (int r = 2; r < HUFF_NT; r++) {
            if (t == 0) S.n_live = 0;
            __syncthreads();
            if (!S.W.done[t]) S.live[atomicAdd(&S.n_live, 1u)] = (uint16_t)t;
            __syncthreads();
            const uint32_t n_live = S.n_live;
            if (n_live == 0) break;
            if ((uint32_t)t < n_live) huff_phase_round((int)S.live[t], r, S.W, J, S.T, w0);
            __syncthreads();
        }
        if (w0 + (uint32_t)t < J.nsub) sub_info[w0 + t] = S.W.info[t];
        if (t == 0) {
            const uint32_t last = J.nsub - w0 < (uint32_t)HUFF_NT ? J.nsub - w0 - 1 : HUFF_NT - 1;
            S.W.carry = S.W.info[last].s;
        }
        __syncthreads();
    }
}

// Pass 2: part boundaries and block offsets. One CTA per file. Lane 0 of warp q re-records the first subsequences of part q
// from the true state (all boundaries at once); thread 0 then checks that every walker did start from a state nobody changed
// afterwards (it redoes the walk otherwise: that needs a whole part of subsequences that never fall into step); an exclusive
// scan of the block counts gives every subsequence its first block.
__global__ void __launch_bounds__(1024) huffman_fixup_kernel(const DecImage *images, const DecTabSet *tabsets, const uint8_t *streams,
                                                             const uint32_t *stream_bits, uint32_t max_parts, SubInfo *sub_info_all,
                                                             uint32_t *sub_block0_all, int32_t *status)
{
    __shared__ uint32_t warp_sums[33];
    __shared__ SubState started_from[32];
    const DecImage im = images[blockIdx.x];
    if (im.restart > 0) {                                                 // decoded interval by interval (huffman_rst_kernel)
        if (threadIdx.x == 0) status[blockIdx.x] = 0;
        return;
    }
    const uint8_t *stream = streams + im.stream_off;
    const uint32_t total_bits = stream_bits[blockIdx.x], nsub = (total_bits + SUB_BITS - 1) / SUB_BITS;
    const uint32_t windows = window_count(nsub), parts = part_count(nsub, max_parts);
    SubInfo *sub_info = sub_info_all + im.sub_off;
    uint32_t *sub_block0 = sub_block0_all + im.sub_off;
    const DecTabSet &T = tabsets[im.tabset];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0 && warp >= 1 && warp < parts) {
        const uint32_t j0 = part_first(warp, parts, windows) * (uint32_t)HUFF_NT;
        uint32_t j_end = part_first(warp + 1, parts, windows) * (uint32_t)HUFF_NT;
        j_end = j_end < nsub ? j_end : nsub;
        started_from[warp] = sub_info[j0 - 1].s;
        fixup_walk(stream, total_bits, T, im.bpm, sub_info, j0, j_end);
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (uint32_t q = 1; q < parts; q++) {                            // in order: each check sees the final state before it
            const uint32_t j0 = part_first(q, parts, windows) * (uint32_t)HUFF_NT;
            uint32_t j_end = part_first(q + 1, parts, windows) * (uint32_t)HUFF_NT;
            j_end = j_end < nsub ? j_end : nsub;
            if (!same_state(started_from[q], sub_info[j0 - 1].s)) fixup_walk(stream, total_bits, T, im.bpm, sub_info, j0, j_end);
        }
    __syncthreads();
    uint32_t running = 0;
    for (uint32_t base = 0; base < nsub; base += 1024) {
        const uint32_t j = base + threadIdx.x;
        uint32_t sum;
        const uint32_t ex = dec_cta_scan(j < nsub ? sub_info[j].n : 0u, warp_sums, &sum);
        if (j < nsub) sub_block0[j] = running + ex;
        running += sum;
    }
    // a well-formed stream holds exactly `blocks` blocks (trailing pad bits may decode into at most a few phantom ones)
    if (threadIdx.x == 0) status[blockIdx.x] = running >= (uint32_t)im.blocks ? 0 : -1;
}

// Pass 3: coefficients. grid = (max windows, files): every window of every file is a CTA of its own.
__global__ void __launch_bounds__(HUFF_NT, HUFF_CTAS) huffman_write_kernel(const DecImage *images, const DecTabSet *tabsets, const uint8_t *streams,
                                                                const uint32_t *stream_bits, const SubInfo *sub_info_all,
                                                                const uint32_t *sub_block0_all, int16_t *coef, int16_t *dc)
{
    extern __shared__ __align__(16) uint8_t huff_smem_raw[];
    HuffSmem &S = *reinterpret_cast<HuffSmem *>(huff_smem_raw);
    const int t = (int)threadIdx.x;
    const DecImage im = images[blockIdx.y];
    HuffJob J;
    J.stream = streams + im.stream_off;
    J.staged.words = S.words;
    J.stream_words = (uint32_t)((im.scan_len + 32) >> 2);
    J.total_bits = stream_bits[blockIdx.y];
    J.nsub = (J.total_bits + SUB_BITS - 1) / SUB_BITS;
    J.bpm = im.bpm;
    J.max_blocks = im.blocks;
    J.coef = coef + im.coef_off * 64;
    J.dc = dc + im.coef_off;
    J.heads = &S.heads;
    const uint32_t w0 = blockIdx.x * (uint32_t)HUFF_NT;
    if (w0 >= J.nsub || im.restart > 0) return;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&tabsets[im.tabset]);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&S.T);
        for (int i = t; i < (int)(sizeof(DecTabSet) / 4); i += HUFF_NT) dst[i] = src[i];
    }
    S.heads.q[0][t] = U4{0u, 0u, 0u, 0u};
    S.heads.q[1][t] = U4{0u, 0u, 0u, 0u};
    J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
    stage_window(t, HUFF_NT, S.words, J.stream, J.staged.base_word, J.stream_words);
    __syncthreads();
    huff_write_sub(t, J, S.T, w0, sub_info_all + im.sub_off, sub_block0_all + im.sub_off);
}

// Files with restart intervals: one thread per interval, reading the stream in place. grid = (ceil(max intervals / 128), files).
// Runs after the synchronising kernels (which skip these files and set their status to 0); a short interval flags the file.
__global__ void __launch_bounds__(128) huffman_rst_kernel(const DecImage *images, const DecTabSet *tabsets, const uint8_t *streams,
                                                          const uint32_t *stream_bits, const uint32_t *rst_starts, int16_t *coef,
                                                          int16_t *dc, int32_t *status)
{
    const DecImage im = images[blockIdx.y];
    if (im.restart <= 0) return;
    const int mcus = im.mcux * im.mcuy, n_int = (mcus + im.restart - 1) / im.restart;
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= n_int) return;
    const uint32_t total_bits = stream_bits[blockIdx.y];
    const uint32_t *starts = rst_starts + im.rst_off;
    const uint32_t p0 = k == 0 ? 0u : starts[k] * 8u;
    if (k > 0 && starts[k] == 0) {                                        // fewer markers in the data than the header promises
        status[blockIdx.y] = -1;
        return;
    }
    uint32_t limit = total_bits;
    if (k + 1 < n_int && starts[k + 1] != 0 && starts[k + 1] * 8u < limit) limit = starts[k + 1] * 8u;
    const int first_mcu = k * im.restart, n_mcu = mcus - first_mcu < im.restart ? mcus - first_mcu : im.restart;
    const int64_t block0 = im.coef_off + (int64_t)first_mcu * im.bpm;
    ByteStream bs;
    bs.data = streams + im.stream_off;
    const int done = decode_interval(bs, p0, limit, tabsets[im.tabset], im.bpm, n_mcu * im.bpm, coef + block0 * 64, dc + block0);
    if (done != n_mcu * im.bpm) status[blockIdx.y] = -1;
}

// DC differences -> values. One CTA per file; thread t owns MCU chunk_base + t, three CTA scans per chunk of 1024 MCUs.
// (files with restart intervals already hold values: huffman_rst_kernel)
__global__ void __launch_bounds__(1024) dc_kernel(const DecImage *images, int16_t *dc)
{
    __shared__ uint32_t warp_sums[33];
    const DecImage im = images[blockIdx.x];
    if (im.restart > 0) return;
    int16_t *base = dc + im.coef_off;
    const int mcus = im.mcux * im.mcuy;
    int run[3] = {0, 0, 0};
    for (int m0 = 0; m0 < mcus; m0 += 1024) {
        const int m = m0 + (int)threadIdx.x;
        int16_t *mc = base + (int64_t)m * im.bpm;
        int d[3] = {0, 0, 0};
        if (m < mcus) {
            if (im.bpm == 1) d[0] = mc[0];
            else {
                const int ny = im.bpm - 2;
                for (int i = 0; i < ny; i++) d[0] += mc[i];
                d[1] = mc[ny];
                d[2] = mc[ny + 1];
            }
        }
        int pred[3];
        for (int c = 0; c < (im.bpm == 1 ? 1 : 3); c++) {
            uint32_t sum;
            const uint32_t ex = dec_cta_scan((uint32_t)d[c], warp_sums, &sum);     // two's complement: wraps like int
            pred[c] = run[c] + (int)ex;
            run[c] += (int)sum;
        }
        if (m < mcus) dc_apply_mcu(mc, im.bpm, pred[0], pred[1], pred[2]);
    }
}

// 64 blocks per CTA, 4 threads per block. The 8 KB of coefficients come in with 128-bit loads and are scattered into natural
// order on the way into shared memory (one 16-bit store per coefficient, once), so that both passes work on packed words.
// grid = (ceil(max blocks / 64), files)
__global__ void __launch_bounds__(256) idct_kernel(const DecImage *images, const uint16_t *qtabs, const int16_t *coef, const int16_t *dc,
                                                   uint8_t *planes)
{
    __shared__ __align__(16) int16_t nat[64][64 + 8];                      // natural order; 144-byte block stride
    __shared__ __align__(16) int16_t ws[64][64 + 8];
    __shared__ __align__(16) uint16_t qt[2][64];
    __shared__ uint8_t z2n[64];
    const DecImage im = images[blockIdx.y];
    const int g0 = (int)blockIdx.x * 64;
    if (g0 >= im.blocks) return;
    const int nb = im.blocks - g0 < 64 ? im.blocks - g0 : 64;
    if (threadIdx.x < 64) z2n[threadIdx.x] = kZigzagToNaturalDev[threadIdx.x];
    if (threadIdx.x < 128) (&qt[0][0])[threadIdx.x] = qtabs[(int64_t)im.qt * 128 + threadIdx.x];
    __syncthreads();
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(coef + (im.coef_off + g0) * 64);
        for (int i = threadIdx.x; i < nb * 8; i += 256) {                  // 8 consecutive zigzag positions of one block
            const uint4 v = __ldg(src + i);
            const int b = i >> 3, k0 = (i & 7) * 8;
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 8; e++) nat[b][z2n[k0 + e]] = (int16_t)(w[e >> 1] >> (16 * (e & 1)));
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < nb) nat[threadIdx.x][0] = dc[im.coef_off + g0 + threadIdx.x];        // DC values live in their own array
    __syncthreads();
    const int lb = (int)threadIdx.x >> 2, j = (int)threadIdx.x & 3;
    const bool active = lb < nb;
    int pitch = 0, comp = 0;
    int64_t off = 0;
    if (active) {
        off = block_dest(im, g0 + lb, pitch, comp);
        idct_cols(nat[lb], qt[comp ? 1 : 0], j, ws[lb]);
    }
    __syncwarp();
    if (active) idct_rows(ws[lb], j, planes + im.plane_off + off, pitch);
}

// one thread per 8 pixels of a row. grid = (ceil(max pixel groups / 256), files)
__global__ void __launch_bounds__(256) colour_kernel(const DecImage *images, const uint8_t *planes, uint8_t *rgb_out, uint8_t *gray_out)
{
    const DecImage im = images[blockIdx.y];
    const int groups = (im.w + 7) >> 3;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= (int64_t)im.h * groups) return;
    const int y = (int)(i / groups), x0 = 8 * (int)(i - (int64_t)y * groups);
    const uint8_t *pl = planes + im.plane_off;
    const int nvalid = im.w - x0 < 8 ? im.w - x0 : 8;
    const int64_t px = (int64_t)y * im.w + x0;
    if (im.gray_off >= 0) {
        uint8_t *d = gray_out + im.gray_off + px;
        const uint2 v = *reinterpret_cast<const uint2 *>(pl + (int64_t)y * im.yw + x0);          // plane rows are 8-byte aligned
        if (nvalid == 8 && (reinterpret_cast<uintptr_t>(d) & 7) == 0) *reinterpret_cast<uint2 *>(d) = v;
        else
            for (int k = 0; k < nvalid; k++) d[k] = (uint8_t)((k < 4 ? v.x : v.y) >> (8 * (k & 3)));
    }
    if (im.rgb_off >= 0) {
        alignas(8) uint8_t o[24];
        uint8_t *d = rgb_out + im.rgb_off + 3 * px;
        const int wc = (im.w + 1) >> 1, cx0 = x0 >> 1;
        if (im.ncomp == 3 && im.hs == 2 && im.vs == 2 && cx0 + 4 <= wc && nvalid == 8) {
            // 4:2:0 unit whose four chroma columns all exist (every unit of a file but the last one or two of a row): the fused
            // kernel's arithmetic for the same two steps — triangle filter as one dot product per sample (v5::upsample8_fast),
            // reconstruction with the rounding folded into the luma word and a saturating pack — 22 instead of 55 instructions
            // per pixel. Same values: both are libjpeg's h2v2 fancy upsampling and YCbCr -> RGB (SURVEY App. A.7 / A.8).
            const uint8_t *cbp = pl + (int64_t)im.yw * im.yh, *crp = cbp + (int64_t)im.cw * im.ch;
            const int hc = (im.h + 1) >> 1, r = y >> 1;
            int nb = (y & 1) ? r + 1 : r - 1;
            nb = nb < 0 ? 0 : (nb > hc - 1 ? hc - 1 : nb);
            const bool le = cx0 == 0, re = cx0 + 4 >= wc;
            // upsample8_fast loads the words beside the unit's own even when an edge flag makes it ignore them: before a row's first
            // word that is the row above (or the plane in front), after its last word the row below — or, in the last row of the Cr
            // plane, whatever follows the image's planes: that one unit takes the general path
            const bool last = r == im.ch - 1 || nb == im.ch - 1;
            int cb[8], cr[8];
            if (last && cx0 + 4 >= im.cw) {
                pixels8_rgb(im, pl, x0, y, o);
            } else {
                v5::upsample8_fast(cbp + (int64_t)r * im.cw + cx0, cbp + (int64_t)nb * im.cw + cx0, le, re, cb);
                v5::upsample8_fast(crp + (int64_t)r * im.cw + cx0, crp + (int64_t)nb * im.cw + cx0, le, re, cr);
                const uint2 yv = *reinterpret_cast<const uint2 *>(pl + (int64_t)y * im.yw + x0);
                const uint32_t ydw[2] = {yv.x, yv.y};
                int rec[24];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int ykr = (int)v5::prmt(ydw[k >> 2], v5::sel_const(v5::SEL_HALF), 0x4054u + ((uint32_t)(k & 3) << 8));   // bytes: 00 80 Y 00
                    rec[3 * k] = (91881 * cr[k] + ykr) >> 16;
                    rec[3 * k + 1] = (-22554 * cb[k] + (-46802 * cr[k] + ykr)) >> 16;
                    rec[3 * k + 2] = (116130 * cb[k] + ykr) >> 16;
                }
                uint32_t *ow32 = reinterpret_cast<uint32_t *>(o);
#pragma unroll
                for (int i = 0; i < 6; i++) ow32[i] = v5::pack4sat(rec[4 * i], rec[4 * i + 1], rec[4 * i + 2], rec[4 * i + 3]);
            }
        } else {
            pixels8_rgb(im, pl, x0, y, o);
        }
        if (nvalid == 8 && (reinterpret_cast<uintptr_t>(d) & 7) == 0) {
            const uint2 *ow = reinterpret_cast<const uint2 *>(o);
            reinterpret_cast<uint2 *>(d)[0] = ow[0];
            reinterpret_cast<uint2 *>(d)[1] = ow[1];
            reinterpret_cast<uint2 *>(d)[2] = ow[2];
        } else {
            for (int k = 0; k < 3 * nvalid; k++) d[k] = o[k];
        }
    }
}
#endif  // __CUDACC__

}  // namespace v5j
