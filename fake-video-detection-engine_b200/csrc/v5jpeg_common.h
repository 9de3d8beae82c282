// v5jpeg_common.h — tables, header writer and header parser of the baseline-JPEG codec rows (SURVEY.md §8f-2, §8f-3).
//
// What the reference does with Pillow / OpenCV around the ELA arithmetic (nodes/V_nodes/v5_texture_ela.py):
//   :64  Image.open(crop).convert('RGB')        decode      :66-67 original.save(tmp,'JPEG',quality=90)   encode
//   :83  cv2.imread(crop, IMREAD_GRAYSCALE)     decode      :80-81 enhanced_diff.save(ela_i.jpg)           encode (q75)
//                                                           :90-91 cv2.imwrite(fft_i.jpg, spectrum)        encode (q95, gray)
// Both libraries drive libjpeg-turbo with its defaults: baseline sequential, Annex K tables, 4:2:0 for colour, JFIF 1.01
// header. Host-side pieces only in this file (plain C++, also compiled by g++ for tests/emu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <vector>

namespace v5j {

// zigzag position -> natural (row-major) index, T.81 Figure A.6
static const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// T.81 Annex K.3.3 typical Huffman tables: [0] luminance, [1] chrominance
static const uint8_t kDcBits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
static const uint8_t kDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t kAcBits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125}, {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119}};
static const uint8_t kAcVals[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
     0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
     0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
     0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
     0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
     0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
     0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
     0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
     0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
     0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
     0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
     0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
     0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

// ---------------------------------------------------------------------------------------------------- encoder tables
// Entry = (code length << 16) | code, indexed by the symbol (DC: category 0..11; AC: run << 4 | size). T.81 Annex C.
struct EncTables {
    uint32_t dc[2][16];
    uint32_t ac[2][256];
};

inline void canonical_codes(const uint8_t bits[16], const uint8_t *vals, uint32_t *out, int nout)
{
    for (int i = 0; i < nout; i++) out[i] = 0;
    int k = 0;
    uint32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        for (int i = 0; i < bits[len - 1]; i++, k++)
            if (vals[k] < nout) out[vals[k]] = ((uint32_t)len << 16) | code++;
            else code++;
        code <<= 1;
    }
}

inline void standard_enc_tables(EncTables &t)
{
    for (int c = 0; c < 2; c++) {
        canonical_codes(kDcBits[c], kDcVals, t.dc[c], 16);
        canonical_codes(kAcBits[c], kAcVals[c], t.ac[c], 256);
    }
}

// ------------------------------------------------------------------------------------------------------ file header
// SOI, APP0 (JFIF 1.01, aspect 1:1, no thumbnail), DQT per table, SOF0, DHT x 2 per table class, SOS — byte for byte what
// libjpeg emits after jpeg_set_defaults / jpeg_set_quality (what PIL's save and cv2.imwrite produce).
inline void put_u16(std::vector<uint8_t> &o, int v) { o.push_back((uint8_t)(v >> 8)); o.push_back((uint8_t)v); }

inline void put_dht(std::vector<uint8_t> &o, int tc_th, const uint8_t bits[16], const uint8_t *vals)
{
    int n = 0;
    for (int i = 0; i < 16; i++) n += bits[i];
    o.push_back(0xFF); o.push_back(0xC4);
    put_u16(o, 2 + 1 + 16 + n);
    o.push_back((uint8_t)tc_th);
    o.insert(o.end(), bits, bits + 16);
    o.insert(o.end(), vals, vals + n);
}

inline std::vector<uint8_t> file_header(int h, int w, int ncomp, const uint16_t ql[64], const uint16_t qc[64])
{
    static const uint8_t jfif[14] = {'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
    std::vector<uint8_t> o;
    o.reserve(640);
    o.push_back(0xFF); o.push_back(0xD8);
    o.push_back(0xFF); o.push_back(0xE0);
    put_u16(o, 16);
    o.insert(o.end(), jfif, jfif + 14);
    for (int t = 0; t < (ncomp == 3 ? 2 : 1); t++) {
        o.push_back(0xFF); o.push_back(0xDB);
        put_u16(o, 67);
        o.push_back((uint8_t)t);
        for (int i = 0; i < 64; i++) o.push_back((uint8_t)(t ? qc : ql)[kZigzag[i]]);
    }
    o.push_back(0xFF); o.push_back(0xC0);
    put_u16(o, 8 + 3 * ncomp);
    o.push_back(8);
    put_u16(o, h);
    put_u16(o, w);
    o.push_back((uint8_t)ncomp);
    for (int c = 0; c < ncomp; c++) {
        o.push_back((uint8_t)(c + 1));
        o.push_back((uint8_t)(ncomp == 3 && c == 0 ? 0x22 : 0x11));
        o.push_back((uint8_t)(c ? 1 : 0));
    }
    put_dht(o, 0x00, kDcBits[0], kDcVals);
    put_dht(o, 0x10, kAcBits[0], kAcVals[0]);
    if (ncomp == 3) {
        put_dht(o, 0x01, kDcBits[1], kDcVals);
        put_dht(o, 0x11, kAcBits[1], kAcVals[1]);
    }
    o.push_back(0xFF); o.push_back(0xDA);
    put_u16(o, 6 + 2 * ncomp);
    o.push_back((uint8_t)ncomp);
    for (int c = 0; c < ncomp; c++) {
        o.push_back((uint8_t)(c + 1));
        o.push_back((uint8_t)(c ? 0x11 : 0x00));
    }
    o.push_back(0); o.push_back(63); o.push_back(0);
    return o;
}

// ---------------------------------------------------------------------------------------------------- decoder tables
// Huffman decoding by a window of the next stream bits: look[window >> 23] resolves codes of <= 9 bits in one step, longer
// codes take a second table (DecTable::lng) or, for tables whose long codes span too many windows, walk maxcode[] (T.81
// F.2.2.3). What comes back is not the raw symbol but what the decoder does with it, packed:
//   bits  0..4   code length
//   bits  8..11  size   = number of value bits that follow the code (0 = none)
//   bits 16..22  zinc   = how far the zigzag index moves: DC 1; AC run + 1; ZRL (F0) 16; end of block 64
//   bits 24..29  total  = code length + size, what the bit position moves by
// so that DC symbols, AC symbols, ZRL and EOB all run through the same few instructions. 0 = not a short code.
#if defined(__CUDACC__)
#define V5J_HOSTDEV __host__ __device__ __forceinline__
#else
#define V5J_HOSTDEV inline
#endif
V5J_HOSTDEV uint32_t pack_symbol(int sym, int len, bool is_dc)
{
    int size, zinc;
    if (is_dc) {
        size = sym > 15 ? 15 : sym;
        zinc = 1;
    } else {
        size = sym & 15;
        zinc = size ? (sym >> 4) + 1 : ((sym >> 4) == 15 ? 16 : 64);
    }
    return (uint32_t)len | ((uint32_t)size << 8) | ((uint32_t)zinc << 16) | ((uint32_t)(len + size) << 24);
}

// What a file's DHT segments say about one table (T.81 B.2.4.2): 276 bytes. FileInfo keeps these; the decoder tables below
// (6.5 KB each) are only built for the DISTINCT table sets of a call (v5jpeg.cu), not per file.
struct HuffSpec {
    uint8_t bits[16];        // number of codes of length 1..16
    uint8_t vals[256];       // symbols in code order; entries past n are zero
    uint16_t n;
    uint16_t is_dc;
};

constexpr int DEC_LOOK_BITS = 9;
constexpr int DEC_LONG_ENTRIES = 1024;
struct DecTable {
    uint32_t look[1 << DEC_LOOK_BITS];
    // Second level: codes longer than DEC_LOOK_BITS bits. A canonical code orders its words by length, so every such code,
    // left-justified to 16 bits, lies in [long_base, 0xffff]; when that range has at most DEC_LONG_ENTRIES values (Annex K
    // tables: 640 for AC, 128 for DC) lng[window16 - long_base] is the action for it and decoding a long code is one more
    // load — no walk over the lengths, which every lane of a warp paid for whenever one of them met a long code (2 % of the
    // symbols of a quality-95 file: half of all warp steps). long_base = 0x10000: range too large, maxcode[] is walked.
    uint32_t lng[DEC_LONG_ENTRIES];
    uint32_t long_base;
    int32_t maxcode[18];     // maxcode[len] for len 1..16; -1 = no codes of that length
    int32_t valoff[17];      // symbol index = valoff[len] + code
    uint8_t vals[256];
    uint32_t is_dc;
};

// Codes of more than DEC_LOOK_BITS bits by the walk of T.81 F.2.2.3 (only the top 16 bits of the window matter). Codes that do
// not exist decode as symbol 0 with length 16 (libjpeg also substitutes zero for corrupt data; progress is guaranteed either way).
V5J_HOSTDEV uint32_t dec_long_action(const DecTable &t, uint32_t win)
{
    for (int l = DEC_LOOK_BITS + 1; l <= 16; l++) {
        const int32_t code = (int32_t)(win >> (32 - l));
        if (code <= t.maxcode[l]) return pack_symbol(t.vals[(t.valoff[l] + code) & 0xff], l, t.is_dc != 0);
    }
    return pack_symbol(0, 16, t.is_dc != 0);
}

// The canonical code of (bits, vals) is well formed: no length oversubscribed, no more symbols than `nvals`.
inline bool huff_spec_ok(const uint8_t bits[16], int nvals)
{
    if (nvals > 256) return false;
    int k = 0;
    int32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        const int cnt = bits[len - 1];
        if (cnt && (code + cnt > (1 << len) || k + cnt > nvals)) return false;
        code = (code + cnt) << 1;
        k += cnt;
    }
    return true;
}

inline bool make_dec_table(const uint8_t bits[16], const uint8_t *vals, int nvals, bool is_dc, DecTable &t)
{
    memset(&t, 0, sizeof(t));
    if (!huff_spec_ok(bits, nvals)) return false;
    memcpy(t.vals, vals, (size_t)nvals);
    t.is_dc = is_dc ? 1u : 0u;
    t.long_base = 0x10000u;
    int k = 0;
    int32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        if (len == DEC_LOOK_BITS + 1 && code < (1 << len) && 0x10000 - (code << (16 - len)) <= DEC_LONG_ENTRIES)
            t.long_base = (uint32_t)code << (16 - len);      // first word a longer code can have, left-justified
        const int cnt = bits[len - 1];
        if (cnt) {
            t.valoff[len] = k - code;
            if (len <= DEC_LOOK_BITS)
                for (int i = 0; i < cnt; i++) {
                    const int first = (code + i) << (DEC_LOOK_BITS - len);
                    for (int f = 0; f < (1 << (DEC_LOOK_BITS - len)); f++) t.look[first + f] = pack_symbol(vals[k + i], len, is_dc);
                }
            code += cnt;
            k += cnt;
            t.maxcode[len] = code - 1;
        } else {
            t.maxcode[len] = -1;
        }
        code <<= 1;
    }
    t.maxcode[17] = 0x7fffffff;
    for (uint32_t w = t.long_base; w < 0x10000u; w++) t.lng[w - t.long_base] = dec_long_action(t, w << 16);
    return true;
}
inline bool make_dec_table(const HuffSpec &h, DecTable &t) { return make_dec_table(h.bits, h.vals, h.n, h.is_dc != 0, t); }

enum { JPEG_OK = 0, JPEG_CORRUPT = -1, JPEG_UNSUPPORTED = -2 };

// The decoder's Huffman state holds bit positions in the unstuffed entropy-coded segment as 32-bit numbers, and rounds them up
// to whole subsequences: a segment of kMaxScanBytes (2^29 - 2^20 bytes, 511 MiB) or more is refused as unsupported.
constexpr size_t kMaxScanBytes = ((size_t)1 << 29) - ((size_t)1 << 20);

struct FileInfo {
    int h = 0, w = 0, ncomp = 0;
    int hs = 1, vs = 1;       // luma sampling factors = luma blocks per MCU across / down (chroma is always 1 x 1)
    int restart = 0;          // restart interval in MCUs (DRI), 0 = none
    uint16_t qt[2][64];       // natural order: [0] the luma component's table, [1] the chroma components' (same for both)
    HuffSpec dc[2], ac[2];    // [0] luma, [1] chroma (decoder tables: make_dec_table, once per distinct set)
    size_t scan_off = 0, scan_len = 0;   // entropy-coded segment inside the file (stuffed bytes included, EOI excluded)
};

// Parses the marker segments of one file. Supported: 8-bit baseline (SOF0/SOF1 Huffman), one component, or three
// components with the luma sampled 2x2 (4:2:0), 2x1 (4:2:2) or 1x1 (4:4:4) against 1x1 chroma, Cb and Cr sharing tables;
// a single scan; with or without restart intervals. Everything the reference's writers (cv2.imwrite, PIL save) produce by
// default is 4:2:0 without restarts; the other layouts and the restart markers are what PIL's `subsampling=` /
// `restart_marker_blocks=` and cv2's IMWRITE_JPEG_SAMPLING_FACTOR / IMWRITE_JPEG_RST_INTERVAL can ask for.
// Anything else is JPEG_UNSUPPORTED.
inline int parse_file(const uint8_t *d, size_t len, FileInfo &F, bool headers_only = false)
{
    uint16_t qt[4][64];
    bool qt_ok[4] = {false, false, false, false};
    struct Raw { uint8_t bits[16]; uint8_t vals[256]; int n; bool ok; } huff[2][4];
    for (auto &cls : huff) for (auto &t : cls) t.ok = false;
    int hs[3] = {0, 0, 0}, vs[3] = {0, 0, 0}, tq[3] = {0, 0, 0}, td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
    int restart = 0;
    bool have_sof = false, have_sos = false;
    if (!d || len < 4 || d[0] != 0xFF || d[1] != 0xD8) return JPEG_CORRUPT;
    size_t i = 2;
    while (i + 4 <= len) {
        if (d[i] != 0xFF) return JPEG_CORRUPT;
        while (i < len && d[i] == 0xFF) i++;
        if (i >= len) return JPEG_CORRUPT;
        const uint8_t m = d[i++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9 || i + 2 > len) return JPEG_CORRUPT;
        const size_t L = ((size_t)d[i] << 8) | d[i + 1];
        if (L < 2 || i + L > len) return JPEG_CORRUPT;
        const uint8_t *s = d + i + 2;
        const size_t n = L - 2;
        if (m == 0xDB) {
            size_t k = 0;
            while (k < n) {
                const int pq = s[k] >> 4, t = s[k] & 15;
                if (t > 3 || pq > 1 || k + 1 + (size_t)(pq ? 128 : 64) > n) return JPEG_CORRUPT;
                k++;
                for (int z = 0; z < 64; z++) {
                    qt[t][kZigzag[z]] = pq ? (uint16_t)((s[k] << 8) | s[k + 1]) : s[k];
                    k += pq ? 2 : 1;
                }
                qt_ok[t] = true;
            }
        } else if (m == 0xC4) {
            size_t k = 0;
            while (k < n) {
                if (k + 17 > n) return JPEG_CORRUPT;
                const int tc = s[k] >> 4, th = s[k] & 15;
                int cnt = 0;
                for (int b = 0; b < 16; b++) cnt += s[k + 1 + b];
                if (th > 3 || tc > 1 || cnt > 256 || k + 17 + (size_t)cnt > n) return JPEG_CORRUPT;
                Raw &r = huff[tc][th];
                memcpy(r.bits, s + k + 1, 16);
                memcpy(r.vals, s + k + 17, (size_t)cnt);
                r.n = cnt;
                r.ok = true;
                k += 17 + (size_t)cnt;
            }
        } else if (m == 0xC0 || m == 0xC1) {
            if (have_sof || n < 6) return JPEG_CORRUPT;
            if (s[0] != 8) return JPEG_UNSUPPORTED;
            F.h = (s[1] << 8) | s[2];
            F.w = (s[3] << 8) | s[4];
            F.ncomp = s[5];
            if (F.ncomp != 1 && F.ncomp != 3) return JPEG_UNSUPPORTED;
            if (n < 6 + 3 * (size_t)F.ncomp) return JPEG_CORRUPT;
            for (int c = 0; c < F.ncomp; c++) {
                hs[c] = s[7 + 3 * c] >> 4;
                vs[c] = s[7 + 3 * c] & 15;
                tq[c] = s[8 + 3 * c] & 3;
            }
            have_sof = true;
        } else if (m >= 0xC2 && m <= 0xCF && m != 0xC8) {
            return JPEG_UNSUPPORTED;                         // progressive, lossless, hierarchical, arithmetic
        } else if (m == 0xDD) {
            if (n < 2) return JPEG_CORRUPT;
            restart = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {
            if (!have_sof) return JPEG_CORRUPT;
            if (n < 1 || s[0] != F.ncomp) return JPEG_UNSUPPORTED;     // multi-scan files
            if (n < 1 + 2 * (size_t)F.ncomp + 3) return JPEG_CORRUPT;
            for (int c = 0; c < F.ncomp; c++) {
                td[c] = s[2 + 2 * c] >> 4;
                ta[c] = s[2 + 2 * c] & 15;
                if (td[c] > 3 || ta[c] > 3) return JPEG_CORRUPT;
            }
            F.scan_off = i + L;
            have_sos = true;
            break;
        }
        i += L;
    }
    if (!have_sos || F.h <= 0 || F.w <= 0) return JPEG_CORRUPT;
    F.restart = restart;
    F.hs = F.vs = 1;                                         // one component: the scan is not interleaved, MCU = one block
    if (F.ncomp == 3) {
        if (!(hs[1] == 1 && vs[1] == 1 && hs[2] == 1 && vs[2] == 1)) return JPEG_UNSUPPORTED;
        if (!((hs[0] == 2 && vs[0] == 2) || (hs[0] == 2 && vs[0] == 1) || (hs[0] == 1 && vs[0] == 1))) return JPEG_UNSUPPORTED;
        if (tq[1] != tq[2] || td[1] != td[2] || ta[1] != ta[2]) return JPEG_UNSUPPORTED;
        F.hs = hs[0];
        F.vs = vs[0];
    } else if (hs[0] != vs[0]) {
        return JPEG_UNSUPPORTED;
    }
    for (int c = 0; c < (F.ncomp == 3 ? 2 : 1); c++) {
        if (!qt_ok[tq[c]] || !huff[0][td[c]].ok || !huff[1][ta[c]].ok) return JPEG_CORRUPT;
        if (headers_only) continue;
        memcpy(F.qt[c], qt[tq[c]], sizeof(F.qt[c]));
        for (int cls = 0; cls < 2; cls++) {
            const Raw &r = huff[cls][cls ? ta[c] : td[c]];
            if (!huff_spec_ok(r.bits, r.n)) return JPEG_CORRUPT;
            HuffSpec &hsp = cls ? F.ac[c] : F.dc[c];
            memset(&hsp, 0, sizeof(hsp));
            memcpy(hsp.bits, r.bits, 16);
            memcpy(hsp.vals, r.vals, (size_t)r.n);
            hsp.n = (uint16_t)r.n;
            hsp.is_dc = cls ? 0 : 1;
        }
    }
    if (!headers_only && F.ncomp == 1) {
        memcpy(F.qt[1], F.qt[0], sizeof(F.qt[0]));
        F.dc[1] = F.dc[0];
        F.ac[1] = F.ac[0];
    }
    // The entropy-coded segment ends at the first marker that is not a stuffed zero: EOI in a well-formed file. Writers put
    // EOI in the last two bytes, which is checked first; otherwise the segment is searched (memchr: FF bytes are rare).
    size_t e;
    if (len >= F.scan_off + 2 && d[len - 2] == 0xFF && d[len - 1] == 0xD9 && !(len >= F.scan_off + 3 && d[len - 3] == 0xFF)) {
        e = len - 2;
    } else {
        e = F.scan_off;
        for (;;) {
            const void *hit = e + 1 < len ? memchr(d + e, 0xFF, len - 1 - e) : nullptr;
            if (!hit) { e = len; break; }
            e = (size_t)(static_cast<const uint8_t *>(hit) - d);
            if (d[e + 1] != 0x00 && !(restart && d[e + 1] >= 0xD0 && d[e + 1] <= 0xD7)) break;
            e += 2;
        }
    }
    F.scan_len = e - F.scan_off;
    // Every block costs at least two bits (a one-bit DC code and a one-bit end-of-block code): a header that promises more
    // blocks than the data can hold is damaged or truncated, and must not size any buffer.
    {
        const uint64_t mw = 8 * (uint64_t)F.hs, mh = 8 * (uint64_t)F.vs;
        const uint64_t blocks = ((uint64_t)(F.w + mw - 1) / mw) * ((uint64_t)(F.h + mh - 1) / mh) * (F.ncomp == 3 ? (uint64_t)(F.hs * F.vs + 2) : 1);
        if (blocks * 2 > (uint64_t)F.scan_len * 8) return JPEG_CORRUPT;
    }
    return JPEG_OK;
}

}  // namespace v5j
