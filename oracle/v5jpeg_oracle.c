/*
 * oracle/v5jpeg_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C, scalar) of the baseline JPEG codec steps that surround the reference's V5 arithmetic
 * (SURVEY.md §8f-2 and §8f-3; line numbers: /root/reference/nodes/V_nodes/v5_texture_ela.py):
 *
 *     Image.open(crop_path).convert('RGB')            :64   decode of the crop V1 wrote (v1_keyframes_facetrack.py:166)
 *     original.save(tmp, 'JPEG', quality=90)          :66-67 the bit stream the reference writes to temp_ela_i.jpg
 *     enhanced_diff.save(ela_output_path)             :80-81 ela_i.jpg, PIL default quality 75, 4:2:0
 *     cv2.imread(crop_path, cv2.IMREAD_GRAYSCALE)     :83   decode of the crop's luma plane only
 *     cv2.imwrite(fft_output_path, magnitude_u8)      :90-91 fft_i.jpg, OpenCV default quality 95, one component
 *
 * That code lives in Pillow / OpenCV, both bundling libjpeg-turbo — third-party, not under /root/reference. This file
 * restates the published algorithm (ITU-T T.81 baseline sequential DCT, Annex F entropy coding with the Annex K.3
 * tables, JFIF 1.01 wrapper; libjpeg's sample-domain rules per SURVEY.md Appendix A) and is pinned against
 * (a) Pillow and OpenCV running in-process — byte-identical files, pixel-identical decodes (tests/test_jpeg_oracle.py),
 * (b) the artefact files the unmodified reference node wrote (tests/golden/node_case0_ref_fixture, node_golden.json).
 *
 * Supported, because it is what the reference's writers produce: 8-bit baseline, one component, or three components
 * sampled 2x2,1x1,1x1 (4:2:0). The decoder takes any Huffman / quantisation tables and restart intervals.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

void v5o_quant_tables(int quality, uint16_t luma[64], uint16_t chroma[64]);
void v5o_fdct_1d(const int32_t d[8], int32_t o[8], int first);

/* zigzag position -> natural (row-major) index, T.81 Figure A.6 */
static const uint8_t k_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

/* T.81 Annex K.3 typical Huffman tables (what libjpeg emits when optimize_coding is off) */
static const uint8_t k_dc_bits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
static const uint8_t k_dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t k_ac_bits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125}, {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119}};
static const uint8_t k_ac_vals[2][162] = {
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

static inline uint8_t clamp_u8(int32_t v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* ================================================================================================ forward half */
/* fDCT + quantise one 8x8 block of samples (pitch bytes apart) into 64 coefficients, natural order (A.4, A.5). */
static void block_forward(const uint8_t *plane, int pitch, const uint16_t tab[64], int16_t coef[64])
{
    int32_t ws[64], tmp[8], res[8];
    for (int r = 0; r < 8; r++) {
        for (int c = 0; c < 8; c++) tmp[c] = (int32_t)plane[r * pitch + c] - 128;
        v5o_fdct_1d(tmp, res, 1);
        for (int c = 0; c < 8; c++) ws[r * 8 + c] = res[c];
    }
    for (int c = 0; c < 8; c++) {
        for (int r = 0; r < 8; r++) tmp[r] = ws[r * 8 + c];
        v5o_fdct_1d(tmp, res, 0);
        for (int r = 0; r < 8; r++) ws[r * 8 + c] = res[r];
    }
    for (int i = 0; i < 64; i++) {
        int32_t div = (int32_t)tab[i] << 3, c = ws[i], a = c < 0 ? -c : c;
        int32_t q = (a + (div >> 1)) / div;
        coef[i] = (int16_t)(c < 0 ? -q : q);
    }
}

/* Sample planes of the encoder, padded to whole MCUs (A.2, A.3). channels == 1: yp only. */
typedef struct {
    int h, w, ncomp;
    int mcux, mcuy;          /* MCUs per row / column (16x16 for 4:2:0, 8x8 for one component) */
    int yw, yh, cw, ch;      /* padded plane sizes in samples */
    uint8_t *yp, *cbp, *crp;
} planes_t;

static void planes_free(planes_t *P)
{
    free(P->yp); free(P->cbp); free(P->crp);
    P->yp = P->cbp = P->crp = NULL;
}

static int planes_from_image(const uint8_t *img, int h, int w, int channels, int64_t row_stride, planes_t *P)
{
    memset(P, 0, sizeof(*P));
    P->h = h; P->w = w; P->ncomp = channels;
    const int mcu = channels == 3 ? 16 : 8;
    P->mcux = (w + mcu - 1) / mcu; P->mcuy = (h + mcu - 1) / mcu;
    P->yw = P->mcux * mcu; P->yh = P->mcuy * mcu;
    P->yp = malloc((size_t)P->yw * P->yh);
    if (!P->yp) return -1;
    if (channels == 1) {
        for (int y = 0; y < P->yh; y++) {
            const uint8_t *row = img + (int64_t)(y < h ? y : h - 1) * row_stride;
            for (int x = 0; x < P->yw; x++) P->yp[(size_t)y * P->yw + x] = row[x < w ? x : w - 1];
        }
        return 0;
    }
    const int he = h + (h & 1), wm = P->yw;
    P->cw = P->yw / 2; P->ch = P->yh / 2;
    uint8_t *cbf = malloc((size_t)he * wm), *crf = malloc((size_t)he * wm);
    P->cbp = malloc((size_t)P->cw * P->ch); P->crp = malloc((size_t)P->cw * P->ch);
    if (!cbf || !crf || !P->cbp || !P->crp) { free(cbf); free(crf); planes_free(P); return -1; }
    for (int y = 0; y < P->yh; y++) {
        const uint8_t *row = img + (int64_t)(y < h ? y : h - 1) * row_stride;
        for (int x = 0; x < wm; x++) {
            const uint8_t *p = row + 3 * (x < w ? x : w - 1);
            const int32_t r = p[0], g = p[1], b = p[2];
            P->yp[(size_t)y * wm + x] = (uint8_t)((19595 * r + 38470 * g + 7471 * b + 32768) >> 16);
            if (y < he) {
                cbf[(size_t)y * wm + x] = (uint8_t)((-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16);
                crf[(size_t)y * wm + x] = (uint8_t)((32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16);
            }
        }
    }
    for (int y = 0; y < P->ch; y++) {                   /* h2v2 box filter, bias 1,2,1,2; bottom: replicate downsampled row */
        const int sy = y < he / 2 ? y : he / 2 - 1;
        for (int x = 0; x < P->cw; x++) {
            const int bias = (x & 1) ? 2 : 1;
            const uint8_t *a = cbf + (size_t)(2 * sy) * wm + 2 * x, *b = crf + (size_t)(2 * sy) * wm + 2 * x;
            P->cbp[(size_t)y * P->cw + x] = (uint8_t)((a[0] + a[1] + a[wm] + a[wm + 1] + bias) >> 2);
            P->crp[(size_t)y * P->cw + x] = (uint8_t)((b[0] + b[1] + b[wm] + b[wm + 1] + bias) >> 2);
        }
    }
    free(cbf); free(crf);
    return 0;
}

/* ============================================================================================ entropy encoder */
typedef struct {
    uint16_t code[256];
    uint8_t size[256];
} enc_table_t;

/* T.81 Annex C: canonical codes from BITS / HUFFVAL */
static void make_enc_table(const uint8_t bits[16], const uint8_t *vals, enc_table_t *t)
{
    memset(t, 0, sizeof(*t));
    int k = 0;
    uint32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        for (int i = 0; i < bits[len - 1]; i++, k++) {
            t->code[vals[k]] = (uint16_t)code++;
            t->size[vals[k]] = (uint8_t)len;
        }
        code <<= 1;
    }
}

typedef struct {
    uint8_t *out;
    size_t cap, pos;
    uint64_t acc;
    int nbits;
    int overflow;
} bitw_t;

static void put_byte(bitw_t *b, uint8_t v)
{
    if (b->pos < b->cap) b->out[b->pos] = v; else b->overflow = 1;
    b->pos++;
}

static void put_bits(bitw_t *b, uint32_t code, int size)
{
    if (size == 0) return;
    b->acc = (b->acc << size) | (code & ((1u << size) - 1u));
    b->nbits += size;
    while (b->nbits >= 8) {
        const uint8_t v = (uint8_t)(b->acc >> (b->nbits - 8));
        put_byte(b, v);
        if (v == 0xFF) put_byte(b, 0x00);               /* byte stuffing, T.81 F.1.2.3 */
        b->nbits -= 8;
    }
}

static int bit_length(int32_t v)
{
    int n = 0;
    while (v) { n++; v >>= 1; }
    return n;
}

/* T.81 F.1.2: one block, coefficients in natural order */
static void encode_block(bitw_t *b, const int16_t coef[64], int *last_dc, const enc_table_t *dc, const enc_table_t *ac)
{
    int32_t t = coef[0] - *last_dc, t2 = t;
    *last_dc = coef[0];
    if (t < 0) { t = -t; t2--; }
    int nb = bit_length(t);
    put_bits(b, dc->code[nb], dc->size[nb]);
    put_bits(b, (uint32_t)t2, nb);
    int run = 0;
    for (int k = 1; k < 64; k++) {
        t = coef[k_zigzag[k]];
        if (t == 0) { run++; continue; }
        while (run > 15) { put_bits(b, ac->code[0xF0], ac->size[0xF0]); run -= 16; }
        t2 = t;
        if (t < 0) { t = -t; t2--; }
        nb = bit_length(t);
        put_bits(b, ac->code[(run << 4) + nb], ac->size[(run << 4) + nb]);
        put_bits(b, (uint32_t)t2, nb);
        run = 0;
    }
    if (run > 0) put_bits(b, ac->code[0], ac->size[0]);
}

static void put_marker(bitw_t *b, uint8_t m) { put_byte(b, 0xFF); put_byte(b, m); }
static void put_u16(bitw_t *b, int v) { put_byte(b, (uint8_t)(v >> 8)); put_byte(b, (uint8_t)v); }

static void put_dht(bitw_t *b, int tc_th, const uint8_t bits[16], const uint8_t *vals)
{
    int n = 0;
    for (int i = 0; i < 16; i++) n += bits[i];
    put_marker(b, 0xC4);
    put_u16(b, 2 + 1 + 16 + n);
    put_byte(b, (uint8_t)tc_th);
    for (int i = 0; i < 16; i++) put_byte(b, bits[i]);
    for (int i = 0; i < n; i++) put_byte(b, vals[i]);
}

/* The header libjpeg writes for jpeg_set_defaults + jpeg_set_quality (JFIF 1.01, density 1:1, no units). */
static void put_headers(bitw_t *b, int h, int w, int ncomp, const uint16_t ql[64], const uint16_t qc[64])
{
    static const uint8_t jfif[14] = {'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0};
    put_marker(b, 0xD8);
    put_marker(b, 0xE0);
    put_u16(b, 16);
    for (int i = 0; i < 14; i++) put_byte(b, jfif[i]);
    for (int t = 0; t < (ncomp == 3 ? 2 : 1); t++) {
        put_marker(b, 0xDB);
        put_u16(b, 67);
        put_byte(b, (uint8_t)t);
        for (int i = 0; i < 64; i++) put_byte(b, (uint8_t)(t ? qc : ql)[k_zigzag[i]]);
    }
    put_marker(b, 0xC0);
    put_u16(b, 8 + 3 * ncomp);
    put_byte(b, 8);
    put_u16(b, h);
    put_u16(b, w);
    put_byte(b, (uint8_t)ncomp);
    for (int c = 0; c < ncomp; c++) {
        put_byte(b, (uint8_t)(c + 1));
        put_byte(b, (uint8_t)(ncomp == 3 && c == 0 ? 0x22 : 0x11));
        put_byte(b, (uint8_t)(c ? 1 : 0));
    }
    put_dht(b, 0x00, k_dc_bits[0], k_dc_vals);
    put_dht(b, 0x10, k_ac_bits[0], k_ac_vals[0]);
    if (ncomp == 3) {
        put_dht(b, 0x01, k_dc_bits[1], k_dc_vals);
        put_dht(b, 0x11, k_ac_bits[1], k_ac_vals[1]);
    }
    put_marker(b, 0xDA);
    put_u16(b, 6 + 2 * ncomp);
    put_byte(b, (uint8_t)ncomp);
    for (int c = 0; c < ncomp; c++) {
        put_byte(b, (uint8_t)(c + 1));
        put_byte(b, (uint8_t)(c ? 0x11 : 0x00));
    }
    put_byte(b, 0);
    put_byte(b, 63);
    put_byte(b, 0);
}

/*
 * Encode one image (channels 1: gray HW; 3: RGB HWC) exactly as libjpeg does for PIL's Image.save(..., 'JPEG', quality=q)
 * and cv2.imwrite(..., [IMWRITE_JPEG_QUALITY, q]). Returns the file size (also when it exceeds `cap`: nothing beyond cap
 * is written), or -1 on error. coef_out (optional): every block's quantised coefficients in scan order, ZIGZAG order
 * within the block, dummy blocks included — what the GPU coefficient kernel is compared with.
 */
int64_t v5jo_encode(const uint8_t *img, int h, int w, int channels, int64_t row_stride, int quality, uint8_t *out, size_t cap,
                    int16_t *coef_out)
{
    if (!img || h <= 0 || w <= 0 || h > 65535 || w > 65535 || (channels != 1 && channels != 3)) return -1;
    uint16_t ql[64], qc[64];
    v5o_quant_tables(quality, ql, qc);
    planes_t P;
    if (planes_from_image(img, h, w, channels, row_stride, &P)) return -1;
    enc_table_t dc[2], ac[2];
    for (int t = 0; t < 2; t++) {
        make_enc_table(k_dc_bits[t], k_dc_vals, &dc[t]);
        make_enc_table(k_ac_bits[t], k_ac_vals[t], &ac[t]);
    }
    bitw_t B = {out, out ? cap : 0, 0, 0, 0, 0};
    put_headers(&B, h, w, channels, ql, qc);
    int last_dc[3] = {0, 0, 0};
    const int ybw = (w + 7) / 8, ybh = (h + 7) / 8;     /* real luma blocks */
    size_t nblk = 0;
    for (int my = 0; my < P.mcuy; my++)
        for (int mx = 0; mx < P.mcux; mx++) {
            int16_t blk[6][64];
            int nb = 0;
            if (channels == 1) {
                block_forward(P.yp + (size_t)(8 * my) * P.yw + 8 * mx, P.yw, ql, blk[nb++]);
            } else {
                /* libjpeg jccoefct.c compress_data: blocks beyond the component's real block grid are dummies — all zero
                 * except a DC equal to the previous block's (right edge: the block to the left; bottom: the last block of
                 * the block row above inside this MCU) so that they cost two bits each. */
                for (int by = 0; by < 2; by++)
                    for (int bx = 0; bx < 2; bx++, nb++) {
                        const int gy = 2 * my + by, gx = 2 * mx + bx;
                        if (gy < ybh && gx < ybw) {
                            block_forward(P.yp + (size_t)(8 * gy) * P.yw + 8 * gx, P.yw, ql, blk[nb]);
                        } else {
                            memset(blk[nb], 0, sizeof(blk[nb]));
                            blk[nb][0] = blk[nb - 1][0];
                        }
                    }
                block_forward(P.cbp + (size_t)(8 * my) * P.cw + 8 * mx, P.cw, qc, blk[nb++]);
                block_forward(P.crp + (size_t)(8 * my) * P.cw + 8 * mx, P.cw, qc, blk[nb++]);
            }
            for (int i = 0; i < nb; i++) {
                const int comp = channels == 1 ? 0 : (i < 4 ? 0 : i - 3), t = comp ? 1 : 0;
                encode_block(&B, blk[i], &last_dc[comp], &dc[t], &ac[t]);
                if (coef_out)
                    for (int k = 0; k < 64; k++) coef_out[(nblk + i) * 64 + k] = blk[i][k_zigzag[k]];
            }
            nblk += nb;
        }
    if (B.nbits > 0) put_bits(&B, 0x7F, 8 - B.nbits);    /* pad the last byte with one-bits */
    put_marker(&B, 0xD9);
    planes_free(&P);
    return (int64_t)B.pos;
}

/* ==================================================================================================== decoder */
typedef struct {
    /* T.81 F.2.2.3 decoding tables */
    int32_t mincode[17], maxcode[18], valptr[17];
    uint8_t vals[256];
    int present;
} dec_table_t;

static void make_dec_table(const uint8_t bits[16], const uint8_t *vals, int nvals, dec_table_t *t)
{
    memset(t, 0, sizeof(*t));
    memcpy(t->vals, vals, (size_t)nvals);
    int k = 0;
    int32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        if (bits[len - 1]) {
            t->valptr[len] = k;
            t->mincode[len] = code;
            code += bits[len - 1];
            k += bits[len - 1];
            t->maxcode[len] = code - 1;
        } else {
            t->maxcode[len] = -1;
        }
        code <<= 1;
    }
    t->maxcode[17] = 0x7fffffff;
    t->present = 1;
}

typedef struct {
    const uint8_t *p, *end;
    uint32_t acc;
    int nbits;
    int marker;               /* a marker met inside the entropy-coded data (0 = none): zero bits are fed from then on */
} bitr_t;

static int get_bit(bitr_t *b)
{
    if (b->nbits == 0) {
        uint8_t v = 0;
        if (!b->marker && b->p < b->end) {
            v = *b->p++;
            if (v == 0xFF) {
                uint8_t n = b->p < b->end ? *b->p : 0xD9;
                if (n == 0) b->p++;                      /* stuffed zero */
                else { b->marker = n; b->p--; v = 0; }   /* leave the marker in place */
            }
        }
        b->acc = v;
        b->nbits = 8;
    }
    b->nbits--;
    return (int)((b->acc >> b->nbits) & 1u);
}

static int get_bits(bitr_t *b, int n)
{
    int v = 0;
    while (n--) v = (v << 1) | get_bit(b);
    return v;
}

static int decode_symbol(bitr_t *b, const dec_table_t *t)
{
    int32_t code = 0;
    for (int len = 1; len <= 16; len++) {
        code = (code << 1) | get_bit(b);
        if (t->maxcode[len] >= 0 && code <= t->maxcode[len] && code >= t->mincode[len])
            return t->vals[t->valptr[len] + (code - t->mincode[len])];
    }
    return 0;                                            /* corrupt data: libjpeg also substitutes zero */
}

static int extend(int v, int n) { return n && v < (1 << (n - 1)) ? v - (1 << n) + 1 : v; }

typedef struct {
    int h, w, ncomp;
    int hs[3], vs[3], tq[3], td[3], ta[3];
    uint16_t qt[4][64];       /* natural order */
    int qt_present[4];
    dec_table_t dc[4], ac[4];
    int restart_interval;
    size_t scan_off;          /* first byte of entropy-coded data */
    int progressive;
} jhead_t;

static int parse_headers(const uint8_t *d, size_t len, jhead_t *H)
{
    memset(H, 0, sizeof(*H));
    if (len < 4 || d[0] != 0xFF || d[1] != 0xD8) return -1;
    size_t i = 2;
    while (i + 4 <= len) {
        if (d[i] != 0xFF) return -1;
        while (i < len && d[i] == 0xFF) i++;             /* fill bytes */
        if (i >= len) return -1;
        const uint8_t m = d[i++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9 || i + 2 > len) return -1;
        const size_t L = ((size_t)d[i] << 8) | d[i + 1];
        if (L < 2 || i + L > len) return -1;
        const uint8_t *s = d + i + 2;
        const size_t n = L - 2;
        if (m == 0xDB) {
            size_t k = 0;
            while (k < n) {
                const int pq = s[k] >> 4, tq = s[k] & 15;
                if (tq > 3 || k + 1 + (size_t)(pq ? 128 : 64) > n) return -1;
                k++;
                for (int z = 0; z < 64; z++) {
                    H->qt[tq][k_zigzag[z]] = pq ? (uint16_t)((s[k] << 8) | s[k + 1]) : s[k];
                    k += pq ? 2 : 1;
                }
                H->qt_present[tq] = 1;
            }
        } else if (m == 0xC4) {
            size_t k = 0;
            while (k < n) {
                if (k + 17 > n) return -1;
                const int tc = s[k] >> 4, th = s[k] & 15;
                int cnt = 0;
                for (int b = 0; b < 16; b++) cnt += s[k + 1 + b];
                if (th > 3 || tc > 1 || cnt > 256 || k + 17 + (size_t)cnt > n) return -1;
                make_dec_table(s + k + 1, s + k + 17, cnt, tc ? &H->ac[th] : &H->dc[th]);
                k += 17 + (size_t)cnt;
            }
        } else if (m == 0xC0 || m == 0xC1 || m == 0xC2) {
            if (n < 6 || s[0] != 8) return -2;
            H->progressive = m == 0xC2;
            H->h = (s[1] << 8) | s[2];
            H->w = (s[3] << 8) | s[4];
            H->ncomp = s[5];
            if ((H->ncomp != 1 && H->ncomp != 3) || n < 6 + 3 * (size_t)H->ncomp) return -2;
            for (int c = 0; c < H->ncomp; c++) {
                H->hs[c] = s[7 + 3 * c] >> 4;
                H->vs[c] = s[7 + 3 * c] & 15;
                H->tq[c] = s[8 + 3 * c] & 3;
            }
        } else if (m >= 0xC3 && m <= 0xCF && m != 0xC8 && m != 0xCC) {
            return -2;                                   /* lossless / hierarchical / arithmetic: not supported */
        } else if (m == 0xDD) {
            if (n < 2) return -1;
            H->restart_interval = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {
            if (n < 1 || s[0] != H->ncomp || n < 1 + 2 * (size_t)H->ncomp + 3) return -2;
            for (int c = 0; c < H->ncomp; c++) {
                H->td[c] = s[2 + 2 * c] >> 4;
                H->ta[c] = s[2 + 2 * c] & 15;
            }
            H->scan_off = i + L;
            break;
        }
        i += L;
    }
    if (!H->scan_off || H->h <= 0 || H->w <= 0 || H->progressive) return -2;
    /* chroma layouts Pillow / OpenCV can write: 4:2:0 (2x2), 4:2:2 (2x1), 4:4:4 (1x1), chroma components always 1x1 */
    if (H->ncomp == 3 && !(H->hs[1] == 1 && H->vs[1] == 1 && H->hs[2] == 1 && H->vs[2] == 1 &&
                           ((H->hs[0] == 2 && H->vs[0] == 2) || (H->hs[0] == 2 && H->vs[0] == 1) || (H->hs[0] == 1 && H->vs[0] == 1)))) return -2;
    for (int c = 0; c < H->ncomp; c++)
        if (!H->qt_present[H->tq[c]] || !H->dc[H->td[c]].present || !H->ac[H->ta[c]].present) return -1;
    return 0;
}

/* -> 0 and the geometry, -1 corrupt, -2 a JPEG flavour outside the supported set */
int v5jo_info(const uint8_t *data, size_t len, int *h, int *w, int *ncomp)
{
    jhead_t H;
    const int rc = parse_headers(data, len, &H);
    if (rc) return rc;
    *h = H.h; *w = H.w; *ncomp = H.ncomp;
    return 0;
}

/* Luma sampling factors (2x2 = 4:2:0, 2x1 = 4:2:2, 1x1 = 4:4:4 or one component) and the restart interval in MCUs. */
int v5jo_layout(const uint8_t *data, size_t len, int *hs, int *vs, int *restart_interval)
{
    jhead_t H;
    const int rc = parse_headers(data, len, &H);
    if (rc) return rc;
    *hs = H.ncomp == 3 ? H.hs[0] : 1;
    *vs = H.ncomp == 3 ? H.vs[0] : 1;
    *restart_interval = H.restart_interval;
    return 0;
}

/* int16 wrap and saturation */
static inline int32_t w16(int32_t v) { return (int32_t)(int16_t)(uint16_t)(uint32_t)v; }
static inline int32_t sat16(int32_t v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); }

/* One 8-point ISLOW pass (T.81 A.6 with libjpeg's constants) as libjpeg-turbo's x86 SIMD code computes it on int16 inputs:
 * in0 + in4, in0 - in4, in3 + in7 and in1 + in5 are 16-bit lane adds that wrap; every product is a 16 x 16 -> 32-bit
 * multiply-add, so the rest is exact (no 32-bit sum of int16 inputs reaches 2^31). -> (sum + 2^(n-1)) >> n. */
static void simd_idct_1d(const int32_t in[8], int32_t out[8], int n)
{
    const int32_t t0 = w16(in[0] + in[4]) * 8192, t1 = w16(in[0] - in[4]) * 8192;
    const int32_t t2 = in[2] * 4433 + in[6] * (4433 - 15137), t3 = in[2] * (4433 + 6270) + in[6] * 4433;
    const int32_t e10 = t0 + t3, e13 = t0 - t3, e11 = t1 + t2, e12 = t1 - t2;
    const int32_t z3 = w16(in[7] + in[3]), z4 = w16(in[5] + in[1]);
    const int32_t z3b = z3 * (9633 - 16069) + z4 * 9633, z4b = z3 * 9633 + z4 * (9633 - 3196);
    const int32_t o0 = in[7] * (2446 - 7373) + in[1] * -7373 + z3b;
    const int32_t o3 = in[7] * -7373 + in[1] * (12299 - 7373) + z4b;
    const int32_t o1 = in[5] * (16819 - 20995) + in[3] * -20995 + z4b;
    const int32_t o2 = in[5] * -20995 + in[3] * (25172 - 20995) + z3b;
    const int32_t r = 1 << (n - 1);
    out[0] = (e10 + o3 + r) >> n; out[7] = (e10 - o3 + r) >> n;
    out[1] = (e11 + o2 + r) >> n; out[6] = (e11 - o2 + r) >> n;
    out[2] = (e12 + o1 + r) >> n; out[5] = (e12 - o1 + r) >> n;
    out[3] = (e13 + o0 + r) >> n; out[4] = (e13 - o0 + r) >> n;
}

/* Dequantise + IDCT of one block (coefficients natural order) into a plane: ISLOW (A.6) with the arithmetic of libjpeg-turbo's
 * x86 SIMD code, the decode Pillow and OpenCV give on x86-64. Dequantisation keeps the low 16 bits of coefficient x entry, the
 * column-pass outputs saturate to int16 (or, when AC rows 1..7 of the block are all zero, are the dequantised DC << 2 wrapped
 * to 16 bits), the samples saturate to 0..255. On the coefficients of files written from pixels nothing leaves int16 and this
 * is A.6 in wide integers. */
static void block_inverse(const int16_t coef[64], const uint16_t tab[64], uint8_t *plane, int pitch)
{
    int32_t ws[64], tmp[8], res[8];
    int ac = 0;
    for (int k = 8; k < 64; k++) ac |= coef[k];
    for (int c = 0; c < 8; c++) {
        for (int r = 0; r < 8; r++) tmp[r] = w16((int32_t)coef[r * 8 + c] * (int32_t)tab[r * 8 + c]);
        if (ac) {
            simd_idct_1d(tmp, res, 11);
            for (int r = 0; r < 8; r++) ws[r * 8 + c] = sat16(res[r]);
        } else {
            for (int r = 0; r < 8; r++) ws[r * 8 + c] = w16(tmp[0] * 4);
        }
    }
    for (int r = 0; r < 8; r++) {
        simd_idct_1d(&ws[r * 8], res, 18);
        for (int c = 0; c < 8; c++) plane[r * pitch + c] = clamp_u8(res[c] + 128);
    }
}

/*
 * Decode like libjpeg with its defaults (JDCT_ISLOW, fancy upsampling), the way PIL's Image.open(...).convert('RGB')
 * and cv2.imread(..., IMREAD_GRAYSCALE) drive it.
 *   rgb_out : H*W*3 or NULL — a one-component file is replicated into the three channels (PIL L -> RGB)
 *   y_out   : H*W or NULL   — the luma plane alone (what IMREAD_GRAYSCALE / PIL draft('L') return for a colour file)
 *   coef_out: optional, all blocks in scan order, zigzag order inside the block, DC predictions already undone
 */
int v5jo_decode(const uint8_t *data, size_t len, uint8_t *rgb_out, uint8_t *y_out, int16_t *coef_out)
{
    jhead_t H;
    int rc = parse_headers(data, len, &H);
    if (rc) return rc;
    const int h = H.h, w = H.w;
    const int hs = H.ncomp == 3 ? H.hs[0] : 1, vs = H.ncomp == 3 ? H.vs[0] : 1;       /* luma blocks per MCU: hs x vs */
    const int mcux = (w + 8 * hs - 1) / (8 * hs), mcuy = (h + 8 * vs - 1) / (8 * vs);
    const int yw = mcux * 8 * hs, yh = mcuy * 8 * vs, cw = mcux * 8, ch = mcuy * 8;
    uint8_t *yp = malloc((size_t)yw * yh), *cbp = NULL, *crp = NULL;
    if (H.ncomp == 3) { cbp = malloc((size_t)cw * ch); crp = malloc((size_t)cw * ch); }
    if (!yp || (H.ncomp == 3 && (!cbp || !crp))) { free(yp); free(cbp); free(crp); return -1; }
    bitr_t B = {data + H.scan_off, data + len, 0, 0, 0};
    int pred[3] = {0, 0, 0};
    int until_restart = H.restart_interval;
    size_t nblk = 0;
    for (int my = 0; my < mcuy; my++)
        for (int mx = 0; mx < mcux; mx++) {
            if (H.restart_interval && until_restart == 0) {
                B.nbits = 0;                             /* discard padding bits, step over the RSTn marker */
                if (B.marker >= 0xD0 && B.marker <= 0xD7) { B.p += 2; B.marker = 0; }
                else if (B.p + 1 < B.end && B.p[0] == 0xFF && B.p[1] >= 0xD0 && B.p[1] <= 0xD7) B.p += 2;
                pred[0] = pred[1] = pred[2] = 0;
                until_restart = H.restart_interval;
            }
            const int ny = hs * vs, nb = H.ncomp == 3 ? ny + 2 : 1;
            for (int i = 0; i < nb; i++) {
                const int comp = H.ncomp == 1 ? 0 : (i < ny ? 0 : i - ny + 1);
                int16_t coef[64];
                memset(coef, 0, sizeof(coef));
                int s = decode_symbol(&B, &H.dc[H.td[comp]]);
                if (s > 15) s = 15;
                pred[comp] += extend(get_bits(&B, s), s);
                coef[0] = (int16_t)pred[comp];
                for (int k = 1; k < 64; k++) {
                    const int rs = decode_symbol(&B, &H.ac[H.ta[comp]]), r = rs >> 4, sz = rs & 15;
                    if (sz == 0) {
                        if (r != 15) break;              /* EOB */
                        k += 15;                         /* ZRL */
                        continue;
                    }
                    k += r;
                    const int v = extend(get_bits(&B, sz), sz);
                    if (k < 64) coef[k_zigzag[k]] = (int16_t)v;
                }
                if (coef_out)
                    for (int k = 0; k < 64; k++) coef_out[(nblk + (size_t)i) * 64 + k] = coef[k_zigzag[k]];
                if (comp == 0) {
                    const int by = vs * my + i / hs, bx = hs * mx + i % hs;
                    block_inverse(coef, H.qt[H.tq[0]], yp + (size_t)(8 * by) * yw + 8 * bx, yw);
                } else {
                    block_inverse(coef, H.qt[H.tq[comp]], (comp == 1 ? cbp : crp) + (size_t)(8 * my) * cw + 8 * mx, cw);
                }
            }
            nblk += (size_t)nb;
            if (H.restart_interval) until_restart--;
        }
    if (y_out)
        for (int y = 0; y < h; y++) memcpy(y_out + (size_t)y * w, yp + (size_t)y * yw, (size_t)w);
    if (rgb_out && H.ncomp == 1) {
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                const uint8_t v = yp[(size_t)y * yw + x];
                uint8_t *o = rgb_out + ((size_t)y * w + x) * 3;
                o[0] = o[1] = o[2] = v;
            }
    } else if (rgb_out) {
        /* chroma sample for pixel (x, y): libjpeg's upsamplers with do_fancy_upsampling (jdsample.c)
         *   2x2: h2v2 "triangle" filter (SURVEY.md A.7)      2x1: h2v1 fancy, 3/4 : 1/4 along the row      1x1: none
         * both fancy forms fall back to plain replication when the downsampled width is <= 2 */
        const int hc = (h + vs - 1) / vs, wc = (w + hs - 1) / hs;
        for (int y = 0; y < h; y++) {
            int r = y / vs, nbr = r;
            if (vs == 2) {
                nbr = (y & 1) ? r + 1 : r - 1;
                if (nbr < 0) nbr = 0;
                if (nbr > hc - 1) nbr = hc - 1;
            }
            for (int x = 0; x < w; x++) {
                const int cx = x / hs;
                int cb, cr;
                if (hs == 1 || wc <= 2) {
                    cb = cbp[(size_t)r * cw + cx];
                    cr = crp[(size_t)r * cw + cx];
                } else if (vs == 2) {
                    int nx = (x & 1) ? cx + 1 : cx - 1;
                    if (nx < 0) nx = 0;
                    if (nx > wc - 1) nx = wc - 1;
                    const int bias = (x & 1) ? 7 : 8;
                    int32_t s0 = 3 * cbp[(size_t)r * cw + cx] + cbp[(size_t)nbr * cw + cx];
                    int32_t s1 = 3 * cbp[(size_t)r * cw + nx] + cbp[(size_t)nbr * cw + nx];
                    cb = (3 * s0 + s1 + bias) >> 4;
                    s0 = 3 * crp[(size_t)r * cw + cx] + crp[(size_t)nbr * cw + cx];
                    s1 = 3 * crp[(size_t)r * cw + nx] + crp[(size_t)nbr * cw + nx];
                    cr = (3 * s0 + s1 + bias) >> 4;
                } else {                                 /* h2v1 fancy: the first and last output samples copy their input */
                    const int nx = (x & 1) ? cx + 1 : cx - 1;
                    if (nx < 0 || nx > wc - 1) {
                        cb = cbp[(size_t)r * cw + cx];
                        cr = crp[(size_t)r * cw + cx];
                    } else {
                        const int bias = (x & 1) ? 2 : 1;
                        cb = (3 * cbp[(size_t)r * cw + cx] + cbp[(size_t)r * cw + nx] + bias) >> 2;
                        cr = (3 * crp[(size_t)r * cw + cx] + crp[(size_t)r * cw + nx] + bias) >> 2;
                    }
                }
                const int32_t yy = yp[(size_t)y * yw + x], cbd = cb - 128, crd = cr - 128;
                uint8_t *o = rgb_out + ((size_t)y * w + x) * 3;
                o[0] = clamp_u8(yy + ((91881 * crd + 32768) >> 16));
                o[1] = clamp_u8(yy + ((-22554 * cbd - 46802 * crd + 32768) >> 16));
                o[2] = clamp_u8(yy + ((116130 * cbd + 32768) >> 16));
            }
        }
    }
    free(yp); free(cbp); free(crp);
    return 0;
}
