/*
 * oracle/v5ela_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C, scalar, one thread) of the arithmetic behind the reference's V5
 * error-level-analysis step:
 *
 *     original.save(tmp, 'JPEG', quality=q)      nodes/V_nodes/v5_texture_ela.py:66-67
 *     compressed = Image.open(tmp)               nodes/V_nodes/v5_texture_ela.py:68
 *     diff = ImageChops.difference(orig, comp)   nodes/V_nodes/v5_texture_ela.py:70
 *     extrema / max_diff / scale                 nodes/V_nodes/v5_texture_ela.py:72-76
 *     ImageEnhance.Brightness(diff).enhance()    nodes/V_nodes/v5_texture_ela.py:78
 *
 * The arithmetic itself lives in third-party code that is NOT under /root/reference:
 * Pillow (uv.lock pins 11.3.0; this image has 12.2.0) bundling libjpeg-turbo (3.1.x): 8-bit baseline JPEG,
 * 4:2:0 (h2v2) chroma, JDCT_ISLOW, Annex-K tables scaled by quality, fancy upsampling. This file restates
 * that published algorithm from the spec in SURVEY.md Appendix A (A.1 .. A.9); entropy coding is lossless
 * and therefore skipped. It is pinned against (a) Pillow itself running in-process (tests/test_oracle.py)
 * and (b) the golden vectors in tests/golden/ which were produced by executing the unmodified reference node.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may load this.
 *
 * Build: see oracle/Makefile  ->  oracle/libv5ela_oracle.so
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ---- A.1 quantisation tables (Annex K.1 / K.2, natural order) ------------------------------------- */
static const uint8_t k_luma_base[64] = {
    16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
    14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
    18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
    49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const uint8_t k_chroma_base[64] = {
    17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
    24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

void v5o_quant_tables(int quality, uint16_t luma[64], uint16_t chroma[64])
{
    int q = quality < 1 ? 1 : (quality > 100 ? 100 : quality);
    int scale = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int i = 0; i < 64; i++) {
        int l = (k_luma_base[i] * scale + 50) / 100;
        int c = (k_chroma_base[i] * scale + 50) / 100;
        luma[i] = (uint16_t)(l < 1 ? 1 : (l > 255 ? 255 : l));   /* force_baseline */
        chroma[i] = (uint16_t)(c < 1 ? 1 : (c > 255 ? 255 : c));
    }
}

/* ---- A.4 / A.6 islow constants (CONST_BITS = 13) --------------------------------------------------- */
#define C0_298 2446
#define C0_390 3196
#define C0_541 4433
#define C0_765 6270
#define C0_899 7373
#define C1_175 9633
#define C1_501 12299
#define C1_847 15137
#define C1_961 16069
#define C2_053 16819
#define C2_562 20995
#define C3_072 25172

static inline int32_t descale(int32_t x, int n) { return (x + (1 << (n - 1))) >> n; }

/* One 8-point forward pass. first != 0: row pass (n = 11, DC terms << 2); else column pass (n = 15, DC descale 2). */
static void fdct_1d(const int32_t d[8], int32_t o[8], int first)
{
    int32_t t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    int32_t t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    int32_t t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int n = first ? 11 : 15;
    if (first) {
        o[0] = (t10 + t11) * 4;
        o[4] = (t10 - t11) * 4;
    } else {
        o[0] = descale(t10 + t11, 2);
        o[4] = descale(t10 - t11, 2);
    }
    int32_t z1 = (t12 + t13) * C0_541;
    o[2] = descale(z1 + t13 * C0_765, n);
    o[6] = descale(z1 - t12 * C1_847, n);
    int32_t y1 = t4 + t7, y2 = t5 + t6, y3 = t4 + t6, y4 = t5 + t7;
    int32_t y5 = (y3 + y4) * C1_175;
    t4 *= C0_298; t5 *= C2_053; t6 *= C3_072; t7 *= C1_501;
    y1 *= -C0_899; y2 *= -C2_562;
    y3 = y3 * -C1_961 + y5;
    y4 = y4 * -C0_390 + y5;
    o[7] = descale(t4 + y1 + y3, n);
    o[5] = descale(t5 + y2 + y4, n);
    o[3] = descale(t6 + y2 + y3, n);
    o[1] = descale(t7 + y1 + y4, n);
}

/* One 8-point inverse pass with descale amount n (11 for the column pass, 18 for the row pass). */
static void idct_1d(const int32_t in[8], int32_t out[8], int n)
{
    int32_t z1 = (in[2] + in[6]) * C0_541;
    int32_t t2 = z1 - in[6] * C1_847;
    int32_t t3 = z1 + in[2] * C0_765;
    int32_t t0 = (in[0] + in[4]) * 8192;
    int32_t t1 = (in[0] - in[4]) * 8192;
    int32_t t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int32_t u0 = in[7], u1 = in[5], u2 = in[3], u3 = in[1];
    int32_t y1 = u0 + u3, y2 = u1 + u2, y3 = u0 + u2, y4 = u1 + u3;
    int32_t y5 = (y3 + y4) * C1_175;
    u0 *= C0_298; u1 *= C2_053; u2 *= C3_072; u3 *= C1_501;
    y1 *= -C0_899; y2 *= -C2_562;
    y3 = y3 * -C1_961 + y5;
    y4 = y4 * -C0_390 + y5;
    u0 += y1 + y3; u1 += y2 + y4; u2 += y2 + y3; u3 += y1 + y4;
    out[0] = descale(t10 + u3, n); out[7] = descale(t10 - u3, n);
    out[1] = descale(t11 + u2, n); out[6] = descale(t11 - u2, n);
    out[2] = descale(t12 + u1, n); out[5] = descale(t12 - u1, n);
    out[3] = descale(t13 + u0, n); out[4] = descale(t13 - u0, n);
}

static inline uint8_t clamp_u8(int32_t v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* A.4 + A.5 + A.6 on one 8x8 block, in place. `plane` has row pitch `pitch`. Optionally exports the quantised
 * coefficients (64 int16, natural order) for kernel debugging. */
static void block_roundtrip(uint8_t *plane, int pitch, const uint16_t tab[64], int16_t *coef_out)
{
    int32_t ws[64], tmp[8], res[8];
    for (int r = 0; r < 8; r++) {                      /* fDCT pass 1: rows */
        for (int c = 0; c < 8; c++) tmp[c] = (int32_t)plane[r * pitch + c] - 128;
        fdct_1d(tmp, res, 1);
        for (int c = 0; c < 8; c++) ws[r * 8 + c] = res[c];
    }
    for (int c = 0; c < 8; c++) {                      /* fDCT pass 2: columns */
        for (int r = 0; r < 8; r++) tmp[r] = ws[r * 8 + c];
        fdct_1d(tmp, res, 0);
        for (int r = 0; r < 8; r++) ws[r * 8 + c] = res[r];
    }
    for (int i = 0; i < 64; i++) {                     /* A.5 quantise (half away from zero) + dequantise */
        int32_t div = (int32_t)tab[i] << 3, c = ws[i], a = c < 0 ? -c : c;
        int32_t q = (a + (div >> 1)) / div;
        if (c < 0) q = -q;
        if (coef_out) coef_out[i] = (int16_t)q;
        ws[i] = q * (int32_t)tab[i];
    }
    for (int c = 0; c < 8; c++) {                      /* IDCT pass 1: columns */
        for (int r = 0; r < 8; r++) tmp[r] = ws[r * 8 + c];
        idct_1d(tmp, res, 11);
        for (int r = 0; r < 8; r++) ws[r * 8 + c] = res[r];
    }
    for (int r = 0; r < 8; r++) {                      /* IDCT pass 2: rows, +128, clamp */
        idct_1d(&ws[r * 8], res, 18);
        for (int c = 0; c < 8; c++) plane[r * pitch + c] = clamp_u8(res[c] + 128);
    }
}

/* cv2.BORDER_REFLECT_101 index (cv2.Laplacian default border); a length-1 axis maps everything to 0. */
static inline int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

/*
 * The per-frame feature record "V5F v1" (SURVEY.md §8a). Must stay byte-identical to v5ela_record in
 * include/v5ela.h; the test-suite asserts the two sizes agree.
 */
typedef struct {
    uint32_t ela_hist[3][256];
    uint64_t ela_sum[3];
    uint64_t ela_sumsq[3];
    uint64_t tex_sumabs;
    uint64_t tex_sumsq;
    uint16_t tex_maxabs;
    uint8_t ela_max[3];
    uint8_t pad[3];
} v5o_record;

size_t v5o_record_bytes(void) { return sizeof(v5o_record); }

/*
 * Full round trip + residual + record for one H x W RGB frame (HWC uint8, row stride `row_stride` bytes).
 *   residual   : out, H*W*3 (tightly packed), may be NULL
 *   recon      : out, H*W*3 decoded RGB, may be NULL
 *   dbg_y/cb/cr: out, decoded planes Hm*Wm, (Hm/2)*(Wm/2) x2; may be NULL
 * Returns 0, or -1 on allocation failure / bad arguments.
 */
int v5o_analyze_frame(const uint8_t *rgb, int h, int w, int64_t row_stride, int quality, v5o_record *rec,
                      uint8_t *residual, uint8_t *recon, uint8_t *dbg_y, uint8_t *dbg_cb, uint8_t *dbg_cr)
{
    if (!rgb || h <= 0 || w <= 0 || !rec) return -1;
    uint16_t qt_l[64], qt_c[64];
    v5o_quant_tables(quality, qt_l, qt_c);
    const int hm = 16 * ((h + 15) / 16), wm = 16 * ((w + 15) / 16);
    const int hc = (h + 1) / 2, wc = (w + 1) / 2, chp = hm / 2, cwp = wm / 2;
    const int he = h + (h & 1);
    uint8_t *yo = malloc((size_t)h * w);               /* luma of the original, for the texture stats */
    uint8_t *yp = malloc((size_t)hm * wm);
    uint8_t *cbf = malloc((size_t)he * wm), *crf = malloc((size_t)he * wm);
    uint8_t *cbp = malloc((size_t)chp * cwp), *crp = malloc((size_t)chp * cwp);
    if (!yo || !yp || !cbf || !crf || !cbp || !crp) {
        free(yo); free(yp); free(cbf); free(crf); free(cbp); free(crp);
        return -1;
    }
    /* A.2 colour conversion, A.3 edge replication in full-resolution colour space */
    for (int y = 0; y < he; y++) {
        int sy = y < h ? y : h - 1;
        for (int x = 0; x < wm; x++) {
            int sx = x < w ? x : w - 1;
            const uint8_t *p = rgb + (int64_t)sy * row_stride + 3 * sx;
            int32_t r = p[0], g = p[1], b = p[2];
            cbf[(size_t)y * wm + x] = (uint8_t)((-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16);
            crf[(size_t)y * wm + x] = (uint8_t)((32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16);
        }
    }
    for (int y = 0; y < hm; y++) {
        int sy = y < h ? y : h - 1;
        for (int x = 0; x < wm; x++) {
            int sx = x < w ? x : w - 1;
            const uint8_t *p = rgb + (int64_t)sy * row_stride + 3 * sx;
            uint8_t v = (uint8_t)((19595 * p[0] + 38470 * p[1] + 7471 * p[2] + 32768) >> 16);
            yp[(size_t)y * wm + x] = v;
            if (y < h && x < w) yo[(size_t)y * w + x] = v;
        }
    }
    /* A.3 h2v2 box downsample, bias 1,2,1,2 along x; then replicate the DOWNSAMPLED bottom row */
    for (int y = 0; y < chp; y++) {
        int sy = y < he / 2 ? y : he / 2 - 1;
        for (int x = 0; x < cwp; x++) {
            int bias = (x & 1) ? 2 : 1;
            const uint8_t *a = cbf + (size_t)(2 * sy) * wm + 2 * x, *b = crf + (size_t)(2 * sy) * wm + 2 * x;
            cbp[(size_t)y * cwp + x] = (uint8_t)((a[0] + a[1] + a[wm] + a[wm + 1] + bias) >> 2);
            crp[(size_t)y * cwp + x] = (uint8_t)((b[0] + b[1] + b[wm] + b[wm + 1] + bias) >> 2);
        }
    }
    /* A.4-A.6 block round trips */
    for (int by = 0; by < hm; by += 8)
        for (int bx = 0; bx < wm; bx += 8) block_roundtrip(yp + (size_t)by * wm + bx, wm, qt_l, NULL);
    for (int by = 0; by < chp; by += 8)
        for (int bx = 0; bx < cwp; bx += 8) {
            block_roundtrip(cbp + (size_t)by * cwp + bx, cwp, qt_c, NULL);
            block_roundtrip(crp + (size_t)by * cwp + bx, cwp, qt_c, NULL);
        }
    if (dbg_y) memcpy(dbg_y, yp, (size_t)hm * wm);
    if (dbg_cb) memcpy(dbg_cb, cbp, (size_t)chp * cwp);
    if (dbg_cr) memcpy(dbg_cr, crp, (size_t)chp * cwp);

    memset(rec, 0, sizeof(*rec));
    /* A.7 upsample + A.8 colour conversion + A.9 residual, pixel by pixel */
    for (int y = 0; y < h; y++) {
        int r = y >> 1, nb = (y & 1) ? r + 1 : r - 1;
        if (nb < 0) nb = 0;
        if (nb > hc - 1) nb = hc - 1;
        for (int x = 0; x < w; x++) {
            int cx = x >> 1, cb, cr;
            if (wc <= 2) {                              /* libjpeg falls back to plain replication */
                cb = cbp[(size_t)r * cwp + cx];
                cr = crp[(size_t)r * cwp + cx];
            } else {
                int nx = (x & 1) ? cx + 1 : cx - 1;
                if (nx < 0) nx = 0;
                if (nx > wc - 1) nx = wc - 1;
                int bias = (x & 1) ? 7 : 8;
                int32_t s0 = 3 * cbp[(size_t)r * cwp + cx] + cbp[(size_t)nb * cwp + cx];
                int32_t s1 = 3 * cbp[(size_t)r * cwp + nx] + cbp[(size_t)nb * cwp + nx];
                cb = (3 * s0 + s1 + bias) >> 4;
                s0 = 3 * crp[(size_t)r * cwp + cx] + crp[(size_t)nb * cwp + cx];
                s1 = 3 * crp[(size_t)r * cwp + nx] + crp[(size_t)nb * cwp + nx];
                cr = (3 * s0 + s1 + bias) >> 4;
            }
            int32_t yy = yp[(size_t)y * wm + x], cbd = cb - 128, crd = cr - 128;
            uint8_t out[3];
            out[0] = clamp_u8(yy + ((91881 * crd + 32768) >> 16));
            out[1] = clamp_u8(yy + ((-22554 * cbd - 46802 * crd + 32768) >> 16));
            out[2] = clamp_u8(yy + ((116130 * cbd + 32768) >> 16));
            const uint8_t *p = rgb + (int64_t)y * row_stride + 3 * x;
            for (int c = 0; c < 3; c++) {
                int d = (int)p[c] - (int)out[c];
                if (d < 0) d = -d;
                if (residual) residual[((size_t)y * w + x) * 3 + c] = (uint8_t)d;
                if (recon) recon[((size_t)y * w + x) * 3 + c] = out[c];
                rec->ela_hist[c][d]++;
                rec->ela_sum[c] += (uint64_t)d;
                rec->ela_sumsq[c] += (uint64_t)(d * d);
                if (d > rec->ela_max[c]) rec->ela_max[c] = (uint8_t)d;
            }
        }
    }
    /* Texture: L = cv2.Laplacian(Y, CV_16S, ksize=1), BORDER_REFLECT_101, on the luma of the ORIGINAL frame */
    for (int y = 0; y < h; y++) {
        int yu = reflect101(y - 1, h), yd = reflect101(y + 1, h);
        for (int x = 0; x < w; x++) {
            int xl = reflect101(x - 1, w), xr = reflect101(x + 1, w);
            int32_t l = (int32_t)yo[(size_t)yu * w + x] + yo[(size_t)yd * w + x] + yo[(size_t)y * w + xl] +
                        yo[(size_t)y * w + xr] - 4 * (int32_t)yo[(size_t)y * w + x];
            int32_t a = l < 0 ? -l : l;
            rec->tex_sumabs += (uint64_t)a;
            rec->tex_sumsq += (uint64_t)(a * a);
            if (a > rec->tex_maxabs) rec->tex_maxabs = (uint16_t)a;
        }
    }
    free(yo); free(yp); free(cbf); free(crf); free(cbp); free(crp);
    return 0;
}

/* Batch driver: n frames, frame stride in bytes; records n x v5o_record; residual n x H x W x 3 or NULL. */
int v5o_analyze(const uint8_t *rgb, int n, int h, int w, int64_t frame_stride, int64_t row_stride, int quality,
                v5o_record *recs, uint8_t *residual)
{
    for (int i = 0; i < n; i++) {
        int rc = v5o_analyze_frame(rgb + (int64_t)i * frame_stride, h, w, row_stride, quality, recs + i,
                                   residual ? residual + (size_t)i * h * w * 3 : NULL, NULL, NULL, NULL, NULL);
        if (rc) return rc;
    }
    return 0;
}

/* A.9 enhancement LUT: u8(trunc(f32(x) * f32(255.0 / max))) clipped — float32 like Pillow's ImagingBlend. */
void v5o_enhance_lut(int max_diff, uint8_t lut[256])
{
    if (max_diff <= 0) max_diff = 1;
    float scale = (float)(255.0 / (double)max_diff);
    for (int x = 0; x < 256; x++) {
        float v = (float)x * scale;
        lut[x] = (uint8_t)(v <= 0.0f ? 0 : (v >= 255.0f ? 255 : (int)v));
    }
}

/* Exported 1-D pass for the codec restatement (oracle/v5jpeg_oracle.c), which is linked into the same .so. */
void v5o_fdct_1d(const int32_t d[8], int32_t o[8], int first) { fdct_1d(d, o, first); }
