// tests/emu/v5jpeg_emu.cpp — TEST INFRASTRUCTURE: runs the host/device-shared logic of the codec kernels
// (csrc/v5jpeg_enc.cuh, csrc/v5jpeg_dec.cuh compiled by g++) with the threads of a CTA emulated sequentially between
// barriers, so strip/edge/dummy-block indexing, the bit writer and the self-synchronising Huffman decoder can be checked
// against the oracle in a container without a GPU. The prefix sums and the byte (un)stuffing are plain loops here; their
// CUDA versions are covered by the -m gpu tests. NOT a CPU fallback: nothing under fake-video-detection-engine_b200/ loads it.
//
// Build (tests/test_jpeg_emu.py does it): g++ -O2 -shared -fPIC [-DV5J_HUFF_NT=.. -DV5J_SUB_BITS=..] -I include -I <csrc> ...
#include <cstdlib>
#include <cstring>
#include <vector>

#include "v5ela_host.h"
#include "v5jpeg_enc.cuh"
#include "v5jpeg_dec.cuh"

using namespace v5j;

extern "C" int64_t v5jemu_encode(const uint8_t *img, int h, int w, int channels, int64_t row_stride, int quality, uint8_t *out,
                                 int64_t cap, int16_t *coef_out)
{
    const EncGeo g = enc_geo(h, w, channels);
    uint16_t ql[64], qc[64];
    v5plan::quant_tables(quality, ql, qc);
    std::vector<int16_t> coef((size_t)g.blocks * 64);
    CoefParams p;
    memset(&p, 0, sizeof(p));
    p.img = img;
    p.row_stride = row_stride;
    p.coef = coef.data();
    p.g = g;
    make_enc_quant(ql, p.q[0]);
    make_enc_quant(qc, p.q[1]);
    const int per = channels == 3 ? ENC_TM : ENC_BLOCKS;
    CoefSmem *S = (CoefSmem *)aligned_alloc(16, (sizeof(CoefSmem) + 15) & ~(size_t)15);
    for (int my = 0; my < g.mcuy; my++)
        for (int tile_x = 0; tile_x * per < g.mcux; tile_x++) {
            memset(S, 0xA5, sizeof(CoefSmem));                              // poison
            memcpy(S->zz, kZigzag, 64);
            for (int t = 0; t < ENC_NT; t++) coef_load_quant(t, *S, p);
            const int mx0 = tile_x * per, mcus = g.mcux - mx0 < per ? g.mcux - mx0 : per, nblocks = mcus * g.bpm;
            if (channels == 3) {
                for (int t = 0; t < ENC_NT; t++) coef_stage_rgb(t, *S, p, img, tile_x, my);
                for (int t = 0; t < ENC_NT; t++) coef_load_colour(t, *S, p, tile_x, my);
            } else {
                for (int t = 0; t < ENC_NT; t++) coef_load_gray(t, *S, p, img, tile_x, my);
            }
            for (int t = 0; t < ENC_NT; t++) coef_rows(t, *S, g.ncomp, nblocks);
            for (int t = 0; t < ENC_NT; t++) coef_cols(t, *S, p, nblocks);
            int16_t *dst = p.coef + ((int64_t)my * g.mcux + mx0) * g.bpm * 64;
            for (int t = 0; t < ENC_NT; t++) coef_store(t, *S, p, dst, mx0, my, nblocks);
        }
    free(S);
    if (coef_out) memcpy(coef_out, coef.data(), coef.size() * 2);
    EncTables T;
    standard_enc_tables(T);
    std::vector<uint32_t> off((size_t)g.blocks + 1);
    uint32_t total = 0;
    for (int b = 0; b < g.blocks; b++) {
        const int prev = dc_predecessor(b, g.bpm), pred = prev >= 0 ? coef[(size_t)prev * 64] : 0;
        const int t = (g.bpm == 6 && (b % 6) >= 4) ? 1 : 0;
        BitCounter cnt;
        encode_block(&coef[(size_t)b * 64], pred, T.dc[t], T.ac[t], cnt);
        off[b] = total;
        total += cnt.total;
    }
    off[g.blocks] = total;
    std::vector<uint32_t> raw((total + 31) / 32 + 2, 0u);
    for (int b = g.blocks - 1; b >= 0; b--) {                               // any order must work
        const int prev = dc_predecessor(b, g.bpm), pred = prev >= 0 ? coef[(size_t)prev * 64] : 0;
        const int t = (g.bpm == 6 && (b % 6) >= 4) ? 1 : 0;
        BitSink sink;
        sink.init(raw.data(), off[b]);
        encode_block(&coef[(size_t)b * 64], pred, T.dc[t], T.ac[t], sink);
        sink.finish();
    }
    const std::vector<uint8_t> hdr = file_header(h, w, channels, ql, qc);
    std::vector<uint8_t> file(hdr);
    const uint32_t nbytes = (total + 7) / 8;
    for (uint32_t i = 0; i < nbytes; i++) {
        uint8_t v = (uint8_t)(raw[i >> 2] >> (24 - 8 * (i & 3)));
        if (i == nbytes - 1 && (total & 7)) v |= (uint8_t)(0xff >> (total & 7));
        file.push_back(v);
        if (v == 0xff) file.push_back(0);
    }
    file.push_back(0xFF);
    file.push_back(0xD9);
    if ((int64_t)file.size() <= cap) memcpy(out, file.data(), file.size());
    return (int64_t)file.size();
}

// -> 0, or the parse error; rounds_out (optional): the largest number of synchronisation rounds any window needed
// dc_kernel, idct_kernel, colour_kernel: everything after the entropy decoding
static int emu_finish(const DecImage &im, const FileInfo &F, std::vector<int16_t> &coef, std::vector<int16_t> &dcv, bool apply_dc,
                      uint8_t *rgb_out, uint8_t *gray_out, int16_t *coef_out)
{
    int py = 0, pcb = 0, pcr = 0;
    if (apply_dc)                                                           // dc_kernel (files without restart intervals)
        for (int mcu = 0; mcu < im.mcux * im.mcuy; mcu++) dc_apply_mcu(&dcv[(size_t)mcu * im.bpm], im.bpm, py, pcb, pcr);
    for (int g = 0; g < im.blocks; g++) coef[(size_t)g * 64] = dcv[(size_t)g];     // what idct_kernel does while staging a block
    if (coef_out) memcpy(coef_out, coef.data(), coef.size() * 2);
    std::vector<uint8_t> planes((size_t)im.yw * im.yh + 2 * (size_t)im.cw * im.ch);
    for (int g = 0; g < im.blocks; g++) {
        int pitch, comp;
        const int64_t off = block_dest(im, g, pitch, comp);
        alignas(16) int16_t nat[64], ws[64];
        for (int k = 0; k < 64; k++) nat[kZigzag[k]] = coef[(size_t)g * 64 + k];       // the kernel scatters while staging
        alignas(16) uint16_t qt[64];
        memcpy(qt, F.qt[comp ? 1 : 0], sizeof(qt));
        for (int j = 0; j < 4; j++) idct_cols(nat, qt, j, ws);
        for (int j = 0; j < 4; j++) idct_rows(ws, j, planes.data() + off, pitch);
    }
    for (int y = 0; y < im.h; y++)
        for (int x0 = 0; x0 < im.w; x0 += 8) {
            uint8_t o[24], single[3];
            pixels8_rgb(im, planes.data(), x0, y, o);                       // what the kernel runs
            for (int k = 0; k < 8 && x0 + k < im.w; k++) {
                const int x = x0 + k;
                if (gray_out) gray_out[(size_t)y * im.w + x] = planes[(size_t)y * im.yw + x];
                pixel_rgb(im, planes.data(), x, y, single);                 // the one-pixel statement of the same arithmetic
                if (memcmp(single, o + 3 * k, 3)) return -4;
                if (rgb_out) memcpy(rgb_out + ((size_t)y * im.w + x) * 3, o + 3 * k, 3);
            }
        }
    return 0;
}

extern "C" int v5jemu_decode(const uint8_t *data, int64_t len, uint8_t *rgb_out, uint8_t *gray_out, int16_t *coef_out, int *rounds_out)
{
    FileInfo *F = new FileInfo();
    const int rc = parse_file(data, (size_t)len, *F);
    if (rc) { delete F; return rc; }
    DecImage im;
    memset(&im, 0, sizeof(im));
    dec_geometry(im, F->h, F->w, F->ncomp, F->hs, F->vs);
    std::vector<uint8_t> stream;
    std::vector<uint32_t> rst_starts(1, 0u);                                // unstuff_kernel: where every restart interval begins
    for (size_t i = 0; i < F->scan_len; i++) {
        const uint8_t b = data[F->scan_off + i];
        const uint8_t prev = i > 0 ? data[F->scan_off + i - 1] : 0, next = i + 1 < F->scan_len ? data[F->scan_off + i + 1] : 0;
        if (b == 0 && prev == 0xFF) continue;
        if (F->restart && b == 0xFF && next >= 0xD0 && next <= 0xD7) continue;
        if (F->restart && prev == 0xFF && b >= 0xD0 && b <= 0xD7) {
            rst_starts.push_back((uint32_t)stream.size());
            continue;
        }
        stream.push_back(b);
    }
    const uint32_t total_bits = (uint32_t)stream.size() * 8;
    stream.resize(stream.size() + 32, 0);
    DecTabSet *T = new DecTabSet();
    for (int c = 0; c < 2; c++) { make_dec_table(F->dc[c], T->dc[c]); make_dec_table(F->ac[c], T->ac[c]); }
    std::vector<int16_t> coef((size_t)im.blocks * 64, 0);
    std::vector<uint32_t> staged(STAGE_WORDS, 0xA5A5A5A5u);
    HuffJob J;
    J.stream = stream.data();
    J.staged.words = staged.data();
    J.staged.base_word = 0;
    J.stream_words = (uint32_t)(stream.size() / 4);
    J.total_bits = total_bits;
    J.nsub = (total_bits + SUB_BITS - 1) / SUB_BITS;
    J.bpm = im.bpm;
    J.max_blocks = im.blocks;
    J.coef = coef.data();
    std::vector<int16_t> dcv((size_t)im.blocks, 0);
    J.dc = dcv.data();
    BlockHead *heads = new BlockHead();                                     // (all zero: what the kernels establish before the write pass)
    memset(heads, 0, sizeof(*heads));
    J.heads = heads;
#ifndef V5J_EMU_PARTS
#define V5J_EMU_PARTS 0
#endif
    if (F->restart > 0) {
        // ---- huffman_rst_kernel: one thread per restart interval, DC values written directly
        const int mcus = im.mcux * im.mcuy, n_int = (mcus + F->restart - 1) / F->restart;
        bool ok = (int)rst_starts.size() >= n_int;
        ByteStream bs;
        bs.data = stream.data();
        for (int k = n_int; k-- > 0 && ok;) {                               // any order: the intervals are independent threads
            const uint32_t p0 = rst_starts[(size_t)k] * 8u;
            uint32_t limit = total_bits;
            if (k + 1 < n_int && rst_starts[(size_t)k + 1] * 8u < limit) limit = rst_starts[(size_t)k + 1] * 8u;
            const int first_mcu = k * F->restart, n_mcu = mcus - first_mcu < F->restart ? mcus - first_mcu : F->restart;
            const int64_t block0 = (int64_t)first_mcu * im.bpm;
            ok = decode_interval(bs, p0, limit, *T, im.bpm, n_mcu * im.bpm, coef.data() + block0 * 64, dcv.data() + block0) == n_mcu * im.bpm;
        }
        if (rounds_out) *rounds_out = 0;
        const int rc2 = emu_finish(im, *F, coef, dcv, false, rgb_out, gray_out, coef_out);
        delete T; delete F; delete heads;
        return rc2 ? rc2 : (ok ? 0 : -3);
    }
#if V5J_EMU_PARTS == 0
    // ---- huffman_kernel: one CTA per file, windows in order, coefficients written window by window
    HuffWindow *W = new HuffWindow();
    memset(W, 0xA5, sizeof(*W));
    W->carry.p = 0; W->carry.c = 0; W->carry.z = 0;
    W->base_blocks = 0;
    int max_rounds = 0;
    for (uint32_t w0 = 0; w0 < J.nsub; w0 += HUFF_NT) {
        J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
        for (int t = 0; t < HUFF_NT; t++) stage_window(t, HUFF_NT, staged.data(), J.stream, J.staged.base_word, J.stream_words);
        for (int t = 0; t < HUFF_NT; t++) huff_phase_first(t, *W, J, *T, w0);
        for (int r = 1; r < HUFF_NT; r++) {
            for (int t = 0; t < HUFF_NT; t++) huff_phase_round(t, r, *W, J, *T, w0);
            bool all = true;
            for (int t = 0; t < HUFF_NT; t++) all = all && W->done[t];
            if (r > max_rounds) max_rounds = r;
            if (all) break;
        }
        uint32_t run = W->base_blocks;
        std::vector<uint32_t> b0(HUFF_NT);
        for (int t = 0; t < HUFF_NT; t++) {
            b0[t] = run;
            if (w0 + (uint32_t)t < J.nsub) run += W->info[t].n;
        }
        for (int t = HUFF_NT - 1; t >= 0; t--) huff_phase_write(t, *W, J, *T, w0, b0[t]);
        const uint32_t last = J.nsub - w0 < (uint32_t)HUFF_NT ? J.nsub - w0 - 1 : HUFF_NT - 1;
        W->carry = W->info[last].s;
        W->base_blocks = run;
    }
    const bool ok = W->base_blocks >= (uint32_t)im.blocks;
#else
    // ---- huffman_sync_kernel / huffman_fixup_kernel / huffman_write_kernel
    HuffWindow *W = new HuffWindow();
    int max_rounds = 0;
    // pass 1 (huffman_sync_kernel): the file's windows shared out among `parts` CTAs; part 0 starts true, the others blind
    std::vector<SubInfo> sub_info(J.nsub + 1);
    std::vector<uint32_t> sub_block0(J.nsub + 1, 0xA5A5A5A5u);
    const uint32_t windows = window_count(J.nsub), parts = part_count(J.nsub, V5J_EMU_PARTS);
    for (uint32_t q = parts; q-- > 0;) {                                    // any order: the parts are independent CTAs
        memset(W, 0xA5, sizeof(*W));
        const uint32_t w_first = part_first(q, parts, windows), w_end = part_first(q + 1, parts, windows);
        W->carry.p = w_first * (uint32_t)HUFF_NT * SUB_BITS; W->carry.c = 0; W->carry.z = 0;
        for (uint32_t w = w_first; w < w_end; w++) {
            const uint32_t w0 = w * (uint32_t)HUFF_NT;
            J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
            for (int t = 0; t < HUFF_NT; t++) stage_window(t, HUFF_NT, staged.data(), J.stream, J.staged.base_word, J.stream_words);
            for (int t = 0; t < HUFF_NT; t++) huff_phase_first(t, *W, J, *T, w0);
            for (int r = 1; r < HUFF_NT; r++) {
                for (int t = 0; t < HUFF_NT; t++) huff_phase_round(t, r, *W, J, *T, w0);
                bool all = true;
                for (int t = 0; t < HUFF_NT; t++) all = all && W->done[t];
                if (r > max_rounds) max_rounds = r;
                if (all) break;
            }
            for (int t = 0; t < HUFF_NT; t++)
                if (w0 + (uint32_t)t < J.nsub) sub_info[w0 + t] = W->info[t];
            const uint32_t last = J.nsub - w0 < (uint32_t)HUFF_NT ? J.nsub - w0 - 1 : HUFF_NT - 1;
            W->carry = W->info[last].s;
        }
    }
    // pass 2 (huffman_fixup_kernel): all boundary walks from the recorded states, then the in-order check, then the scan
    std::vector<SubState> started_from(parts + 1);
    auto bounds = [&](uint32_t q, uint32_t &j0, uint32_t &j_end) {
        j0 = part_first(q, parts, windows) * (uint32_t)HUFF_NT;
        j_end = part_first(q + 1, parts, windows) * (uint32_t)HUFF_NT;
        j_end = j_end < J.nsub ? j_end : J.nsub;
    };
    for (uint32_t q = 1; q < parts; q++) started_from[q] = sub_info[part_first(q, parts, windows) * (uint32_t)HUFF_NT - 1].s;
    for (uint32_t q = parts; q-- > 1;) {                                    // "concurrent": each from the state it saw at the start
        uint32_t j0, j_end;
        bounds(q, j0, j_end);
        SubInfo saved = sub_info[j0 - 1];
        sub_info[j0 - 1].s = started_from[q];
        fixup_walk(J.stream, J.total_bits, *T, J.bpm, sub_info.data(), j0, j_end);
        sub_info[j0 - 1] = saved;
    }
    for (uint32_t q = 1; q < parts; q++) {
        uint32_t j0, j_end;
        bounds(q, j0, j_end);
        if (!same_state(started_from[q], sub_info[j0 - 1].s)) fixup_walk(J.stream, J.total_bits, *T, J.bpm, sub_info.data(), j0, j_end);
    }
    uint32_t total_blocks = 0;
    for (uint32_t j = 0; j < J.nsub; j++) {
        sub_block0[j] = total_blocks;
        total_blocks += sub_info[j].n;
    }
    // pass 3 (huffman_write_kernel): one CTA per window
    for (uint32_t w = windows; w-- > 0;) {
        const uint32_t w0 = w * (uint32_t)HUFF_NT;
        J.staged.base_word = w0 * (uint32_t)SUB_WORDS;
        for (int t = 0; t < HUFF_NT; t++) stage_window(t, HUFF_NT, staged.data(), J.stream, J.staged.base_word, J.stream_words);
        for (int t = HUFF_NT - 1; t >= 0; t--) huff_write_sub(t, J, *T, w0, sub_info.data(), sub_block0.data());
    }
    const bool ok = total_blocks >= (uint32_t)im.blocks;
#endif
    if (rounds_out) *rounds_out = max_rounds;
    const int rc2 = emu_finish(im, *F, coef, dcv, true, rgb_out, gray_out, coef_out);
    bool heads_clean = true;                                                // every write pass must leave the block heads zeroed
    for (size_t i = 0; i < sizeof(BlockHead); i++) heads_clean = heads_clean && reinterpret_cast<const uint8_t *>(heads)[i] == 0;
    delete W; delete T; delete F; delete heads;
    return rc2 ? rc2 : (ok ? (heads_clean ? 0 : -4) : -3);
}

extern "C" int v5jemu_info(const uint8_t *data, int64_t len, int *h, int *w, int *ncomp)
{
    FileInfo *F = new FileInfo();
    const int rc = parse_file(data, (size_t)len, *F);
    if (!rc) { *h = F->h; *w = F->w; *ncomp = F->ncomp; }
    delete F;
    return rc;
}

// huff_action of the decoder table built from (bits, vals) for `count` 32-bit windows; returns the table's long_base
// (0x10000 = the long codes are walked), -1 for a table make_dec_table refuses.
extern "C" int v5jemu_huff_actions(const uint8_t *bits, const uint8_t *vals, int nvals, int is_dc, const uint32_t *windows, int count, uint32_t *actions)
{
    DecTable *t = new DecTable();
    if (!make_dec_table(bits, vals, nvals, is_dc != 0, *t)) { delete t; return -1; }
    for (int i = 0; i < count; i++) actions[i] = huff_action(*t, windows[i]);
    const int lb = (int)t->long_base;
    delete t;
    return lb;
}
