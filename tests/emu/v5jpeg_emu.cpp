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
#include "v5jpeg_plan.h"

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

// parts: 0 = huffman_kernel (one CTA per file), otherwise the three-launch flow with the file's windows shared out among up to
// `parts` CTAs (the plan's DecChunk::one_launch / parts)
extern "C" int v5jemu_decode(const uint8_t *data, int64_t len, uint8_t *rgb_out, uint8_t *gray_out, int16_t *coef_out, int *rounds_out,
                             int parts_wanted)
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
    HuffWindow *W = new HuffWindow();
    int max_rounds = 0;
    bool ok;
    if (parts_wanted == 0) {
        // ---- huffman_kernel: one CTA per file, windows in order, coefficients written window by window
        memset(W, 0xA5, sizeof(*W));
        W->carry.p = 0; W->carry.c = 0; W->carry.z = 0;
        W->base_blocks = 0;
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
        ok = W->base_blocks >= (uint32_t)im.blocks;
    } else {
        // ---- huffman_sync_kernel / huffman_fixup_kernel / huffman_write_kernel
        // pass 1 (huffman_sync_kernel): the file's windows shared out among `parts` CTAs; part 0 starts true, the others blind
        std::vector<SubInfo> sub_info(J.nsub + 1);
        std::vector<uint32_t> sub_block0(J.nsub + 1, 0xA5A5A5A5u);
        const uint32_t windows = window_count(J.nsub), parts = part_count(J.nsub, (uint32_t)parts_wanted);
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
        ok = total_blocks >= (uint32_t)im.blocks;
    }
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

// The decoder's plan of a call (v5j::plan_decode) as the library makes it, summarised for the tests. Returns the plan's status;
// *n_chunks, *bad_file. Per chunk k (up to max_chunks), chunk_rows[PLAN_ROW * k ..]:
//   files, first file, off_tab, off_q, off_scan, stage_bytes, host_stage_bytes, upload runs, scan_bytes, stream_bytes, coef_blocks,
//   plane_bytes, subs, rst_entries, max_windows, max_intervals, max_blocks, max_groups, one_launch, parts, launches,
//   hash of the DecImage table, hash of the upload runs (host addresses relative to files[0])
// Per file i, file_rows[FILE_ROW * i ..]: chunk, position in the chunk, tabset, qt, rgb_off, gray_off, scan_off, rst_off.
// Per upload run (up to max_runs; *n_runs counts them all), run_rows[4 * r ..]: chunk, device offset, host address - files[0], bytes.
constexpr int PLAN_ROW = 23, FILE_ROW = 8;

static uint64_t fnv(uint64_t hsh, int64_t v)
{
    for (int b = 0; b < 8; b++) hsh = (hsh ^ (uint8_t)((uint64_t)v >> (8 * b))) * 0x100000001b3ull;
    return hsh;
}

extern "C" int v5jemu_plan_decode(const uint8_t *const *files, const int64_t *lens, int n, const int64_t *rgb_offsets,
                                  const int64_t *gray_offsets, int want_rgb, int want_gray, int all_pinned, int sm_count, int huff_path,
                                  int huff_parts, int64_t chunk_bytes, int64_t *chunk_rows, int max_chunks, int64_t *file_rows,
                                  int64_t *run_rows, int max_runs, int *n_chunks, int *n_runs, int *bad_file)
{
    v5j::DecodeCall c;
    c.files = files;
    c.lens = lens;
    c.n = n;
    c.rgb_offsets = rgb_offsets;
    c.gray_offsets = gray_offsets;
    c.want_rgb = want_rgb != 0;
    c.want_gray = want_gray != 0;
    c.all_pinned = all_pinned != 0;
    c.sm_count = sm_count;
    c.huff_path = huff_path;
    c.huff_parts = huff_parts;
    c.threads = 4;
    c.chunk_bytes = (size_t)chunk_bytes;
    v5j::DecodePlan *P = new v5j::DecodePlan();
    v5j::plan_decode(c, *P);
    *bad_file = P->bad_file;
    *n_chunks = (int)P->chunks.size();
    *n_runs = 0;
    const intptr_t base = n > 0 ? reinterpret_cast<intptr_t>(files[0]) : 0;
    for (size_t k = 0; P->status == V5ELA_OK && k < P->chunks.size(); k++) {
        const v5j::DecChunk &C = P->chunks[k];
        uint64_t h_img = 0xcbf29ce484222325ull, h_run = 0xcbf29ce484222325ull;
        for (size_t j = 0; j < C.images.size(); j++) {
            const DecImage &im = C.images[j];
            for (int64_t v : {(int64_t)im.h, (int64_t)im.w, (int64_t)im.ncomp, (int64_t)im.hs, (int64_t)im.vs, (int64_t)im.mcux, (int64_t)im.mcuy,
                              (int64_t)im.bpm, (int64_t)im.blocks, (int64_t)im.restart, (int64_t)im.rst_off, (int64_t)im.tabset, (int64_t)im.qt,
                              (int64_t)im.yw, (int64_t)im.yh, (int64_t)im.cw, (int64_t)im.ch, im.scan_off, im.scan_len, im.stream_off, im.coef_off,
                              im.sub_off, im.plane_off, im.rgb_off, im.gray_off})
                h_img = fnv(h_img, v);
            int64_t *f = file_rows + (size_t)FILE_ROW * C.file_index[j];
            const int64_t row[FILE_ROW] = {(int64_t)k, (int64_t)j, im.tabset, im.qt, im.rgb_off, im.gray_off, im.scan_off, im.rst_off};
            memcpy(f, row, sizeof(row));
        }
        for (const v5j::UploadRun &r : C.runs) {
            const int64_t rel = (int64_t)(reinterpret_cast<intptr_t>(r.src) - base);
            h_run = fnv(fnv(fnv(h_run, (int64_t)r.dev_off), rel), (int64_t)r.bytes);
            if (*n_runs < max_runs) {
                const int64_t row[4] = {(int64_t)k, (int64_t)r.dev_off, rel, (int64_t)r.bytes};
                memcpy(run_rows + 4 * (size_t)*n_runs, row, sizeof(row));
            }
            ++*n_runs;
        }
        if ((int)k >= max_chunks) continue;
        const int64_t row[PLAN_ROW] = {(int64_t)C.images.size(), C.file_index[0], (int64_t)C.off_tab, (int64_t)C.off_q, (int64_t)C.off_scan,
                                       (int64_t)C.stage_bytes, (int64_t)C.host_stage_bytes, (int64_t)C.runs.size(), (int64_t)C.scan_bytes,
                                       (int64_t)C.stream_bytes, (int64_t)C.coef_blocks, (int64_t)C.plane_bytes, (int64_t)C.subs,
                                       (int64_t)C.rst_entries, C.max_windows, C.max_intervals, C.max_blocks, C.max_groups, C.one_launch,
                                       C.parts, C.launches, (int64_t)(h_img >> 1), (int64_t)(h_run >> 1)};
        memcpy(chunk_rows + (size_t)PLAN_ROW * k, row, sizeof(row));
    }
    const int rc = P->status;
    delete P;
    return rc;
}
