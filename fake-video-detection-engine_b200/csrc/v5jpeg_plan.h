// v5jpeg_plan.h — the decoder's launch plan: every file parsed once, table sets de-duplicated, the batch cut into chunks, each
// chunk's staging layout, upload runs, workspace sizes and Huffman path, all decided on the host before anything touches the
// device. Host only, no CUDA runtime calls: shared by both decode entry points (v5jpeg.cu) and the CPU emulator (tests/emu).
#pragma once
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "v5ela.h"
#include "v5jpeg_common.h"
#include "v5jpeg_dec.cuh"

namespace v5j {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Host-side helper threads for header parsing and the staging copy of large batches (a 1080p file is ~0.5 MB): up to `threads`
// of them, and none below 4 MB of work.
template <class Fn>
void parallel_for(int n, size_t bytes_hint, int threads, Fn fn)
{
    const int nt = threads > n ? n : threads;
    if (nt <= 1 || bytes_hint < ((size_t)4 << 20)) {
        for (int i = 0; i < n; i++) fn(i);
        return;
    }
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; t++)
        pool.emplace_back([=]() {
            for (int i = t; i < n; i += nt) fn(i);
        });
    for (auto &th : pool) th.join();
}

// One decode call as the caller gives it.
struct DecodeCall {
    const uint8_t *const *files = nullptr;
    const int64_t *lens = nullptr;
    int n = 0;
    const int64_t *rgb_offsets = nullptr, *gray_offsets = nullptr;   // output positions (bytes); null = tightly packed in file order
    bool want_rgb = false, want_gray = false;
    bool all_pinned = false;   // the first and last byte of every file are page-locked: files are uploaded from where they are
    int sm_count = 0;
    int huff_path = 0;         // 0: chosen per chunk; 1: the one-launch Huffman path; 3: the three-launch path
    int huff_parts = 0;        // parts per file of the three-launch path, 1..16; anything else: chosen per chunk
    int threads = 1;           // helper threads (parallel_for)
    size_t chunk_bytes = 0;    // workspace per chunk: streams, coefficients and planes stay under it
    // Coefficients only (v5ela_jpeg_dct_stats): the decode stops after dc_kernel and the DCT statistics kernels run instead
    // of the inverse DCT and colour conversion; no sample planes. want_map adds the double-compression map, file i's at
    // element offset map_offsets[i] (null = packed in file order).
    bool coef_only = false, want_map = false;
    const int64_t *map_offsets = nullptr;
};

// One host-to-device copy of pinned file bytes: `bytes` from `src` to `dev_off` inside the chunk's staging buffer.
struct UploadRun {
    size_t dev_off;
    const uint8_t *src;
    size_t bytes;
};

// One chunk of files, decoded by one launch sequence.
struct DecChunk {
    std::vector<DecImage> images;              // as uploaded: scan_off is relative to the staging buffer
    std::vector<int> file_index;               // the file of each image: consecutive files, in file order
    std::vector<int64_t> map_off;              // coefficient-only calls with a map: where each image's map starts (elements)
    // staging layout: descriptors (off_img) | table sets | quantisation tables | map offsets (coefficient-only calls with a
    // map, one int64 per image) | scan segments
    size_t off_img = 0, off_tab = 0, off_q = 0, off_map = 0, off_scan = 0;
    size_t stage_bytes = 0;                    // the device staging buffer
    size_t host_stage_bytes = 0;               // what goes through the pinned host staging buffer (all of it for pageable files)
    std::vector<UploadRun> runs;               // pinned files: copied from the caller's memory, one run per group of close files
    // workspace
    size_t scan_bytes = 0, stream_bytes = 0, coef_blocks = 0, plane_bytes = 0, subs = 0;
    size_t rst_entries = 0;                    // interval starts of the files with restart markers
    uint32_t max_windows = 1;
    int max_intervals = 0;
    int max_blocks = 0;
    int max_luma_blocks = 0;                   // real luma blocks of the largest image (coefficient-only calls)
    int64_t max_groups = 0;                    // 8-pixel groups of the largest image
    // Huffman decoding: one CTA per file in one launch, or a file's windows shared out among `parts` CTAs in three launches
    bool one_launch = true;
    unsigned parts = 1;
    int launches = 0;                          // kernel launches of the chunk
};

struct DecodePlan {
    int status = V5ELA_OK;                     // V5ELA_OK, or why the call is refused ...
    const char *error = "";
    int bad_file = -1;                         // ... and the file it is refused for (-1: none named)
    std::vector<FileInfo> info;                // per file
    std::vector<DecTabSet> tabsets;            // the distinct Huffman table sets of the call (usually one)
    std::vector<std::vector<uint16_t>> qsets;  // the distinct quantisation table pairs (2 x 64 entries)
    std::vector<DecChunk> chunks;
};

inline void refuse(DecodePlan &P, int status, const char *error, int file)
{
    P.status = status;
    P.error = error;
    P.bad_file = file;
}

// Plans call c into P. P.status says whether the call can go ahead; nothing is planned past a refusal.
inline void plan_decode(const DecodeCall &c, DecodePlan &P)
{
    const int n = c.n;
    P = DecodePlan();
    // ---- parse every file; unique Huffman table sets and quantisation table pairs
    size_t total_len = 0;
    for (int i = 0; i < n; i++) {
        if (!c.files[i] || c.lens[i] <= 0) return refuse(P, V5ELA_ERR_INVALID, "null or empty file", -1);
        total_len += (size_t)c.lens[i];
    }
    P.info.resize((size_t)n);
    std::vector<int> tab_of((size_t)n), q_of((size_t)n), parse_rc((size_t)n);
    parallel_for(n, total_len, c.threads, [&](int i) { parse_rc[(size_t)i] = parse_file(c.files[i], (size_t)c.lens[i], P.info[(size_t)i]); });
    std::vector<HuffSpecSet> specsets;         // decoder tables are built for these only
    for (int i = 0; i < n; i++) {
        const int prc = parse_rc[(size_t)i];
        if (prc == JPEG_UNSUPPORTED)
            return refuse(P, V5ELA_ERR_UNSUPPORTED, "not an 8-bit baseline one-component / 4:2:0 / 4:2:2 / 4:4:4 JPEG", i);
        if (prc != JPEG_OK) return refuse(P, V5ELA_ERR_INVALID, "corrupt JPEG headers", i);
        if (P.info[(size_t)i].scan_len >= kMaxScanBytes)
            return refuse(P, V5ELA_ERR_UNSUPPORTED, "entropy-coded segment of 2^29 - 2^20 bytes or more", i);
        if ((c.rgb_offsets && c.rgb_offsets[i] < 0) || (c.gray_offsets && c.gray_offsets[i] < 0) ||
            (c.want_map && c.map_offsets && c.map_offsets[i] < 0))
            return refuse(P, V5ELA_ERR_INVALID, "negative output offset", i);
        const FileInfo &F = P.info[(size_t)i];
        HuffSpecSet ts;                        // (HuffSpec has no padding bytes and parse_file zeroes what it does not fill)
        ts.dc[0] = F.dc[0]; ts.dc[1] = F.dc[1]; ts.ac[0] = F.ac[0]; ts.ac[1] = F.ac[1];
        int found = -1;
        for (size_t k = specsets.size(); k-- > 0 && found < 0;)
            if (!memcmp(&specsets[k], &ts, sizeof(ts))) found = (int)k;
        if (found < 0) { specsets.push_back(ts); found = (int)specsets.size() - 1; }
        tab_of[(size_t)i] = found;
        std::vector<uint16_t> q(128);
        memcpy(q.data(), F.qt[0], 128);
        memcpy(q.data() + 64, F.qt[1], 128);
        found = -1;
        for (size_t k = 0; k < P.qsets.size() && found < 0; k++)
            if (P.qsets[k] == q) found = (int)k;
        if (found < 0) { P.qsets.push_back(q); found = (int)P.qsets.size() - 1; }
        q_of[(size_t)i] = found;
    }
    P.tabsets.resize(specsets.size());
    for (size_t k = 0; k < specsets.size(); k++) make_tabset(specsets[k], P.tabsets[k]);   // (parse_file has validated every table)

    // ---- chunks of files whose workspace stays under c.chunk_bytes (a 1080p file needs ~11 MB: coefficients, planes, streams)
    P.chunks.resize(1);
    int64_t rgb_run = 0, gray_run = 0, map_run = 0;
    for (int i = 0; i < n; i++) {
        const FileInfo &F = P.info[(size_t)i];
        DecImage im;
        memset(&im, 0, sizeof(im));
        dec_geometry(im, F.h, F.w, F.ncomp, F.hs, F.vs);
        im.tabset = tab_of[(size_t)i];
        im.qt = q_of[(size_t)i];
        const size_t planes = c.coef_only ? 0 : (size_t)im.yw * im.yh + 2 * (size_t)im.cw * im.ch;
        const size_t need = F.scan_len * 2 + (size_t)im.blocks * 128 + planes + 256;
        DecChunk *C = &P.chunks.back();
        if (!C->images.empty() && (C->scan_bytes * 2 + C->coef_blocks * 128 + C->plane_bytes + need > c.chunk_bytes || C->images.size() >= 65535)) {
            P.chunks.emplace_back();
            C = &P.chunks.back();
        }
        // Pinned files that follow each other in host memory keep their relative distance on the device, so that the whole run
        // goes up in one copy — which also copies the bytes between two scan segments: the next file's header (its first and
        // last byte are known to be pinned, see all_pinned) and the padding between the files, which is only accepted when it is
        // shorter than a page: every byte of it then shares a page with a byte of one of the two files, so the copy can touch
        // neither unmapped nor foreign memory. Files further apart get a copy of their own. scan_bytes = end of the used scan area.
        size_t start = align_up(C->scan_bytes, 16);
        const uint8_t *cur = c.files[i] + F.scan_off;
        bool contig = false;
        if (c.all_pinned && !C->images.empty()) {
            const int pi = C->file_index.back();
            const uint8_t *prev_end = c.files[pi] + P.info[(size_t)pi].scan_off + P.info[(size_t)pi].scan_len;
            const uint8_t *prev_file_end = c.files[pi] + c.lens[pi];
            if (cur >= prev_end && c.files[i] >= prev_file_end && (size_t)(c.files[i] - prev_file_end) < 4096) {
                contig = true;
                start = (size_t)(C->images.back().scan_off + C->images.back().scan_len) + (size_t)(cur - prev_end);
            }
        }
        if (contig) C->runs.back().bytes = start + F.scan_len - C->runs.back().dev_off;
        else if (c.all_pinned) C->runs.push_back({start, cur, F.scan_len});
        im.scan_off = (int64_t)start;          // relative to the scan area of the staging buffer (fixed up below)
        im.scan_len = (int64_t)F.scan_len;
        im.stream_off = (int64_t)C->stream_bytes;
        im.coef_off = (int64_t)C->coef_blocks;
        im.sub_off = (int64_t)C->subs;
        const size_t nsub_max = (F.scan_len * 8 + SUB_BITS - 1) / SUB_BITS + 1;
        C->subs += nsub_max;
        const uint32_t wmax = (uint32_t)((nsub_max + HUFF_NT - 1) / HUFF_NT);
        if (wmax > C->max_windows) C->max_windows = wmax;
        if (F.restart > 0) {                   // restart intervals: one start position per interval
            const int n_int = (im.mcux * im.mcuy + F.restart - 1) / F.restart;
            im.restart = F.restart;
            im.rst_off = (int32_t)C->rst_entries;
            C->rst_entries += (size_t)n_int;
            if (n_int > C->max_intervals) C->max_intervals = n_int;
        }
        im.plane_off = (int64_t)C->plane_bytes;
        im.rgb_off = c.want_rgb ? (c.rgb_offsets ? c.rgb_offsets[i] : rgb_run) : -1;
        im.gray_off = c.want_gray ? (c.gray_offsets ? c.gray_offsets[i] : gray_run) : -1;
        rgb_run += (int64_t)F.h * F.w * 3;
        gray_run += (int64_t)F.h * F.w;
        const int luma_blocks = ((F.h + 7) / 8) * ((F.w + 7) / 8);
        if (c.want_map) C->map_off.push_back(c.map_offsets ? c.map_offsets[i] : map_run);
        map_run += luma_blocks;
        if (luma_blocks > C->max_luma_blocks) C->max_luma_blocks = luma_blocks;
        C->scan_bytes = start + F.scan_len;
        C->stream_bytes += align_up(F.scan_len + 32, 16);
        C->coef_blocks += (size_t)im.blocks;
        C->plane_bytes += align_up(planes, 16);
        if (im.blocks > C->max_blocks) C->max_blocks = im.blocks;
        if ((int64_t)F.h * ((F.w + 7) / 8) > C->max_groups) C->max_groups = (int64_t)F.h * ((F.w + 7) / 8);
        C->images.push_back(im);
        C->file_index.push_back(i);
    }

    for (DecChunk &C : P.chunks) {
        const int cn = (int)C.images.size();
        C.off_img = 0;
        C.off_tab = align_up(sizeof(DecImage) * (size_t)cn, 16);
        C.off_q = C.off_tab + align_up(sizeof(DecTabSet) * P.tabsets.size(), 16);
        C.off_map = C.off_q + align_up(256 * P.qsets.size(), 16);
        C.off_scan = C.off_map + (c.want_map ? align_up(sizeof(int64_t) * (size_t)cn, 16) : 0);
        C.stage_bytes = C.off_scan + align_up(C.scan_bytes, 16);
        // Files in pinned (page-locked) host memory are copied to the device straight from where they are — the caller keeps
        // them alive until the stream has been synchronised; pageable files go through the handle's pinned staging buffer.
        C.host_stage_bytes = c.all_pinned ? C.off_scan : C.stage_bytes;
        for (DecImage &im : C.images) im.scan_off += (int64_t)C.off_scan;
        for (UploadRun &r : C.runs) r.dev_off += C.off_scan;
        // Huffman decoding in three launches: synchronisation (the windows of a file shared out among `parts` CTAs so that a
        // small batch still fills the GPU), boundary fix-up + block offsets, then one CTA per window writes coefficients.
        // (a batch of at least one file per SM gains nothing from splitting files: parts = 1, no blind starts, no fix-up walks)
        unsigned parts = (unsigned)(c.sm_count / cn);
        parts = parts < 1 ? 1 : (parts > 16 ? 16 : parts);
        parts = parts > C.max_windows ? C.max_windows : parts;
        if (c.huff_parts >= 1 && c.huff_parts <= 16) parts = (unsigned)c.huff_parts > C.max_windows ? C.max_windows : (unsigned)c.huff_parts;
        C.parts = parts;
        // nothing to gain from splitting when there is no room for two parts per file, or no file has more than one window
        C.one_launch = c.huff_path ? c.huff_path == 1 : (c.sm_count / cn < 2 || C.max_windows < 2);
        // unstuff, Huffman (1 or 3), dc, then idct + colour, or the statistics: histogram (+ tables and map)
        C.launches = (C.one_launch ? 3 : 5) + (C.max_intervals > 0 ? 1 : 0) + (c.coef_only ? (c.want_map ? 3 : 1) : 2);
    }
}

}  // namespace v5j
