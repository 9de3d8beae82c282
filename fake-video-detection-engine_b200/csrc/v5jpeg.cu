// v5jpeg.cu — codec rows of libv5ela.so (SURVEY.md §8f-2 decode, §8f-3 encode): C-ABI entry points v5ela_jpeg_*.
// Kernels: v5jpeg_enc.cuh, v5jpeg_dec.cuh. Host-side header writing / parsing: v5jpeg_common.h.
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

#include "v5ela.h"
#include "v5ela_handle.h"
#include "v5ela_host.h"
#include "v5jpeg_common.h"
#include "v5jpeg_enc.cuh"
#include "v5jpeg_dec.cuh"

using namespace v5host;

struct v5jpeg_state {
    // encoder
    v5j::EncTables *d_enc_tabs = nullptr;
    uint8_t *d_header = nullptr;
    void *d_coef = nullptr, *d_bitoff = nullptr, *d_total = nullptr, *d_raw = nullptr;
    size_t coef_cap = 0, bitoff_cap = 0, total_cap = 0, raw_cap = 0;
    // host-buffer entry points
    uint8_t *d_img = nullptr, *d_out = nullptr;
    int32_t *d_sizes = nullptr;
    size_t img_cap = 0, out_cap = 0, sizes_cap = 0;
    // decoder: one pinned staging buffer (descriptors | table sets | quantisation tables | scan segments) mirrored on the
    // device, plus the per-batch workspace (unstuffed streams, coefficients, sample planes)
    // Two of each, used alternately: the upload of one batch (on upload_stream) overlaps the kernels of the previous one.
    uint8_t *stage_host[2] = {nullptr, nullptr}, *d_stage[2] = {nullptr, nullptr};
    size_t stage_host_cap[2] = {0, 0}, stage_cap[2] = {0, 0};
    cudaEvent_t uploaded[2] = {nullptr, nullptr};   // the upload into d_stage[b] (and out of stage_host[b]) has completed
    cudaEvent_t consumed[2] = {nullptr, nullptr};   // the kernels that read d_stage[b] have completed
    cudaStream_t upload_stream = nullptr;
    int toggle = 0;
    void *d_streams = nullptr, *d_dcoef = nullptr, *d_planes = nullptr, *d_bits = nullptr, *d_status = nullptr, *d_dc = nullptr;
    void *d_sub_info = nullptr, *d_sub_block0 = nullptr, *d_rst = nullptr;
    size_t rst_cap = 0;
    size_t streams_cap = 0, dcoef_cap = 0, planes_cap = 0, bits_cap = 0, status_cap = 0, dc_cap = 0, sub_info_cap = 0, sub_block0_cap = 0;
    uint8_t *d_dec_rgb = nullptr, *d_dec_gray = nullptr;
    int32_t *d_dec_status = nullptr;
    size_t dec_rgb_cap = 0, dec_gray_cap = 0, dec_status_cap = 0;
};

void v5jpeg_release(v5ela_handle *h)
{
    v5jpeg_state *s = h->jpeg;
    if (!s) return;
    cudaFree(s->d_enc_tabs);
    cudaFree(s->d_header);
    cudaFree(s->d_coef);
    cudaFree(s->d_bitoff);
    cudaFree(s->d_total);
    cudaFree(s->d_raw);
    cudaFree(s->d_img);
    cudaFree(s->d_out);
    cudaFree(s->d_sizes);
    for (int b = 0; b < 2; b++) {
        if (s->stage_host[b]) cudaFreeHost(s->stage_host[b]);
        if (s->uploaded[b]) cudaEventDestroy(s->uploaded[b]);
        if (s->consumed[b]) cudaEventDestroy(s->consumed[b]);
        cudaFree(s->d_stage[b]);
    }
    if (s->upload_stream) cudaStreamDestroy(s->upload_stream);
    cudaFree(s->d_streams);
    cudaFree(s->d_dcoef);
    cudaFree(s->d_planes);
    cudaFree(s->d_bits);
    cudaFree(s->d_status);
    cudaFree(s->d_dc);
    cudaFree(s->d_sub_info);
    cudaFree(s->d_sub_block0);
    cudaFree(s->d_rst);
    cudaFree(s->d_dec_rgb);
    cudaFree(s->d_dec_gray);
    cudaFree(s->d_dec_status);
    delete s;
    h->jpeg = nullptr;
}

namespace {

int jpeg_state(v5ela_handle *h, v5jpeg_state **out)
{
    if (!h->jpeg) {
        h->jpeg = new (std::nothrow) v5jpeg_state();
        if (!h->jpeg) return fail(h, V5ELA_ERR_NOMEM, "v5ela_jpeg: out of host memory%s");
    }
    *out = h->jpeg;
    return 0;
}

constexpr int kHeaderMax = 1024;

}  // namespace

extern "C" {

int64_t v5ela_jpeg_bound(int height, int width, int channels)
{
    if (height <= 0 || width <= 0 || (channels != 1 && channels != 3)) return V5ELA_ERR_INVALID;
    // worst case per block: DC 9 + 11 bits, 63 x (16 + 10) bits, every byte stuffed
    return (int64_t)v5j::enc_geo(height, width, channels).blocks * 416 + kHeaderMax;
}

static int v5ela_jpeg_encode_impl(v5ela_handle *h, const uint8_t *d_img, int n, int height, int width, int channels,
                      int64_t frame_stride_bytes, int64_t row_stride_bytes, int quality, uint8_t *d_out,
                      int64_t out_stride_bytes, int32_t *d_sizes, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!d_img || !d_out || !d_sizes || n < 0 || height <= 0 || width <= 0 || height > 65535 || width > 65535 ||
        (channels != 1 && channels != 3) || quality < 1 || quality > 100 || row_stride_bytes < (int64_t)width * channels ||
        (n > 1 && frame_stride_bytes < row_stride_bytes * (int64_t)height) || out_stride_bytes < kHeaderMax ||
        out_stride_bytes > (int64_t)1 << 30)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_encode: bad pointer, size, stride, channel count or quality%s");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // the codec workspace is handle-owned
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;

    const v5j::EncGeo g = v5j::enc_geo(height, width, channels);
    uint16_t ql[64], qc[64];
    v5plan::quant_tables(quality, ql, qc);
    const std::vector<uint8_t> header = v5j::file_header(height, width, channels, ql, qc);
    if (!s->d_enc_tabs) {
        v5j::EncTables tabs;
        v5j::standard_enc_tables(tabs);
        V5_CUDA(h, cudaMalloc(&s->d_enc_tabs, sizeof(tabs)));
        V5_CUDA(h, cudaMemcpyAsync(s->d_enc_tabs, &tabs, sizeof(tabs), cudaMemcpyHostToDevice, st));
        V5_CUDA(h, cudaMalloc(&s->d_header, kHeaderMax));
    }
    V5_CUDA(h, cudaMemcpyAsync(s->d_header, header.data(), header.size(), cudaMemcpyHostToDevice, st));

    // images per pass: keep the workspace (coefficients 128 B/block, offsets, unstuffed stream) under ~8 GiB (one pass for a
    // few hundred 1080p frames: the per-image-CTA kernels cost the same for 8 images as for 148)
    const int64_t raw_words = (out_stride_bytes + 3) / 4;
    const size_t per_image = (size_t)g.blocks * (128 + 4) + (size_t)raw_words * 4 + 16;
    int chunk = (int)(((size_t)8 << 30) / per_image);
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    if (chunk > 65535) chunk = 65535;
    if ((rc = ensure(h, &s->d_coef, &s->coef_cap, (size_t)chunk * g.blocks * 128))) return rc;
    if ((rc = ensure(h, &s->d_bitoff, &s->bitoff_cap, (size_t)chunk * g.blocks * 4))) return rc;
    if ((rc = ensure(h, &s->d_total, &s->total_cap, (size_t)chunk * 4))) return rc;
    if ((rc = ensure(h, &s->d_raw, &s->raw_cap, (size_t)chunk * raw_words * 4))) return rc;

    v5j::CoefParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.frame_stride = frame_stride_bytes;
    cp.row_stride = row_stride_bytes;
    cp.coef = static_cast<int16_t *>(s->d_coef);
    cp.g = g;
    v5j::make_enc_quant(ql, cp.q[0]);
    v5j::make_enc_quant(qc, cp.q[1]);
    const int per_strip = channels == 3 ? v5j::ENC_TM : v5j::ENC_BLOCKS;
    const unsigned tiles_x = (unsigned)((g.mcux + per_strip - 1) / per_strip);

    for (int f0 = 0; f0 < n; f0 += chunk) {
        const int fn = f0 + chunk <= n ? chunk : n - f0;
        cp.img = d_img + (int64_t)f0 * frame_stride_bytes;
        v5j::coef_kernel<<<dim3(tiles_x, (unsigned)g.mcuy, (unsigned)fn), v5j::ENC_NT, 0, st>>>(cp);
        V5_CUDA(h, cudaGetLastError());
        v5j::EntropyParams ep;
        ep.coef = cp.coef;
        ep.bitoff = static_cast<uint32_t *>(s->d_bitoff);
        ep.total_bits = static_cast<uint32_t *>(s->d_total);
        ep.raw = static_cast<uint32_t *>(s->d_raw);
        ep.raw_words = raw_words;
        ep.blocks = g.blocks;
        ep.bpm = g.bpm;
        ep.n = fn;
        const dim3 eg((unsigned)((g.blocks + 127) / 128), (unsigned)fn);
        v5j::entropy_kernel<false><<<eg, 128, 0, st>>>(ep, s->d_enc_tabs);
        V5_CUDA(h, cudaGetLastError());
        v5j::scan_kernel<<<fn, 1024, 0, st>>>(ep);
        V5_CUDA(h, cudaGetLastError());
        V5_CUDA(h, cudaMemsetAsync(s->d_raw, 0, (size_t)fn * raw_words * 4, st));
        v5j::entropy_kernel<true><<<eg, 128, 0, st>>>(ep, s->d_enc_tabs);
        V5_CUDA(h, cudaGetLastError());
        v5j::StuffParams sp;
        sp.raw = ep.raw;
        sp.raw_words = raw_words;
        sp.total_bits = ep.total_bits;
        sp.header = s->d_header;
        sp.header_len = (int)header.size();
        sp.out = d_out + (int64_t)f0 * out_stride_bytes;
        sp.out_stride = out_stride_bytes;
        sp.sizes = d_sizes + f0;
        v5j::stuff_kernel<<<fn, 1024, 0, st>>>(sp);
        V5_CUDA(h, cudaGetLastError());
        h->launches += 5;
    }
    return V5ELA_OK;
}

static int v5ela_jpeg_encode_host_impl(v5ela_handle *h, const uint8_t *img_host, int n, int height, int width, int channels, int quality,
                           uint8_t *out_host, int64_t out_stride_bytes, int32_t *sizes_host)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!img_host || !out_host || !sizes_host || n < 0 || height <= 0 || width <= 0 || (channels != 1 && channels != 3) ||
        out_stride_bytes < kHeaderMax)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_encode_host: bad pointer, size or channel count%s");
    DeviceGuard guard(h->device);
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;
    if (!h->own_stream) V5_CUDA(h, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    cudaStream_t st = h->own_stream;
    const size_t fbytes = (size_t)height * width * channels;
    if ((rc = ensure(h, (void **)&s->d_img, &s->img_cap, fbytes * n))) return rc;
    if ((rc = ensure(h, (void **)&s->d_out, &s->out_cap, (size_t)out_stride_bytes * n))) return rc;
    if ((rc = ensure(h, (void **)&s->d_sizes, &s->sizes_cap, sizeof(int32_t) * (size_t)n))) return rc;
    V5_CUDA(h, cudaMemcpyAsync(s->d_img, img_host, fbytes * n, cudaMemcpyHostToDevice, st));
    rc = v5ela_jpeg_encode(h, s->d_img, n, height, width, channels, (int64_t)fbytes, (int64_t)width * channels, quality,
                           s->d_out, out_stride_bytes, s->d_sizes, st);
    if (rc) return rc;
    V5_CUDA(h, cudaMemcpyAsync(sizes_host, s->d_sizes, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    V5_CUDA(h, cudaStreamSynchronize(st));
    for (int i = 0; i < n; i++) {                               // only the bytes that make up each file come back
        const int64_t sz = sizes_host[i] <= out_stride_bytes ? sizes_host[i] : 0;
        if (sz) V5_CUDA(h, cudaMemcpyAsync(out_host + (int64_t)i * out_stride_bytes, s->d_out + (int64_t)i * out_stride_bytes,
                                           (size_t)sz, cudaMemcpyDeviceToHost, st));
    }
    V5_CUDA(h, cudaStreamSynchronize(st));
    return V5ELA_OK;
}


// ---------------------------------------------------------------------------------------------------------- decode
int v5ela_jpeg_info(const uint8_t *file_host, int64_t len, int *height, int *width, int *channels)
{
    if (!file_host || len <= 0 || !height || !width || !channels) return V5ELA_ERR_INVALID;
    v5j::FileInfo *F = new (std::nothrow) v5j::FileInfo();
    if (!F) return V5ELA_ERR_NOMEM;
    const int rc = v5j::parse_file(file_host, (size_t)len, *F, true);
    if (rc == v5j::JPEG_OK) {
        *height = F->h;
        *width = F->w;
        *channels = F->ncomp;
    }
    delete F;
    return rc == v5j::JPEG_OK ? V5ELA_OK : (rc == v5j::JPEG_UNSUPPORTED ? V5ELA_ERR_UNSUPPORTED : V5ELA_ERR_INVALID);
}

/* n files at once: dims_out[3 i .. 3 i + 2] = height, width, channels of file i. Stops at the first unreadable file and returns
 * its status; *bad_index (optional) names it. */
static int v5ela_jpeg_info_batch_impl(const uint8_t *const *files_host, const int64_t *lens, int n, int32_t *dims_out, int *bad_index)
{
    if (!files_host || !lens || n < 0 || !dims_out) return V5ELA_ERR_INVALID;
    for (int i = 0; i < n; i++) {
        int hh = 0, ww = 0, cc = 0;
        const int rc = files_host[i] ? v5ela_jpeg_info(files_host[i], lens[i], &hh, &ww, &cc) : V5ELA_ERR_INVALID;
        if (rc) {
            if (bad_index) *bad_index = i;
            return rc;
        }
        dims_out[3 * i] = hh;
        dims_out[3 * i + 1] = ww;
        dims_out[3 * i + 2] = cc;
    }
    return V5ELA_OK;
}

}  // extern "C"

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Host-side helper threads for header parsing and the staging copy of large batches (a 1080p file is ~0.5 MB).
template <class Fn>
void parallel_for(int n, size_t bytes_hint, Fn fn)
{
    int nt = (int)std::thread::hardware_concurrency();
    nt = nt > 8 ? 8 : nt;
    if (const char *env = getenv("V5ELA_HOST_THREADS")) {       // several processes per host (one per GPU): share the cores out
        const int v = atoi(env);
        if (v >= 1 && v < nt) nt = v;
    }
    if (nt > n) nt = n;
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

bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

struct DecPlan {                               // host-side description of one chunk of files
    std::vector<v5j::DecImage> images;
    std::vector<int> file_index;
    std::vector<char> contiguous;              // file k follows file k-1 in host memory closely enough to share one upload
    size_t scan_bytes = 0, stream_bytes = 0, coef_blocks = 0, plane_bytes = 0, subs = 0;
    uint32_t max_windows = 1;
    size_t rst_entries = 0;                    // interval starts of the files with restart markers
    int max_intervals = 0;
    int max_blocks = 0;
    int64_t max_groups = 0;                    // 8-pixel groups of the largest image
};

}  // namespace

extern "C" {

static int v5ela_jpeg_decode_impl(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *d_rgb,
                      const int64_t *rgb_offsets, uint8_t *d_gray, const int64_t *gray_offsets, int32_t *d_status,
                      void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!files_host || !lens || n < 0 || (!d_rgb && !d_gray))
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode: bad pointer or count%s");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // the codec workspace is handle-owned
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;
    if (!s->upload_stream) {
        V5_CUDA(h, cudaStreamCreateWithFlags(&s->upload_stream, cudaStreamNonBlocking));
        for (int b = 0; b < 2; b++) {
            V5_CUDA(h, cudaEventCreateWithFlags(&s->uploaded[b], cudaEventDisableTiming));
            V5_CUDA(h, cudaEventCreateWithFlags(&s->consumed[b], cudaEventDisableTiming));
        }
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_sync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
    }

    // ---- parse every file; unique Huffman table sets and quantisation table pairs
    std::vector<v5j::FileInfo> info((size_t)n);
    std::vector<v5j::HuffSpecSet> specsets;                    // distinct table sets of the call (usually one): decoder tables are built for these only
    std::vector<std::vector<uint16_t>> qsets;
    std::vector<int> tab_of((size_t)n), q_of((size_t)n), parse_rc((size_t)n);
    size_t total_len = 0;
    bool all_pinned = true;
    for (int i = 0; i < n; i++) {
        if (!files_host[i] || lens[i] <= 0) return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode: null or empty file%s");
        total_len += (size_t)lens[i];
        all_pinned = all_pinned && is_pinned(files_host[i]) && is_pinned(files_host[i] + (lens[i] > 0 ? lens[i] - 1 : 0));   // first and last byte
    }
    parallel_for(n, total_len, [&](int i) { parse_rc[(size_t)i] = v5j::parse_file(files_host[i], (size_t)lens[i], info[(size_t)i]); });
    for (int i = 0; i < n; i++) {
        const int prc = parse_rc[(size_t)i];
        if (prc != v5j::JPEG_OK) {
            char which[64];
            snprintf(which, sizeof(which), " (file %d)", i);
            return prc == v5j::JPEG_UNSUPPORTED
                       ? fail(h, V5ELA_ERR_UNSUPPORTED, "v5ela_jpeg_decode: not an 8-bit baseline one-component / 4:2:0 / 4:2:2 / 4:4:4 JPEG%s", which)
                       : fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode: corrupt JPEG headers%s", which);
        }
        v5j::HuffSpecSet ts;                                    // (HuffSpec has no padding bytes and parse_file zeroes what it does not fill)
        ts.dc[0] = info[i].dc[0]; ts.dc[1] = info[i].dc[1]; ts.ac[0] = info[i].ac[0]; ts.ac[1] = info[i].ac[1];
        int found = -1;
        for (size_t k = specsets.size(); k-- > 0 && found < 0;)
            if (!memcmp(&specsets[k], &ts, sizeof(ts))) found = (int)k;
        if (found < 0) { specsets.push_back(ts); found = (int)specsets.size() - 1; }
        tab_of[i] = found;
        std::vector<uint16_t> q(128);
        memcpy(q.data(), info[i].qt[0], 128);
        memcpy(q.data() + 64, info[i].qt[1], 128);
        found = -1;
        for (size_t k = 0; k < qsets.size() && found < 0; k++)
            if (qsets[k] == q) found = (int)k;
        if (found < 0) { qsets.push_back(q); found = (int)qsets.size() - 1; }
        q_of[i] = found;
    }

    std::vector<v5j::DecTabSet> tabsets(specsets.size());
    for (size_t k = 0; k < specsets.size(); k++) v5j::make_tabset(specsets[k], tabsets[k]);   // (parse_file has validated every table)

    // ---- chunks of files whose workspace stays under ~8 GiB (a 1080p file needs ~11 MB: coefficients, planes, streams)
    std::vector<DecPlan> plans(1);
    int64_t rgb_run = 0, gray_run = 0;
    for (int i = 0; i < n; i++) {
        const v5j::FileInfo &F = info[i];
        v5j::DecImage im;
        memset(&im, 0, sizeof(im));
        v5j::dec_geometry(im, F.h, F.w, F.ncomp, F.hs, F.vs);
        im.tabset = tab_of[i];
        im.qt = q_of[i];
        const size_t planes = (size_t)im.yw * im.yh + 2 * (size_t)im.cw * im.ch;
        const size_t need = F.scan_len * 2 + (size_t)im.blocks * 128 + planes + 256;
        DecPlan *P = &plans.back();
        if (!P->images.empty() && (P->scan_bytes * 2 + P->coef_blocks * 128 + P->plane_bytes + need > ((size_t)8 << 30) || P->images.size() >= 65535)) {
            plans.emplace_back();
            P = &plans.back();
        }
        // Pinned files that follow each other in host memory keep their relative distance on the device, so that the whole run
        // goes up in one copy — which also copies the bytes between two scan segments: the next file's header (its first and
        // last byte are known to be pinned, see all_pinned) and the padding between the files, which is only accepted when it is
        // shorter than a page: every byte of it then shares a page with a byte of one of the two files, so the copy can touch
        // neither unmapped nor foreign memory. Files further apart get a copy of their own. scan_bytes = end of the used scan area.
        size_t start = align_up(P->scan_bytes, 16);
        char contig = 0;
        if (all_pinned && !P->images.empty()) {
            const int pi = P->file_index.back();
            const uint8_t *prev_end = files_host[pi] + info[(size_t)pi].scan_off + info[(size_t)pi].scan_len;
            const uint8_t *cur = files_host[i] + F.scan_off;
            const uint8_t *prev_file_end = files_host[pi] + lens[pi];
            if (cur >= prev_end && files_host[i] >= prev_file_end && (size_t)(files_host[i] - prev_file_end) < 4096) {
                contig = 1;
                start = (size_t)(P->images.back().scan_off + P->images.back().scan_len) + (size_t)(cur - prev_end);
            }
        }
        P->contiguous.push_back(contig);
        im.scan_off = (int64_t)start;                  // relative to the scan area of the staging buffer (fixed up below)
        im.scan_len = (int64_t)F.scan_len;
        im.stream_off = (int64_t)P->stream_bytes;
        im.coef_off = (int64_t)P->coef_blocks;
        im.sub_off = (int64_t)P->subs;
        const size_t nsub_max = (F.scan_len * 8 + v5j::SUB_BITS - 1) / v5j::SUB_BITS + 1;
        P->subs += nsub_max;
        const uint32_t wmax = (uint32_t)((nsub_max + v5j::HUFF_NT - 1) / v5j::HUFF_NT);
        if (wmax > P->max_windows) P->max_windows = wmax;
        if (F.restart > 0) {                           // restart intervals: one start position per interval
            const int n_int = (im.mcux * im.mcuy + F.restart - 1) / F.restart;
            im.restart = F.restart;
            im.rst_off = (int32_t)P->rst_entries;
            P->rst_entries += (size_t)n_int;
            if (n_int > P->max_intervals) P->max_intervals = n_int;
        }
        im.plane_off = (int64_t)P->plane_bytes;
        im.rgb_off = d_rgb ? (rgb_offsets ? rgb_offsets[i] : rgb_run) : -1;
        im.gray_off = d_gray ? (gray_offsets ? gray_offsets[i] : gray_run) : -1;
        rgb_run += (int64_t)F.h * F.w * 3;
        gray_run += (int64_t)F.h * F.w;
        P->scan_bytes = start + F.scan_len;
        P->stream_bytes += align_up(F.scan_len + 32, 16);
        P->coef_blocks += (size_t)im.blocks;
        P->plane_bytes += align_up(planes, 16);
        if (im.blocks > P->max_blocks) P->max_blocks = im.blocks;
        if ((int64_t)F.h * ((F.w + 7) / 8) > P->max_groups) P->max_groups = (int64_t)F.h * ((F.w + 7) / 8);
        P->images.push_back(im);
        P->file_index.push_back(i);
    }

    for (DecPlan &P : plans) {
        const int cn = (int)P.images.size();
        // staging layout: descriptors | table sets | quantisation tables | scan segments
        const size_t off_img = 0, off_tab = align_up(sizeof(v5j::DecImage) * (size_t)cn, 16);
        const size_t off_q = off_tab + align_up(sizeof(v5j::DecTabSet) * tabsets.size(), 16);
        const size_t off_scan = off_q + align_up(256 * qsets.size(), 16);
        const size_t stage_bytes = off_scan + align_up(P.scan_bytes, 16);
        // Files in pinned (page-locked) host memory are copied to the device straight from where they are — the caller keeps
        // them alive until the stream has been synchronised; pageable files go through the handle's pinned staging buffer.
        const size_t host_stage_bytes = all_pinned ? off_scan : stage_bytes;
        const int b = s->toggle;
        s->toggle ^= 1;
        cudaStream_t up = s->upload_stream;
        // host: the previous upload out of stage_host[b] is over; device: the kernels that read d_stage[b] are over
        V5_CUDA(h, cudaEventSynchronize(s->uploaded[b]));
        if (s->stage_host_cap[b] < host_stage_bytes) {
            if (s->stage_host[b]) cudaFreeHost(s->stage_host[b]);
            s->stage_host[b] = nullptr;
            s->stage_host_cap[b] = 0;
            V5_CUDA(h, cudaHostAlloc((void **)&s->stage_host[b], host_stage_bytes + host_stage_bytes / 4, cudaHostAllocDefault));
            s->stage_host_cap[b] = host_stage_bytes + host_stage_bytes / 4;
        }
        if ((rc = ensure(h, (void **)&s->d_stage[b], &s->stage_cap[b], stage_bytes))) return rc;
        if ((rc = ensure(h, &s->d_streams, &s->streams_cap, P.stream_bytes))) return rc;
        if ((rc = ensure(h, &s->d_dcoef, &s->dcoef_cap, P.coef_blocks * 128))) return rc;
        if ((rc = ensure(h, &s->d_planes, &s->planes_cap, P.plane_bytes))) return rc;
        if ((rc = ensure(h, &s->d_bits, &s->bits_cap, sizeof(uint32_t) * (size_t)cn))) return rc;
        if ((rc = ensure(h, &s->d_status, &s->status_cap, sizeof(int32_t) * (size_t)cn))) return rc;
        if ((rc = ensure(h, &s->d_dc, &s->dc_cap, sizeof(int16_t) * P.coef_blocks))) return rc;
        if ((rc = ensure(h, &s->d_sub_info, &s->sub_info_cap, sizeof(v5j::SubInfo) * P.subs))) return rc;
        if ((rc = ensure(h, &s->d_sub_block0, &s->sub_block0_cap, sizeof(uint32_t) * P.subs))) return rc;
        if ((rc = ensure(h, &s->d_rst, &s->rst_cap, sizeof(uint32_t) * (P.rst_entries + 1)))) return rc;
        uint8_t *stage_host = s->stage_host[b], *d_stage = s->d_stage[b];
        for (int k = 0; k < cn; k++) P.images[(size_t)k].scan_off += (int64_t)off_scan;
        if (!all_pinned)
            parallel_for(cn, P.scan_bytes, [&](int k) {   // every scan segment to its planned place in the staging buffer
                const v5j::DecImage &im = P.images[(size_t)k];
                const int fi = P.file_index[(size_t)k];
                memcpy(stage_host + im.scan_off, files_host[fi] + info[(size_t)fi].scan_off, (size_t)im.scan_len);
            });
        memcpy(stage_host + off_img, P.images.data(), sizeof(v5j::DecImage) * (size_t)cn);
        memcpy(stage_host + off_tab, tabsets.data(), sizeof(v5j::DecTabSet) * tabsets.size());
        for (size_t k = 0; k < qsets.size(); k++) memcpy(stage_host + off_q + 256 * k, qsets[k].data(), 256);
        V5_CUDA(h, cudaStreamWaitEvent(up, s->consumed[b], 0));
        V5_CUDA(h, cudaMemcpyAsync(d_stage, stage_host, host_stage_bytes, cudaMemcpyHostToDevice, up));
        if (all_pinned) {
            // one copy per file, or per run of files that also sit back to back in host memory (a loader's arena): the
            // device layout was planned with the same gaps, so a run is a single contiguous range
            for (int k = 0; k < cn;) {
                int e = k + 1;
                while (e < cn && P.contiguous[(size_t)e]) e++;
                const v5j::DecImage &first = P.images[(size_t)k], &last = P.images[(size_t)e - 1];
                const int fi = P.file_index[(size_t)k];
                const size_t bytes = (size_t)(last.scan_off + last.scan_len - first.scan_off);
                V5_CUDA(h, cudaMemcpyAsync(d_stage + first.scan_off, files_host[fi] + info[(size_t)fi].scan_off, bytes,
                                           cudaMemcpyHostToDevice, up));
                k = e;
            }
        }
        V5_CUDA(h, cudaEventRecord(s->uploaded[b], up));
        V5_CUDA(h, cudaStreamWaitEvent(st, s->uploaded[b], 0));
        V5_CUDA(h, cudaStreamWaitEvent(st, s->consumed[b ^ 1], 0));      // the shared workspace: previous batch (any stream) is done
        V5_CUDA(h, cudaMemsetAsync(s->d_streams, 0, P.stream_bytes, st));
        V5_CUDA(h, cudaMemsetAsync(s->d_dcoef, 0, P.coef_blocks * 128, st));
        V5_CUDA(h, cudaMemsetAsync(s->d_dc, 0, sizeof(int16_t) * P.coef_blocks, st));
        if (P.rst_entries) V5_CUDA(h, cudaMemsetAsync(s->d_rst, 0, sizeof(uint32_t) * P.rst_entries, st));

        const v5j::DecImage *d_images = reinterpret_cast<const v5j::DecImage *>(d_stage + off_img);
        const v5j::DecTabSet *d_tabs = reinterpret_cast<const v5j::DecTabSet *>(d_stage + off_tab);
        const uint16_t *d_q = reinterpret_cast<const uint16_t *>(d_stage + off_q);
        uint32_t *d_bits = static_cast<uint32_t *>(s->d_bits);
        int32_t *d_st = static_cast<int32_t *>(s->d_status);
        v5j::unstuff_kernel<<<cn, 1024, 0, st>>>(d_images, d_stage, static_cast<uint8_t *>(s->d_streams), d_bits, static_cast<uint32_t *>(s->d_rst));
        V5_CUDA(h, cudaGetLastError());
        // Huffman decoding in three launches: synchronisation (the windows of a file shared out among `parts` CTAs so that a
        // small batch still fills the GPU), boundary fix-up + block offsets, then one CTA per window writes coefficients.
        // (a batch of at least one file per SM gains nothing from splitting files: parts = 1, no blind starts, no fix-up walks)
        unsigned parts = (unsigned)(h->sm_count / cn);
        parts = parts < 1 ? 1 : (parts > 16 ? 16 : parts);
        parts = parts > P.max_windows ? P.max_windows : parts;
        const uint8_t *d_str = static_cast<const uint8_t *>(s->d_streams);
        v5j::SubInfo *d_sub_info = static_cast<v5j::SubInfo *>(s->d_sub_info);
        uint32_t *d_sub_block0 = static_cast<uint32_t *>(s->d_sub_block0);
        const char *force = getenv("V5ELA_HUFF_PATH");                    // tests: "one" / "three" force a path
        if (const char *fp = getenv("V5ELA_HUFF_PARTS")) {                 // experiments: parts per file of the three-launch path
            const int v = atoi(fp);
            if (v >= 1 && v <= 16) parts = (unsigned)v > P.max_windows ? P.max_windows : (unsigned)v;
        }
        // nothing to gain from splitting when there is no room for two parts per file, or no file has more than one window
        const bool one_launch = force ? force[0] == 'o' : (h->sm_count / cn < 2 || P.max_windows < 2);
        if (one_launch) {
            v5j::huffman_kernel<<<cn, v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(d_images, d_tabs, d_str, d_bits, static_cast<int16_t *>(s->d_dcoef),
                                                                            static_cast<int16_t *>(s->d_dc), d_st);
            V5_CUDA(h, cudaGetLastError());
        } else {
            v5j::huffman_sync_kernel<<<dim3(parts, (unsigned)cn), v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(d_images, d_tabs, d_str, d_bits, d_sub_info);
            V5_CUDA(h, cudaGetLastError());
            v5j::huffman_fixup_kernel<<<cn, 1024, 0, st>>>(d_images, d_tabs, d_str, d_bits, parts, d_sub_info, d_sub_block0, d_st);
            V5_CUDA(h, cudaGetLastError());
            v5j::huffman_write_kernel<<<dim3(P.max_windows, (unsigned)cn), v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(
                d_images, d_tabs, d_str, d_bits, d_sub_info, d_sub_block0, static_cast<int16_t *>(s->d_dcoef), static_cast<int16_t *>(s->d_dc));
            V5_CUDA(h, cudaGetLastError());
        }
        if (P.max_intervals > 0) {                                         // files with restart intervals: one thread per interval
            v5j::huffman_rst_kernel<<<dim3((unsigned)((P.max_intervals + 127) / 128), (unsigned)cn), 128, 0, st>>>(
                d_images, d_tabs, d_str, d_bits, static_cast<const uint32_t *>(s->d_rst), static_cast<int16_t *>(s->d_dcoef),
                static_cast<int16_t *>(s->d_dc), d_st);
            V5_CUDA(h, cudaGetLastError());
            h->launches += 1;
        }
        v5j::dc_kernel<<<cn, 1024, 0, st>>>(d_images, static_cast<int16_t *>(s->d_dc));
        V5_CUDA(h, cudaGetLastError());
        v5j::idct_kernel<<<dim3((unsigned)((P.max_blocks + 63) / 64), (unsigned)cn), 256, 0, st>>>(
            d_images, d_q, static_cast<const int16_t *>(s->d_dcoef), static_cast<const int16_t *>(s->d_dc), static_cast<uint8_t *>(s->d_planes));
        V5_CUDA(h, cudaGetLastError());
        v5j::colour_kernel<<<dim3((unsigned)((P.max_groups + 255) / 256), (unsigned)cn), 256, 0, st>>>(
            d_images, static_cast<const uint8_t *>(s->d_planes), d_rgb, d_gray);
        V5_CUDA(h, cudaGetLastError());
        if (d_status)                                                      // chunks keep file order: one contiguous range
            V5_CUDA(h, cudaMemcpyAsync(d_status + P.file_index[0], d_st, sizeof(int32_t) * (size_t)cn, cudaMemcpyDeviceToDevice, st));
        V5_CUDA(h, cudaEventRecord(s->consumed[b], st));
        h->launches += one_launch ? 5 : 7;
    }
    return V5ELA_OK;
}

static int v5ela_jpeg_decode_host_impl(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *rgb_host,
                           const int64_t *rgb_offsets, uint8_t *gray_host, const int64_t *gray_offsets)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!files_host || !lens || n < 0 || (!rgb_host && !gray_host))
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: bad pointer or count%s");
    DeviceGuard guard(h->device);
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;
    if (!h->own_stream) V5_CUDA(h, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    cudaStream_t st = h->own_stream;
    // output extents: the caller's offsets, or tight packing in file order
    std::vector<int64_t> px((size_t)n);
    int64_t rgb_end = 0, gray_end = 0, run = 0;
    for (int i = 0; i < n; i++) {
        int hh, ww, cc;
        if (!files_host[i] || (rc = v5ela_jpeg_info(files_host[i], lens[i], &hh, &ww, &cc)))
            return fail(h, rc ? rc : V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: unreadable JPEG headers%s");
        px[(size_t)i] = (int64_t)hh * ww;
        const int64_t ro = rgb_offsets ? rgb_offsets[i] : 3 * run, go = gray_offsets ? gray_offsets[i] : run;
        if (ro < 0 || go < 0) return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: negative output offset%s");
        if (ro + 3 * px[(size_t)i] > rgb_end) rgb_end = ro + 3 * px[(size_t)i];
        if (go + px[(size_t)i] > gray_end) gray_end = go + px[(size_t)i];
        run += px[(size_t)i];
    }
    if (rgb_host && (rc = ensure(h, (void **)&s->d_dec_rgb, &s->dec_rgb_cap, (size_t)rgb_end))) return rc;
    if (gray_host && (rc = ensure(h, (void **)&s->d_dec_gray, &s->dec_gray_cap, (size_t)gray_end))) return rc;
    std::vector<int32_t> status((size_t)n, 0);
    if ((rc = ensure(h, (void **)&s->d_dec_status, &s->dec_status_cap, sizeof(int32_t) * (size_t)n))) return rc;
    int32_t *d_status = s->d_dec_status;
    rc = v5ela_jpeg_decode(h, files_host, lens, n, rgb_host ? s->d_dec_rgb : nullptr, rgb_offsets, gray_host ? s->d_dec_gray : nullptr,
                           gray_offsets, d_status, st);
    if (rc == V5ELA_OK) {
        cudaMemcpyAsync(status.data(), d_status, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st);
        run = 0;
        for (int i = 0; i < n; i++) {
            const int64_t ro = rgb_offsets ? rgb_offsets[i] : 3 * run, go = gray_offsets ? gray_offsets[i] : run;
            if (rgb_host) cudaMemcpyAsync(rgb_host + ro, s->d_dec_rgb + ro, (size_t)(3 * px[(size_t)i]), cudaMemcpyDeviceToHost, st);
            if (gray_host) cudaMemcpyAsync(gray_host + go, s->d_dec_gray + go, (size_t)px[(size_t)i], cudaMemcpyDeviceToHost, st);
            run += px[(size_t)i];
        }
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = fail(h, V5ELA_ERR_CUDA, "v5ela_jpeg_decode_host: %s", cudaGetErrorString(e));
    }
    if (rc) return rc;
    for (int i = 0; i < n; i++)
        if (status[(size_t)i] != 0) {
            char which[64];
            snprintf(which, sizeof(which), " (file %d)", i);
            return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: entropy-coded data ends early or is corrupt%s", which);
        }
    return V5ELA_OK;
}


// ---- the exported entry points: nothing may unwind through the C ABI (std::vector / std::thread inside the implementations can throw)
#define V5J_GUARD(h, call)                                                                       \
    try {                                                                                        \
        return call;                                                                             \
    } catch (const std::bad_alloc &) {                                                           \
        return fail((h), V5ELA_ERR_NOMEM, "out of host memory%s");                               \
    } catch (const std::exception &e) {                                                          \
        return fail((h), V5ELA_ERR_INVALID, "host-side failure: %s", e.what());                  \
    } catch (...) {                                                                              \
        return fail((h), V5ELA_ERR_INVALID, "host-side failure%s");                              \
    }

int v5ela_jpeg_encode(v5ela_handle *h, const uint8_t *d_img, int n, int height, int width, int channels, int64_t frame_stride_bytes,
                      int64_t row_stride_bytes, int quality, uint8_t *d_out, int64_t out_stride_bytes, int32_t *d_sizes, void *cuda_stream)
{
    V5J_GUARD(h, v5ela_jpeg_encode_impl(h, d_img, n, height, width, channels, frame_stride_bytes, row_stride_bytes, quality, d_out,
                                        out_stride_bytes, d_sizes, cuda_stream))
}

int v5ela_jpeg_encode_host(v5ela_handle *h, const uint8_t *img_host, int n, int height, int width, int channels, int quality,
                           uint8_t *out_host, int64_t out_stride_bytes, int32_t *sizes_host)
{
    V5J_GUARD(h, v5ela_jpeg_encode_host_impl(h, img_host, n, height, width, channels, quality, out_host, out_stride_bytes, sizes_host))
}

int v5ela_jpeg_info_batch(const uint8_t *const *files_host, const int64_t *lens, int n, int32_t *dims_out, int *bad_index)
{
    V5J_GUARD(static_cast<v5ela_handle *>(nullptr), v5ela_jpeg_info_batch_impl(files_host, lens, n, dims_out, bad_index))
}

int v5ela_jpeg_decode(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *d_rgb,
                      const int64_t *rgb_offsets, uint8_t *d_gray, const int64_t *gray_offsets, int32_t *d_status, void *cuda_stream)
{
    V5J_GUARD(h, v5ela_jpeg_decode_impl(h, files_host, lens, n, d_rgb, rgb_offsets, d_gray, gray_offsets, d_status, cuda_stream))
}

int v5ela_jpeg_decode_host(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *rgb_host,
                           const int64_t *rgb_offsets, uint8_t *gray_host, const int64_t *gray_offsets)
{
    V5J_GUARD(h, v5ela_jpeg_decode_host_impl(h, files_host, lens, n, rgb_host, rgb_offsets, gray_host, gray_offsets))
}

}  // extern "C"
