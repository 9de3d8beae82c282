// v5jpeg.cu — codec rows of libv5ela.so (SURVEY.md §8f-2 decode, §8f-3 encode): C-ABI entry points v5ela_jpeg_*.
// Kernels: v5jpeg_enc.cuh, v5jpeg_dec.cuh. Host-side header writing / parsing: v5jpeg_common.h. The decoder's launch plan (files
// parsed once, chunks, staging layout, upload runs, Huffman path; negative output offsets refused): v5jpeg_plan.h, which both
// decode entry points run through run_plan.
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
#include "v5jpeg_plan.h"

using namespace v5host;

struct v5jpeg_state {
    // encoder
    DeviceBuf<v5j::EncTables> d_enc_tabs;
    DeviceBuf<uint8_t> d_header;
    DeviceBuf<int16_t> d_coef;
    DeviceBuf<uint32_t> d_bitoff, d_total, d_raw;
    // host-buffer entry points
    DeviceBuf<uint8_t> d_img, d_out;
    DeviceBuf<int32_t> d_sizes;
    // decoder: one pinned staging buffer (descriptors | table sets | quantisation tables | scan segments) mirrored on the
    // device, plus the per-batch workspace (unstuffed streams, coefficients, sample planes)
    // Two of each, used alternately: the upload of one batch (on upload_stream) overlaps the kernels of the previous one.
    PinnedBuf stage_host[2];
    DeviceBuf<uint8_t> d_stage[2];
    Event uploaded[2];                     // the upload into d_stage[b] (and out of stage_host[b]) has completed
    Event consumed[2];                     // the kernels that read d_stage[b] have completed
    Stream upload_stream;
    int toggle = 0;
    DeviceBuf<uint8_t> d_streams, d_planes;
    DeviceBuf<int16_t> d_dcoef, d_dc;
    DeviceBuf<uint32_t> d_bits, d_sub_block0, d_rst;
    DeviceBuf<int32_t> d_status;
    DeviceBuf<v5j::SubInfo> d_sub_info;
    DeviceBuf<uint8_t> d_dec_rgb, d_dec_gray;
    DeviceBuf<int32_t> d_dec_status;
};

void v5host::JpegStateDelete::operator()(v5jpeg_state *s) const { delete s; }

namespace {

int jpeg_state(v5ela_handle *h, v5jpeg_state **out)
{
    if (!h->jpeg) {
        h->jpeg.reset(new (std::nothrow) v5jpeg_state());
        if (!h->jpeg) return fail(h, V5ELA_ERR_NOMEM, "v5ela_jpeg: out of host memory%s");
    }
    *out = h->jpeg.get();
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

int v5ela_jpeg_encode(v5ela_handle *h, const uint8_t *d_img, int n, int height, int width, int channels, int64_t frame_stride_bytes,
                      int64_t row_stride_bytes, int quality, uint8_t *d_out, int64_t out_stride_bytes, int32_t *d_sizes, void *cuda_stream)
try {
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
        if ((rc = s->d_enc_tabs.ensure(h, sizeof(tabs)))) return rc;
        V5_CUDA(h, cudaMemcpyAsync(s->d_enc_tabs, &tabs, sizeof(tabs), cudaMemcpyHostToDevice, st));
        if ((rc = s->d_header.ensure(h, kHeaderMax))) return rc;
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
    if ((rc = s->d_coef.ensure(h, (size_t)chunk * g.blocks * 128))) return rc;
    if ((rc = s->d_bitoff.ensure(h, (size_t)chunk * g.blocks * 4))) return rc;
    if ((rc = s->d_total.ensure(h, (size_t)chunk * 4))) return rc;
    if ((rc = s->d_raw.ensure(h, (size_t)chunk * raw_words * 4))) return rc;

    v5j::CoefParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.frame_stride = frame_stride_bytes;
    cp.row_stride = row_stride_bytes;
    cp.coef = s->d_coef;
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
        ep.bitoff = s->d_bitoff;
        ep.total_bits = s->d_total;
        ep.raw = s->d_raw;
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
} V5_CATCH(h)

int v5ela_jpeg_encode_host(v5ela_handle *h, const uint8_t *img_host, int n, int height, int width, int channels, int quality,
                           uint8_t *out_host, int64_t out_stride_bytes, int32_t *sizes_host)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!img_host || !out_host || !sizes_host || n < 0 || height <= 0 || width <= 0 || (channels != 1 && channels != 3) ||
        out_stride_bytes < kHeaderMax)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_encode_host: bad pointer, size or channel count%s");
    DeviceGuard guard(h->device);
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    const size_t fbytes = (size_t)height * width * channels;
    if ((rc = s->d_img.ensure(h, fbytes * n))) return rc;
    if ((rc = s->d_out.ensure(h, (size_t)out_stride_bytes * n))) return rc;
    if ((rc = s->d_sizes.ensure(h, sizeof(int32_t) * (size_t)n))) return rc;
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
} V5_CATCH(h)


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
int v5ela_jpeg_info_batch(const uint8_t *const *files_host, const int64_t *lens, int n, int32_t *dims_out, int *bad_index)
try {
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
} V5_CATCH(nullptr)

}  // extern "C"

namespace {

bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// A decode call with the environment's knobs, read on every call: the helper threads, a forced Huffman path and part count.
v5j::DecodeCall decode_call(const v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, const int64_t *rgb_offsets,
                            const int64_t *gray_offsets, bool want_rgb, bool want_gray)
{
    v5j::DecodeCall c;
    c.files = files_host;
    c.lens = lens;
    c.n = n;
    c.rgb_offsets = rgb_offsets;
    c.gray_offsets = gray_offsets;
    c.want_rgb = want_rgb;
    c.want_gray = want_gray;
    c.all_pinned = true;
    for (int i = 0; i < n && c.all_pinned; i++)               // first and last byte
        c.all_pinned = files_host[i] && lens[i] > 0 && is_pinned(files_host[i]) && is_pinned(files_host[i] + lens[i] - 1);
    c.sm_count = h->sm_count;
    if (const char *force = getenv("V5ELA_HUFF_PATH")) c.huff_path = force[0] == 'o' ? 1 : 3;   // tests: "one" / "three" force a path
    if (const char *fp = getenv("V5ELA_HUFF_PARTS")) c.huff_parts = atoi(fp);                  // experiments: parts per file of the three-launch path
    int nt = (int)std::thread::hardware_concurrency();
    nt = nt > 8 ? 8 : nt;
    if (const char *env = getenv("V5ELA_HOST_THREADS")) {       // several processes per host (one per GPU): share the cores out
        const int v = atoi(env);
        if (v >= 1 && v < nt) nt = v;
    }
    c.threads = nt;
    c.chunk_bytes = (size_t)8 << 30;
    return c;
}

int refused(v5ela_handle *h, const char *entry, const v5j::DecodePlan &P)
{
    char which[64] = "";
    if (P.bad_file >= 0) snprintf(which, sizeof(which), " (file %d)", P.bad_file);
    char msg[256];
    snprintf(msg, sizeof(msg), "%s: %s%s", entry, P.error, which);
    return fail(h, P.status, "%s", msg);
}

// Runs plan P of call c on stream st: per chunk, the workspaces, the staging buffer, the upload and the launches.
int run_plan(v5ela_handle *h, v5jpeg_state *s, const v5j::DecodeCall &c, const v5j::DecodePlan &P, uint8_t *d_rgb, uint8_t *d_gray,
             int32_t *d_status, cudaStream_t st)
{
    int rc;
    if (!s->upload_stream) {
        V5_CUDA(h, s->upload_stream.create());
        for (int b = 0; b < 2; b++) {
            V5_CUDA(h, s->uploaded[b].create());
            V5_CUDA(h, s->consumed[b].create());
        }
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_sync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
        V5_CUDA(h, cudaFuncSetAttribute(v5j::huffman_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(v5j::HuffSmem)));
    }
    for (const v5j::DecChunk &C : P.chunks) {
        const int cn = (int)C.images.size();
        const int b = s->toggle;
        s->toggle ^= 1;
        cudaStream_t up = s->upload_stream;
        // host: the previous upload out of stage_host[b] is over; device: the kernels that read d_stage[b] are over
        V5_CUDA(h, cudaEventSynchronize(s->uploaded[b]));
        if ((rc = s->stage_host[b].ensure(h, C.host_stage_bytes, C.host_stage_bytes + C.host_stage_bytes / 4))) return rc;
        if ((rc = s->d_stage[b].ensure(h, C.stage_bytes))) return rc;
        if ((rc = s->d_streams.ensure(h, C.stream_bytes))) return rc;
        if ((rc = s->d_dcoef.ensure(h, C.coef_blocks * 128))) return rc;
        if ((rc = s->d_planes.ensure(h, C.plane_bytes))) return rc;
        if ((rc = s->d_bits.ensure(h, sizeof(uint32_t) * (size_t)cn))) return rc;
        if ((rc = s->d_status.ensure(h, sizeof(int32_t) * (size_t)cn))) return rc;
        if ((rc = s->d_dc.ensure(h, sizeof(int16_t) * C.coef_blocks))) return rc;
        if ((rc = s->d_sub_info.ensure(h, sizeof(v5j::SubInfo) * C.subs))) return rc;
        if ((rc = s->d_sub_block0.ensure(h, sizeof(uint32_t) * C.subs))) return rc;
        if ((rc = s->d_rst.ensure(h, sizeof(uint32_t) * (C.rst_entries + 1)))) return rc;
        uint8_t *stage_host = s->stage_host[b], *d_stage = s->d_stage[b];
        if (!c.all_pinned)
            v5j::parallel_for(cn, C.scan_bytes, c.threads, [&](int k) {   // every scan segment to its planned place in the staging buffer
                const v5j::DecImage &im = C.images[(size_t)k];
                const int fi = C.file_index[(size_t)k];
                memcpy(stage_host + im.scan_off, c.files[fi] + P.info[(size_t)fi].scan_off, (size_t)im.scan_len);
            });
        memcpy(stage_host + C.off_img, C.images.data(), sizeof(v5j::DecImage) * (size_t)cn);
        memcpy(stage_host + C.off_tab, P.tabsets.data(), sizeof(v5j::DecTabSet) * P.tabsets.size());
        for (size_t k = 0; k < P.qsets.size(); k++) memcpy(stage_host + C.off_q + 256 * k, P.qsets[k].data(), 256);
        V5_CUDA(h, cudaStreamWaitEvent(up, s->consumed[b], 0));
        V5_CUDA(h, cudaMemcpyAsync(d_stage, stage_host, C.host_stage_bytes, cudaMemcpyHostToDevice, up));
        for (const v5j::UploadRun &r : C.runs)
            V5_CUDA(h, cudaMemcpyAsync(d_stage + r.dev_off, r.src, r.bytes, cudaMemcpyHostToDevice, up));
        V5_CUDA(h, cudaEventRecord(s->uploaded[b], up));
        V5_CUDA(h, cudaStreamWaitEvent(st, s->uploaded[b], 0));
        V5_CUDA(h, cudaStreamWaitEvent(st, s->consumed[b ^ 1], 0));      // the shared workspace: previous batch (any stream) is done
        V5_CUDA(h, cudaMemsetAsync(s->d_streams, 0, C.stream_bytes, st));
        V5_CUDA(h, cudaMemsetAsync(s->d_dcoef, 0, C.coef_blocks * 128, st));
        V5_CUDA(h, cudaMemsetAsync(s->d_dc, 0, sizeof(int16_t) * C.coef_blocks, st));
        if (C.rst_entries) V5_CUDA(h, cudaMemsetAsync(s->d_rst, 0, sizeof(uint32_t) * C.rst_entries, st));

        const v5j::DecImage *d_images = reinterpret_cast<const v5j::DecImage *>(d_stage + C.off_img);
        const v5j::DecTabSet *d_tabs = reinterpret_cast<const v5j::DecTabSet *>(d_stage + C.off_tab);
        const uint16_t *d_q = reinterpret_cast<const uint16_t *>(d_stage + C.off_q);
        uint32_t *d_bits = s->d_bits;
        int32_t *d_st = s->d_status;
        const uint8_t *d_str = s->d_streams;
        v5j::SubInfo *d_sub_info = s->d_sub_info;
        uint32_t *d_sub_block0 = s->d_sub_block0;
        v5j::unstuff_kernel<<<cn, 1024, 0, st>>>(d_images, d_stage, s->d_streams, d_bits, s->d_rst);
        V5_CUDA(h, cudaGetLastError());
        if (C.one_launch) {
            v5j::huffman_kernel<<<cn, v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(d_images, d_tabs, d_str, d_bits, s->d_dcoef, s->d_dc, d_st);
            V5_CUDA(h, cudaGetLastError());
        } else {
            v5j::huffman_sync_kernel<<<dim3(C.parts, (unsigned)cn), v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(d_images, d_tabs, d_str, d_bits, d_sub_info);
            V5_CUDA(h, cudaGetLastError());
            v5j::huffman_fixup_kernel<<<cn, 1024, 0, st>>>(d_images, d_tabs, d_str, d_bits, C.parts, d_sub_info, d_sub_block0, d_st);
            V5_CUDA(h, cudaGetLastError());
            v5j::huffman_write_kernel<<<dim3(C.max_windows, (unsigned)cn), v5j::HUFF_NT, sizeof(v5j::HuffSmem), st>>>(
                d_images, d_tabs, d_str, d_bits, d_sub_info, d_sub_block0, s->d_dcoef, s->d_dc);
            V5_CUDA(h, cudaGetLastError());
        }
        if (C.max_intervals > 0) {                                         // files with restart intervals: one thread per interval
            v5j::huffman_rst_kernel<<<dim3((unsigned)((C.max_intervals + 127) / 128), (unsigned)cn), 128, 0, st>>>(
                d_images, d_tabs, d_str, d_bits, s->d_rst, s->d_dcoef, s->d_dc, d_st);
            V5_CUDA(h, cudaGetLastError());
        }
        v5j::dc_kernel<<<cn, 1024, 0, st>>>(d_images, s->d_dc);
        V5_CUDA(h, cudaGetLastError());
        v5j::idct_kernel<<<dim3((unsigned)((C.max_blocks + 63) / 64), (unsigned)cn), 256, 0, st>>>(
            d_images, d_q, s->d_dcoef, s->d_dc, s->d_planes);
        V5_CUDA(h, cudaGetLastError());
        v5j::colour_kernel<<<dim3((unsigned)((C.max_groups + 255) / 256), (unsigned)cn), 256, 0, st>>>(
            d_images, s->d_planes, d_rgb, d_gray);
        V5_CUDA(h, cudaGetLastError());
        if (d_status)                                                      // chunks keep file order: one contiguous range
            V5_CUDA(h, cudaMemcpyAsync(d_status + C.file_index[0], d_st, sizeof(int32_t) * (size_t)cn, cudaMemcpyDeviceToDevice, st));
        V5_CUDA(h, cudaEventRecord(s->consumed[b], st));
        h->launches += C.launches;
    }
    return V5ELA_OK;
}

}  // namespace

extern "C" {

int v5ela_jpeg_decode(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *d_rgb,
                      const int64_t *rgb_offsets, uint8_t *d_gray, const int64_t *gray_offsets, int32_t *d_status, void *cuda_stream)
try {
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
    const v5j::DecodeCall c = decode_call(h, files_host, lens, n, rgb_offsets, gray_offsets, d_rgb != nullptr, d_gray != nullptr);
    v5j::DecodePlan P;
    v5j::plan_decode(c, P);
    if (P.status) return refused(h, "v5ela_jpeg_decode", P);
    return run_plan(h, s, c, P, d_rgb, d_gray, d_status, st);
} V5_CATCH(h)

int v5ela_jpeg_decode_host(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint8_t *rgb_host,
                           const int64_t *rgb_offsets, uint8_t *gray_host, const int64_t *gray_offsets)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!files_host || !lens || n < 0 || (!rgb_host && !gray_host))
        return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: bad pointer or count%s");
    DeviceGuard guard(h->device);
    v5jpeg_state *s;
    int rc;
    if ((rc = jpeg_state(h, &s))) return rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    const v5j::DecodeCall c = decode_call(h, files_host, lens, n, rgb_offsets, gray_offsets, rgb_host != nullptr, gray_host != nullptr);
    v5j::DecodePlan P;
    v5j::plan_decode(c, P);
    if (P.status) return refused(h, "v5ela_jpeg_decode_host", P);
    int64_t rgb_end = 0, gray_end = 0;                          // output extents on the device, from the plan's offsets
    for (const v5j::DecChunk &C : P.chunks)
        for (const v5j::DecImage &im : C.images) {
            const int64_t px = (int64_t)im.h * im.w;
            if (im.rgb_off + 3 * px > rgb_end) rgb_end = im.rgb_off + 3 * px;
            if (im.gray_off + px > gray_end) gray_end = im.gray_off + px;
        }
    if (rgb_host && (rc = s->d_dec_rgb.ensure(h, (size_t)rgb_end))) return rc;
    if (gray_host && (rc = s->d_dec_gray.ensure(h, (size_t)gray_end))) return rc;
    if ((rc = s->d_dec_status.ensure(h, sizeof(int32_t) * (size_t)n))) return rc;
    ScratchOrder order(h, st);                                  // the codec workspace is handle-owned
    if ((rc = run_plan(h, s, c, P, rgb_host ? static_cast<uint8_t *>(s->d_dec_rgb) : nullptr,
                       gray_host ? static_cast<uint8_t *>(s->d_dec_gray) : nullptr, s->d_dec_status, st)))
        return rc;
    std::vector<int32_t> status((size_t)n, 0);
    V5_CUDA(h, cudaMemcpyAsync(status.data(), s->d_dec_status, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    for (const v5j::DecChunk &C : P.chunks)
        for (const v5j::DecImage &im : C.images) {
            const size_t px = (size_t)im.h * im.w;
            if (rgb_host) V5_CUDA(h, cudaMemcpyAsync(rgb_host + im.rgb_off, s->d_dec_rgb + im.rgb_off, 3 * px, cudaMemcpyDeviceToHost, st));
            if (gray_host) V5_CUDA(h, cudaMemcpyAsync(gray_host + im.gray_off, s->d_dec_gray + im.gray_off, px, cudaMemcpyDeviceToHost, st));
        }
    V5_CUDA(h, cudaStreamSynchronize(st));
    for (int i = 0; i < n; i++)
        if (status[(size_t)i] != 0) {
            char which[64];
            snprintf(which, sizeof(which), " (file %d)", i);
            return fail(h, V5ELA_ERR_INVALID, "v5ela_jpeg_decode_host: entropy-coded data ends early or is corrupt%s", which);
        }
    return V5ELA_OK;
} V5_CATCH(h)

}  // extern "C"
