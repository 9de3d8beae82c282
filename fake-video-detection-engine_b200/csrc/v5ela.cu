// v5ela.cu — kernels + C ABI (include/v5ela.h) of libv5ela.so. sm_100a only.
//
// Launch sequence of one v5ela_analyze call (all on the caller's stream, no host sync, no allocation):
//   1. cudaMemsetAsync(records)                      records are accumulated with atomics by several CTAs per frame
//   2. ela_fused_kernel   (persistent, 2 CTAs / SM)  everything per pixel — see v5ela_device.cuh
//   3. ela_finalize_kernel (1 warp per frame-channel) ela_sum / ela_sumsq / ela_max from the histogram
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

#include "v5ela.h"
#include "v5ela_launch.cuh"
#include "v5ela_fft.cuh"

static_assert(sizeof(v5ela_record) == 3144, "V5F v1 record layout");

namespace v5 {

// One warp per (frame, channel): ela_sum = sum b*hist[b], ela_sumsq = sum b^2*hist[b], ela_max = highest non-empty bin.
__global__ void __launch_bounds__(96) ela_finalize_kernel(v5ela_record *recs, int n)
{
    const int frame = blockIdx.x, c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (frame >= n) return;
    v5ela_record &r = recs[frame];
    unsigned long long s = 0, sq = 0;
    int mx = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int b = lane + 32 * i;
        const unsigned long long cnt = r.ela_hist[c][b];
        s += cnt * (unsigned long long)b;
        sq += cnt * (unsigned long long)(b * b);
        if (cnt) mx = b;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) {
        r.ela_sum[c] = s;
        r.ela_sumsq[c] = sq;
    }
    __syncthreads();                       // tex_maxabs shares its 32-bit word with ela_max[0..1]: plain byte stores
    if (lane == 0) r.ela_max[c] = (uint8_t)mx;
}

// ImageEnhance.Brightness(diff).enhance(255.0/max_diff) (v5_texture_ela.py:74-78): a per-frame 256-entry float32 LUT.
__global__ void __launch_bounds__(256) ela_enhance_kernel(const uint8_t *__restrict__ resid, const v5ela_record *recs,
                                                         uint8_t *__restrict__ out, long long bytes_per_frame)
{
    __shared__ uint8_t lut[256];
    const int frame = blockIdx.y;
    const v5ela_record &r = recs[frame];
    int m = max((int)r.ela_max[0], max((int)r.ela_max[1], (int)r.ela_max[2]));
    if (m == 0) m = 1;
    const float scale = (float)(255.0 / (double)m);
    {
        const float v = (float)threadIdx.x * scale;
        lut[threadIdx.x] = (uint8_t)(v <= 0.0f ? 0 : (v >= 255.0f ? 255 : (int)v));
    }
    __syncthreads();
    const uint8_t *src = resid + (long long)frame * bytes_per_frame;
    uint8_t *dst = out + (long long)frame * bytes_per_frame;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if ((((uintptr_t)src | (uintptr_t)dst) & 15) == 0) {
        const long long nvec = bytes_per_frame >> 4;
        for (long long v = i; v < nvec; v += stride) {
            uint4 w = reinterpret_cast<const uint4 *>(src)[v];
            uint32_t *pw = reinterpret_cast<uint32_t *>(&w);
#pragma unroll
            for (int k = 0; k < 4; k++)
                pw[k] = lut[pw[k] & 0xff] | (lut[(pw[k] >> 8) & 0xff] << 8) | (lut[(pw[k] >> 16) & 0xff] << 16) |
                        (lut[pw[k] >> 24] << 24);
            reinterpret_cast<uint4 *>(dst)[v] = w;
        }
        for (long long b = (nvec << 4) + i; b < bytes_per_frame; b += stride) dst[b] = lut[src[b]];
    } else {
        for (long long b = i; b < bytes_per_frame; b += stride) dst[b] = lut[src[b]];
    }
}

// The same for a ragged batch: one (source, destination, byte count) entry per frame; frames without an enhanced map have bytes = 0.
struct EnhDesc { const uint8_t *src; uint8_t *dst; long long bytes; };
__global__ void __launch_bounds__(256) ela_enhance_ragged_kernel(const EnhDesc *tab, const v5ela_record *recs)
{
    __shared__ uint8_t lut[256];
    const EnhDesc d = tab[blockIdx.y];
    if (d.bytes == 0) return;
    const v5ela_record &r = recs[blockIdx.y];
    int m = max((int)r.ela_max[0], max((int)r.ela_max[1], (int)r.ela_max[2]));
    if (m == 0) m = 1;
    const float scale = (float)(255.0 / (double)m);
    {
        const float v = (float)threadIdx.x * scale;
        lut[threadIdx.x] = (uint8_t)(v <= 0.0f ? 0 : (v >= 255.0f ? 255 : (int)v));
    }
    __syncthreads();
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < d.bytes; b += (long long)gridDim.x * blockDim.x)
        d.dst[b] = lut[d.src[b]];
}

// Per-video aggregation: out[g] = combine(records[g*group .. (g+1)*group)). One CTA per group, 786 32-bit words.
__global__ void __launch_bounds__(256) ela_reduce_kernel(const v5ela_record *recs, int group, v5ela_record *out)
{
    const v5ela_record *src = recs + (long long)blockIdx.x * group;
    v5ela_record &dst = out[blockIdx.x];
    for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) {        // 32-bit bins: a group of more than 2^32 - 1 pixels saturates
        unsigned long long s = 0;
        for (int k = 0; k < group; k++) s += (&src[k].ela_hist[0][0])[i];
        (&dst.ela_hist[0][0])[i] = s > 0xffffffffull ? 0xffffffffu : (uint32_t)s;
    }
    if (threadIdx.x < 8) {                 // ela_sum[3], ela_sumsq[3], tex_sumabs, tex_sumsq are 8 consecutive u64
        unsigned long long s = 0;
        for (int k = 0; k < group; k++) s += (&src[k].ela_sum[0])[threadIdx.x];
        (&dst.ela_sum[0])[threadIdx.x] = s;
    } else if (threadIdx.x == 8) {
        int m = 0;
        for (int k = 0; k < group; k++) m = max(m, (int)src[k].tex_maxabs);
        dst.tex_maxabs = (uint16_t)m;
    } else if (threadIdx.x >= 9 && threadIdx.x < 12) {
        const int c = threadIdx.x - 9;
        int m = 0;
        for (int k = 0; k < group; k++) m = max(m, (int)src[k].ela_max[c]);
        dst.ela_max[c] = (uint8_t)m;
        dst.pad[c] = 0;
    }
}

}  // namespace v5

namespace v5m {                                         // v5ela_mma.cu: the launcher of the tensor-core build
cudaError_t prepare();
int launch(const v5plan::KParams &p, int inst, long long total, int max_ctas, cudaStream_t st, cudaEvent_t ev_start, cudaEvent_t ev_stop);
}

// ======================================================================================================= C ABI
#include "v5ela_handle.h"
using namespace v5host;

// The two builds of the fused kernel, indexed by v5ela_handle::block_stage.
static const struct {
    cudaError_t (*prepare)();
    int (*launch)(const v5plan::KParams &, int, long long, int, cudaStream_t, cudaEvent_t, cudaEvent_t);
} fused_builds[2] = {{v5::prepare, v5::launch}, {v5m::prepare, v5m::launch}};
static_assert(V5ELA_BLOCKS_SMEM == 0 && V5ELA_BLOCKS_MMA == 1, "fused_builds");

// Launches the planned fused kernel with the handle's block stage, then the finalize kernel: the tail of every analyze call.
static int launch_fused(v5ela_handle *h, const v5plan::KParams &p, int inst, long long total, cudaStream_t st)
{
    const bool prof = h->profiling && h->prof_used + 2 <= h->prof_events.size();
    const int rc = fused_builds[h->block_stage].launch(p, inst, total, h->sm_count * h->ctas_per_sm, st,
                                                       prof ? static_cast<cudaEvent_t>(h->prof_events[h->prof_used]) : nullptr,
                                                       prof ? static_cast<cudaEvent_t>(h->prof_events[h->prof_used + 1]) : nullptr);
    if (rc != 0) return fail(h, V5ELA_ERR_CUDA, "fused kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
    if (inst != v5plan::INST_SWEEP) h->last_inst = inst == v5plan::INST_RAGGED ? V5ELA_INST_GENERAL : inst;
    if (prof) h->prof_used += 2;
    v5::ela_finalize_kernel<<<p.n, 96, 0, st>>>(p.records, p.n);
    V5_CUDA(h, cudaGetLastError());
    h->launches += 2;
    return V5ELA_OK;
}

// The handle's table staging buffer (h_table) and its device copy (d_table), both at least `need` bytes, ready to be refilled: waits,
// on the host, until the previous call's upload out of h_table has completed.
static int staging_table(v5ela_handle *h, size_t need)
{
    int rc;
    if (h->h_table.capacity() < need || h->d_table.capacity() < need) {   // the staging buffer and its device copy grow together
        if (h->ev_table) cudaEventSynchronize(h->ev_table);
        h->h_table.reset();
        h->d_table.reset();
        const size_t cap = need < 4096 ? 4096 : need * 2;
        if ((rc = h->h_table.ensure(h, need, cap)) || (rc = h->d_table.ensure(h, cap))) return rc;
    }
    V5_CUDA(h, h->ev_table.create());
    V5_CUDA(h, cudaEventSynchronize(h->ev_table));
    return 0;
}

extern "C" {

int v5ela_abi_version(void) { return V5ELA_ABI_VERSION; }
size_t v5ela_record_bytes(void) { return sizeof(v5ela_record); }

const char *v5ela_status_string(int status)
{
    switch (status) {
        case V5ELA_OK: return "ok";
        case V5ELA_ERR_INVALID: return "invalid argument";
        case V5ELA_ERR_CUDA: return "CUDA error";
        case V5ELA_ERR_NO_DEVICE: return "no sm_100 CUDA device";
        case V5ELA_ERR_NOMEM: return "out of memory";
        case V5ELA_ERR_UNSUPPORTED: return "unsupported JPEG flavour";
        default: return "unknown status";
    }
}

int v5ela_create(int device, v5ela_handle **out)
{
    if (!out) return V5ELA_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return V5ELA_ERR_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return V5ELA_ERR_NO_DEVICE;
    if (prop.major != 10) return V5ELA_ERR_NO_DEVICE;       // the library carries sm_100a SASS only
    v5ela_handle *h = new (std::nothrow) v5ela_handle();
    if (!h) return V5ELA_ERR_NOMEM;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    v5plan::quant_tables(h->quality, h->luma, h->chroma);
    DeviceGuard guard(device);
    if (fused_builds[0].prepare() != cudaSuccess || fused_builds[1].prepare() != cudaSuccess) {
        delete h;
        return V5ELA_ERR_CUDA;
    }
    {   // per-lane operand fragments of the tensor-core block stage: 32 x 128 bytes, fixed for the life of the handle
        v5plan::LaneConsts lc[32];
        if (!v5::mma::make_lane_consts(lc) || h->d_lane_consts.ensure(h, sizeof(lc)) != 0 ||
            cudaMemcpy(h->d_lane_consts, lc, sizeof(lc), cudaMemcpyHostToDevice) != cudaSuccess) {
            delete h;
            return V5ELA_ERR_CUDA;
        }
    }
    const char *env = getenv("V5ELA_SEG_ROWS");
    if (env) h->seg_rows = atoi(env);
    env = getenv("V5ELA_DECOMP");                             // tuning knob: "rounds,tail_seg_rows,tail_eighths"
    if (env && sscanf(env, "%d,%d,%d", &h->decomp[0], &h->decomp[1], &h->decomp[2]) == 3 && h->decomp[0] >= 1 && h->decomp[1] >= 4)
        h->decomp_set = true;
    env = getenv("V5ELA_CTAS_PER_SM");                        // tuning knob: launch fewer persistent CTAs than fit
    if (env && atoi(env) >= 1 && atoi(env) <= v5plan::MIN_CTAS) h->ctas_per_sm = atoi(env);
    env = getenv("V5ELA_BLOCK_STAGE");                        // "mma" / "smem": default block stage of new handles (A/B runs)
    if (env) h->block_stage = !strcmp(env, "mma") ? V5ELA_BLOCKS_MMA : (!strcmp(env, "smem") ? V5ELA_BLOCKS_SMEM : h->block_stage);
    env = getenv("V5ELA_HOST_CHUNK");
    if (env) h->host_chunk_frames = atoi(env);
    *out = h;
    return V5ELA_OK;
}

int v5ela_destroy(v5ela_handle *h)
{
    if (!h) return V5ELA_ERR_INVALID;
    DeviceGuard guard(h->device);                                // the members release what they own on the handle's device
    delete h;
    return V5ELA_OK;
}

const char *v5ela_last_error(const v5ela_handle *h) { return h ? h->err : "null handle"; }

int v5ela_set_quality(v5ela_handle *h, int quality)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (quality < 1 || quality > 100) return fail(h, V5ELA_ERR_INVALID, "quality must be in 1..100%s");
    h->quality = quality;
    v5plan::quant_tables(quality, h->luma, h->chroma);
    return V5ELA_OK;
}

int v5ela_get_quality(const v5ela_handle *h) { return h ? h->quality : V5ELA_ERR_INVALID; }

int v5ela_get_quant_tables(const v5ela_handle *h, uint16_t luma_host[64], uint16_t chroma_host[64])
{
    if (!h || !luma_host || !chroma_host) return V5ELA_ERR_INVALID;
    memcpy(luma_host, h->luma, sizeof(h->luma));
    memcpy(chroma_host, h->chroma, sizeof(h->chroma));
    return V5ELA_OK;
}

int v5ela_analyze(v5ela_handle *h, const uint8_t *d_rgb, int n, int height, int width, int64_t frame_stride_bytes,
                  int64_t row_stride_bytes, void *d_records, uint8_t *d_residual, void *cuda_stream)
{
    return v5ela_analyze_ex(h, d_rgb, n, height, width, frame_stride_bytes, row_stride_bytes, d_records, d_residual, nullptr, cuda_stream);
}

int v5ela_analyze_ex(v5ela_handle *h, const uint8_t *d_rgb, int n, int height, int width, int64_t frame_stride_bytes,
                     int64_t row_stride_bytes, void *d_records, uint8_t *d_residual, uint32_t *d_tex_hist, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // the ticket counter is handle-owned
    if (const int rc = h->d_ticket.ensure(h, sizeof(unsigned int))) return rc;
    v5plan::KParams p;
    if (v5plan::fill_params(p, d_rgb, n, height, width, frame_stride_bytes, row_stride_bytes, static_cast<v5ela_record *>(d_records),
                            d_residual, h->quality, h->seg_rows, 2 * h->sm_count * h->ctas_per_sm, h->decomp_set ? h->decomp : nullptr) != 0)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze: bad pointer, size or stride%s");
    const long long total = v5plan::total_work_items(p);
    if (total > 0x7fffffffLL) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze: batch too large%s");
    p.tex_hist = d_tex_hist;
    p.ticket = h->d_ticket;
    p.lane_consts = h->d_lane_consts;
    V5_CUDA(h, cudaMemsetAsync(h->d_ticket, 0, sizeof(unsigned int), st));
    V5_CUDA(h, cudaMemsetAsync(d_records, 0, sizeof(v5ela_record) * (size_t)n, st));
    if (d_tex_hist) V5_CUDA(h, cudaMemsetAsync(d_tex_hist, 0, sizeof(uint32_t) * 256 * (size_t)n, st));
    return launch_fused(h, p, v5plan::choose_instantiation(p), total, st);
}

int v5ela_analyze_ragged(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, void *d_records, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!frames_host || !d_records || n < 0) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged: bad pointer or count%s");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // ticket counter and frame table are handle-owned
    int rc;
    if ((rc = h->d_ticket.ensure(h, sizeof(unsigned int)))) return rc;
    const size_t desc_bytes = (sizeof(v5plan::FrameDesc) * (size_t)n + 15) / 16 * 16, need = desc_bytes + sizeof(v5::EnhDesc) * (size_t)n;
    if ((rc = staging_table(h, need))) return rc;
    long long total = 0;
    rc = v5plan::plan_ragged(reinterpret_cast<v5plan::FrameDesc *>(static_cast<uint8_t *>(h->h_table)), frames_host, n, h->seg_rows,
                             2 * h->sm_count * h->ctas_per_sm, &total);
    if (rc == -1) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged: bad pointer, size or stride in a frame descriptor%s");
    if (rc == -2) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged: batch too large%s");
    v5::EnhDesc *et = reinterpret_cast<v5::EnhDesc *>(h->h_table + desc_bytes);
    bool any_enh = false;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        et[i].src = f.residual ? f.residual : f.enhanced;
        et[i].dst = f.enhanced;
        et[i].bytes = f.enhanced ? (long long)f.height * f.width * 3 : 0;
        any_enh = any_enh || f.enhanced;
    }
    V5_CUDA(h, cudaMemcpyAsync(h->d_table, h->h_table, need, cudaMemcpyHostToDevice, st));
    V5_CUDA(h, cudaEventRecord(h->ev_table, st));
    V5_CUDA(h, cudaMemsetAsync(h->d_ticket, 0, sizeof(unsigned int), st));
    V5_CUDA(h, cudaMemsetAsync(d_records, 0, sizeof(v5ela_record) * (size_t)n, st));
    v5plan::KParams p;
    memset(&p, 0, sizeof(p));
    p.records = static_cast<v5ela_record *>(d_records);
    p.n = n;
    p.ticket = h->d_ticket;
    p.lane_consts = h->d_lane_consts;
    p.frames = reinterpret_cast<const v5plan::FrameDesc *>(static_cast<uint8_t *>(h->d_table));
    v5plan::fill_quant(p.q, h->quality);
    if ((rc = launch_fused(h, p, v5plan::choose_instantiation(p), total, st))) return rc;
    if (any_enh) {
        if (n > 65535) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged: more than 65535 frames with enhanced maps%s");
        v5::ela_enhance_ragged_kernel<<<dim3(32, (unsigned)n), 256, 0, st>>>(
            reinterpret_cast<const v5::EnhDesc *>(h->d_table + desc_bytes), static_cast<const v5ela_record *>(d_records));
        V5_CUDA(h, cudaGetLastError());
        h->launches += 1;
    }
    return V5ELA_OK;
}

int v5ela_analyze_ragged_host(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, void *records_host)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!frames_host || !records_host || n < 0) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged_host: bad pointer or count%s");
    DeviceGuard guard(h->device);
    int rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    ScratchOrder order(h, st);
    // device arena: per frame the pixels (rows packed), then the maps it asked for; every part 256-byte aligned
    std::vector<v5ela_frame_desc> dev((size_t)n);
    std::vector<size_t> off_in((size_t)n), off_res((size_t)n), off_enh((size_t)n);
    size_t total = 0;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        if (!f.rgb || f.height <= 0 || f.width <= 0 || f.height > 65536 || f.width > 65536 || f.row_stride_bytes < (int64_t)3 * f.width)
            return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_ragged_host: bad pointer, size or stride in a frame descriptor%s");
        const size_t bytes = ((size_t)f.height * f.width * 3 + 255) / 256 * 256;
        off_in[i] = total; total += bytes;
        off_res[i] = total; total += (f.residual || f.enhanced) ? bytes : 0;
        off_enh[i] = total; total += f.enhanced ? bytes : 0;
    }
    if ((rc = h->d_in.ensure(h, total))) return rc;
    if ((rc = h->d_rec.ensure(h, sizeof(v5ela_record) * (size_t)n))) return rc;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        V5_CUDA(h, cudaMemcpy2DAsync(h->d_in + off_in[i], (size_t)3 * f.width, f.rgb, (size_t)f.row_stride_bytes, (size_t)3 * f.width,
                                     (size_t)f.height, cudaMemcpyHostToDevice, st));
        dev[i].rgb = h->d_in + off_in[i];
        dev[i].height = f.height; dev[i].width = f.width;
        dev[i].row_stride_bytes = (int64_t)3 * f.width;
        dev[i].residual = (f.residual || f.enhanced) ? h->d_in + off_res[i] : nullptr;
        dev[i].enhanced = f.enhanced ? h->d_in + off_enh[i] : nullptr;
    }
    rc = v5ela_analyze_ragged(h, dev.data(), n, h->d_rec, st);
    if (rc) return rc;
    V5_CUDA(h, cudaMemcpyAsync(records_host, h->d_rec, sizeof(v5ela_record) * (size_t)n, cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        const size_t bytes = (size_t)f.height * f.width * 3;
        if (f.residual) V5_CUDA(h, cudaMemcpyAsync(f.residual, h->d_in + off_res[i], bytes, cudaMemcpyDeviceToHost, st));
        if (f.enhanced) V5_CUDA(h, cudaMemcpyAsync(f.enhanced, h->d_in + off_enh[i], bytes, cudaMemcpyDeviceToHost, st));
    }
    V5_CUDA(h, cudaStreamSynchronize(st));
    return V5ELA_OK;
} V5_CATCH(h)

// The sweep's refusal, in v5ela_last_error: the frame or the quality index it names.
static int sweep_refused(v5ela_handle *h, const char *fn, const v5plan::SweepPlan &P)
{
    if (P.bad_frame >= 0) snprintf(h->err, sizeof(h->err), "%s: frame %d: %s", fn, P.bad_frame, P.error);
    else if (P.bad_quality >= 0) snprintf(h->err, sizeof(h->err), "%s: quality %d: %s", fn, P.bad_quality, P.error);
    else snprintf(h->err, sizeof(h->err), "%s: %s", fn, P.error);
    return P.status;
}

int v5ela_analyze_sweep(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, const int *qualities_host, int nq, void *d_records,
                        uint32_t *d_ghost, void *cuda_stream)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!d_records) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_sweep: null record array%s");
    v5plan::SweepPlan P;
    v5plan::plan_sweep(P, frames_host, n, qualities_host, nq, d_ghost, h->seg_rows, 2 * h->sm_count * h->ctas_per_sm);
    if (P.status) return sweep_refused(h, "v5ela_analyze_sweep", P);
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // ticket counter and tables are handle-owned
    int rc;
    if ((rc = h->d_ticket.ensure(h, sizeof(unsigned int)))) return rc;
    if ((rc = staging_table(h, P.table_bytes))) return rc;
    uint8_t *tab = h->h_table;
    memcpy(tab, P.frames.data(), sizeof(v5plan::FrameDesc) * P.frames.size());
    memcpy(tab + P.off_entries, P.entries.data(), sizeof(v5plan::SweepEntry) * P.entries.size());
    memcpy(tab + P.off_quant, P.quant.data(), sizeof(v5plan::QuantTab) * P.quant.size());
    const size_t records = P.frames.size();
    V5_CUDA(h, cudaMemcpyAsync(h->d_table, h->h_table, P.table_bytes, cudaMemcpyHostToDevice, st));
    V5_CUDA(h, cudaEventRecord(h->ev_table, st));
    V5_CUDA(h, cudaMemsetAsync(h->d_ticket, 0, sizeof(unsigned int), st));
    V5_CUDA(h, cudaMemsetAsync(d_records, 0, sizeof(v5ela_record) * records, st));
    v5plan::KParams p;
    memset(&p, 0, sizeof(p));
    p.records = static_cast<v5ela_record *>(d_records);
    p.n = (int)records;
    p.ticket = h->d_ticket;
    p.lane_consts = h->d_lane_consts;
    p.frames = reinterpret_cast<const v5plan::FrameDesc *>(static_cast<uint8_t *>(h->d_table));   // the sweep's tables behind it
    return launch_fused(h, p, v5plan::INST_SWEEP, P.total, st);
} V5_CATCH(h)

int v5ela_analyze_sweep_host(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, const int *qualities_host, int nq,
                             void *records_host, uint32_t *ghost_host)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!records_host) return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_sweep_host: null record array%s");
    {   // refuse before anything is copied (the device call plans the same entries again, over the uploaded pixels)
        v5plan::SweepPlan P;
        v5plan::plan_sweep(P, frames_host, n, qualities_host, nq, nullptr, h->seg_rows, 2 * h->sm_count * h->ctas_per_sm);
        if (P.status) return sweep_refused(h, "v5ela_analyze_sweep_host", P);
    }
    DeviceGuard guard(h->device);
    int rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    ScratchOrder order(h, st);
    // device arena: per frame its pixels (rows packed), 256-byte aligned; each frame goes up once for all qualities
    std::vector<v5ela_frame_desc> dev((size_t)n);
    std::vector<size_t> off((size_t)n);
    size_t total = 0, maps = 0;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        off[(size_t)i] = total;
        total += ((size_t)f.height * f.width * 3 + 255) / 256 * 256;
        maps += (size_t)((f.height + 15) / 16) * ((f.width + 15) / 16);
    }
    const size_t records = (size_t)n * nq;
    if ((rc = h->d_in.ensure(h, total)) || (rc = h->d_rec.ensure(h, sizeof(v5ela_record) * records))) return rc;
    if (ghost_host && (rc = h->d_ghost.ensure(h, sizeof(uint32_t) * maps * nq))) return rc;
    for (int i = 0; i < n; i++) {
        const v5ela_frame_desc &f = frames_host[i];
        V5_CUDA(h, cudaMemcpy2DAsync(h->d_in + off[(size_t)i], (size_t)3 * f.width, f.rgb, (size_t)f.row_stride_bytes, (size_t)3 * f.width,
                                     (size_t)f.height, cudaMemcpyHostToDevice, st));
        dev[(size_t)i] = v5ela_frame_desc{h->d_in + off[(size_t)i], f.height, f.width, (int64_t)3 * f.width, nullptr, nullptr};
    }
    if ((rc = v5ela_analyze_sweep(h, dev.data(), n, qualities_host, nq, h->d_rec, ghost_host ? (uint32_t *)h->d_ghost : nullptr, st))) return rc;
    V5_CUDA(h, cudaMemcpyAsync(records_host, h->d_rec, sizeof(v5ela_record) * records, cudaMemcpyDeviceToHost, st));
    if (ghost_host) V5_CUDA(h, cudaMemcpyAsync(ghost_host, h->d_ghost, sizeof(uint32_t) * maps * nq, cudaMemcpyDeviceToHost, st));
    V5_CUDA(h, cudaStreamSynchronize(st));
    return V5ELA_OK;
} V5_CATCH(h)

int v5ela_enhance(v5ela_handle *h, const uint8_t *d_residual, const void *d_records, int n, int height, int width,
                  uint8_t *d_enhanced, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!d_residual || !d_records || !d_enhanced || n < 0 || height <= 0 || width <= 0)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_enhance: bad pointer or size%s");
    DeviceGuard guard(h->device);
    const long long bytes = (long long)height * width * 3;
    long long bx = (bytes / 16 + 255) / 256;
    if (bx < 1) bx = 1;
    if (bx > 4LL * h->sm_count) bx = 4LL * h->sm_count;
    if (n > 65535) return fail(h, V5ELA_ERR_INVALID, "v5ela_enhance: more than 65535 frames per call%s");
    v5::ela_enhance_kernel<<<dim3((unsigned)bx, (unsigned)n), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        d_residual, static_cast<const v5ela_record *>(d_records), d_enhanced, bytes);
    V5_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return V5ELA_OK;
}

int v5ela_reduce_records(v5ela_handle *h, const void *d_records, int n, int group, void *d_out, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!d_records || !d_out || n < 0 || group <= 0 || n % group != 0)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_reduce_records: n must be a positive multiple of group%s");
    DeviceGuard guard(h->device);
    v5::ela_reduce_kernel<<<n / group, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        static_cast<const v5ela_record *>(d_records), group, static_cast<v5ela_record *>(d_out));
    V5_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return V5ELA_OK;
}

int v5ela_analyze_host(v5ela_handle *h, const uint8_t *rgb_host, int n, int height, int width, void *records_host,
                       uint8_t *residual_host_or_null, uint8_t *enhanced_host_or_null, void *cuda_stream)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!rgb_host || !records_host || n < 0 || height <= 0 || width <= 0)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_analyze_host: bad pointer or size%s");
    DeviceGuard guard(h->device);
    int rc;
    cudaStream_t own;
    if ((rc = internal_stream(h, &own))) return rc;
    V5_CUDA(h, h->copy_stream.create());
    V5_CUDA(h, h->work_stream.create());
    V5_CUDA(h, h->ev_fork.create());
    V5_CUDA(h, h->ev_join_copy.create());
    V5_CUDA(h, h->ev_join_work.create());
    const size_t fbytes = (size_t)height * width * 3, in_bytes = fbytes * n, rec_bytes = sizeof(v5ela_record) * (size_t)n;
    const bool want_map = residual_host_or_null || enhanced_host_or_null;
    if ((rc = h->d_in.ensure(h, in_bytes))) return rc;
    if ((rc = h->d_rec.ensure(h, rec_bytes))) return rc;
    if (want_map && (rc = h->d_res.ensure(h, in_bytes))) return rc;
    if (enhanced_host_or_null && (rc = h->d_enh.ensure(h, in_bytes))) return rc;

    // chunking: ~64 MB of frames per chunk keeps the copy engine and the SMs both busy
    int chunk = h->host_chunk_frames > 0 ? h->host_chunk_frames : (int)((64u << 20) / fbytes);
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    const int n_chunks = (n + chunk - 1) / chunk;
    while ((int)h->ev_chunk.size() < n_chunks) {
        Event e;
        V5_CUDA(h, e.create());
        h->ev_chunk.push_back(std::move(e));
    }
    cudaStream_t user = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : own;
    cudaStream_t cs = h->copy_stream, ws = h->work_stream;
    ScratchOrder order(h, user);                                // d_in / d_rec / d_res / d_enh and the two internal streams
    V5_CUDA(h, cudaEventRecord(h->ev_fork, user));
    V5_CUDA(h, cudaStreamWaitEvent(cs, h->ev_fork, 0));
    V5_CUDA(h, cudaStreamWaitEvent(ws, h->ev_fork, 0));
    for (int c = 0; c < n_chunks; c++) {
        const int f0 = c * chunk, fn = (f0 + chunk <= n ? chunk : n - f0);
        const size_t off = fbytes * f0, bytes = fbytes * fn, roff = sizeof(v5ela_record) * (size_t)f0;
        V5_CUDA(h, cudaMemcpyAsync(h->d_in + off, rgb_host + off, bytes, cudaMemcpyHostToDevice, cs));
        V5_CUDA(h, cudaEventRecord(h->ev_chunk[c], cs));
        V5_CUDA(h, cudaStreamWaitEvent(ws, h->ev_chunk[c], 0));
        rc = v5ela_analyze(h, h->d_in + off, fn, height, width, (int64_t)fbytes, (int64_t)width * 3, h->d_rec + roff,
                           want_map ? h->d_res + off : nullptr, ws);
        if (rc) return rc;
        if (residual_host_or_null)
            V5_CUDA(h, cudaMemcpyAsync(residual_host_or_null + off, h->d_res + off, bytes, cudaMemcpyDeviceToHost, ws));
        if (enhanced_host_or_null) {
            rc = v5ela_enhance(h, h->d_res + off, h->d_rec + roff, fn, height, width, h->d_enh + off, ws);
            if (rc) return rc;
            V5_CUDA(h, cudaMemcpyAsync(enhanced_host_or_null + off, h->d_enh + off, bytes, cudaMemcpyDeviceToHost, ws));
        }
    }
    V5_CUDA(h, cudaMemcpyAsync(records_host, h->d_rec, rec_bytes, cudaMemcpyDeviceToHost, ws));
    V5_CUDA(h, cudaEventRecord(h->ev_join_copy, cs));
    V5_CUDA(h, cudaEventRecord(h->ev_join_work, ws));
    V5_CUDA(h, cudaStreamWaitEvent(user, h->ev_join_copy, 0));
    V5_CUDA(h, cudaStreamWaitEvent(user, h->ev_join_work, 0));
    if (!cuda_stream) V5_CUDA(h, cudaStreamSynchronize(user));
    return V5ELA_OK;
} V5_CATCH(h)

// threads per CTA of the FFT kernels: 256; 512 measured no faster (profiles/r02/spectrum.txt). V5ELA_FFT_THREADS overrides
// (tuning knob: 128 / 256 / 512)
static unsigned fft_threads(int points)
{
    if (const char *env = getenv("V5ELA_FFT_THREADS")) {
        const int v = atoi(env);
        if (v == 128 || v == 256 || v == 512) return (unsigned)v;
    }
    (void)points;
    return 256u;
}

// V5ELA_FFT=0 sends every frame down the exact-size DFT (tests compare the two paths); read on every call.
static bool fft_enabled()
{
    const char *env = getenv("V5ELA_FFT");
    return !(env && atoi(env) == 0);
}

// Workspace cap of one pass of a spectrum call: ~1 GiB of float64 intermediates, or V5ELA_SPEC_CHUNK_MB (tuning knob).
static size_t spec_chunk_bytes()
{
    if (const char *env = getenv("V5ELA_SPEC_CHUNK_MB")) {
        const long v = atol(env);
        if (v >= 1 && v <= 4096) return (size_t)v << 20;
    }
    return (size_t)1 << 30;
}

int v5ela_spectrum(v5ela_handle *h, const uint8_t *d_gray, int n, int height, int width, int64_t frame_stride_bytes,
                   int64_t row_stride_bytes, uint8_t *d_out, void *cuda_stream)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!d_gray || !d_out || n < 0 || height <= 0 || width <= 0 || height > 65536 || width > 65536 ||
        row_stride_bytes < width || (n > 1 && frame_stride_bytes < row_stride_bytes * (int64_t)height))
        return fail(h, V5ELA_ERR_INVALID, "v5ela_spectrum: bad pointer, size or stride%s");
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // twiddle tables, d_g / d_ms / d_minmax
    const int wh = width / 2 + 1;
    int rc;
    if (h->tw_w_n != width) {
        if ((rc = h->tw_w.ensure(h, sizeof(double2) * (size_t)width))) return rc;
        v5fft::twiddle_kernel<<<(width + 255) / 256, 256, 0, st>>>(h->tw_w, width);
        h->tw_w_n = width;
        h->launches++;
    }
    if (h->tw_h_n != height) {
        if ((rc = h->tw_h.ensure(h, sizeof(double2) * (size_t)height))) return rc;
        v5fft::twiddle_kernel<<<(height + 255) / 256, 256, 0, st>>>(h->tw_h, height);
        h->tw_h_n = height;
        h->launches++;
    }
    // frames per pass: keep the float64 workspace (24 bytes per half-spectrum sample) under ~1 GiB. Smaller, L2-sized passes were
    // measured and are SLOWER (profiles/r02/spectrum.txt: 64 MB -10 %, 32 MB -25 %): the passes are bound by their own latency chains,
    // not by where the intermediate lives.
    const size_t per_frame = (size_t)height * wh;
    int chunk = (int)(spec_chunk_bytes() / (per_frame * 24));
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    if (chunk > 65535) chunk = 65535;
    if ((rc = h->d_g.ensure(h, per_frame * 16 * chunk))) return rc;
    if ((rc = h->d_ms.ensure(h, per_frame * 8 * chunk))) return rc;
    if ((rc = h->d_minmax.ensure(h, sizeof(unsigned long long) * 2 * (size_t)chunk))) return rc;
    const dim3 grid((wh + v5fft::TILE - 1) / v5fft::TILE, (height + v5fft::TILE - 1) / v5fft::TILE, 1);
    // Sizes with only 2/3/5 as prime factors take the shared-memory FFT; anything else (crops are arbitrary) the exact-size
    // DFT products (v5fft::fft_path).
    v5fft::FftPlan plan_w, plan_h;
    v5fft::FftShape shape;
    const bool fast = v5fft::fft_path(fft_enabled(), height, width, plan_w, plan_h, shape) && n <= 65535;
    const int cc = shape.cc;
    const size_t rows_smem = shape.rows_smem, cols_smem = shape.cols_smem;
    if (fast && !h->fft_attr_set) {
        V5_CUDA(h, cudaFuncSetAttribute(v5fft::fft_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 << 10));
        V5_CUDA(h, cudaFuncSetAttribute(v5fft::fft_cols_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 << 10));
        h->fft_attr_set = true;
    }
    for (int f0 = 0; f0 < n; f0 += chunk) {
        const int fn = f0 + chunk <= n ? chunk : n - f0;
        // min/max slots: {~0, 0} per frame
        V5_CUDA(h, cudaMemsetAsync(h->d_minmax, 0, sizeof(unsigned long long) * 2 * (size_t)fn, st));
        V5_CUDA(h, cudaMemset2DAsync(h->d_minmax, 16, 0xff, 8, (size_t)fn, st));
        if (fast) {
            v5fft::fft_rows_kernel<<<dim3((unsigned)((height + 1) / 2), (unsigned)fn), fft_threads(width), rows_smem, st>>>(
                d_gray + (int64_t)f0 * frame_stride_bytes, frame_stride_bytes, row_stride_bytes, height, width, wh, plan_w, h->tw_w, h->d_g);
            V5_CUDA(h, cudaGetLastError());
            v5fft::fft_cols_kernel<<<dim3((unsigned)((wh + cc - 1) / cc), (unsigned)fn), fft_threads(cc * height), cols_smem, st>>>(
                h->d_g, height, wh, cc, plan_h, h->tw_h, h->d_ms, h->d_minmax);
            V5_CUDA(h, cudaGetLastError());
        } else {
            dim3 gr = grid;
            gr.z = (unsigned)fn;
            v5fft::dft_rows_kernel<<<gr, 256, 0, st>>>(d_gray + (int64_t)f0 * frame_stride_bytes, frame_stride_bytes, row_stride_bytes,
                                                       height, width, wh, h->tw_w, h->d_g);
            V5_CUDA(h, cudaGetLastError());
            v5fft::dft_cols_kernel<<<gr, 256, 0, st>>>(h->d_g, height, wh, h->tw_h, h->d_ms, h->d_minmax);
            V5_CUDA(h, cudaGetLastError());
        }
        // every CTA walks ~16 rows: the per-thread set-up (the double-precision 255 / (max - min)) is paid once per 16 pixels
        const unsigned bx = (unsigned)((width + 255) / 256);
        unsigned by = (unsigned)((height + 15) / 16);
        by = by < 1 ? 1 : (by > 65535 ? 65535 : by);
        v5fft::spectrum_image_kernel<<<dim3(bx, by, (unsigned)fn), 256, 0, st>>>(h->d_ms, h->d_minmax, height, width, wh,
                                                                                  d_out + (int64_t)f0 * height * width);
        V5_CUDA(h, cudaGetLastError());
        h->launches += 3;
    }
    return V5ELA_OK;
}

int v5ela_spectrum_host(v5ela_handle *h, const uint8_t *gray_host, int n, int height, int width, uint8_t *out_host)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!gray_host || !out_host || n < 0 || height <= 0 || width <= 0)
        return fail(h, V5ELA_ERR_INVALID, "v5ela_spectrum_host: bad pointer or size%s");
    DeviceGuard guard(h->device);
    int rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    const size_t bytes = (size_t)n * height * width;
    if ((rc = h->d_gray.ensure(h, bytes))) return rc;
    if ((rc = h->d_spec.ensure(h, bytes))) return rc;
    V5_CUDA(h, cudaMemcpyAsync(h->d_gray, gray_host, bytes, cudaMemcpyHostToDevice, st));
    rc = v5ela_spectrum(h, h->d_gray, n, height, width, (int64_t)height * width, width, h->d_spec, st);
    if (rc) return rc;
    V5_CUDA(h, cudaMemcpyAsync(out_host, h->d_spec, bytes, cudaMemcpyDeviceToHost, st));
    V5_CUDA(h, cudaStreamSynchronize(st));
    return V5ELA_OK;
}

int v5ela_spectrum_ragged(v5ela_handle *h, const v5ela_gray_desc *frames_host, int n, void *cuda_stream)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    v5fft::SpecPlan P;
    v5fft::plan_spectrum_ragged(frames_host, n, fft_enabled(), spec_chunk_bytes(), P);
    if (P.status) {
        if (P.bad_frame >= 0) snprintf(h->err, sizeof(h->err), "v5ela_spectrum_ragged: frame %d: %s", P.bad_frame, P.error);
        else snprintf(h->err, sizeof(h->err), "v5ela_spectrum_ragged: %s", P.error);
        return P.status;
    }
    DeviceGuard guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ScratchOrder order(h, st);                                  // twiddle arena, d_g / d_ms / d_minmax, plan table
    int rc;
    if ((rc = h->tw_rag.ensure(h, sizeof(double2) * P.tw_elems)) || (rc = h->d_g.ensure(h, sizeof(double2) * P.g_max)) ||
        (rc = h->d_ms.ensure(h, sizeof(double) * P.ms_max)) || (rc = h->d_minmax.ensure(h, sizeof(unsigned long long) * 2 * (size_t)P.mm_max)))
        return rc;
    const size_t need = P.table_bytes;
    if ((rc = staging_table(h, need))) return rc;
    uint8_t *tab = h->h_table;
    memcpy(tab + P.off_sizes, P.sizes.data(), sizeof(v5fft::SpecSize) * P.sizes.size());
    memcpy(tab + P.off_frames, P.frames.data(), sizeof(v5fft::SpecFrame) * P.frames.size());
    memcpy(tab + P.off_tw_base, P.tw_base.data(), sizeof(uint32_t) * P.tw_base.size());
    memcpy(tab + P.off_bases, P.bases.data(), sizeof(uint32_t) * P.bases.size());
    V5_CUDA(h, cudaMemcpyAsync(h->d_table, h->h_table, need, cudaMemcpyHostToDevice, st));
    V5_CUDA(h, cudaEventRecord(h->ev_table, st));
    if (!h->fft_rag_attr_set) {
        V5_CUDA(h, cudaFuncSetAttribute(v5fft::fft_rows_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v5fft::FFT_SMEM_MAX));
        V5_CUDA(h, cudaFuncSetAttribute(v5fft::fft_cols_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v5fft::FFT_SMEM_MAX));
        h->fft_rag_attr_set = true;
    }
    const uint8_t *dt = h->d_table;
    const auto *sizes = reinterpret_cast<const v5fft::SpecSize *>(dt + P.off_sizes);
    const auto *frames = reinterpret_cast<const v5fft::SpecFrame *>(dt + P.off_frames);
    const auto *bases = reinterpret_cast<const uint32_t *>(dt + P.off_bases);
    v5fft::twiddle_ragged_kernel<<<P.tw_base.back(), 256, 0, st>>>(sizes, (int)P.sizes.size(), reinterpret_cast<const uint32_t *>(dt + P.off_tw_base),
                                                                   h->tw_rag);
    V5_CUDA(h, cudaGetLastError());
    h->launches++;
    for (const v5fft::SpecChunk &C : P.chunks) {
        const v5fft::SpecFrame *cf = frames + C.f0;
        const uint32_t *base = bases + C.off_base;
        auto kind = [&](int k) { return base + (size_t)k * (C.n + 1); };
        // min/max slots: {~0, 0} per frame
        V5_CUDA(h, cudaMemsetAsync(h->d_minmax, 0, sizeof(unsigned long long) * 2 * (size_t)C.n, st));
        V5_CUDA(h, cudaMemset2DAsync(h->d_minmax, 16, 0xff, 8, (size_t)C.n, st));
        if (C.ctas[v5fft::L_FFT_ROWS]) {
            v5fft::fft_rows_ragged_kernel<<<C.ctas[v5fft::L_FFT_ROWS], 256, C.rows_smem, st>>>(cf, C.n, kind(v5fft::L_FFT_ROWS), sizes, h->tw_rag, h->d_g);
            V5_CUDA(h, cudaGetLastError());
            v5fft::fft_cols_ragged_kernel<<<C.ctas[v5fft::L_FFT_COLS], 256, C.cols_smem, st>>>(cf, C.n, kind(v5fft::L_FFT_COLS), sizes, h->tw_rag, h->d_g,
                                                                                              h->d_ms, h->d_minmax);
            V5_CUDA(h, cudaGetLastError());
            h->launches += 2;
        }
        if (C.ctas[v5fft::L_DFT_ROWS]) {
            v5fft::dft_rows_ragged_kernel<<<C.ctas[v5fft::L_DFT_ROWS], 256, 0, st>>>(cf, C.n, kind(v5fft::L_DFT_ROWS), sizes, h->tw_rag, h->d_g);
            V5_CUDA(h, cudaGetLastError());
            v5fft::dft_cols_ragged_kernel<<<C.ctas[v5fft::L_DFT_COLS], 256, 0, st>>>(cf, C.n, kind(v5fft::L_DFT_COLS), sizes, h->tw_rag, h->d_g, h->d_ms,
                                                                                    h->d_minmax);
            V5_CUDA(h, cudaGetLastError());
            h->launches += 2;
        }
        v5fft::spectrum_image_ragged_kernel<<<C.ctas[v5fft::L_IMAGE], 256, 0, st>>>(cf, C.n, kind(v5fft::L_IMAGE), h->d_ms, h->d_minmax);
        V5_CUDA(h, cudaGetLastError());
        h->launches++;
    }
    return V5ELA_OK;
} V5_CATCH(h)

int v5ela_spectrum_ragged_host(v5ela_handle *h, const v5ela_gray_desc *frames_host, int n)
try {
    if (!h) return V5ELA_ERR_INVALID;
    if (n == 0) return V5ELA_OK;
    if (!frames_host || n < 0) return fail(h, V5ELA_ERR_INVALID, "v5ela_spectrum_ragged_host: null descriptor array or negative count%s");
    // device arena: per image its pixels (rows packed), 256-byte aligned; the images' spectra at the same offsets of d_spec
    std::vector<v5ela_gray_desc> dev((size_t)n);
    std::vector<size_t> off((size_t)n);
    size_t total = 0;
    for (int i = 0; i < n; i++) {
        if (const char *why = v5fft::gray_desc_error(frames_host[i])) {
            snprintf(h->err, sizeof(h->err), "v5ela_spectrum_ragged_host: frame %d: %s", i, why);
            return V5ELA_ERR_INVALID;
        }
        off[(size_t)i] = total;
        total += ((size_t)frames_host[i].height * frames_host[i].width + 255) / 256 * 256;
    }
    DeviceGuard guard(h->device);
    int rc;
    cudaStream_t st;
    if ((rc = internal_stream(h, &st))) return rc;
    ScratchOrder order(h, st);                                  // d_gray / d_spec
    if ((rc = h->d_gray.ensure(h, total)) || (rc = h->d_spec.ensure(h, total))) return rc;
    for (int i = 0; i < n; i++) {
        const v5ela_gray_desc &f = frames_host[i];
        V5_CUDA(h, cudaMemcpy2DAsync(h->d_gray + off[(size_t)i], (size_t)f.width, f.gray, (size_t)f.row_stride_bytes, (size_t)f.width,
                                     (size_t)f.height, cudaMemcpyHostToDevice, st));
        dev[(size_t)i].gray = h->d_gray + off[(size_t)i];
        dev[(size_t)i].height = f.height;
        dev[(size_t)i].width = f.width;
        dev[(size_t)i].row_stride_bytes = f.width;
        dev[(size_t)i].out = h->d_spec + off[(size_t)i];
    }
    if ((rc = v5ela_spectrum_ragged(h, dev.data(), n, st))) return rc;
    for (int i = 0; i < n; i++) {
        const v5ela_gray_desc &f = frames_host[i];
        V5_CUDA(h, cudaMemcpyAsync(f.out, h->d_spec + off[(size_t)i], (size_t)f.height * f.width, cudaMemcpyDeviceToHost, st));
    }
    V5_CUDA(h, cudaStreamSynchronize(st));
    return V5ELA_OK;
} V5_CATCH(h)

int v5ela_profile_enable(v5ela_handle *h, int enable)
try {
    if (!h) return V5ELA_ERR_INVALID;
    DeviceGuard guard(h->device);
    if (enable && h->prof_events.empty()) {
        h->prof_events.resize(8192);
        for (Event &e : h->prof_events) V5_CUDA(h, e.create(cudaEventDefault));
    }
    h->profiling = enable != 0;
    return V5ELA_OK;
} V5_CATCH(h)

int v5ela_profile_read(v5ela_handle *h, double *fused_ms_sum, int64_t *fused_launches, int reset)
{
    if (!h || !fused_ms_sum || !fused_launches) return V5ELA_ERR_INVALID;
    DeviceGuard guard(h->device);
    double sum = 0.0;
    for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
        float ms = 0.f;
        V5_CUDA(h, cudaEventSynchronize(h->prof_events[i + 1]));
        V5_CUDA(h, cudaEventElapsedTime(&ms, h->prof_events[i], h->prof_events[i + 1]));
        sum += ms;
    }
    *fused_ms_sum = sum;
    *fused_launches = (int64_t)(h->prof_used / 2);
    if (reset) h->prof_used = 0;
    return V5ELA_OK;
}

int64_t v5ela_launch_count(const v5ela_handle *h) { return h ? h->launches : 0; }

int v5ela_last_instantiation(const v5ela_handle *h) { return h ? h->last_inst : V5ELA_ERR_INVALID; }

int v5ela_set_block_stage(v5ela_handle *h, int mode)
{
    if (!h) return V5ELA_ERR_INVALID;
    if (mode != V5ELA_BLOCKS_SMEM && mode != V5ELA_BLOCKS_MMA) return fail(h, V5ELA_ERR_INVALID, "block stage must be V5ELA_BLOCKS_SMEM or V5ELA_BLOCKS_MMA%s");
    h->block_stage = mode;
    return V5ELA_OK;
}

int v5ela_get_block_stage(const v5ela_handle *h) { return h ? h->block_stage : V5ELA_ERR_INVALID; }


}  // extern "C"
