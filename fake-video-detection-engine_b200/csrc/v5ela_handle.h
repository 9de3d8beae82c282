// v5ela_handle.h — the handle behind the C ABI (include/v5ela.h) and small host helpers shared by the translation units
// of libv5ela.so (v5ela.cu: ELA + spectrum; v5jpeg.cu: codec rows).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <vector>

#include "v5ela.h"
#include "v5ela_device.cuh"

struct v5ela_handle {
    int device = 0;
    int quality = 90;
    int sm_count = 0;
    int seg_rows = 0;                      // 0 = default
    int decomp[3] = {0, 0, 0};             // V5ELA_DECOMP=a,b,c development knob (fill_params' tune); decomp_set = it was given
    bool decomp_set = false;
    int ctas_per_sm = v5plan::MIN_CTAS;
    int64_t launches = 0;
    int last_inst = -1;                    // V5ELA_INST_* of the most recent fused-kernel launch
    cudaStream_t own_stream = nullptr;     // v5ela_analyze_host with a NULL stream
    cudaStream_t copy_stream = nullptr, work_stream = nullptr;   // chunk pipeline of v5ela_analyze_host
    cudaEvent_t ev_fork = nullptr, ev_join_copy = nullptr, ev_join_work = nullptr;
    std::vector<cudaEvent_t> ev_chunk;     // "chunk c has landed" events
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;  // pairs (start, stop) around the fused kernel
    size_t prof_used = 0;
    int host_chunk_frames = 0;             // 0 = auto
    uint8_t *d_in = nullptr, *d_res = nullptr, *d_enh = nullptr;
    void *d_rec = nullptr;
    unsigned int *d_ticket = nullptr;
    // ragged batches: the kernel's frame table (+ the enhancement kernel's table behind it), pinned host staging and device copy
    void *h_table = nullptr, *d_table = nullptr;
    size_t table_cap = 0;
    cudaEvent_t ev_table = nullptr;        // the last upload out of h_table has completed
    v5plan::LaneConsts *d_lane_consts = nullptr;   // 32 entries: operand fragments of the tensor-core block stage (v5ela_dctmma.cuh)
    int block_stage = V5ELA_BLOCKS_DEFAULT; // which build of the fused kernel analyze launches (v5ela_set_block_stage)
    size_t d_in_cap = 0, d_res_cap = 0, d_enh_cap = 0, d_rec_cap = 0;
    // spectrum path (v5ela_fft.cuh): twiddle tables for the last (width, height), DFT workspace
    double2 *tw_w = nullptr, *tw_h = nullptr;
    int tw_w_n = 0, tw_h_n = 0;
    bool fft_attr_set = false;
    size_t tw_w_cap = 0, tw_h_cap = 0;
    void *d_g = nullptr, *d_ms = nullptr, *d_minmax = nullptr;
    size_t d_g_cap = 0, d_ms_cap = 0, d_minmax_cap = 0;
    uint8_t *d_gray = nullptr, *d_spec = nullptr;
    size_t d_gray_cap = 0, d_spec_cap = 0;
    uint16_t luma[64], chroma[64];
    struct v5jpeg_state *jpeg = nullptr;   // codec workspace, owned by v5jpeg.cu (created on first use)
    // Scratch owned by the handle (ticket counter, host-path / spectrum / codec workspaces) is reused by every call. Calls on ONE
    // stream are ordered by the stream; a call on another stream than the previous one first waits for that call's last launch.
    cudaEvent_t ev_scratch = nullptr;
    cudaStream_t scratch_stream = nullptr;
    bool scratch_used = false;
    char err[512] = {0};
};

void v5jpeg_release(v5ela_handle *h);      // v5jpeg.cu: frees h->jpeg (device set by the caller)

namespace v5host {

inline int fail(v5ela_handle *h, int code, const char *fmt, const char *detail = "")
{
    if (h) snprintf(h->err, sizeof(h->err), fmt, detail);
    return code;
}

#define V5_CUDA(h, call)                                                                    \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) return fail((h), V5ELA_ERR_CUDA, #call ": %s", cudaGetErrorString(e_)); \
    } while (0)

// RAII around an entry point that touches handle-owned scratch on stream `st` (see v5ela_handle::ev_scratch).
struct ScratchOrder {
    v5ela_handle *h;
    cudaStream_t st;
    ScratchOrder(v5ela_handle *handle, cudaStream_t stream) : h(handle), st(stream)
    {
        if (h->scratch_used && h->scratch_stream != st) cudaStreamWaitEvent(st, h->ev_scratch, 0);
    }
    ~ScratchOrder()
    {
        if (!h->ev_scratch && cudaEventCreateWithFlags(&h->ev_scratch, cudaEventDisableTiming) != cudaSuccess) return;
        if (cudaEventRecord(h->ev_scratch, st) == cudaSuccess) {
            h->scratch_stream = st;
            h->scratch_used = true;
        }
    }
    ScratchOrder(const ScratchOrder &) = delete;
    ScratchOrder &operator=(const ScratchOrder &) = delete;
};

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

inline int ensure(v5ela_handle *h, void **ptr, size_t *cap, size_t need)
{
    if (*cap >= need) return 0;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr;
    *cap = 0;
    V5_CUDA(h, cudaMalloc(ptr, need));
    *cap = need;
    return 0;
}

}  // namespace v5host
