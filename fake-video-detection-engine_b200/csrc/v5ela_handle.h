// v5ela_handle.h — the handle behind the C ABI (include/v5ela.h) and small host helpers shared by the translation units
// of libv5ela.so (v5ela.cu: ELA + spectrum; v5jpeg.cu: codec rows).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <exception>
#include <memory>
#include <new>
#include <vector>

#include "v5ela.h"
#include "v5ela_device.cuh"

struct v5jpeg_state;

namespace v5host {

// The resources a handle owns. Each member is created or grown on first use and released by its destructor, so adding a
// workspace to the handle (or to the codec state) is adding one member. v5ela_destroy deletes the handle with its device current.

// Device memory for T, grown by ensure(): below `need` bytes it frees the old buffer and allocates exactly `need` bytes.
template <class T>
class DeviceBuf {
  public:
    DeviceBuf() = default;
    DeviceBuf(const DeviceBuf &) = delete;
    DeviceBuf &operator=(const DeviceBuf &) = delete;
    ~DeviceBuf() { reset(); }
    operator T *() const { return p_; }
    size_t capacity() const { return cap_; }
    void reset()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    int ensure(v5ela_handle *h, size_t need);

  private:
    T *p_ = nullptr;
    size_t cap_ = 0;
};

// Pinned host memory, grown by ensure(): below `need` bytes it frees the old buffer and allocates `alloc` (>= need) bytes, so
// that each caller keeps its own growth rule.
class PinnedBuf {
  public:
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf &) = delete;
    PinnedBuf &operator=(const PinnedBuf &) = delete;
    ~PinnedBuf() { reset(); }
    operator uint8_t *() const { return p_; }
    size_t capacity() const { return cap_; }
    void reset()
    {
        if (p_) cudaFreeHost(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    int ensure(v5ela_handle *h, size_t need, size_t alloc);

  private:
    uint8_t *p_ = nullptr;
    size_t cap_ = 0;
};

// A non-blocking stream; create() does nothing once it exists.
class Stream {
  public:
    Stream() = default;
    Stream(const Stream &) = delete;
    Stream &operator=(const Stream &) = delete;
    ~Stream() { if (s_) cudaStreamDestroy(s_); }
    operator cudaStream_t() const { return s_; }
    cudaError_t create() { return s_ ? cudaSuccess : cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking); }

  private:
    cudaStream_t s_ = nullptr;
};

// An event; create() does nothing once it exists. Movable, so that the handle can keep a growing std::vector of them.
class Event {
  public:
    Event() = default;
    Event(Event &&o) noexcept : e_(o.e_) { o.e_ = nullptr; }
    Event &operator=(Event &&) = delete;
    ~Event() { if (e_) cudaEventDestroy(e_); }
    operator cudaEvent_t() const { return e_; }
    cudaError_t create(unsigned flags = cudaEventDisableTiming) { return e_ ? cudaSuccess : cudaEventCreateWithFlags(&e_, flags); }

  private:
    cudaEvent_t e_ = nullptr;
};

// The codec workspace is defined in v5jpeg.cu; the handle owns it through a unique_ptr with this deleter (defined there too).
struct JpegStateDelete {
    void operator()(v5jpeg_state *s) const;
};

}  // namespace v5host

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
    v5host::Stream own_stream;             // see internal_stream
    v5host::Stream copy_stream, work_stream;   // chunk pipeline of v5ela_analyze_host
    v5host::Event ev_fork, ev_join_copy, ev_join_work;
    std::vector<v5host::Event> ev_chunk;   // "chunk c has landed" events
    bool profiling = false;
    std::vector<v5host::Event> prof_events;   // pairs (start, stop) around the fused kernel
    size_t prof_used = 0;
    int host_chunk_frames = 0;             // 0 = auto
    v5host::DeviceBuf<uint8_t> d_in, d_res, d_enh, d_rec;
    v5host::DeviceBuf<uint32_t> d_ghost;   // v5ela_analyze_sweep_host: the ghost maps
    v5host::DeviceBuf<unsigned int> d_ticket;
    // ragged batches and sweeps: the kernel's frame table (+ the enhancement kernel's, or the sweep's, tables behind it), pinned host
    // staging and device copy
    v5host::PinnedBuf h_table;
    v5host::DeviceBuf<uint8_t> d_table;
    v5host::Event ev_table;                // the last upload out of h_table has completed
    v5host::DeviceBuf<v5plan::LaneConsts> d_lane_consts;   // 32 entries: operand fragments of the tensor-core block stage (v5ela_dctmma.cuh)
    int block_stage = V5ELA_BLOCKS_DEFAULT; // which build of the fused kernel analyze launches (v5ela_set_block_stage)
    // spectrum path (v5ela_fft.cuh): twiddle tables for the last (width, height), DFT workspace
    v5host::DeviceBuf<double2> tw_w, tw_h;
    int tw_w_n = 0, tw_h_n = 0;
    bool fft_attr_set = false;             // the four FFT kernels may take FFT_SMEM_MAX of dynamic shared memory
    v5host::DeviceBuf<double2> tw_rag;     // ragged spectrum calls: the twiddle tables of the call's distinct sides
    v5host::DeviceBuf<double2> d_g;
    v5host::DeviceBuf<double> d_ms;
    v5host::DeviceBuf<unsigned long long> d_minmax;
    v5host::DeviceBuf<uint8_t> d_gray, d_spec;
    uint16_t luma[64], chroma[64];
    std::unique_ptr<v5jpeg_state, v5host::JpegStateDelete> jpeg;   // codec workspace (v5jpeg.cu), created on first use
    // Scratch owned by the handle (ticket counter, host-path / spectrum / codec workspaces) is reused by every call. Calls on ONE
    // stream are ordered by the stream; a call on another stream than the previous one first waits for that call's last launch.
    v5host::Event ev_scratch;
    cudaStream_t scratch_stream = nullptr;
    bool scratch_used = false;
    char err[512] = {0};
};

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

// The handlers of every extern "C" entry point whose host code can throw (std::vector, std::thread): the entry point is a
// function-try-block, `int v5ela_x(...) try { ... } V5_CATCH(h)`, so that no C++ exception crosses the C ABI.
#define V5_CATCH(h)                                                                              \
    catch (const std::bad_alloc &) {                                                             \
        return v5host::fail((h), V5ELA_ERR_NOMEM, "out of host memory%s");                       \
    } catch (const std::exception &e) {                                                          \
        return v5host::fail((h), V5ELA_ERR_INVALID, "host-side failure: %s", e.what());          \
    } catch (...) {                                                                              \
        return v5host::fail((h), V5ELA_ERR_INVALID, "host-side failure%s");                      \
    }

template <class T>
int DeviceBuf<T>::ensure(v5ela_handle *h, size_t need)
{
    if (cap_ >= need) return 0;
    reset();
    const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&p_), need);
    if (e != cudaSuccess) {
        p_ = nullptr;
        return fail(h, V5ELA_ERR_CUDA, "cudaMalloc(ptr, need): %s", cudaGetErrorString(e));
    }
    cap_ = need;
    return 0;
}

inline int PinnedBuf::ensure(v5ela_handle *h, size_t need, size_t alloc)
{
    if (cap_ >= need) return 0;
    reset();
    const cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&p_), alloc);
    if (e != cudaSuccess) {
        p_ = nullptr;
        return fail(h, V5ELA_ERR_CUDA, "cudaMallocHost(ptr, alloc): %s", cudaGetErrorString(e));
    }
    cap_ = alloc;
    return 0;
}

// The stream of the synchronous _host entry points and of v5ela_analyze_host without a stream, created on first use.
inline int internal_stream(v5ela_handle *h, cudaStream_t *st)
{
    V5_CUDA(h, h->own_stream.create());
    *st = h->own_stream;
    return 0;
}

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
        if (h->ev_scratch.create() != cudaSuccess) return;
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

}  // namespace v5host
