/*
 * include/v5ela.h — C ABI of libv5ela.so: the B200 (sm_100a) implementation of the V5 texture/ELA hot path of
 * MrBottleTree/fake-video-detection-engine.
 *
 * The reference has no FFI for this path (it is pure Python); its only interface is the LangGraph node callable
 * `run(state)` (nodes/V_nodes/v5_texture_ela.py:13, registered at main.py:304). This ABI is what the replacement
 * node module binds with ctypes (fake-video-detection-engine_b200/v5ela/_abi.py; INTEGRATION.md shows the stub).
 * Each entry point cites the reference lines whose work it takes over.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative v5ela_status; no exceptions
 * cross the boundary; v5ela_last_error() gives a handle-owned message. All image/record pointers are DEVICE
 * pointers owned by the caller unless the name says `host`. Calls are asynchronous on the given CUDA stream and do
 * not synchronise or allocate after the first call at a given geometry. A handle is bound to one device and is not
 * thread-safe; the library is (one handle per thread). One thread may use its handle on several CUDA streams: the handle owns
 * scratch memory (work-item counter, host-path / spectrum / codec workspaces) that every call reuses, so a call issued on another
 * stream than the previous call first waits — on the device, cudaStreamWaitEvent, no host synchronisation — for that call's
 * last launch. Calls on one stream are ordered by the stream itself. Caller-owned buffers are the caller's to order.
 */
#ifndef V5ELA_H
#define V5ELA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define V5ELA_ABI_VERSION 1

#if defined(__GNUC__)
#define V5ELA_API __attribute__((visibility("default")))
#else
#define V5ELA_API
#endif

typedef enum {
    V5ELA_OK = 0,
    V5ELA_ERR_INVALID = -1,     /* bad argument (null pointer, non-positive size, bad stride, quality outside 1..100) */
    V5ELA_ERR_CUDA = -2,        /* a CUDA runtime call failed; see v5ela_last_error */
    V5ELA_ERR_NO_DEVICE = -3,   /* no CUDA device / device is not compute capability 10.x */
    V5ELA_ERR_NOMEM = -4,
    V5ELA_ERR_UNSUPPORTED = -5  /* a JPEG file outside the supported set (see v5ela_jpeg_decode) */
} v5ela_status;

/*
 * Per-frame feature record "V5F v1" (SURVEY.md §8a), 3144 bytes, little endian, no implicit padding.
 *   ela_*   : statistics of the residual |orig - jpeg_roundtrip(orig, q)| per RGB channel.
 *             max over channels of ela_max is the reference's `max_diff` before its 0 -> 1 fix
 *             (v5_texture_ela.py:72-75); 255.0/max is its `scale` (v5…:76).
 *   tex_*   : statistics of L = Laplacian(Y) (kernel [0 1 0; 1 -4 1; 0 1 0], BORDER_REFLECT_101) on the libjpeg luma
 *             of the original frame — build-defined high-pass texture response (north_star), oracle =
 *             cv2.Laplacian(Y, CV_16S, ksize=1).
 */
typedef struct v5ela_record {
    uint32_t ela_hist[3][256];  /* np.bincount(residual[..., c]) */
    uint64_t ela_sum[3];        /* sum of residual values */
    uint64_t ela_sumsq[3];      /* sum of squared residual values */
    uint64_t tex_sumabs;        /* sum |L| */
    uint64_t tex_sumsq;         /* sum L^2 */
    uint16_t tex_maxabs;        /* max |L| */
    uint8_t  ela_max[3];        /* max residual per channel */
    uint8_t  pad[3];
} v5ela_record;

typedef struct v5ela_handle v5ela_handle;

/* Library identification. */
V5ELA_API int         v5ela_abi_version(void);
V5ELA_API size_t      v5ela_record_bytes(void);                       /* == sizeof(v5ela_record) == 3144 */
V5ELA_API const char *v5ela_status_string(int status);

/* Handle life cycle. `device` is a CUDA ordinal. The handle owns quantisation tables and a small workspace. */
V5ELA_API int         v5ela_create(int device, v5ela_handle **out);
V5ELA_API int         v5ela_destroy(v5ela_handle *h);
V5ELA_API const char *v5ela_last_error(const v5ela_handle *h);

/*
 * JPEG quality of the simulated re-encode. Replaces the literal in `original.save(path, 'JPEG', quality=90)`
 * (v5_texture_ela.py:67): builds libjpeg's Annex-K tables scaled by `quality` (1..100, baseline-forced) and the exact
 * reciprocal constants the kernel divides with. Default after create: 90.
 */
V5ELA_API int v5ela_set_quality(v5ela_handle *h, int quality);
V5ELA_API int v5ela_get_quality(const v5ela_handle *h);
/* Copies the 64+64 table entries (natural order) to HOST arrays; what PIL reports as Image.quantization. */
V5ELA_API int v5ela_get_quant_tables(const v5ela_handle *h, uint16_t luma_host[64], uint16_t chroma_host[64]);

/*
 * The hot path. For each of `n` RGB frames (uint8, HWC, `row_stride_bytes` between rows, `frame_stride_bytes`
 * between frames) performs, in one fused kernel, what the reference does with
 *   original.save(tmp, 'JPEG', quality=q); compressed = Image.open(tmp)      v5_texture_ela.py:66-68
 *   diff = ImageChops.difference(original, compressed)                       v5_texture_ela.py:70
 *   extrema = diff.getextrema(); max_diff = max(...)                         v5_texture_ela.py:72-73
 * i.e. libjpeg's RGB->YCbCr, h2v2 chroma downsample, 8x8 ISLOW forward DCT, quantise, dequantise, ISLOW inverse DCT,
 * h2v2 fancy upsample, YCbCr->RGB, abs-diff — bit-exact — and reduces the residual and the luma Laplacian into one
 * v5ela_record per frame.
 *   d_records  : n x sizeof(v5ela_record) bytes, overwritten.
 *   d_residual : optional (may be NULL): n x h x w x 3 tightly packed residual map (`diff`).
 * No host synchronisation; ordering follows `cuda_stream` (a cudaStream_t passed as void*; NULL = legacy default).
 */
V5ELA_API int v5ela_analyze(v5ela_handle *h, const uint8_t *d_rgb, int n, int height, int width,
                  int64_t frame_stride_bytes, int64_t row_stride_bytes,
                  void *d_records, uint8_t *d_residual, void *cuda_stream);

/*
 * The same call with the record table's optional texture histogram (SURVEY.md §8a, `tex_hist[256]`):
 *   d_tex_hist : optional (may be NULL): n x 256 uint32, overwritten with
 *                np.bincount(np.minimum(np.abs(cv2.Laplacian(Y, cv2.CV_16S, ksize=1)), 255), minlength=256)
 *                of each frame's luma (the Laplacian behind tex_sumabs / tex_sumsq / tex_maxabs).
 * Asking for it selects a kernel instantiation with one more shared-memory increment per pixel; NULL is v5ela_analyze.
 */
V5ELA_API int v5ela_analyze_ex(v5ela_handle *h, const uint8_t *d_rgb, int n, int height, int width,
                     int64_t frame_stride_bytes, int64_t row_stride_bytes,
                     void *d_records, uint8_t *d_residual, uint32_t *d_tex_hist, void *cuda_stream);

/*
 * The same analysis for a RAGGED batch — frames of different sizes in ONE launch. This is the reference node's real input: at
 * most three face crops of different sizes per call (v5_texture_ela.py:42, 56-64), cut by V1 with its 20 % padding rule
 * (v1_keyframes_facetrack.py:144-166). Every frame brings its own pointer, size and row stride; record i belongs to frame i.
 *   frames_host : HOST array of n descriptors whose pointers are DEVICE pointers (frames may live anywhere: separate allocations,
 *                 strided views into one keyframe, ...). residual / enhanced are optional per frame: tightly packed h*w*3 maps,
 *                 `diff` (v5…:70) and `ImageEnhance.Brightness(diff).enhance(255.0 / max_diff)` (v5…:74-78); they may alias.
 *   d_records   : n records, overwritten.
 * The descriptor table goes to the device through a small pinned staging buffer inside the handle (the only host work besides
 * filling it; before refilling it the call waits, on the host, for the PREVIOUS ragged call's table upload — a few microseconds
 * of copy, normally long finished). Otherwise asynchronous on `cuda_stream`; launches: memsets, the fused kernel, the finalize kernel and — only when a frame
 * asks for an enhanced map — one enhancement kernel per 65535 frames of the batch.
 */
typedef struct v5ela_frame_desc {
    const uint8_t *rgb;         /* uint8 HWC RGB */
    int32_t height, width;
    int64_t row_stride_bytes;   /* >= 3 * width */
    uint8_t *residual;          /* optional */
    uint8_t *enhanced;          /* optional */
} v5ela_frame_desc;
V5ELA_API int v5ela_analyze_ragged(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, void *d_records, void *cuda_stream);
/* The same with HOST pointers in the descriptors and a HOST record array (what the drop-in node calls for its <= 3 crops): one
 * packed upload, one launch sequence, one download; synchronises before returning. */
V5ELA_API int v5ela_analyze_ragged_host(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, void *records_host);

/*
 * A quality SWEEP — n frames of any sizes, each analysed at nq JPEG qualities, in ONE launch sequence — and, optionally, the
 * JPEG-ghost map of every (quality, frame) (Farid, "Exposing Digital Forgeries from JPEG Ghosts", 2009): a region that was saved at
 * quality q0 before is almost a fixed point of a re-save at q0, so where the residual is smallest over q says what its earlier
 * quality was; a pasted region with another compression history shows its minimum at another q.
 *   frames_host   : HOST array of n descriptors whose pointers are DEVICE pointers (as v5ela_analyze_ragged takes them); residual
 *                   and enhanced must be NULL.
 *   qualities_host: HOST array of nq qualities, each in 1..100, 1 <= nq <= 100; duplicates are allowed. The handle's own quality
 *                   (v5ela_set_quality) is neither used nor changed.
 *   d_records     : n * nq records, overwritten: record [q * n + i] is byte-identical to v5ela_analyze_ragged of frame i alone at
 *                   quality qualities_host[q] (and to v5ela_analyze of it).
 *   d_ghost       : optional (may be NULL), uint32: per (quality, frame) one ceil(h/16) x ceil(w/16) map, map (q, i) at element
 *                   q * M + sum_{j<i} m_j, m_j = ceil(h_j/16) * ceil(w_j/16), M = sum_j m_j; entry (by, bx) = sum over the image
 *                   pixels of MCU (by, bx) of sum_c residual_c^2 (residual as in v5ela_analyze).
 * A null array, n < 0, nq outside 1..100, a quality outside 1..100, a descriptor v5ela_analyze_ragged would refuse, a non-NULL
 * residual or enhanced pointer, or more than 2^31 - 1 work items is refused with V5ELA_ERR_INVALID before anything is launched or
 * copied; v5ela_last_error names the frame or the quality index. n == 0 returns V5ELA_OK.
 * Ordering as for v5ela_analyze_ragged (the tables go up through the same staging buffer). Launches: the sweep kernel and the
 * finalize kernel, whatever n and nq. v5ela_last_instantiation is left as it is.
 */
V5ELA_API int v5ela_analyze_sweep(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, const int *qualities_host, int nq,
                                  void *d_records, uint32_t *d_ghost, void *cuda_stream);
/* The same with HOST pointers in the descriptors and HOST records / maps: each frame uploaded once, one launch sequence, one download;
 * synchronises before returning. */
V5ELA_API int v5ela_analyze_sweep_host(v5ela_handle *h, const v5ela_frame_desc *frames_host, int n, const int *qualities_host, int nq,
                                       void *records_host, uint32_t *ghost_host);

/*
 * Brightness enhancement of the residual map: `ImageEnhance.Brightness(diff).enhance(255.0 / max_diff)`
 * (v5_texture_ela.py:74-78) == u8(trunc(f32(x) * f32(scale))) clipped, with max_diff read per frame from the records
 * produced by v5ela_analyze on the same stream (0 -> 1 fix applied). d_enhanced may alias d_residual. Any n: one launch per
 * 65535 frames.
 */
V5ELA_API int v5ela_enhance(v5ela_handle *h, const uint8_t *d_residual, const void *d_records, int n, int height, int width,
                  uint8_t *d_enhanced, void *cuda_stream);

/*
 * Per-group aggregation of records (per-video features, BASELINE.json config 4): out[g] = sum of histograms and sums,
 * max of maxima over records [g*group, (g+1)*group). n must be a multiple of `group`. d_out: (n/group) records.
 * The histogram bins stay 32-bit: a bin that would exceed 2^32 - 1 (groups of more than ~2071 frames of 1080p) saturates at that
 * value instead of wrapping; the 64-bit sums are exact.
 */
V5ELA_API int v5ela_reduce_records(v5ela_handle *h, const void *d_records, int n, int group, void *d_out, void *cuda_stream);

/*
 * The reference-facing entry point for callers that hold HOST memory (the drop-in node, the end-to-end benchmark):
 * same work as v5ela_analyze, but copies the frames in, and the records (and the optional residual / enhanced maps)
 * back. The batch is cut into chunks whose host->device copies overlap the kernels of the previous chunk (two internal
 * streams forked from / joined to `cuda_stream`). Host buffers should be pinned (cudaHostAlloc / torch pin_memory) for
 * the copies to be asynchronous and full speed.
 *   cuda_stream == NULL : runs on an internal stream and SYNCHRONISES before returning (outputs valid on return).
 *   cuda_stream != NULL : fully asynchronous; outputs are valid once the caller has synchronised that stream.
 */
V5ELA_API int v5ela_analyze_host(v5ela_handle *h, const uint8_t *rgb_host, int n, int height, int width,
                       void *records_host, uint8_t *residual_host_or_null, uint8_t *enhanced_host_or_null,
                       void *cuda_stream);

/*
 * The reference's "texture" artefact, SURVEY.md §8f-1 (v5_texture_ela.py:84-88):
 *   f = np.fft.fft2(gray); fshift = np.fft.fftshift(f); ms = 20*np.log(np.abs(fshift)+1);
 *   cv2.normalize(ms, None, 0, 255, cv2.NORM_MINMAX, dtype=cv2.CV_8U)
 * for `n` single-channel uint8 images of any size (float64 DFT, exact sizes, no padding). d_out: n x h x w uint8,
 * tightly packed. Parity: within 1 grey level of NumPy/OpenCV (summation order differs from pocketfft).
 */
V5ELA_API int v5ela_spectrum(v5ela_handle *h, const uint8_t *d_gray, int n, int height, int width,
                   int64_t frame_stride_bytes, int64_t row_stride_bytes, uint8_t *d_out, void *cuda_stream);
/* Same with HOST buffers (what the drop-in node calls); synchronises before returning. */
V5ELA_API int v5ela_spectrum_host(v5ela_handle *h, const uint8_t *gray_host, int n, int height, int width,
                        uint8_t *out_host);

/*
 * The same spectrum for a RAGGED batch — images of different sizes in ONE launch sequence: the node's face crops (v5…:83-91),
 * or any number of crops of mixed sizes. Output i is byte-identical to what v5ela_spectrum writes for image i alone: every
 * image takes the path the uniform call would take (the shared-memory FFT when both sides have only 2, 3 and 5 as prime
 * factors, otherwise the exact-size DFT; V5ELA_FFT=0 forces the DFT for all), with the same float64 arithmetic.
 *   frames_host : HOST array of n descriptors whose pointers are DEVICE pointers; `out` is height * width bytes, tightly packed.
 * A null array, n < 0, or a descriptor with a null pointer, a non-positive size, a side over 65536 or a row stride smaller
 * than the width is refused with V5ELA_ERR_INVALID before anything is launched; v5ela_last_error names the frame.
 * The call plans everything on the host (twiddle tables of the distinct sides, chunks under the same workspace cap as
 * v5ela_spectrum, the CTAs of every launch), uploads the plan through the handle's staging buffer (waiting first, on the host,
 * for the previous ragged call's table upload, as v5ela_analyze_ragged does) and is otherwise asynchronous on `cuda_stream`.
 * Launches: one twiddle kernel per call; per chunk two FFT kernels if an image there takes the FFT, two DFT kernels if one
 * takes the DFT, and the image kernel. The twiddle tables v5ela_spectrum caches are left as they are.
 */
typedef struct v5ela_gray_desc {
    const uint8_t *gray;        /* uint8 HW, one channel */
    int32_t height, width;
    int64_t row_stride_bytes;   /* >= width */
    uint8_t *out;               /* height * width uint8, tightly packed */
} v5ela_gray_desc;
V5ELA_API int v5ela_spectrum_ragged(v5ela_handle *h, const v5ela_gray_desc *frames_host, int n, void *cuda_stream);
/* The same with HOST pointers in the descriptors: one upload per image into one packed device arena, one launch sequence, one
 * download per image; synchronises before returning. */
V5ELA_API int v5ela_spectrum_ragged_host(v5ela_handle *h, const v5ela_gray_desc *frames_host, int n);

/*
 * ---- Codec rows (SURVEY.md §8f-2, §8f-3): the JPEG files on either side of the ELA arithmetic, on the GPU ----------------
 *
 * Encoder: what the reference writes with PIL / OpenCV — `original.save(tmp,'JPEG',quality=90)` (v5_texture_ela.py:66-67),
 * `enhanced_diff.save(ela_i.jpg)` (v5…:80-81, PIL default quality 75) and `cv2.imwrite(fft_i.jpg, spectrum)` (v5…:90-91, OpenCV
 * default quality 95, one component) — byte-identical to libjpeg's output: baseline sequential, Annex K tables scaled by
 * `quality`, 4:2:0 for three channels, the standard Huffman tables, JFIF 1.01 header.
 *   d_img      : n images, uint8, `channels` = 1 (HW) or 3 (HWC, RGB), all height x width; sides up to 65535.
 *   d_out      : n x out_stride_bytes (at most 1 GiB); file i starts at d_out + i * out_stride_bytes. Every file that fits comes
 *                out right, however long its entropy-coded stream (up to 2^33 bits).
 *   d_sizes    : n file sizes. A size larger than out_stride_bytes means that file did not fit and its bytes are undefined;
 *                v5ela_jpeg_bound() is a capacity that always fits (it is ~13 bytes per pixel; real files are far smaller).
 * Asynchronous on `cuda_stream`; owns a workspace inside the handle.
 */
V5ELA_API int64_t v5ela_jpeg_bound(int height, int width, int channels);
V5ELA_API int v5ela_jpeg_encode(v5ela_handle *h, const uint8_t *d_img, int n, int height, int width, int channels,
                      int64_t frame_stride_bytes, int64_t row_stride_bytes, int quality,
                      uint8_t *d_out, int64_t out_stride_bytes, int32_t *d_sizes, void *cuda_stream);
/* Same with HOST buffers (what the drop-in node calls); synchronises before returning. */
V5ELA_API int v5ela_jpeg_encode_host(v5ela_handle *h, const uint8_t *img_host, int n, int height, int width, int channels,
                           int quality, uint8_t *out_host, int64_t out_stride_bytes, int32_t *sizes_host);

/*
 * Decoder: what the reference reads with `Image.open(crop_path).convert('RGB')` (v5_texture_ela.py:64) and
 * `cv2.imread(crop_path, cv2.IMREAD_GRAYSCALE)` (v5…:83) — the crops V1 wrote with cv2.imwrite (v1_keyframes_facetrack.py:166).
 * Pixel-identical to libjpeg's defaults (ISLOW inverse DCT, fancy upsampling) as Pillow and OpenCV run them on x86-64, i.e.
 * libjpeg-turbo's x86 SIMD inverse DCT: its 16-bit arithmetic (dequantisation modulo 2^16, some sums wrapping, saturation
 * between the passes) is reproduced exactly. Files written from pixels never reach that range; blocks a file can still carry
 * (AC values near +-1023, large or 16-bit quantisation entries) decode differently in libjpeg-turbo's plain C path, which
 * this decoder does not follow. Supported: 8-bit baseline Huffman files with
 * one component, or three components with the luma sampled 2x2 (4:2:0), 2x1 (4:2:2) or 1x1 (4:4:4) against 1x1 chroma; one
 * scan; any Huffman / quantisation tables (16-bit ones under SOF1 too); with or without restart intervals; an entropy-coded segment (stuffed bytes
 * included) of less than 2^29 - 2^20 bytes (511 MiB; the decoder's Huffman state holds 32-bit bit positions) — everything
 * PIL's and OpenCV's writers produce by default (4:2:0, no restarts) plus what their sampling and restart options add. Anything
 * else (progressive, other sampling factors, CMYK, 12-bit, arithmetic coding, larger entropy-coded segments) returns
 * V5ELA_ERR_UNSUPPORTED before anything is uploaded or launched, and v5ela_last_error names the file.
 *   files_host / lens : n complete JPEG files in HOST memory (they come from disk); sizes may differ from file to file.
 *             Files that all live in page-locked memory (cudaHostAlloc / cudaHostRegister / torch pin_memory) are copied
 *             to the device asynchronously from where they are — keep them alive until the stream has been synchronised;
 *             pageable files are staged through a pinned buffer inside the handle before the call returns.
 *   d_rgb   : optional DEVICE buffer; file i is decoded to RGB (HWC; a one-component file is replicated) at byte offset
 *             rgb_offsets[i], or tightly packed in file order when rgb_offsets is NULL. A negative offset is refused with
 *             V5ELA_ERR_INVALID (v5ela_last_error names the file) before anything is launched.
 *   d_gray  : optional DEVICE buffer; the luma plane alone (what IMREAD_GRAYSCALE returns), offsets likewise.
 *   d_status: optional DEVICE array of n ints: 0, or -1 when the entropy-coded data of that file ended early (or a restart
 *             marker is missing).
 * Header parsing and the staging copy happen on the calling thread; the decode itself is asynchronous on `cuda_stream`.
 * The compressed bytes are uploaded on an internal stream as soon as the call is made (so the upload of one batch overlaps
 * the kernels of the previous one): the files must be complete in host memory at that moment.
 */
V5ELA_API int v5ela_jpeg_info(const uint8_t *file_host, int64_t len, int *height, int *width, int *channels);
/* The same for n files in one call: dims_out[3i .. 3i+2] = height, width, channels; stops at the first unreadable file,
 * returns its status and (optionally) its index. */
V5ELA_API int v5ela_jpeg_info_batch(const uint8_t *const *files_host, const int64_t *lens, int n, int32_t *dims_out, int *bad_index);
V5ELA_API int v5ela_jpeg_decode(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n,
                      uint8_t *d_rgb, const int64_t *rgb_offsets, uint8_t *d_gray, const int64_t *gray_offsets,
                      int32_t *d_status, void *cuda_stream);
/* Same with HOST outputs; synchronises, and reports truncated / corrupt entropy data as V5ELA_ERR_INVALID. */
V5ELA_API int v5ela_jpeg_decode_host(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n,
                           uint8_t *rgb_host, const int64_t *rgb_offsets, uint8_t *gray_host, const int64_t *gray_offsets);

/*
 * DCT statistics of JPEG files (DESIGN.md §4.8): what the decoder reads from the files before any pixel exists — the quantised
 * coefficients and quantisation tables — as per-frequency histograms, and a per-block map of aligned double JPEG compression
 * (Popescu & Farid 2004; Lin, He, Tang & Tang 2009). The files, the supported set, the refusals (V5ELA_ERR_UNSUPPORTED naming
 * the file), the staging of pinned and pageable files and the Huffman decoding are v5ela_jpeg_decode's; the decode stops once
 * the coefficients are known (no inverse DCT, no colour conversion).
 *   d_hist  : DEVICE uint32 [n][3][64][129]. Entry [i][c][k][v + 64] counts the blocks of component c (0 Y, 1 Cb, 2 Cr) of file i
 *             whose quantised coefficient at NATURAL-order position k equals v, values clamped to -64 .. 64 (the end bins
 *             saturate). k = 0 is the DC value with the prediction undone. Only real blocks count: bx < ceil(ceil(W h_c / h_max) / 8),
 *             by < ceil(ceil(H v_c / v_max) / 8); the padding blocks of the MCU grid do not. A one-component file leaves c = 1, 2 zero.
 *   d_qtab  : optional DEVICE uint16 [n][3][64]: each component's quantisation table, natural order, as the file's DQT gives it
 *             (zero for the components a one-component file lacks).
 *   d_map   : optional DEVICE float32 maps, one per file with one entry per real luma 8x8 block (ceil(H/8) rows of ceil(W/8)):
 *             the posterior that the block was NOT aligned-double-compressed. File i's map starts at element map_offsets[i], or
 *             the maps are packed in file order when map_offsets is NULL; a negative offset is refused with V5ELA_ERR_INVALID
 *             before anything is launched. The estimator, per file, for the 15 luma AC frequencies k at zigzag positions 1..15:
 *               h = the luma histogram of k, g(v) = h(v) + h(-v) for v = 1..63, N = sum g; N < 64: p_k = 1. Otherwise, with
 *               r(v) = g(v) - (g(v-1) + g(v+1)) / 2 (v = 2..62) and S(p) = |sum r(v) e^{-2 pi i v / p}| / max(sum |r|, 1) for
 *               p = 2..12, p* = argmax S (the smaller p on ties) and p_k = p* if S(p*) >= 0.5 and sum |r| >= 0.05 N, else 1.
 *               P_u(v) = h(v) / (sum of h over the p_k bins from p_k floor(v / p_k) on, clipped to -63..63), 1 / p_k where that
 *               sum is 0; the clamped values +-64 use the entries of +-63. P_t = 1 / p_k.
 *               map = 1 / (1 + exp(sum over the k with p_k > 1 of log P_u(v_k) - log P_t)), 0.5 when no k has p_k > 1.
 *   d_status: optional DEVICE int32 [n], as v5ela_jpeg_decode's.
 * Asynchronous on `cuda_stream`; the workspace is the decoder's, inside the handle.
 */
V5ELA_API int v5ela_jpeg_dct_stats(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n, uint32_t *d_hist,
                                   uint16_t *d_qtab, float *d_map, const int64_t *map_offsets, int32_t *d_status, void *cuda_stream);
/* Same with HOST outputs (map offsets likewise); synchronises, and reports truncated / corrupt entropy data as V5ELA_ERR_INVALID. */
V5ELA_API int v5ela_jpeg_dct_stats_host(v5ela_handle *h, const uint8_t *const *files_host, const int64_t *lens, int n,
                                        uint32_t *hist_host, uint16_t *qtab_host, float *map_host, const int64_t *map_offsets);
/* The IJG quality 1..100 whose tables (libjpeg's jpeg_set_quality, baseline-forced: what v5ela_set_quality derives) equal
 * luma[64] and, unless chroma is NULL, chroma[64] (natural order, as in d_qtab); 0 when no quality does. No device needed. */
V5ELA_API int v5ela_jpeg_ijg_quality(const uint16_t luma[64], const uint16_t *chroma);

/*
 * Measurement hook: while enabled, every v5ela_analyze records a CUDA event pair around the fused kernel on the launch
 * stream. v5ela_profile_read waits for the recorded events, returns the summed kernel time and launch count since the
 * last reset, and optionally resets. Used by bench.py for the roofline line; off by default.
 */
V5ELA_API int v5ela_profile_enable(v5ela_handle *h, int enable);
V5ELA_API int v5ela_profile_read(v5ela_handle *h, double *fused_ms_sum, int64_t *fused_launches, int reset);

/*
 * Which instantiation of the fused kernel the most recent v5ela_analyze / v5ela_analyze_ex call on this handle launched
 * (same arithmetic, different edge handling — csrc/v5ela_device.cuh): V5ELA_INST_GENERAL any size / stride / outputs,
 * V5ELA_INST_FAST width % 16 == 0, 16-byte aligned frames, records only (every BASELINE.json config), V5ELA_INST_TEXHIST
 * general + tex_hist. -1 before the first call. Tests and bench.py use it to prove which code they measured.
 */
#define V5ELA_INST_GENERAL 0
#define V5ELA_INST_FAST 1
#define V5ELA_INST_TEXHIST 2
V5ELA_API int v5ela_last_instantiation(const v5ela_handle *h);

/*
 * The 8x8 block stage of the fused kernel (fDCT -> quantise -> dequantise -> IDCT) exists in two bit-identical builds:
 *   V5ELA_BLOCKS_SMEM  four threads per block, ISLOW butterflies in registers, two shared-memory transposes (kernel v10);
 *   V5ELA_BLOCKS_MMA   the four passes as int8 limb-split tensor-core contractions (mma.sync.m16n8k16, SASS IMMA), a warp per pair
 *                      of blocks, everything in registers (csrc/v5ela_dctmma.cuh): 17 % fewer instructions per pixel.
 * They run within 3 % of each other on every frame geometry measured (360p .. 4K, profiles/r02/variants.txt section 8; DESIGN.md
 * 4.4 says why); V5ELA_BLOCKS_DEFAULT is what a new handle uses. Results do not depend on the choice.
 */
#define V5ELA_BLOCKS_SMEM 0
#define V5ELA_BLOCKS_MMA 1
#define V5ELA_BLOCKS_DEFAULT V5ELA_BLOCKS_SMEM
V5ELA_API int v5ela_set_block_stage(v5ela_handle *h, int mode);
V5ELA_API int v5ela_get_block_stage(const v5ela_handle *h);

/* Number of kernel launches issued through this handle since creation (bench.py's gpu_launches evidence). */
V5ELA_API int64_t v5ela_launch_count(const v5ela_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* V5ELA_H */
