// v5ela_fft.cuh — the reference's "texture" artefact (v5_texture_ela.py:83-91) on the GPU:
//     f = np.fft.fft2(gray); fshift = np.fft.fftshift(f); ms = 20*np.log(np.abs(fshift) + 1)
//     out = cv2.normalize(ms, None, 0, 255, cv2.NORM_MINMAX, dtype=cv2.CV_8U)
// Face crops have arbitrary sizes (prime widths included), so the 2-D DFT is evaluated as two exact-size float64
// matrix products with twiddle factors from an N-entry table (index (j*k) mod N kept by integer addition — no argument
// reduction error): rows real -> half spectrum (Hermitian symmetry), then columns complex -> complex fused with
// |F|, 20*ln(|F|+1) and the per-frame min/max; a last kernel normalises, shifts (fftshift) and mirrors the half
// spectrum into the uint8 image. float64 throughout like NumPy; parity target is +-1 LSB of the uint8 image (the
// reference's pocketfft sums in a different order), SURVEY.md §8f-1.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "v5ela_spec_plan.h"                                    // FftPlan, make_plan, TILE, the ragged plan

namespace v5fft {

// tw[m] = exp(-2*pi*i*m/n)
__global__ void twiddle_kernel(double2 *tw, int n)
{
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tw[m] = make_double2(c, -s);
}

constexpr int KC = 32;       // reduction chunk staged in shared memory

// G[y][v] = sum_x gray[y][x] * twW[(x*v) mod W],  v in [0, W/2]
__global__ void __launch_bounds__(256) dft_rows_kernel(const uint8_t *__restrict__ gray, int64_t frame_stride, int64_t row_stride,
                                                       int h, int w, int wh, const double2 *__restrict__ tw, double2 *__restrict__ g)
{
    __shared__ double xs[TILE][KC + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int y0 = blockIdx.y * TILE, v0 = blockIdx.x * TILE;
    const uint8_t *src = gray + (int64_t)blockIdx.z * frame_stride;
    const int va = v0 + tx, vb = v0 + tx + 16;
    int ia = 0, ib = 0;                                         // (x * v) mod w for the two columns of this thread
    const int sa = va % w, sb = vb % w;
    double2 acc[2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
    for (int x0 = 0; x0 < w; x0 += KC) {
        for (int i = threadIdx.x; i < TILE * KC; i += 256) {
            const int r = i / KC, c = i - r * KC;
            const int y = y0 + r, x = x0 + c;
            xs[r][c] = (y < h && x < w) ? (double)src[(int64_t)y * row_stride + x] : 0.0;
        }
        __syncthreads();
        const int kn = min(KC, w - x0);
        for (int k = 0; k < kn; k++) {
            const double2 ta = tw[ia], tb = tw[ib];
            const double xa = xs[ty][k], xb = xs[ty + 16][k];
            acc[0][0].x = fma(xa, ta.x, acc[0][0].x); acc[0][0].y = fma(xa, ta.y, acc[0][0].y);
            acc[0][1].x = fma(xa, tb.x, acc[0][1].x); acc[0][1].y = fma(xa, tb.y, acc[0][1].y);
            acc[1][0].x = fma(xb, ta.x, acc[1][0].x); acc[1][0].y = fma(xb, ta.y, acc[1][0].y);
            acc[1][1].x = fma(xb, tb.x, acc[1][1].x); acc[1][1].y = fma(xb, tb.y, acc[1][1].y);
            ia += sa; ia = ia >= w ? ia - w : ia;
            ib += sb; ib = ib >= w ? ib - w : ib;
        }
        __syncthreads();
    }
    double2 *dst = g + (int64_t)blockIdx.z * h * wh;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int y = y0 + ty + 16 * i;
        if (y >= h) continue;
        if (va < wh) dst[(int64_t)y * wh + va] = acc[i][0];
        if (vb < wh) dst[(int64_t)y * wh + vb] = acc[i][1];
    }
}

// ms[u][v] = 20*ln(|sum_y G[y][v] * twH[(u*y) mod H]| + 1); per-frame min/max as ordered uint64 (ms >= 0)
__global__ void __launch_bounds__(256) dft_cols_kernel(const double2 *__restrict__ g, int h, int wh, const double2 *__restrict__ tw,
                                                       double *__restrict__ ms, unsigned long long *__restrict__ minmax)
{
    __shared__ double2 gs[KC][TILE + 1];
    __shared__ unsigned long long smin, smax;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int u0 = blockIdx.y * TILE, v0 = blockIdx.x * TILE;
    const double2 *src = g + (int64_t)blockIdx.z * h * wh;
    if (threadIdx.x == 0) { smin = ~0ull; smax = 0ull; }
    const int ua = u0 + ty, ub = u0 + ty + 16;
    int ia = 0, ib = 0;
    const int sa = ua % h, sb = ub % h;
    double2 acc[2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
    for (int y0 = 0; y0 < h; y0 += KC) {
        for (int i = threadIdx.x; i < KC * TILE; i += 256) {
            const int r = i / TILE, c = i - r * TILE;
            const int y = y0 + r, v = v0 + c;
            gs[r][c] = (y < h && v < wh) ? src[(int64_t)y * wh + v] : make_double2(0.0, 0.0);
        }
        __syncthreads();
        const int kn = min(KC, h - y0);
        for (int k = 0; k < kn; k++) {
            const double2 ta = tw[ia], tb = tw[ib];
            const double2 ga = gs[k][tx], gb = gs[k][tx + 16];
            // (a + ib)(c + id) = (ac - bd) + i(ad + bc)
            acc[0][0].x = fma(ga.x, ta.x, fma(-ga.y, ta.y, acc[0][0].x)); acc[0][0].y = fma(ga.x, ta.y, fma(ga.y, ta.x, acc[0][0].y));
            acc[0][1].x = fma(gb.x, ta.x, fma(-gb.y, ta.y, acc[0][1].x)); acc[0][1].y = fma(gb.x, ta.y, fma(gb.y, ta.x, acc[0][1].y));
            acc[1][0].x = fma(ga.x, tb.x, fma(-ga.y, tb.y, acc[1][0].x)); acc[1][0].y = fma(ga.x, tb.y, fma(ga.y, tb.x, acc[1][0].y));
            acc[1][1].x = fma(gb.x, tb.x, fma(-gb.y, tb.y, acc[1][1].x)); acc[1][1].y = fma(gb.x, tb.y, fma(gb.y, tb.x, acc[1][1].y));
            ia += sa; ia = ia >= h ? ia - h : ia;
            ib += sb; ib = ib >= h ? ib - h : ib;
        }
        __syncthreads();
    }
    double *dst = ms + (int64_t)blockIdx.z * h * wh;
    unsigned long long lo = ~0ull, hi = 0ull;
#pragma unroll
    for (int i = 0; i < 2; i++) {
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int u = u0 + ty + 16 * i, v = v0 + tx + 16 * j;
            if (u >= h || v >= wh) continue;
            const double m = 20.0 * log(hypot(acc[i][j].x, acc[i][j].y) + 1.0);
            dst[(int64_t)u * wh + v] = m;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(m);
            lo = bits < lo ? bits : lo;
            hi = bits > hi ? bits : hi;
        }
    }
    atomicMin(&smin, lo);
    atomicMax(&smax, hi);
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicMin(&minmax[2 * blockIdx.z], smin);
        atomicMax(&minmax[2 * blockIdx.z + 1], smax);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Fast path for sizes whose prime factors are all in {2, 3, 5} (every common video size): mixed-radix (5, 3, 4, 2) Stockham
// autosort FFT in shared memory, float64. One stage of radix r over a sequence of current length n and stride s
// (n * s == N): for p in [0, n/r), q in [0, s):
//     a_t = x[q + s*(p + t*n/r)],  b_u = (sum_t a_t w_r^{t u}) * exp(-2 pi i p u s / N),  y[q + s*(r*p + u)] = b_u
// then n /= r, s *= r and the buffers swap. p*u*s < N, so the twiddle is a direct index into the N-entry table.
// (FftPlan, recip_u16 and make_plan live in v5ela_spec_plan.h)
__device__ __forceinline__ int div_u16(int a, uint32_t inv) { return (int)__umulhi((uint32_t)a, inv); }

__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cmul(double2 a, double2 b)
{
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ double2 mul_neg_i(double2 a) { return make_double2(a.y, -a.x); }   // -i * a

// All stages of `nseq` sequences of length plan.n stored one after the other in x (work buffer y). Returns the buffer
// that holds the result. Must be called by every thread of the CTA.
__device__ double2 *stockham(double2 *x, double2 *y, int nseq, const FftPlan &plan, const double2 *__restrict__ tw)
{
    const int N = plan.n;
    int n = N, s = 1;
    for (int st = 0; st < plan.nst; st++) {
        const int r = plan.radix[st], m = n / r, per_seq = N / r;
        const uint32_t inv_s = plan.inv_s[st], inv_ps = plan.inv_per_seq[st];
        for (int wi = threadIdx.x; wi < nseq * per_seq; wi += blockDim.x) {     // wi < 4 * 32768: both divisions through reciprocals
            const int seq = (nseq == 1 || per_seq == 1) ? (nseq == 1 ? 0 : wi) : div_u16(wi, inv_ps), idx = wi - seq * per_seq;
            const int p = s == 1 ? idx : div_u16(idx, inv_s), q = idx - p * s;      // (the reciprocal of 1 does not fit 32 bits)
            const double2 *xi = x + seq * N + q + s * p;
            double2 *yo = y + seq * N + q + s * r * p;
            const int ms_ = s * m;                              // input stride between the r operands
            if (r == 2) {
                const double2 a0 = xi[0], a1 = xi[ms_];
                yo[0] = cadd(a0, a1);
                yo[s] = cmul(csub(a0, a1), tw[p * s]);
            } else if (r == 4) {
                const double2 a0 = xi[0], a1 = xi[ms_], a2 = xi[2 * ms_], a3 = xi[3 * ms_];
                const double2 t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = mul_neg_i(csub(a1, a3));
                yo[0] = cadd(t0, t2);
                yo[s] = cmul(cadd(t1, t3), tw[p * s]);
                yo[2 * s] = cmul(csub(t0, t2), tw[2 * p * s]);
                yo[3 * s] = cmul(csub(t1, t3), tw[3 * p * s]);
            } else if (r == 3) {
                const double2 a0 = xi[0], a1 = xi[ms_], a2 = xi[2 * ms_];
                const double2 t1 = cadd(a1, a2);
                const double2 t2 = make_double2(a0.x - 0.5 * t1.x, a0.y - 0.5 * t1.y);
                const double2 d = csub(a1, a2);
                const double2 e = mul_neg_i(make_double2(0.86602540378443864676 * d.x, 0.86602540378443864676 * d.y));
                yo[0] = cadd(a0, t1);
                yo[s] = cmul(cadd(t2, e), tw[p * s]);
                yo[2 * s] = cmul(csub(t2, e), tw[2 * p * s]);
            } else {                                            // r == 5
                const double c1 = 0.30901699437494742410, c2 = -0.80901699437494742410;
                const double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;
                const double2 a0 = xi[0], a1 = xi[ms_], a2 = xi[2 * ms_], a3 = xi[3 * ms_], a4 = xi[4 * ms_];
                const double2 t1 = cadd(a1, a4), t2 = cadd(a2, a3), t3 = csub(a1, a4), t4 = csub(a2, a3);
                const double2 m1 = make_double2(a0.x + c1 * t1.x + c2 * t2.x, a0.y + c1 * t1.y + c2 * t2.y);
                const double2 m2 = make_double2(a0.x + c2 * t1.x + c1 * t2.x, a0.y + c2 * t1.y + c1 * t2.y);
                const double2 n1 = mul_neg_i(make_double2(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y));
                const double2 n2 = mul_neg_i(make_double2(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y));
                yo[0] = make_double2(a0.x + t1.x + t2.x, a0.y + t1.y + t2.y);
                yo[s] = cmul(cadd(m1, n1), tw[p * s]);
                yo[2 * s] = cmul(cadd(m2, n2), tw[2 * p * s]);
                yo[3 * s] = cmul(csub(m2, n2), tw[3 * p * s]);
                yo[4 * s] = cmul(csub(m1, n1), tw[4 * p * s]);
            }
        }
        __syncthreads();
        double2 *t = x;
        x = y;
        y = t;
        n = m;
        s *= r;
    }
    return x;
}

// Rows: two real rows ride in one complex transform (z = a + i b); the half spectra of both are separated with
// A_k = (Z_k + conj(Z_{N-k}))/2, B_k = (Z_k - conj(Z_{N-k}))/(2i).
__global__ void __launch_bounds__(512) fft_rows_kernel(const uint8_t *__restrict__ gray, int64_t frame_stride, int64_t row_stride,
                                                       int h, int w, int wh, const __grid_constant__ FftPlan plan,
                                                       const double2 *__restrict__ tw, double2 *__restrict__ g)
{
    extern __shared__ double2 fbuf[];
    const int y0 = 2 * blockIdx.x, y1 = y0 + 1;
    const uint8_t *src = gray + (int64_t)blockIdx.y * frame_stride;
    // all of a thread's pixels are requested before the first one is converted (memory-level parallelism: the kernel is latency-bound)
    const uint8_t *r0 = src + (int64_t)y0 * row_stride, *r1 = src + (int64_t)(y1 < h ? y1 : y0) * row_stride;
    for (int xb = 0; xb < w; xb += 4 * blockDim.x) {
        uint8_t a[4], b[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int x = xb + j * blockDim.x + threadIdx.x;
            a[j] = x < w ? r0[x] : 0;
            b[j] = x < w ? r1[x] : 0;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int x = xb + j * blockDim.x + threadIdx.x;
            if (x < w) fbuf[x] = make_double2((double)a[j], y1 < h ? (double)b[j] : 0.0);
        }
    }
    __syncthreads();
    const double2 *res = stockham(fbuf, fbuf + w, 1, plan, tw);
    double2 *ga = g + ((int64_t)blockIdx.y * h + y0) * wh;
    for (int k = threadIdx.x; k < wh; k += blockDim.x) {
        const double2 zk = res[k], zn = res[k == 0 ? 0 : w - k];
        ga[k] = make_double2(0.5 * (zk.x + zn.x), 0.5 * (zk.y - zn.y));
        if (y1 < h) ga[wh + k] = make_double2(0.5 * (zk.y + zn.y), 0.5 * (zn.x - zk.x));
    }
}

// 20 ln(sqrt(s) + 1) for s = re^2 + im^2 in [0, 2^67), absolute error < 2e-13 (the uint8 image has ~1.5 units per grey level, so
// a pixel would need to sit within 1e-13 of a rounding boundary to differ from the library functions' result). The library's
// sqrt() and log() — general-purpose, every special case handled — were ~60 % of fft_cols_kernel's instructions.
//   sqrt(s) = s rsqrt(s): a few ulp, and a relative error eps of sqrt(s) is an absolute error of at most 20 eps in the result.
//   ln x, x = t + 1 = 2^e m, m in [1, 2): the top 7 mantissa bits pick c_i = 1 + (i + 1/2)/128; q = m / c_i - 1 through a tabulated
//   reciprocal (|q| <= 2^-8, one FMA), ln m = -ln(1/c_i) + ln(1 + q) with the tabulated value taken of the ROUNDED reciprocal (so its
//   rounding costs nothing) and a degree-6 Taylor polynomial (next term 2e-18).
struct LogTab {
    double inv_c[128], neg_ln_inv_c[128];
};
__device__ __forceinline__ void logtab_fill(LogTab &t)                     // every thread of the CTA; a barrier must follow
{
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
        const double ic = 1.0 / (1.0 + ((double)i + 0.5) * (1.0 / 128.0));
        t.inv_c[i] = ic;
        t.neg_ln_inv_c[i] = -log(ic);
    }
}
__device__ __forceinline__ double log_magnitude20(const LogTab &t, double s)
{
    s = fmax(s, 1e-300);                                                    // s = 0: sqrt -> 1e-150, x = 1 exactly
    const double m = s * rsqrt(s);                                          // a relative error eps here is an absolute 20 eps in the result
    const long long b = __double_as_longlong(m + 1.0);
    const int e = (int)(b >> 52) - 1023, i = (int)(b >> 45) & 127;
    const double mant = __longlong_as_double((b & 0x000fffffffffffffll) | 0x3ff0000000000000ll);
    const double q = fma(mant, t.inv_c[i], -1.0);
    double p = fma(q, -1.0 / 6.0, 0.2);
    p = fma(q, p, -0.25);
    p = fma(q, p, 1.0 / 3.0);
    p = fma(q, p, -0.5);
    p = fma(q, p, 1.0);
    // |.|: for x = 1 the two halves cancel to +-1e-19, and the per-frame minimum is taken on the bit patterns of non-negative values
    return 20.0 * fabs(fma((double)e, 0.69314718055994530942, t.neg_ln_inv_c[i]) + p * q);
}

// Columns: `cc` adjacent columns per CTA (cc * 16 contiguous bytes per row), transform, then |F|, 20 ln(|F|+1), min/max.
__global__ void __launch_bounds__(512) fft_cols_kernel(const double2 *__restrict__ g, int h, int wh, int cc,
                                                       const __grid_constant__ FftPlan plan, const double2 *__restrict__ tw,
                                                       double *__restrict__ ms, unsigned long long *__restrict__ minmax)
{
    extern __shared__ double2 fbuf[];
    __shared__ unsigned long long smin, smax;
    __shared__ LogTab logtab;
    if (threadIdx.x == 0) { smin = ~0ull; smax = 0ull; }
    logtab_fill(logtab);
    const int v0 = blockIdx.x * cc;
    const double2 *src = g + (int64_t)blockIdx.y * h * wh;
    const int csh = cc == 4 ? 2 : (cc == 2 ? 1 : 0);              // cc is 1, 2 or 4 (host): i / cc and i % cc are a shift and a mask
    for (int ib = 0; ib < h * cc; ib += 4 * blockDim.x) {          // four loads in flight per thread before the first store
        double2 t[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = ib + j * blockDim.x + threadIdx.x;
            const int y = i >> csh, c = i & (cc - 1);
            t[j] = (i < h * cc && v0 + c < wh) ? src[(int64_t)y * wh + v0 + c] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = ib + j * blockDim.x + threadIdx.x;
            const int y = i >> csh, c = i & (cc - 1);
            if (i < h * cc) fbuf[c * h + y] = t[j];
        }
    }
    __syncthreads();
    const double2 *res = stockham(fbuf, fbuf + cc * h, cc, plan, tw);
    double *dst = ms + (int64_t)blockIdx.y * h * wh;
    unsigned long long lo = ~0ull, hi = 0ull;
    for (int i = threadIdx.x; i < h * cc; i += blockDim.x) {
        const int u = i >> csh, c = i & (cc - 1);
        if (v0 + c >= wh) continue;
        const double2 f = res[c * h + u];
        // |F| <= 255 H W < 2^33: the squares cannot overflow or underflow harmfully, so re^2 + im^2 needs none of hypot()'s scaling
        const double m = log_magnitude20(logtab, fma(f.x, f.x, f.y * f.y));
        dst[(int64_t)u * wh + v0 + c] = m;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(m);
        lo = bits < lo ? bits : lo;
        hi = bits > hi ? bits : hi;
    }
    atomicMin(&smin, lo);
    atomicMax(&smax, hi);
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicMin(&minmax[2 * blockIdx.y], smin);
        atomicMax(&minmax[2 * blockIdx.y + 1], smax);
    }
}

// out[i][j] = u8(rint(ms_shifted[i][j] * scale + shift)), cv2.normalize(NORM_MINMAX, 0..255) + np.fft.fftshift.
// grid (column blocks, rows, frames): no index divisions.
__global__ void __launch_bounds__(256) spectrum_image_kernel(const double *__restrict__ ms, const unsigned long long *__restrict__ minmax,
                                                             int h, int w, int wh, uint8_t *__restrict__ out)
{
    const int frame = blockIdx.z;
    const double mn = __longlong_as_double((long long)minmax[2 * frame]), mx = __longlong_as_double((long long)minmax[2 * frame + 1]);
    const double scale = (mx - mn) > 2.220446049250313e-16 ? 255.0 / (mx - mn) : 0.0;   // cv::normalize: DBL_EPSILON guard
    const double shift = 0.0 - mn * scale;
    const double *src = ms + (int64_t)frame * h * wh;
    uint8_t *dst = out + (int64_t)frame * h * w;
    for (int i = blockIdx.y; i < h; i += gridDim.y) {
        int u0 = i - h / 2;                                      // fftshift: y[i] = x[(i - n//2) mod n]
        u0 = u0 < 0 ? u0 + h : u0;
        const int um = u0 == 0 ? 0 : h - u0;                     // Hermitian mirror row: |F[u][v]| = |F[-u][-v]|
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < w; j += gridDim.x * blockDim.x) {
            int v = j - w / 2;
            v = v < 0 ? v + w : v;
            const int u = v >= wh ? um : u0;
            v = v >= wh ? w - v : v;
            double r = rint(__dadd_rn(__dmul_rn(src[(int64_t)u * wh + v], scale), shift));   // cvRound: ties to even
            r = r < 0.0 ? 0.0 : (r > 255.0 ? 255.0 : r);
            dst[(int64_t)i * w + j] = (uint8_t)r;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Ragged calls (v5ela_spectrum_ragged): frames of different sizes in one launch sequence, planned on the host
// (v5ela_spec_plan.h). Each kernel flattens its grid in x; a CTA finds its frame through the chunk's CTA prefix table
// (cta_frame) and then runs the body of the uniform kernel above for that frame, with the frame's FftPlan read from the size
// table instead of a __grid_constant__. The bodies are copies, not shared functions, so that the uniform kernels' code stays
// exactly as it is; every arithmetic step is the same, so every frame's image is byte-identical to v5ela_spectrum's.

// The twiddle tables of every distinct side of the call, back to back in one arena: blockDim.x entries per CTA.
__global__ void __launch_bounds__(256) twiddle_ragged_kernel(const SpecSize *__restrict__ sizes, int ns, const uint32_t *__restrict__ base,
                                                             double2 *__restrict__ tw)
{
    const int k = cta_frame(base, ns, blockIdx.x);
    const int n = sizes[k].n;
    const int m = (int)(blockIdx.x - base[k]) * blockDim.x + threadIdx.x;
    if (m >= n) return;
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tw[sizes[k].tw + m] = make_double2(c, -s);
}

// dft_rows_kernel for one TILE x TILE output tile of one frame
__global__ void __launch_bounds__(256) dft_rows_ragged_kernel(const SpecFrame *__restrict__ frames, int nf, const uint32_t *__restrict__ base,
                                                              const SpecSize *__restrict__ sizes, const double2 *__restrict__ tw_arena,
                                                              double2 *__restrict__ g)
{
    __shared__ double xs[TILE][KC + 1];
    const int fi = cta_frame(base, nf, blockIdx.x);
    const SpecFrame f = frames[fi];
    const int local = (int)(blockIdx.x - base[fi]), ty_ = local / f.gx;
    const int h = f.h, w = f.w, wh = f.wh;
    const int64_t row_stride = f.row_stride;
    const double2 *__restrict__ tw = tw_arena + sizes[f.sw].tw;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int y0 = ty_ * TILE, v0 = (local - ty_ * f.gx) * TILE;
    const uint8_t *src = f.gray;
    const int va = v0 + tx, vb = v0 + tx + 16;
    int ia = 0, ib = 0;
    const int sa = va % w, sb = vb % w;
    double2 acc[2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
    for (int x0 = 0; x0 < w; x0 += KC) {
        for (int i = threadIdx.x; i < TILE * KC; i += 256) {
            const int r = i / KC, c = i - r * KC;
            const int y = y0 + r, x = x0 + c;
            xs[r][c] = (y < h && x < w) ? (double)src[(int64_t)y * row_stride + x] : 0.0;
        }
        __syncthreads();
        const int kn = min(KC, w - x0);
        for (int k = 0; k < kn; k++) {
            const double2 ta = tw[ia], tb = tw[ib];
            const double xa = xs[ty][k], xb = xs[ty + 16][k];
            acc[0][0].x = fma(xa, ta.x, acc[0][0].x); acc[0][0].y = fma(xa, ta.y, acc[0][0].y);
            acc[0][1].x = fma(xa, tb.x, acc[0][1].x); acc[0][1].y = fma(xa, tb.y, acc[0][1].y);
            acc[1][0].x = fma(xb, ta.x, acc[1][0].x); acc[1][0].y = fma(xb, ta.y, acc[1][0].y);
            acc[1][1].x = fma(xb, tb.x, acc[1][1].x); acc[1][1].y = fma(xb, tb.y, acc[1][1].y);
            ia += sa; ia = ia >= w ? ia - w : ia;
            ib += sb; ib = ib >= w ? ib - w : ib;
        }
        __syncthreads();
    }
    double2 *dst = g + f.g_off;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int y = y0 + ty + 16 * i;
        if (y >= h) continue;
        if (va < wh) dst[(int64_t)y * wh + va] = acc[i][0];
        if (vb < wh) dst[(int64_t)y * wh + vb] = acc[i][1];
    }
}

// dft_cols_kernel for one TILE x TILE output tile of one frame
__global__ void __launch_bounds__(256) dft_cols_ragged_kernel(const SpecFrame *__restrict__ frames, int nf, const uint32_t *__restrict__ base,
                                                              const SpecSize *__restrict__ sizes, const double2 *__restrict__ tw_arena,
                                                              const double2 *__restrict__ g, double *__restrict__ ms,
                                                              unsigned long long *__restrict__ minmax)
{
    __shared__ double2 gs[KC][TILE + 1];
    __shared__ unsigned long long smin, smax;
    const int fi = cta_frame(base, nf, blockIdx.x);
    const SpecFrame f = frames[fi];
    const int local = (int)(blockIdx.x - base[fi]), ty_ = local / f.gx;
    const int h = f.h, wh = f.wh;
    const double2 *__restrict__ tw = tw_arena + sizes[f.sh].tw;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int u0 = ty_ * TILE, v0 = (local - ty_ * f.gx) * TILE;
    const double2 *src = g + f.g_off;
    if (threadIdx.x == 0) { smin = ~0ull; smax = 0ull; }
    const int ua = u0 + ty, ub = u0 + ty + 16;
    int ia = 0, ib = 0;
    const int sa = ua % h, sb = ub % h;
    double2 acc[2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
    for (int y0 = 0; y0 < h; y0 += KC) {
        for (int i = threadIdx.x; i < KC * TILE; i += 256) {
            const int r = i / TILE, c = i - r * TILE;
            const int y = y0 + r, v = v0 + c;
            gs[r][c] = (y < h && v < wh) ? src[(int64_t)y * wh + v] : make_double2(0.0, 0.0);
        }
        __syncthreads();
        const int kn = min(KC, h - y0);
        for (int k = 0; k < kn; k++) {
            const double2 ta = tw[ia], tb = tw[ib];
            const double2 ga = gs[k][tx], gb = gs[k][tx + 16];
            acc[0][0].x = fma(ga.x, ta.x, fma(-ga.y, ta.y, acc[0][0].x)); acc[0][0].y = fma(ga.x, ta.y, fma(ga.y, ta.x, acc[0][0].y));
            acc[0][1].x = fma(gb.x, ta.x, fma(-gb.y, ta.y, acc[0][1].x)); acc[0][1].y = fma(gb.x, ta.y, fma(gb.y, ta.x, acc[0][1].y));
            acc[1][0].x = fma(ga.x, tb.x, fma(-ga.y, tb.y, acc[1][0].x)); acc[1][0].y = fma(ga.x, tb.y, fma(ga.y, tb.x, acc[1][0].y));
            acc[1][1].x = fma(gb.x, tb.x, fma(-gb.y, tb.y, acc[1][1].x)); acc[1][1].y = fma(gb.x, tb.y, fma(gb.y, tb.x, acc[1][1].y));
            ia += sa; ia = ia >= h ? ia - h : ia;
            ib += sb; ib = ib >= h ? ib - h : ib;
        }
        __syncthreads();
    }
    double *dst = ms + f.ms_off;
    unsigned long long lo = ~0ull, hi = 0ull;
#pragma unroll
    for (int i = 0; i < 2; i++) {
#pragma unroll
        for (int j = 0; j < 2; j++) {
            const int u = u0 + ty + 16 * i, v = v0 + tx + 16 * j;
            if (u >= h || v >= wh) continue;
            const double m = 20.0 * log(hypot(acc[i][j].x, acc[i][j].y) + 1.0);
            dst[(int64_t)u * wh + v] = m;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(m);
            lo = bits < lo ? bits : lo;
            hi = bits > hi ? bits : hi;
        }
    }
    atomicMin(&smin, lo);
    atomicMax(&smax, hi);
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicMin(&minmax[2 * f.mm], smin);
        atomicMax(&minmax[2 * f.mm + 1], smax);
    }
}

// fft_rows_kernel for one pair of rows of one frame
__global__ void __launch_bounds__(512) fft_rows_ragged_kernel(const SpecFrame *__restrict__ frames, int nf, const uint32_t *__restrict__ base,
                                                              const SpecSize *__restrict__ sizes, const double2 *__restrict__ tw_arena,
                                                              double2 *__restrict__ g)
{
    extern __shared__ double2 fbuf[];
    const int fi = cta_frame(base, nf, blockIdx.x);
    const SpecFrame f = frames[fi];
    const int h = f.h, w = f.w, wh = f.wh;
    const SpecSize &sz = sizes[f.sw];
    const int y0 = 2 * (int)(blockIdx.x - base[fi]), y1 = y0 + 1;
    const uint8_t *src = f.gray;
    const uint8_t *r0 = src + (int64_t)y0 * f.row_stride, *r1 = src + (int64_t)(y1 < h ? y1 : y0) * f.row_stride;
    for (int xb = 0; xb < w; xb += 4 * blockDim.x) {
        uint8_t a[4], b[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int x = xb + j * blockDim.x + threadIdx.x;
            a[j] = x < w ? r0[x] : 0;
            b[j] = x < w ? r1[x] : 0;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int x = xb + j * blockDim.x + threadIdx.x;
            if (x < w) fbuf[x] = make_double2((double)a[j], y1 < h ? (double)b[j] : 0.0);
        }
    }
    __syncthreads();
    const double2 *res = stockham(fbuf, fbuf + w, 1, sz.plan, tw_arena + sz.tw);
    double2 *ga = g + f.g_off + (int64_t)y0 * wh;
    for (int k = threadIdx.x; k < wh; k += blockDim.x) {
        const double2 zk = res[k], zn = res[k == 0 ? 0 : w - k];
        ga[k] = make_double2(0.5 * (zk.x + zn.x), 0.5 * (zk.y - zn.y));
        if (y1 < h) ga[wh + k] = make_double2(0.5 * (zk.y + zn.y), 0.5 * (zn.x - zk.x));
    }
}

// fft_cols_kernel for cc adjacent columns of one frame
__global__ void __launch_bounds__(512) fft_cols_ragged_kernel(const SpecFrame *__restrict__ frames, int nf, const uint32_t *__restrict__ base,
                                                              const SpecSize *__restrict__ sizes, const double2 *__restrict__ tw_arena,
                                                              const double2 *__restrict__ g, double *__restrict__ ms,
                                                              unsigned long long *__restrict__ minmax)
{
    extern __shared__ double2 fbuf[];
    __shared__ unsigned long long smin, smax;
    __shared__ LogTab logtab;
    if (threadIdx.x == 0) { smin = ~0ull; smax = 0ull; }
    logtab_fill(logtab);
    const int fi = cta_frame(base, nf, blockIdx.x);
    const SpecFrame f = frames[fi];
    const int h = f.h, wh = f.wh, cc = f.cc;
    const SpecSize &sz = sizes[f.sh];
    const int v0 = (int)(blockIdx.x - base[fi]) * cc;
    const double2 *src = g + f.g_off;
    const int csh = cc == 4 ? 2 : (cc == 2 ? 1 : 0);
    for (int ib = 0; ib < h * cc; ib += 4 * blockDim.x) {
        double2 t[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = ib + j * blockDim.x + threadIdx.x;
            const int y = i >> csh, c = i & (cc - 1);
            t[j] = (i < h * cc && v0 + c < wh) ? src[(int64_t)y * wh + v0 + c] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = ib + j * blockDim.x + threadIdx.x;
            const int y = i >> csh, c = i & (cc - 1);
            if (i < h * cc) fbuf[c * h + y] = t[j];
        }
    }
    __syncthreads();
    const double2 *res = stockham(fbuf, fbuf + cc * h, cc, sz.plan, tw_arena + sz.tw);
    double *dst = ms + f.ms_off;
    unsigned long long lo = ~0ull, hi = 0ull;
    for (int i = threadIdx.x; i < h * cc; i += blockDim.x) {
        const int u = i >> csh, c = i & (cc - 1);
        if (v0 + c >= wh) continue;
        const double2 fv = res[c * h + u];
        const double m = log_magnitude20(logtab, fma(fv.x, fv.x, fv.y * fv.y));
        dst[(int64_t)u * wh + v0 + c] = m;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(m);
        lo = bits < lo ? bits : lo;
        hi = bits > hi ? bits : hi;
    }
    atomicMin(&smin, lo);
    atomicMax(&smax, hi);
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicMin(&minmax[2 * f.mm], smin);
        atomicMax(&minmax[2 * f.mm + 1], smax);
    }
}

// spectrum_image_kernel for one (column block, row block) of one frame: f.bx x f.by CTAs per frame
__global__ void __launch_bounds__(256) spectrum_image_ragged_kernel(const SpecFrame *__restrict__ frames, int nf, const uint32_t *__restrict__ base,
                                                                    const double *__restrict__ ms,
                                                                    const unsigned long long *__restrict__ minmax)
{
    const int fi = cta_frame(base, nf, blockIdx.x);
    const SpecFrame f = frames[fi];
    const int local = (int)(blockIdx.x - base[fi]), by_ = local / f.bx, bx_ = local - by_ * f.bx;
    const int h = f.h, w = f.w, wh = f.wh;
    const double mn = __longlong_as_double((long long)minmax[2 * f.mm]), mx = __longlong_as_double((long long)minmax[2 * f.mm + 1]);
    const double scale = (mx - mn) > 2.220446049250313e-16 ? 255.0 / (mx - mn) : 0.0;
    const double shift = 0.0 - mn * scale;
    const double *src = ms + f.ms_off;
    uint8_t *dst = f.out;
    for (int i = by_; i < h; i += f.by) {
        int u0 = i - h / 2;
        u0 = u0 < 0 ? u0 + h : u0;
        const int um = u0 == 0 ? 0 : h - u0;
        for (int j = bx_ * blockDim.x + threadIdx.x; j < w; j += f.bx * blockDim.x) {
            int v = j - w / 2;
            v = v < 0 ? v + w : v;
            const int u = v >= wh ? um : u0;
            v = v >= wh ? w - v : v;
            double r = rint(__dadd_rn(__dmul_rn(src[(int64_t)u * wh + v], scale), shift));
            r = r < 0.0 ? 0.0 : (r > 255.0 ? 255.0 : r);
            dst[(int64_t)i * w + j] = (uint8_t)r;
        }
    }
}

}  // namespace v5fft
