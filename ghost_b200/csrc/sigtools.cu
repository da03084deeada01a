// Device versions of the ghost.sigtools helpers (SURVEY.md section 8(f), "next" rows):
//
//   fastconv_scipy / fastconv_fftw   ghost/sigtools/convolution.py:16-216  -> gcwt_fastconv
//   chirpz_dft                       ghost/sigtools/fourier.py:9-48        -> gcwt_dft
//   analytic_signal_scipy / _fftw    ghost/sigtools/analytic.py:15-112     -> gcwt_analytic_signal
//
// All in complex128 like the reference.  They share the batched power-of-two Stockham FFT of
// the generic CWT path; lengths that are not a power of two go through Bluestein's chirp-z
// identity (what chirpz_dft does on the CPU) with exact integer phase reduction.
//
// Reductions of a result on the device, so that only the reduced array crosses the link: moments and
// time pooling for displays, scale-averaged band power (band_reduce_kernel) and event-locked power and phase
// (event_reduce_kernel).
#include "plan.h"
#include "common.cuh"
#include "fft_global.cuh"
#include <algorithm>
#include <string>
#include <vector>

namespace gcwt {

typedef double2 C;

// e^{sign * i * pi * j^2 / n} with j^2 reduced mod 2n in integers
__device__ __forceinline__ C chirp(int64_t j, int64_t n, int sign) {
    const int64_t r = (j % (2 * n)) * (j % (2 * n)) % (2 * n);
    C w;
    sincospi((double)sign * (double)r / (double)n, &w.y, &w.x);
    return w;
}

__global__ void st_pad_real(const double* __restrict__ x, int64_t n, C* __restrict__ out, int64_t m) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[i] = make_double2(i < n ? x[i] : 0.0, 0.0);
}

__global__ void st_pad_complex(const C* __restrict__ x, int64_t n, C* __restrict__ out, int64_t m) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[i] = i < n ? x[i] : make_double2(0.0, 0.0);
}

__global__ void st_mul(C* __restrict__ a, const C* __restrict__ b, int64_t m, double scale) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) {
        const C p = cmul(a[i], b[i]);
        a[i] = make_double2(p.x * scale, p.y * scale);
    }
}

__global__ void st_scale(C* __restrict__ a, int64_t m, double scale) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) a[i] = make_double2(a[i].x * scale, a[i].y * scale);
}

__global__ void st_bluestein_pre(const C* __restrict__ x, int64_t n, C* __restrict__ a, int64_t m, int sign) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) a[i] = i < n ? cmul(x[i], chirp(i, n, sign)) : make_double2(0.0, 0.0);
}

__global__ void st_bluestein_kernel(C* __restrict__ b, int64_t n, int64_t m, int sign) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    C v = make_double2(0.0, 0.0);
    if (i < n) v = chirp(i, n, -sign);
    else if (m - i < n) v = chirp(m - i, n, -sign);
    b[i] = v;
}

__global__ void st_bluestein_post(const C* __restrict__ conv, int64_t n, C* __restrict__ out, int sign, double scale) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) {
        const C p = cmul(conv[k], chirp(k, n, sign));
        out[k] = make_double2(p.x * scale, p.y * scale);
    }
}

// scipy.signal.hilbert weights: 1 at DC (and Nyquist for even n), 2 for positive, 0 for negative frequencies
__global__ void st_hilbert_weights(C* __restrict__ X, int64_t n) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double w;
    if (k == 0 || (2 * k == n)) w = 1.0;
    else if (2 * k < n) w = 2.0;
    else w = 0.0;
    X[k] = make_double2(X[k].x * w, X[k].y * w);
}

static inline unsigned nblk(int64_t m) { return (unsigned)((m + 255) / 256); }

// Cyclic convolution of two m-point buffers (m a power of two): forward transforms of a and b, their product
// scaled by 1/m, inverse transform.  `t` is a third m-point buffer; all three are overwritten, and the one that
// holds the result is returned.
static C* cyclic_conv(C* a, C* b, C* t, int64_t m) {
    C* spare = t;
    fft_batched<-1>(a, spare, (int)m, 1, 0);
    fft_batched<-1>(b, spare, (int)m, 1, 0);
    st_mul<<<nblk(m), 256>>>(a, b, m, 1.0 / (double)m);
    count_launch();
    fft_batched<+1>(a, spare, (int)m, 1, 0);
    return a;
}

// DFT of arbitrary length n (device in -> device out), sign = -1 forward / +1 backward (unscaled).
static int dft_any(const C* d_in, int64_t n, int sign, C* d_out) {
    if (n > (int64_t(1) << 26)) { set_error("sigtools: transform too long"); return GCWT_ERR_UNSUPPORTED; }
    const bool pow2 = (n & (n - 1)) == 0;
    if (pow2) {
        DevBuf t; int rc = t.alloc(sizeof(C) * n); if (rc) return rc;
        GCWT_CUDA_OK(cudaMemcpy(d_out, d_in, sizeof(C) * n, cudaMemcpyDeviceToDevice));
        C* res = d_out;
        C* spare = t.c();
        if (sign < 0) fft_batched<-1>(res, spare, (int)n, 1, 0); else fft_batched<+1>(res, spare, (int)n, 1, 0);
        if (res != d_out) GCWT_CUDA_OK(cudaMemcpy(d_out, res, sizeof(C) * n, cudaMemcpyDeviceToDevice));
        return GCWT_OK;
    }
    const int64_t m = int64_t(1) << ilog2_ceil(2 * n - 1);
    DevBuf a, b, t;
    int rc = a.alloc(sizeof(C) * m); if (rc) return rc;
    rc = b.alloc(sizeof(C) * m); if (rc) return rc;
    rc = t.alloc(sizeof(C) * m); if (rc) return rc;
    st_bluestein_pre<<<nblk(m), 256>>>(d_in, n, a.c(), m, sign);
    st_bluestein_kernel<<<nblk(m), 256>>>(b.c(), n, m, sign);
    count_launch(2);
    const C* conv = cyclic_conv(a.c(), b.c(), t.c(), m);
    st_bluestein_post<<<nblk(n), 256>>>(conv, n, d_out, sign, 1.0);
    count_launch();
    GCWT_CUDA_OK(cudaGetLastError());
    GCWT_CUDA_OK(cudaDeviceSynchronize());
    return GCWT_OK;
}

int sig_dft_host(const double* x_host, int64_t n, int sign, double* out_host) {
    DevBuf in, out;
    int rc = in.alloc(sizeof(C) * n); if (rc) return rc;
    rc = out.alloc(sizeof(C) * n); if (rc) return rc;
    GCWT_CUDA_OK(cudaMemcpy(in.p, x_host, sizeof(C) * n, cudaMemcpyHostToDevice));
    rc = dft_any(in.c(), n, sign, out.c()); if (rc) return rc;
    GCWT_CUDA_OK(cudaMemcpy(out_host, out.p, sizeof(C) * n, cudaMemcpyDeviceToHost));
    return GCWT_OK;
}

int sig_analytic_host(const double* x_host, int64_t n, double* out_host) {
    DevBuf xr, a, b;
    int rc = xr.alloc(sizeof(double) * n); if (rc) return rc;
    rc = a.alloc(sizeof(C) * n); if (rc) return rc;
    rc = b.alloc(sizeof(C) * n); if (rc) return rc;
    GCWT_CUDA_OK(cudaMemcpy(xr.p, x_host, sizeof(double) * n, cudaMemcpyHostToDevice));
    st_pad_real<<<nblk(n), 256>>>((const double*)xr.p, n, a.c(), n);
    count_launch();
    rc = dft_any(a.c(), n, -1, b.c()); if (rc) return rc;
    st_hilbert_weights<<<nblk(n), 256>>>(b.c(), n);
    count_launch();
    rc = dft_any(b.c(), n, +1, a.c()); if (rc) return rc;
    st_scale<<<nblk(n), 256>>>(a.c(), n, 1.0 / (double)n);
    count_launch();
    GCWT_CUDA_OK(cudaGetLastError());
    GCWT_CUDA_OK(cudaMemcpy(out_host, a.p, sizeof(C) * n, cudaMemcpyDeviceToHost));
    return GCWT_OK;
}

// Full linear convolution (n + m - 1 complex outputs) of complex signal and kernel.
int sig_fastconv_host(const double* sig_host, int sig_complex, int64_t n, const double* ker_host, int ker_complex,
                      int64_t m, double* out_host) {
    const int64_t tot = n + m - 1;
    if (tot > (int64_t(1) << 26)) { set_error("fastconv: n + m - 1 above 2^26, convolve in blocks"); return GCWT_ERR_UNSUPPORTED; }
    const int64_t nfft = int64_t(1) << ilog2_ceil(tot);
    DevBuf raw_s, raw_k, a, b, t;
    int rc = raw_s.alloc(sizeof(double) * n * (sig_complex ? 2 : 1)); if (rc) return rc;
    rc = raw_k.alloc(sizeof(double) * m * (ker_complex ? 2 : 1)); if (rc) return rc;
    rc = a.alloc(sizeof(C) * nfft); if (rc) return rc;
    rc = b.alloc(sizeof(C) * nfft); if (rc) return rc;
    rc = t.alloc(sizeof(C) * nfft); if (rc) return rc;
    GCWT_CUDA_OK(cudaMemcpy(raw_s.p, sig_host, sizeof(double) * n * (sig_complex ? 2 : 1), cudaMemcpyHostToDevice));
    GCWT_CUDA_OK(cudaMemcpy(raw_k.p, ker_host, sizeof(double) * m * (ker_complex ? 2 : 1), cudaMemcpyHostToDevice));
    if (sig_complex) st_pad_complex<<<nblk(nfft), 256>>>((const C*)raw_s.p, n, a.c(), nfft);
    else st_pad_real<<<nblk(nfft), 256>>>((const double*)raw_s.p, n, a.c(), nfft);
    if (ker_complex) st_pad_complex<<<nblk(nfft), 256>>>((const C*)raw_k.p, m, b.c(), nfft);
    else st_pad_real<<<nblk(nfft), 256>>>((const double*)raw_k.p, m, b.c(), nfft);
    count_launch(2);
    const C* res = cyclic_conv(a.c(), b.c(), t.c(), nfft);
    GCWT_CUDA_OK(cudaGetLastError());
    GCWT_CUDA_OK(cudaMemcpy(out_host, res, sizeof(C) * tot, cudaMemcpyDeviceToHost));
    return GCWT_OK;
}

// ---------------------------------------------------------------------------- moments
// sum and sum of squares (of x, or of x^2 when `square`) in fp64: the global mean / std that
// plot(standardize=True) needs (ghost/wave/transforms.py:360-366) without a host pass.
template <typename T>
__global__ void moments_kernel(const T* __restrict__ x, int64_t n, int square, double* __restrict__ acc) {
    double s1 = 0.0, s2 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = (double)x[i];
        if (square) v *= v;
        s1 += v;
        s2 += v * v;
    }
    __shared__ double sh1[256], sh2[256];
    sh1[threadIdx.x] = s1; sh2[threadIdx.x] = s2;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k) { sh1[threadIdx.x] += sh1[threadIdx.x + k]; sh2[threadIdx.x] += sh2[threadIdx.x + k]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { atomicAdd(acc, sh1[0]); atomicAdd(acc + 1, sh2[0]); }
}

int sig_moments(const void* x_dev, int type, int64_t n, int square, double* out_host, cudaStream_t st) {
    DevBuf buf;
    { int rc = buf.alloc(2 * sizeof(double)); if (rc) return rc; }
    double* d = buf.as<double>();
    GCWT_CUDA_OK(cudaMemsetAsync(d, 0, 2 * sizeof(double), st));
    const unsigned blocks = (unsigned)std::min<int64_t>(148 * 8, (n + 255) / 256);
    if (type == GCWT_F32) moments_kernel<float><<<blocks, 256, 0, st>>>((const float*)x_dev, n, square, d);
    else moments_kernel<double><<<blocks, 256, 0, st>>>((const double*)x_dev, n, square, d);
    count_launch();
    GCWT_CUDA_OK(cudaGetLastError());
    double h[2];
    GCWT_CUDA_OK(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, st));
    GCWT_CUDA_OK(cudaStreamSynchronize(st));
    const double mean = h[0] / (double)n;
    double var = h[1] / (double)n - mean * mean;
    if (var < 0.0) var = 0.0;
    out_host[0] = mean;
    out_host[1] = sqrt(var);
    return GCWT_OK;
}

// ----------------------------------------------------------------------------- pooling for display
// plot() draws contourf over the whole (scales, samples) array (ghost/wave/transforms.py:356-367,395-396);
// a display has a few thousand columns.  One warp reduces one bin of `width` consecutive samples of one
// row to its mean or maximum (of x, or of x^2 for power from amplitude), accumulating in fp64: the
// consumer then pulls (rows x bins) values over PCIe instead of 4 bytes per coefficient.
template <typename T>
__global__ void __launch_bounds__(256)
pool_rows_kernel(const T* __restrict__ x, int64_t row_stride, int64_t n_cols, int64_t width, int mode, int square,
                 double* __restrict__ out, int64_t out_stride, int64_t n_bins) {
    const int64_t bin = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bin >= n_bins) return;
    const int64_t lo = bin * width, hi = min(n_cols, lo + width);
    const T* row = x + (int64_t)blockIdx.y * row_stride;
    double acc = mode == 1 ? -1.0e300 : 0.0;
    for (int64_t i = lo + lane; i < hi; i += 32) {
        double v = (double)row[i];
        if (square) v *= v;
        acc = mode == 1 ? fmax(acc, v) : acc + v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double other = __shfl_xor_sync(0xffffffffu, acc, o);
        acc = mode == 1 ? fmax(acc, other) : acc + other;
    }
    if (lane == 0) out[(int64_t)blockIdx.y * out_stride + bin] = mode == 1 ? acc : acc / (double)(hi - lo);
}

int pool_rows_launch(const void* x_dev, int type, int64_t n_rows, int64_t n_cols, int64_t row_stride, int64_t width,
                     int mode, int square, double* out_dev, int64_t out_stride, cudaStream_t st) {
    if (n_rows <= 0 || n_cols <= 0 || width <= 0 || (mode != 0 && mode != 1)) { set_error("pool_rows: bad argument"); return GCWT_ERR_ARG; }
    const int64_t n_bins = (n_cols + width - 1) / width;
    for (int64_t r0 = 0; r0 < n_rows; r0 += 65535) {                 // gridDim.y limit
        const int64_t rows = std::min<int64_t>(65535, n_rows - r0);
        dim3 grid((unsigned)((n_bins + 7) / 8), (unsigned)rows);
        if (type == GCWT_F32)
            pool_rows_kernel<float><<<grid, 256, 0, st>>>((const float*)x_dev + r0 * row_stride, row_stride, n_cols, width, mode,
                                                          square, out_dev + r0 * out_stride, out_stride, n_bins);
        else
            pool_rows_kernel<double><<<grid, 256, 0, st>>>((const double*)x_dev + r0 * row_stride, row_stride, n_cols, width,
                                                           mode, square, out_dev + r0 * out_stride, out_stride, n_bins);
        count_launch();
    }
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// ----------------------------------------------------------------------------- scale-averaged band power
// Band power over time (theta, gamma, ripple envelopes) averages |W|^2 over the adjacent scales of a band.
// One thread owns VEC consecutive samples of one (channel, band) and walks the band's rows: a pure streaming
// read of 16-byte loads when the rows are aligned, accumulated in fp64 with explicit fma so that the vector
// and scalar paths give the same bits.  Overlapping bands re-read their shared rows.
__device__ __forceinline__ double mag2(float v, bool power) { const double d = v; return power ? d : d * d; }
__device__ __forceinline__ double mag2(double v, bool power) { return power ? v : v * v; }
__device__ __forceinline__ double mag2(float2 v, bool) { const double re = v.x, im = v.y; return fma(re, re, im * im); }
__device__ __forceinline__ double mag2(double2 v, bool) { return fma(v.x, v.x, v.y * v.y); }

template <typename In, typename Out, int VEC, bool POWER>
__global__ void __launch_bounds__(256)
band_reduce_kernel(const In* __restrict__ x, int64_t n, int64_t s_stride, int64_t c_stride, Out* __restrict__ out,
                   int64_t ob_stride, int64_t oc_stride, const __grid_constant__ BandTable tab) {
    struct alignas(sizeof(In) * VEC) InV { In v[VEC]; };
    struct alignas(sizeof(Out) * VEC) OutV { Out v[VEC]; };
    const int b = blockIdx.z;
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    if (i0 >= n) return;
    const int cnt = tab.count[b];
    const double* w = tab.w + tab.off[b];
    const In* row = x + (int64_t)blockIdx.y * c_stride + (int64_t)tab.first[b] * s_stride + i0;
    Out* dst = out + (int64_t)blockIdx.y * oc_stride + (int64_t)b * ob_stride + i0;
    double acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.0;
    if (i0 + VEC <= n) {
#pragma unroll 4
        for (int k = 0; k < cnt; ++k) {
            const InV v = *reinterpret_cast<const InV*>(row + (int64_t)k * s_stride);
            const double wk = w[k];
#pragma unroll
            for (int j = 0; j < VEC; ++j) acc[j] = fma(wk, mag2(v.v[j], POWER), acc[j]);
        }
        OutV o;
#pragma unroll
        for (int j = 0; j < VEC; ++j) o.v[j] = (Out)acc[j];
        *reinterpret_cast<OutV*>(dst) = o;
    } else {                                                         // the row's last, partial vector
        const int m = (int)(n - i0);
        for (int k = 0; k < cnt; ++k)
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                if (j < m) acc[j] = fma(w[k], mag2(row[(int64_t)k * s_stride + j], POWER), acc[j]);
#pragma unroll
        for (int j = 0; j < VEC; ++j)
            if (j < m) dst[j] = (Out)acc[j];
    }
}

int band_table_build(int n_bands, const int32_t* first, const int32_t* count, const double* weights, BandTable* tab,
                     const char* who) {
    const std::string pre = std::string(who) + ": ";
    if (!first || !count || !weights) { set_error(pre + "band_first / band_count / weights is NULL"); return GCWT_ERR_ARG; }
    if (n_bands < 1 || n_bands > kMaxBands) {
        set_error(pre + "n_bands must be 1 .. " + std::to_string(kMaxBands) + " (got " + std::to_string(n_bands) + ")");
        return GCWT_ERR_ARG;
    }
    tab->n_bands = n_bands;
    tab->rows = 0;
    int off = 0;
    for (int b = 0; b < n_bands; ++b) {
        if (first[b] < 0 || count[b] < 1) {
            set_error(pre + "band " + std::to_string(b) + " needs first >= 0 and count >= 1 (got first " +
                      std::to_string(first[b]) + ", count " + std::to_string(count[b]) + ")");
            return GCWT_ERR_ARG;
        }
        if (count[b] > kMaxBandEntries - off) {
            set_error(pre + "the bands hold more than " + std::to_string(kMaxBandEntries) + " (band, scale) entries");
            return GCWT_ERR_ARG;
        }
        tab->first[b] = first[b];
        tab->count[b] = count[b];
        tab->off[b] = off;
        for (int k = 0; k < count[b]; ++k) tab->w[off + k] = weights[off + k];
        off += count[b];
        tab->rows = std::max<int32_t>(tab->rows, (int32_t)std::min<int64_t>((int64_t)first[b] + count[b], INT32_MAX));
    }
    return GCWT_OK;
}

template <typename In, typename Out, int VEC>
static void band_launch(const void* x, int kind, int64_t n_ch, int64_t n, int64_t s_stride, int64_t c_stride,
                        const BandTable& tab, void* out, int64_t ob_stride, int64_t oc_stride, cudaStream_t st) {
    for (int64_t c0 = 0; c0 < n_ch; c0 += 65535) {                   // gridDim.y limit
        const int64_t rows = std::min<int64_t>(65535, n_ch - c0);
        dim3 grid((unsigned)((n + 256 * VEC - 1) / (256 * VEC)), (unsigned)rows, (unsigned)tab.n_bands);
        const In* xs = (const In*)x + c0 * c_stride;
        Out* os = (Out*)out + c0 * oc_stride;
        if (kind == GCWT_OUT_POWER)
            band_reduce_kernel<In, Out, VEC, true><<<grid, 256, 0, st>>>(xs, n, s_stride, c_stride, os, ob_stride, oc_stride, tab);
        else
            band_reduce_kernel<In, Out, VEC, false><<<grid, 256, 0, st>>>(xs, n, s_stride, c_stride, os, ob_stride, oc_stride, tab);
        count_launch();
    }
}

// 16-byte vectors when every row of the input and of the output starts on a vector boundary, else one sample per thread
template <typename In, typename Out>
static void band_dispatch(const void* x, int kind, int64_t n_ch, int64_t n, int64_t s_stride, int64_t c_stride,
                          const BandTable& tab, void* out, int64_t ob_stride, int64_t oc_stride, cudaStream_t st) {
    constexpr int V = 16 / sizeof(In);
    const bool vec = (uintptr_t)x % 16 == 0 && (uintptr_t)out % (sizeof(Out) * V) == 0 && s_stride % V == 0 &&
                     c_stride % V == 0 && ob_stride % V == 0 && oc_stride % V == 0;
    if (vec) band_launch<In, Out, V>(x, kind, n_ch, n, s_stride, c_stride, tab, out, ob_stride, oc_stride, st);
    else band_launch<In, Out, 1>(x, kind, n_ch, n, s_stride, c_stride, tab, out, ob_stride, oc_stride, st);
}

int band_reduce_launch(const void* x_dev, int type, int kind, int64_t n_channels, int64_t n_samples, int64_t s_stride,
                       int64_t c_stride, const BandTable& tab, void* out_dev, int64_t out_b_stride, int64_t out_c_stride,
                       cudaStream_t st) {
    if (n_channels <= 0 || n_samples <= 0) { set_error("band_reduce: empty input"); return GCWT_ERR_ARG; }
    const bool cx = kind == GCWT_OUT_COMPLEX;
    if (type == GCWT_F32) {
        if (cx) band_dispatch<float2, float>(x_dev, kind, n_channels, n_samples, s_stride, c_stride, tab, out_dev, out_b_stride, out_c_stride, st);
        else band_dispatch<float, float>(x_dev, kind, n_channels, n_samples, s_stride, c_stride, tab, out_dev, out_b_stride, out_c_stride, st);
    } else {
        if (cx) band_dispatch<double2, double>(x_dev, kind, n_channels, n_samples, s_stride, c_stride, tab, out_dev, out_b_stride, out_c_stride, st);
        else band_dispatch<double, double>(x_dev, kind, n_channels, n_samples, s_stride, c_stride, tab, out_dev, out_b_stride, out_c_stride, st);
    }
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// ----------------------------------------------------------------------------- event-locked power and phase
// The mean spectrogram around a set of events (stimuli, ripple peaks, trial starts) and the inter-trial phase
// coherence.  A block owns lags [256 x, 256 x + 256) of one (channel, scale); each thread owns one lag and walks
// the events in the order given, so a warp's loads are 32 consecutive samples of the row and every sum has one
// fixed order: no atomics, the same bits on every run.  Events whose sample falls outside the tile
// [sample0, sample0 + n) are skipped, so a caller can drive a result tile by tile into the same accumulator.
__device__ __forceinline__ double2 unit_phase(double2 v) {
    const double m2 = fma(v.x, v.x, v.y * v.y);
    if (!(m2 > 0.0)) return make_double2(0.0, 0.0);                 // |W| = 0 counts, adds nothing
    const double r = rsqrt(m2);                                     // 1 / |W| within 1 ulp, no division slow path
    return make_double2(v.x * r, v.y * r);
}
__device__ __forceinline__ double2 unit_phase(float2 v) { return unit_phase(make_double2(v.x, v.y)); }

template <typename In, bool POWER, bool PHASE>
__global__ void __launch_bounds__(256)
event_reduce_kernel(const In* __restrict__ x, int64_t n, int64_t s_stride, int64_t c_stride, int64_t sample0,
                    const int64_t* __restrict__ events, int64_t n_events, int64_t lag_first, int64_t n_lags,
                    double* __restrict__ acc_power, double2* __restrict__ acc_phase, int64_t as_stride,
                    int64_t ac_stride) {
    const int64_t lag = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (lag >= n_lags) return;
    const In* row = x + (int64_t)blockIdx.z * c_stride + (int64_t)blockIdx.y * s_stride;
    const int64_t shift = lag_first + lag - sample0;
    double p = 0.0, re = 0.0, im = 0.0;
#pragma unroll 4
    for (int64_t e = 0; e < n_events; ++e) {
        const int64_t t = __ldg(events + e) + shift;
        if (t < 0 || t >= n) continue;
        const In v = row[t];
        p += mag2(v, POWER);
        if constexpr (PHASE) {
            const double2 u = unit_phase(v);
            re += u.x;
            im += u.y;
        }
    }
    const int64_t o = (int64_t)blockIdx.z * ac_stride + (int64_t)blockIdx.y * as_stride + lag;
    acc_power[o] += p;
    if constexpr (PHASE) {
        const double2 a = acc_phase[o];
        acc_phase[o] = make_double2(a.x + re, a.y + im);
    }
}

template <typename In, bool POWER, bool PHASE>
static void event_launch(const void* x, int64_t n_ch, int n_scales, int64_t n, int64_t s_stride, int64_t c_stride,
                         int64_t sample0, const int64_t* events, int64_t n_events, int64_t lag_first, int64_t n_lags,
                         double* acc_power, double2* acc_phase, int64_t as_stride, int64_t ac_stride, cudaStream_t st) {
    for (int64_t c0 = 0; c0 < n_ch; c0 += 65535) {                   // gridDim.z limit
        const int64_t rows = std::min<int64_t>(65535, n_ch - c0);
        dim3 grid((unsigned)((n_lags + 255) / 256), (unsigned)n_scales, (unsigned)rows);
        event_reduce_kernel<In, POWER, PHASE><<<grid, 256, 0, st>>>(
            (const In*)x + c0 * c_stride, n, s_stride, c_stride, sample0, events, n_events, lag_first, n_lags,
            acc_power + c0 * ac_stride, PHASE ? acc_phase + c0 * ac_stride : nullptr, as_stride, ac_stride);
        count_launch();
    }
}

int event_reduce_launch(const void* x_dev, int type, int kind, int64_t n_channels, int n_scales, int64_t n_samples,
                        int64_t s_stride, int64_t c_stride, int64_t sample0, const int64_t* events_dev, int64_t n_events,
                        int64_t lag_first, int64_t n_lags, double* acc_power, double2* acc_phase, int64_t as_stride,
                        int64_t ac_stride, cudaStream_t st) {
    if (n_events == 0) return GCWT_OK;
    const bool f32 = type == GCWT_F32;
#define GCWT_EVENTS(In, POWER, PHASE)                                                                                 \
    event_launch<In, POWER, PHASE>(x_dev, n_channels, n_scales, n_samples, s_stride, c_stride, sample0, events_dev, \
                                   n_events, lag_first, n_lags, acc_power, acc_phase, as_stride, ac_stride, st)
    if (kind == GCWT_OUT_COMPLEX) {
        if (acc_phase) { if (f32) GCWT_EVENTS(float2, false, true); else GCWT_EVENTS(double2, false, true); }
        else { if (f32) GCWT_EVENTS(float2, false, false); else GCWT_EVENTS(double2, false, false); }
    } else if (kind == GCWT_OUT_POWER) {
        if (f32) GCWT_EVENTS(float, true, false); else GCWT_EVENTS(double, true, false);
    } else {
        if (f32) GCWT_EVENTS(float, false, false); else GCWT_EVENTS(double, false, false);
    }
#undef GCWT_EVENTS
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

}  // namespace gcwt
