// Generic full-spectrum overlap-save path (global-memory Stockham FFT).
//
// Serves the fp64 plans (parity bar 1e-10 needs the two-sided spectrum of the exact
// filter) and is the fp32 fallback for scales the fused kernels cannot take.  Replaces
// fastconv_scipy's overlap-ADD (ghost/sigtools/convolution.py:63-87) by overlap-SAVE
// with the kernel's transfer function evaluated in closed form on the device instead of
// fft(kernel, n) per block (convolution.py:75).
#include "plan.h"
#include "common.cuh"
#include "multiplier.cuh"
#include "fft_global.cuh"
#include "fft_fourstep.cuh"
#include <algorithm>

namespace gcwt {

// ----------------------------------------------------------------------------- means
template <typename TIn>
__global__ void mean_partial_kernel(const TIn* __restrict__ x, int64_t n, int64_t stride,
                                    double* __restrict__ partial) {
    const int c = blockIdx.y, nb = gridDim.x;
    const TIn* xc = x + (int64_t)c * stride;
    // block ranges start on multiples of 4 samples so that aligned rows can be read as 128-bit vectors
    const int64_t per = (((n + nb - 1) / nb) + 3) & ~int64_t(3);
    const int64_t lo = (int64_t)blockIdx.x * per;
    const int64_t hi = min(n, lo + per);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;              // independent chains: several loads in flight
    int64_t i = lo + threadIdx.x;
    if (sizeof(TIn) == 4 && (((uintptr_t)xc) & 15) == 0 && lo < hi) {
        // fp32 rows: four samples per load, two loads in flight per thread (the kernel is a pure HBM read)
        const float4* v = (const float4*)(xc + lo);
        const int64_t nv = (hi - lo) >> 2;
        int64_t k = threadIdx.x;
        for (; k + blockDim.x < nv; k += 2 * (int64_t)blockDim.x) {
            const float4 p = v[k], q = v[k + blockDim.x];
            a0 += (double)p.x + (double)p.y; a1 += (double)p.z + (double)p.w;
            a2 += (double)q.x + (double)q.y; a3 += (double)q.z + (double)q.w;
        }
        for (; k < nv; k += blockDim.x) {
            const float4 p = v[k];
            a0 += (double)p.x + (double)p.y; a1 += (double)p.z + (double)p.w;
        }
        i = lo + (nv << 2) + threadIdx.x;                        // the (< 4) samples behind the last full vector
    } else {
        for (; i + 3 * (int64_t)blockDim.x < hi; i += 4 * (int64_t)blockDim.x) {
            a0 += (double)xc[i];
            a1 += (double)xc[i + blockDim.x];
            a2 += (double)xc[i + 2 * (int64_t)blockDim.x];
            a3 += (double)xc[i + 3 * (int64_t)blockDim.x];
        }
    }
    for (; i < hi; i += blockDim.x) a0 += (double)xc[i];
    const double acc = (a0 + a1) + (a2 + a3);
    __shared__ double sh[256];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[(int64_t)c * nb + blockIdx.x] = sh[0];
}

// one block per channel: block-wide fp64 reduction of the channel's partial sums
__global__ void __launch_bounds__(128)
mean_final_kernel(const double* __restrict__ partial, int nb, int64_t n,
                  double* __restrict__ means, int n_channels) {
    const int c = blockIdx.x;
    double acc = 0.0;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) acc += partial[(int64_t)c * nb + i];
    __shared__ double sh[128];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) means[c] = sh[0] / (double)n;
}

int means_blocks(int64_t n_samples) {
    int nb = (int)std::min<int64_t>(512, (n_samples + 4095) / 4096);
    return nb < 1 ? 1 : nb;
}

// `partial` is scratch for means_blocks(n_samples) * n_channels doubles (no allocation on the hot path:
// stream-ordered allocations here showed up as milliseconds of jitter per transform)
int means_launch(const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                 int64_t x_stride, double* d_means, double* partial, cudaStream_t st) {
    if (n_channels <= 0 || n_samples <= 0) { set_error("means: empty input"); return GCWT_ERR_ARG; }
    const int nb = means_blocks(n_samples);
    dim3 grid(nb, (unsigned)n_channels);
    if (in_type == GCWT_F32)
        mean_partial_kernel<float><<<grid, 256, 0, st>>>((const float*)x, n_samples, x_stride, partial);
    else
        mean_partial_kernel<double><<<grid, 256, 0, st>>>((const double*)x, n_samples, x_stride, partial);
    mean_final_kernel<<<(unsigned)n_channels, 128, 0, st>>>(partial, nb, n_samples, d_means, (int)n_channels);
    count_launch(2);
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// ----------------------------------------------------------------------------- load
template <typename TIn>
__global__ void generic_load_kernel(const TIn* __restrict__ x, int64_t x_stride, int64_t n,
                                    int64_t halo_l, int64_t halo_r, const double* __restrict__ means,
                                    double2* __restrict__ dst, int nfft,
                                    int64_t hop, int64_t offset, int64_t item0, int64_t n_chunks) {
    const int64_t item = item0 + blockIdx.y;
    const int64_t c = item / n_chunks, q = item % n_chunks;
    const int64_t t0 = q * hop - offset;
    const double mu = means[c];
    const TIn* xc = x + c * x_stride;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nfft; i += gridDim.x * blockDim.x) {
        const int64_t t = t0 + i;
        double v = 0.0;
        if (t >= -halo_l && t < n + halo_r) v = (double)xc[t] - mu;
        dst[(int64_t)blockIdx.y * nfft + i] = make_double2(v, 0.0);
    }
}

// ----------------------------------------------------------------------------- response
// H_s on the n-point grid, scaled by 1/n.  Kernel (2)'s multiplier, evaluated in registers.
// p2 >= 0: position j holds bin k1 + 2^p1 * k2 with k1 = j >> p2, k2 = j & (2^p2 - 1) (four-step order)
__global__ void generic_response_kernel(const ScaleInfo* __restrict__ scales,
                                        const double* __restrict__ terms,
                                        const int* __restrict__ ids, int nfft,
                                        double2* __restrict__ H, int p1 = -1, int p2 = -1) {
    const int pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= nfft) return;
    const int j = p2 < 0 ? pos : (pos >> p2) + ((pos & ((1 << p2) - 1)) << p1);
    const ScaleInfo sc = scales[ids ? ids[blockIdx.y] : (int)blockIdx.y];
    H[(int64_t)blockIdx.y * nfft + pos] = morse_transfer(j, nfft, sc.L, sc.k_first, sc.n_terms, terms + sc.term_off,
                                                         (double)nfft);
}

__global__ void generic_multiply_kernel(const double2* __restrict__ Y, const double2* __restrict__ H,
                                        double2* __restrict__ Z, int nfft, int sb) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nfft) return;
    const int s = blockIdx.y, ib = blockIdx.z;
    Z[((int64_t)ib * sb + s) * nfft + j] = cmul(Y[(int64_t)ib * nfft + j], H[(int64_t)s * nfft + j]);
}

// ----------------------------------------------------------------------------- epilogue
template <typename TOut, int KIND>
__global__ void generic_epilogue_kernel(const double2* __restrict__ Z, int nfft,
                                        int64_t item0, int64_t n_chunks, int64_t hop, int64_t offset,
                                        int64_t n, const int* __restrict__ ids, int sb, void* out,
                                        int64_t s_stride, int64_t c_stride) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hop) return;
    const int s = blockIdx.y, ib = blockIdx.z;
    const int64_t item = item0 + ib;
    const int64_t c = item / n_chunks, q = item % n_chunks;
    const int64_t t = q * hop + i;
    if (t >= n) return;
    const double2 v = Z[((int64_t)ib * sb + s) * nfft + offset + i];
    const int64_t o = c * c_stride + (int64_t)ids[s] * s_stride + t;
    typedef typename cplx_of<TOut>::type CO;
    if (KIND == GCWT_OUT_COMPLEX) ((CO*)out)[o] = mk<TOut>((TOut)v.x, (TOut)v.y);
    else if (KIND == GCWT_OUT_AMPLITUDE) ((TOut*)out)[o] = (TOut)sqrt(v.x * v.x + v.y * v.y);
    else ((TOut*)out)[o] = (TOut)(v.x * v.x + v.y * v.y);
}

// ----------------------------------------------------------------------------- drivers
// One generic call: the scales `ids` of every channel, chunked for overlap-save.  Input samples are TIn, the
// arithmetic is fp64 and the coefficients are stored as TOut (fp32 plans: fp64 arithmetic with an fp32 store).
struct GenericCall {
    gcwt_plan* p;
    const std::vector<int>& ids;
    const void* x;
    int64_t n_channels, n, x_stride, halo_l, halo_r;
    const double* d_means;
    void* out;
    int64_t s_stride, c_stride;
    cudaStream_t st;
    int64_t nfft, offset, hop, n_chunks, n_items;   // chunk geometry
};

std::vector<SmemKernel> fourstep_kernels() {
    std::vector<SmemKernel> k = {{(const void*)fs_forward_cols_kernel<float>, kFourStepSmem},
                                 {(const void*)fs_forward_cols_kernel<double>, kFourStepSmem},
                                 {(const void*)fs_forward_rows_kernel, kFourStepSmem},
                                 {(const void*)fs_inverse_rows_kernel, kFourStepSmem}};
    for (int kind = GCWT_OUT_COMPLEX; kind <= GCWT_OUT_POWER; ++kind)
        with_kind(kind, [&](auto K) {
            k.push_back({(const void*)fs_inverse_cols_kernel<float, K>, kFourStepSmem});
            k.push_back({(const void*)fs_inverse_cols_kernel<double, K>, kFourStepSmem});
        });
    return k;
}

// 2^11 <= nfft <= 2^20: the four-step FFT with shared-memory sub-transforms (fft_fourstep.cuh)
template <typename TIn, typename TOut>
static int run_fourstep(const GenericCall& g) {
    gcwt_plan* p = g.p;
    const std::vector<int>& ids = g.ids;
    const int ns = (int)ids.size();
    const int64_t nfft = g.nfft;
    const FourStep fs(nfft);
    cudaStream_t st = g.st;
    // ---- tables ------------------------------------------------------------------------------
    if (!p->d_tw1k) {
        std::vector<double2> tw(1024);
        for (int j = 0; j < 1024; ++j) {
            // exact octant symmetry is not needed: fp64 sin / cos of an exactly representable multiple of pi / 512
            tw[j] = make_double2(std::cos(-2.0 * M_PI * j / 1024.0), std::sin(-2.0 * M_PI * j / 1024.0));
        }
        GCWT_CUDA_OK(cudaMalloc((void**)&p->d_tw1k, sizeof(double2) * 1024));
        GCWT_CUDA_OK(cudaMemcpyAsync(p->d_tw1k, tw.data(), sizeof(double2) * 1024, cudaMemcpyHostToDevice, st));
        GCWT_CUDA_OK(cudaStreamSynchronize(st));
        GCWT_CUDA_OK(cudaMalloc((void**)&p->d_tw_fine, sizeof(double2) * 1024));
    }
    if (p->tw_fine_n != nfft) {
        fs_fine_twiddle_kernel<<<4, 256, 0, st>>>(fs.p, p->d_tw_fine);
        count_launch();
        p->tw_fine_n = nfft;
    }
    // ---- batch geometry --------------------------------------------------------------------------
    const size_t row = (size_t)nfft * sizeof(double2);
    // intermediate of one launch pair.  Measured on config 5: 32 ... 96 MB (L2-sized) 21.3 ms, 192 MB 19.9, 512 MB 19.3 --
    // the kernels are bound by shared-memory wavefronts, not by HBM, so fewer and larger launches win
    const size_t t_budget = (size_t)512 << 20;
    const int ib = (int)std::max<int64_t>(1, std::min<int64_t>(g.n_items, (int64_t)(((size_t)256 << 20) / row)));
    const int sb = (int)std::max<int64_t>(1, std::min<int64_t>(ns, (int64_t)(t_budget / (row * ib))));
    // the responses of a whole plan are cached when they fit (they depend on the scale and nfft only)
    bool contiguous = true;
    for (int i = 1; i < ns; ++i) contiguous = contiguous && ids[i] == ids[i - 1] + 1;
    const bool cache = contiguous && ns == p->n_scales && (size_t)p->n_scales * row <= ((size_t)4 << 30);
    if (cache && p->hcache_n != nfft) {
        if (p->d_hcache) { GCWT_CUDA_OK(cudaStreamSynchronize(st)); cudaFree(p->d_hcache); p->d_hcache = nullptr; p->hcache_n = 0; }
        if (cudaMalloc((void**)&p->d_hcache, (size_t)p->n_scales * row) == cudaSuccess) {
            generic_response_kernel<<<dim3((unsigned)((nfft + 255) / 256), p->n_scales), 256, 0, st>>>(
                p->d_scales, p->d_terms, nullptr, (int)nfft, p->d_hcache, fs.p1, fs.p2);
            count_launch();
            p->hcache_n = nfft;
        } else {
            cudaGetLastError();
        }
    }
    const bool cached = cache && p->hcache_n == nfft;
    // layout: U[ib] | Y[ib] | T[ib*sb] | H[sb] (unless cached) | ids[ns]
    const size_t need = row * ((size_t)2 * ib + (size_t)ib * sb + (cached ? 0 : sb)) + sizeof(int) * ns + 256;
    int rc = ensure_workspace(p, need);
    if (rc) return rc;
    char* w = (char*)p->ws.ptr;
    double2* U = (double2*)w;      w += row * ib;
    double2* Y = (double2*)w;      w += row * ib;
    double2* T = (double2*)w;      w += row * (size_t)ib * sb;
    double2* Hb = (double2*)w;     if (!cached) w += row * sb;
    int* d_ids = (int*)w;
    GCWT_CUDA_OK(cudaMemcpyAsync(d_ids, ids.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, st));

    FourStepParams fp;
    fp.p = fs.p; fp.p1 = fs.p1; fp.p2 = fs.p2; fp.tw = p->d_tw1k; fp.tw_fine = p->d_tw_fine;
    fp.n_chunks = g.n_chunks; fp.hop = g.hop; fp.offset = g.offset; fp.n = g.n; fp.halo_l = g.halo_l; fp.halo_r = g.halo_r;
    const unsigned col_blocks = (unsigned)(fs.n2 / fs.cols_per_block), row_blocks = (unsigned)(fs.n1 / fs.rows_per_block);
    for (int64_t i0 = 0; i0 < g.n_items; i0 += ib) {
        const int ibn = (int)std::min<int64_t>(ib, g.n_items - i0);
        fp.item0 = i0; fp.n_items = ibn;
        fs_forward_cols_kernel<TIn><<<col_blocks * ibn, 256, kFourStepSmem, st>>>(fp, (const TIn*)g.x, g.x_stride, g.d_means, U);
        fs_forward_rows_kernel<<<row_blocks * ibn, 256, kFourStepSmem, st>>>(fp, U, Y);
        count_launch(2);
        for (int s0 = 0; s0 < ns; s0 += sb) {
            const int sbn = std::min(sb, ns - s0);
            const double2* H = cached ? p->d_hcache + ((int64_t)ids[s0] << fs.p) : Hb;
            if (!cached) {
                generic_response_kernel<<<dim3((unsigned)((nfft + 255) / 256), sbn), 256, 0, st>>>(
                    p->d_scales, p->d_terms, d_ids + s0, (int)nfft, Hb, fs.p1, fs.p2);
                count_launch();
            }
            fs_inverse_rows_kernel<<<dim3(row_blocks * ibn, sbn), 256, kFourStepSmem, st>>>(fp, Y, H, T, sbn);
            with_kind(p->out_kind, [&](auto K) {
                fs_inverse_cols_kernel<TOut, K><<<dim3(col_blocks * ibn, sbn), 256, kFourStepSmem, st>>>(
                    fp, T, sbn, d_ids + s0, g.out, g.s_stride, g.c_stride);
            });
            count_launch(2);
        }
    }
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// every other nfft: radix-16/8/4/2 passes through global memory (fft_global.cuh)
template <typename TIn, typename TOut>
static int run_stockham(const GenericCall& g) {
    gcwt_plan* p = g.p;
    const int ns = (int)g.ids.size();
    const int64_t nfft = g.nfft;
    cudaStream_t st = g.st;
    const size_t row = (size_t)nfft * sizeof(double2);
    const size_t budget = (size_t)1 << 30;
    // few scales (the accuracy guard re-computing a handful of pairs): batch more chunks per launch instead
    int ib = (int)std::min<int64_t>(g.n_items, std::max<int64_t>(4, std::min<int64_t>(32, (int64_t)(budget / (6 * row * std::min(ns, 4))))));
    int sb = (int)std::min<int64_t>(ns, std::max<int64_t>(1, (int64_t)(budget / (2 * row * ib))));
    sb = std::min(sb, 1024);
    // layout: Y[ib] | H[sb] | Za[ib*sb] | Zb[ib*sb] | ids[ns] | Yscratch[ib]
    const size_t need = row * ((size_t)ib * 2 + sb + 2 * (size_t)ib * sb) + sizeof(int) * ns + 256;
    int rc = ensure_workspace(p, need);
    if (rc) return rc;
    char* w = (char*)p->ws.ptr;
    double2* Y = (double2*)w;     w += row * ib;
    double2* Y2 = (double2*)w;    w += row * ib;
    double2* H = (double2*)w;     w += row * sb;
    double2* Za = (double2*)w;    w += row * (size_t)ib * sb;
    double2* Zb = (double2*)w;    w += row * (size_t)ib * sb;
    int* d_ids = (int*)w;
    GCWT_CUDA_OK(cudaMemcpyAsync(d_ids, g.ids.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, st));

    const int tpb = 256;
    const unsigned gx = (unsigned)((nfft + tpb - 1) / tpb);
    for (int s0 = 0; s0 < ns; s0 += sb) {
        const int sbn = std::min(sb, ns - s0);
        generic_response_kernel<<<dim3(gx, sbn), tpb, 0, st>>>(p->d_scales, p->d_terms, d_ids + s0, (int)nfft, H);
        count_launch();
        for (int64_t i0 = 0; i0 < g.n_items; i0 += ib) {
            const int ibn = (int)std::min<int64_t>(ib, g.n_items - i0);
            generic_load_kernel<TIn><<<dim3(std::min(gx, 1024u), ibn), tpb, 0, st>>>(
                (const TIn*)g.x, g.x_stride, g.n, g.halo_l, g.halo_r, g.d_means, Y, (int)nfft, g.hop, g.offset, i0, g.n_chunks);
            count_launch();
            double2* ya = Y; double2* yb = Y2;
            fft_batched<-1>(ya, yb, (int)nfft, ibn, st);
            generic_multiply_kernel<<<dim3(gx, sbn, ibn), tpb, 0, st>>>(ya, H, Za, (int)nfft, sbn);
            count_launch();
            double2* za = Za; double2* zb = Zb;
            fft_batched<+1>(za, zb, (int)nfft, ibn * sbn, st);
            const dim3 ge((unsigned)((g.hop + tpb - 1) / tpb), sbn, ibn);
            with_kind(p->out_kind, [&](auto K) {
                generic_epilogue_kernel<TOut, K><<<ge, tpb, 0, st>>>(
                    za, (int)nfft, i0, g.n_chunks, g.hop, g.offset, g.n, d_ids + s0, sbn, g.out, g.s_stride, g.c_stride);
            });
            count_launch();
        }
    }
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// fp64 plans, and in fp32 plans the scales the fused kernels cannot take (wavelets whose truncated kernels are
// genuinely broadband, GCWT_FLAG_FORCE_GENERIC) and the pairs the accuracy guard re-computes.  Always fp64
// arithmetic: a full-spectrum fp32 transform has no guard of its own against recordings whose energy sits far
// from a scale's band (errors of 1e-4 ... 1e-3 there), and the fp64 four-step path is the faster one anyway.
int generic_execute(gcwt_plan* p, const std::vector<int>& ids, const void* x, int in_type,
                    int64_t n_channels, int64_t n_samples, int64_t x_stride, int64_t halo_l,
                    int64_t halo_r, const double* d_means, void* out, int64_t s_stride,
                    int64_t c_stride, cudaStream_t st) {
    if (ids.empty()) return GCWT_OK;
    int64_t lmax = 1;
    for (int id : ids) lmax = std::max<int64_t>(lmax, p->scales[id].L);
    // chunk geometry: one chunk when the whole segment fits a 2^20-point transform
    int64_t nfft;
    if (n_samples + lmax - 1 <= (int64_t(1) << 20)) nfft = int64_t(1) << ilog2_ceil(n_samples + lmax - 1);
    else nfft = std::max<int64_t>(int64_t(1) << 17, int64_t(1) << ilog2_ceil(4 * lmax));
    if (nfft > (int64_t(1) << 26)) { set_error("generic path: kernel too long"); return GCWT_ERR_UNSUPPORTED; }
    if (nfft < 16) nfft = 16;
    const int64_t hop = nfft - (lmax - 1), n_chunks = (n_samples + hop - 1) / hop;
    const GenericCall g{p, ids, x, n_channels, n_samples, x_stride, halo_l, halo_r, d_means, out, s_stride, c_stride, st,
                        nfft, lmax / 2, hop, n_chunks, n_channels * n_chunks};
    const auto by_type = [](int type, auto f) { return type == GCWT_F32 ? f(float()) : f(double()); };
    return by_type(in_type, [&](auto tin) {
        return by_type(p->compute_type, [&](auto tout) {
            using TIn = decltype(tin);
            using TOut = decltype(tout);
            return FourStep::usable(nfft) ? run_fourstep<TIn, TOut>(g) : run_stockham<TIn, TOut>(g);
        });
    });
}

// ----------------------------------------------------------------------------- probe
__global__ void filter_response_kernel(int64_t L, int k_first, int n_terms, const double* __restrict__ terms,
                                       int64_t nfft, int64_t first_bin, int64_t n_bins,
                                       double2* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bins) return;
    out[i] = morse_transfer(first_bin + i, nfft, L, k_first, n_terms, terms, 1.0);
}

int filter_response_device(int64_t L, int k_first, int n_terms, const double* terms_host, int64_t nfft,
                           int64_t first_bin, int64_t n_bins, double* out_host) {
    DevBuf terms, out;
    { int rc = terms.alloc(sizeof(double) * n_terms); if (rc) return rc; }
    { int rc = out.alloc(sizeof(double2) * n_bins); if (rc) return rc; }
    GCWT_CUDA_OK(cudaMemcpy(terms.p, terms_host, sizeof(double) * n_terms, cudaMemcpyHostToDevice));
    filter_response_kernel<<<(unsigned)((n_bins + 255) / 256), 256>>>(L, k_first, n_terms, terms.as<double>(), nfft,
                                                                       first_bin, n_bins, out.as<double2>());
    count_launch();
    GCWT_CUDA_OK(cudaGetLastError());
    GCWT_CUDA_OK(cudaMemcpy(out_host, out.p, sizeof(double2) * n_bins, cudaMemcpyDeviceToHost));
    return GCWT_OK;
}

// psi_L[n] = (1/L) sum_k X[k] e^{2 pi i k (n + (L+1)/2) / L}; phase kept as an exact
// integer: 2 k (n + (L+1)/2) / L = k (2n + L + 1) / L half-turns.
__global__ void morse_kernel_kernel(int64_t L, int k_first, int n_terms, const double* __restrict__ terms,
                                    double2* __restrict__ out) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= L) return;
    double re = 0.0, im = 0.0;
    for (int t = 0; t < n_terms; ++t) {
        const int64_t k = k_first + t;
        const int64_t num = (k * ((2 * n + L + 1) % (2 * L))) % (2 * L);
        double s, c;
        sincospi((double)num / (double)L, &s, &c);
        re += terms[t] * c;
        im += terms[t] * s;
    }
    out[n] = make_double2(re / (double)L, im / (double)L);
}

int morse_kernel_device(int64_t L, int k_first, int n_terms, const double* terms_host, double* out_host) {
    DevBuf terms, out;
    { int rc = terms.alloc(sizeof(double) * n_terms); if (rc) return rc; }
    { int rc = out.alloc(sizeof(double2) * L); if (rc) return rc; }
    GCWT_CUDA_OK(cudaMemcpy(terms.p, terms_host, sizeof(double) * n_terms, cudaMemcpyHostToDevice));
    morse_kernel_kernel<<<(unsigned)((L + 255) / 256), 256>>>(L, k_first, n_terms, terms.as<double>(), out.as<double2>());
    count_launch();
    GCWT_CUDA_OK(cudaGetLastError());
    GCWT_CUDA_OK(cudaMemcpy(out_host, out.p, sizeof(double2) * L, cudaMemcpyDeviceToHost));
    return GCWT_OK;
}

}  // namespace gcwt
