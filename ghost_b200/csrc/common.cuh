// Shared device helpers for the ghost_b200 CWT kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include <type_traits>
#include "../../include/ghost_cwt.h"

namespace gcwt {

// ---------------------------------------------------------------- errors
void set_error(const std::string& msg);     // defined in cabi.cu (thread-local)

#define GCWT_CUDA_OK(expr)                                                        \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) {                                                  \
            gcwt::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));  \
            return GCWT_ERR_CUDA;                                                 \
        }                                                                         \
    } while (0)

// scratch device memory of the stand-alone helpers: freed on every return path
struct DevBuf {
    void* p = nullptr;
    DevBuf() {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); set_error("device allocation of scratch memory failed"); return GCWT_ERR_NOMEM; }
        return GCWT_OK;
    }
    double2* c() { return (double2*)p; }
    template <typename T> T* as() const { return (T*)p; }
};

// ---------------------------------------------------------------- complex
template <typename T> struct cplx_of;
template <> struct cplx_of<float>  { typedef float2  type; };
template <> struct cplx_of<double> { typedef double2 type; };

template <typename T> __host__ __device__ __forceinline__
typename cplx_of<T>::type mk(T re, T im) { typename cplx_of<T>::type r; r.x = re; r.y = im; return r; }

template <typename C> __device__ __forceinline__ C cadd(C a, C b) { a.x += b.x; a.y += b.y; return a; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { a.x -= b.x; a.y -= b.y; return a; }
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
    C r;
    r.x = a.x * b.x - a.y * b.y;
    r.y = a.x * b.y + a.y * b.x;
    return r;
}
// multiply by +i / -i
template <int SIGN, typename C> __device__ __forceinline__ C mul_i(C a) {
    C r;
    if (SIGN > 0) { r.x = -a.y; r.y = a.x; } else { r.x = a.y; r.y = -a.x; }
    return r;
}

// e^{i * pi * x}: x is exact (dyadic) in all our call sites
__device__ __forceinline__ float2  expipi(float x)  { float2 r;  sincospif(x, &r.y, &r.x); return r; }
__device__ __forceinline__ double2 expipi(double x) { double2 r; sincospi(x, &r.y, &r.x);  return r; }

// ---------------------------------------------------------------- small DFTs
// All transforms: b[n] = sum_k a[k] e^{SIGN * 2 pi i k n / R}, natural order in and out.
template <int SIGN, typename C> __device__ __forceinline__ void dft2(C& a0, C& a1) {
    C t = a0;
    a0 = cadd(t, a1);
    a1 = csub(t, a1);
}

template <int SIGN, typename C> __device__ __forceinline__ void dft4(C& a0, C& a1, C& a2, C& a3) {
    C s02 = cadd(a0, a2), d02 = csub(a0, a2);
    C s13 = cadd(a1, a3), d13 = mul_i<SIGN>(csub(a1, a3));
    a0 = cadd(s02, s13);
    a2 = csub(s02, s13);
    a1 = cadd(d02, d13);
    a3 = csub(d02, d13);
}

template <int SIGN, typename C> __device__ __forceinline__ void dft8(C* a) {
    typedef decltype(a[0].x) T;
    const T h = (T)0.70710678118654752440;
    // 2 x dft4 over even / odd inputs, then radix-2 combine
    dft4<SIGN>(a[0], a[2], a[4], a[6]);
    dft4<SIGN>(a[1], a[3], a[5], a[7]);
    // twiddles W8^n on odd branch, n = 0..3
    C t1, t2, t3;
    if (SIGN > 0) {
        t1.x = (a[3].x - a[3].y) * h; t1.y = (a[3].x + a[3].y) * h;     // * e^{+i pi/4}
        t3.x = (-a[7].x - a[7].y) * h; t3.y = (a[7].x - a[7].y) * h;    // * e^{+i 3pi/4}
    } else {
        t1.x = (a[3].x + a[3].y) * h; t1.y = (a[3].y - a[3].x) * h;     // * e^{-i pi/4}
        t3.x = (a[7].y - a[7].x) * h; t3.y = (-a[7].x - a[7].y) * h;    // * e^{-i 3pi/4}
    }
    t2 = mul_i<SIGN>(a[5]);
    C e0 = a[0], e1 = a[2], e2 = a[4], e3 = a[6], o0 = a[1];
    a[0] = cadd(e0, o0); a[4] = csub(e0, o0);
    a[1] = cadd(e1, t1); a[5] = csub(e1, t1);
    a[2] = cadd(e2, t2); a[6] = csub(e2, t2);
    a[3] = cadd(e3, t3); a[7] = csub(e3, t3);
}

// 16-point DFT as 4 x 4.  k = k0 + 4 k1, n = na + 4 nb.
template <int SIGN, typename C> __device__ __forceinline__ void dft16(C* a) {
    typedef decltype(a[0].x) T;
    const T c1 = (T)0.92387953251128675613;   // cos(pi/8)
    const T s1 = (T)0.38268343236508977173;   // sin(pi/8)
    const T h  = (T)0.70710678118654752440;
    // stage 1: for each k0, 4-point DFT over k1 (inputs a[k0], a[k0+4], a[k0+8], a[k0+12]);
    // result index na stored at a[k0 + 4*na]
#pragma unroll
    for (int k0 = 0; k0 < 4; ++k0) dft4<SIGN>(a[k0], a[k0 + 4], a[k0 + 8], a[k0 + 12]);
    // twiddle W16^{k0*na}
    const T sg = (SIGN > 0) ? (T)1 : (T)-1;
    const C w1 = mk<T>(c1, sg * s1), w2 = mk<T>(h, sg * h), w3 = mk<T>(s1, sg * c1);
    const C w6 = mk<T>(-h, sg * h), w9 = mk<T>(-c1, -sg * s1);
    a[1 + 4 * 1] = cmul(a[1 + 4 * 1], w1);
    a[2 + 4 * 1] = cmul(a[2 + 4 * 1], w2);
    a[3 + 4 * 1] = cmul(a[3 + 4 * 1], w3);
    a[1 + 4 * 2] = cmul(a[1 + 4 * 2], w2);
    a[2 + 4 * 2] = mul_i<SIGN>(a[2 + 4 * 2]);           // W16^4
    a[3 + 4 * 2] = cmul(a[3 + 4 * 2], w6);
    a[1 + 4 * 3] = cmul(a[1 + 4 * 3], w3);
    a[2 + 4 * 3] = cmul(a[2 + 4 * 3], w6);
    a[3 + 4 * 3] = cmul(a[3 + 4 * 3], w9);
    // stage 2: for each na, 4-point DFT over k0 (inputs a[0+4na..3+4na]); output nb at a[4na + nb]
#pragma unroll
    for (int na = 0; na < 4; ++na) dft4<SIGN>(a[4 * na], a[4 * na + 1], a[4 * na + 2], a[4 * na + 3]);
    // now a[4*na + nb] holds output n = na + 4*nb: transpose to natural order
#pragma unroll
    for (int na = 0; na < 4; ++na)
#pragma unroll
        for (int nb = na + 1; nb < 4; ++nb) {
            C t = a[4 * na + nb];
            a[4 * na + nb] = a[4 * nb + na];
            a[4 * nb + na] = t;
        }
}

template <int R, int SIGN, typename C> struct small_dft;
template <int SIGN, typename C> struct small_dft<2, SIGN, C>  { static __device__ __forceinline__ void run(C* a) { dft2<SIGN>(a[0], a[1]); } };
template <int SIGN, typename C> struct small_dft<4, SIGN, C>  { static __device__ __forceinline__ void run(C* a) { dft4<SIGN>(a[0], a[1], a[2], a[3]); } };
template <int SIGN, typename C> struct small_dft<8, SIGN, C>  { static __device__ __forceinline__ void run(C* a) { dft8<SIGN>(a); } };
template <int SIGN, typename C> struct small_dft<16, SIGN, C> { static __device__ __forceinline__ void run(C* a) { dft16<SIGN>(a); } };

static inline int ilog2_ceil(int64_t v) { int l = 0; while ((int64_t(1) << l) < v) ++l; return l; }

// ---------------------------------------------------------------- output kind
template <int V> using IntC = std::integral_constant<int, V>;

// The run-time output kind as a template argument: calls f(IntC<KIND>()), where any kind other than complex and
// amplitude is power.  COMPLEX = false for kernels that have no complex-output instance.
template <bool COMPLEX = true, typename F>
static void with_kind(int kind, const F& f) {
    if constexpr (COMPLEX)
        if (kind == GCWT_OUT_COMPLEX) return f(IntC<GCWT_OUT_COMPLEX>());
    if (kind == GCWT_OUT_AMPLITUDE) f(IntC<GCWT_OUT_AMPLITUDE>());
    else f(IntC<GCWT_OUT_POWER>());
}

}  // namespace gcwt
