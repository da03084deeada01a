// Exact frequency response of the reference's L-tap Morse kernel.
//
// The reference builds each scale's FIR kernel as the L-point inverse DFT of the
// sampled Morse spectrum X[k] with a centring phase (ghost/wave/morseutils.py:145-149)
// and convolves with a "same" slice that advances by (L-1)//2
// (ghost/sigtools/convolution.py:79-87).  That kernel is a sum of a few dozen complex
// exponentials under a rectangular window, so its transfer function has the closed form
//
//   H(w) = e^{-i w / 2 * [L even]} * G(w),
//   G(w) = sum_k X[k] * sin(L (w - w_k) / 2) / (L sin((w - w_k) / 2)),   w_k = 2 pi k / L
//
// (SURVEY.md fact 5 / Appendix A; derivation in DESIGN.md).  On a DFT grid w = 2 pi j / n
// every phase is a ratio of integers, (w - w_k)/2 = pi (j L - k n) / (n L), which we keep
// exact in 64-bit integers so that the 0/0 limit at coincident grid points and the
// near-cancelling denominators are evaluated to full precision.
#pragma once
#include "common.cuh"

namespace gcwt {

// sin(pi * num / den) with integer range reduction; den > 0.
__host__ __device__ inline double sinpi_ratio(int64_t num, int64_t den) {
    int64_t two = 2 * den;
    num %= two;
    if (num < 0) num += two;              // [0, 2 den)
    double sign = 1.0;
    if (num >= den) { num -= den; sign = -1.0; }   // sin(pi + x) = -sin x
    if (2 * num > den) num = den - num;            // sin(pi - x) = sin x
    double x = (double)num / (double)den;          // [0, 0.5]
#ifdef __CUDA_ARCH__
    return sign * sinpi(x);
#else
    return sign * sin(3.14159265358979323846 * x);
#endif
}

// Real zero-phase part G at bin j of an n-point grid.
__host__ __device__ inline double morse_response(int64_t j, int64_t n, int64_t L,
                                                 int k_first, int n_terms, const double* X) {
    const double sN = sinpi_ratio(j * L, n);       // sin(L w / 2)
    const int64_t den = n * L;
    double acc = 0.0;
    for (int t = 0; t < n_terms; ++t) {
        const int64_t k = k_first + t;
        const int64_t num = j * L - k * n;
        if (num == 0) return X[t];                 // on an L-grid point: exactly X[k]
        const double d = (double)L * sinpi_ratio(num, den);
        const double term = sN / d * X[t];
        acc += (k & 1) ? -term : term;
    }
    return acc;
}

// H at bin j of an n-point grid, divided by `div`: G with the half-sample delay of an even-L kernel.
__device__ inline double2 morse_transfer(int64_t j, int64_t n, int64_t L, int k_first, int n_terms, const double* X,
                                         double div) {
    const double g = morse_response(j, n, L, k_first, n_terms, X) / div;
    if (L & 1) return make_double2(g, 0.0);
    double s, c;
    sincospi(-(double)(j % (2 * n)) / (double)n, &s, &c);
    return make_double2(g * c, g * s);
}

}  // namespace gcwt
