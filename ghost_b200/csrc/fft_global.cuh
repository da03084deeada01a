// Batched power-of-two complex128 FFT through global memory (radix-16/8/4/2 Stockham autosort passes).
// Shared by the generic CWT path and the sigtools helpers.
#pragma once
#include "plan.h"
#include "common.cuh"
#include <algorithm>

namespace gcwt {

// ----------------------------------------------------------------------------- FFT pass
// One radix-R Stockham autosort pass over `batch` transforms of length n.
template <int R, int SIGN>
__global__ void stockham_pass_kernel(const double2* __restrict__ in, double2* __restrict__ out, int n, int ns) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = n / R;
    if (j >= m) return;
    const int64_t base = (int64_t)blockIdx.y * n;
    const int k = j % ns;
    double2 v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = in[base + j + (int64_t)r * m];
    if (ns > 1) {
        const int span = ns * R;
#pragma unroll
        for (int r = 1; r < R; ++r) {
            const int e = (int)(((int64_t)r * k) % span);
            v[r] = cmul(v[r], expipi((double)(SIGN * 2) * (double)e / (double)span));
        }
    }
    small_dft<R, SIGN, double2>::run(v);
    const int64_t j0 = (int64_t)(j - k) * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) out[base + j0 + (int64_t)r * ns] = v[r];
}

template <int SIGN>
static void fft_batched(double2*& a, double2*& b, int n, int batch, cudaStream_t st) {
    // result ends up in `a` (pointers are swapped as passes go)
    int lg = ilog2_ceil(n);
    int ns = 1;
    while (lg > 0) {
        int r = lg >= 4 ? 16 : (1 << lg);
        const int m = n / r;
        dim3 grid((m + 127) / 128, batch);
        switch (r) {
            case 16: stockham_pass_kernel<16, SIGN><<<grid, 128, 0, st>>>(a, b, n, ns); break;
            case 8:  stockham_pass_kernel<8, SIGN><<<grid, 128, 0, st>>>(a, b, n, ns); break;
            case 4:  stockham_pass_kernel<4, SIGN><<<grid, 128, 0, st>>>(a, b, n, ns); break;
            default: stockham_pass_kernel<2, SIGN><<<grid, 128, 0, st>>>(a, b, n, ns); break;
        }
        count_launch();
        std::swap(a, b);
        ns *= r;
        lg -= (r == 16 ? 4 : lg);
    }
}

}  // namespace gcwt
