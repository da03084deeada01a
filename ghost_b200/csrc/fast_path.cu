// fp32 fast path: half-band decimation pyramid + fused overlap-save kernels.
//
// One fused kernel per scale class does, for a chunk of the recording that stays in
// shared memory: (1) forward FFT of the chunk, (2) multiply by each scale's exact filter
// response (closed form of the reference's L-tap Morse kernel, see multiplier.cuh),
// (3) inverse FFT per scale and (4) the |W| / |W|^2 / complex epilogue straight to the
// output rows.  No wavelet bank of size scales x N and no intermediate spectrum ever
// touches HBM (north-star kernels (1)-(3)).
//
// Wavelets are band-pass: a scale whose response lives below pi/(2 D) is computed from
// the recording decimated by D = 2^level (zero-phase half-band cascade, exactly
// compensated in the multiplier), so that every chunk needs only kBins = 256 spectrum
// bins however long the kernel is (L reaches 236 760 taps at 30 kHz).  The inverse
// transform back to the full sample rate is a 256*P-point FFT with 256 non-zero inputs:
// output sample n = n1*P + n2 is the n1-th output of a 256-point FFT of the spectrum
// times the phase ramp e^{2 pi i m n2 / (256 P)}.  Each lane of a warp owns one column
// n2, so stores are contiguous runs across lanes.
//
// Kernels: pyramid_kernel (decimation), fused_full_kernel (full rate, 4096-point chunks),
// fused_banded_kernel (exact pruned inverse, any output kind), and for amplitude / power the two
// coarse-grid + interpolation kernels fused_interp_kernel (U = D/2, 8 least-squares taps) and
// fused_wide2_kernel (levels 2-3, U = D, 12 taps, 2048-sample chunks with the spectrum in registers).
//
// Replaces ghost/sigtools/convolution.py:63-87 (fastconv overlap-add), morseutils.py:
// 115-151 (kernel synthesis) and transforms.py:142-143,202-204 (mean removal, abs).
#include "plan.h"
#include "common.cuh"
#include "multiplier.cuh"
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <type_traits>

namespace gcwt {

constexpr int kMaxFastLevel = 14;       // chunk of 1024 << 14 samples: phases stay exact in fp32
constexpr int kMaxFullScales = 64;
constexpr double kMaxHaloFrac = 0.45;   // (L-1) / chunk must stay below this

__constant__ float c_halfband[kHalfbandOdd];
// polyphase taps for the small coarse spacings U = 4, 8 (constant-bank operands of the FMAs)
constexpr int kSmallCoef = (4 + 8) * kInterpT;
__constant__ float c_interp_small[kSmallCoef];
// wide-spacing classes: U = 4 (level 2) and U = 8 (level 3), kWideT taps
constexpr int kWideCoef = (4 + 8) * kWideT;
__constant__ float c_interp_wide[kWideCoef];

// ============================================================================ planner
static double bessel_i0(double x) {
    double sum = 1.0, term = 1.0;
    const double q = x * x / 4.0;
    for (int k = 1; k < 200; ++k) {
        term *= q / ((double)k * (double)k);
        sum += term;
        if (term < 1e-18 * sum) break;
    }
    return sum;
}

static void design_halfband(double* odd /*kHalfbandOdd*/) {
    const int T = kHalfbandT;
    const double atten = 140.0;
    const double beta = 0.1102 * (atten - 8.7);
    const double i0b = bessel_i0(beta);
    double sum = 0.0;
    for (int k = 0; k < kHalfbandOdd; ++k) {
        const int t = 2 * k + 1;
        const double r = (double)t / (double)T;
        const double win = bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
        const double x = M_PI * t / 2.0;
        odd[k] = 0.5 * std::sin(x) / x * win;
        sum += 2.0 * odd[k];
    }
    for (int k = 0; k < kHalfbandOdd; ++k) odd[k] *= 0.5 / sum;      // unit DC gain
    // The device applies the taps in fp32.  Plain rounding leaves sum(odd) - 0.25 ~ 1e-8, i.e. a gain of
    // ~2e-8 at the input Nyquist frequency instead of the exact zero a half-band filter has there -- the
    // floor of the alias rejection of every stage but the last two.  Round greedily instead, largest
    // tap first, each one absorbing what the previous roundings left: the fp32 taps then sum to 0.25 to
    // ~1e-14 and the response near Nyquist is again quadratic in the distance from it.
    long double done = 0.0L;
    for (int k = 0; k < kHalfbandOdd; ++k) {
        long double rest = 0.0L;
        for (int j = k + 1; j < kHalfbandOdd; ++j) rest += (long double)odd[j];
        const float f = (float)(0.25L - done - rest);
        odd[k] = (double)f;
        done += (long double)f;
    }
}

static double halfband_gain(const double* odd, double theta) {
    double g = 0.5;                       // the device applies the taps rounded to fp32
    for (int k = 0; k < kHalfbandOdd; ++k) g += 2.0 * (double)(float)odd[k] * std::cos((2 * k + 1) * theta);
    return g;
}

// ---- plan-time evaluation of the exact responses, on the device ------------------------------
// Per scale: kBins values on each candidate grid 1024 << level (level = kMinFastLevel ...
// kMaxFastLevel) followed by kFullN values on the 4096-point grid.
constexpr int kPlanLevels = kMaxFastLevel - kMinFastLevel + 1;
constexpr int kWide2Levels = kWideMaxLevel - kMinFastLevel + 1;      // levels that may run fused_wide2_kernel
constexpr int kPlanRow = kPlanLevels * kBins + kFullN + kWide2Levels * 2 * kBins;

__global__ void plan_response_kernel(const ScaleInfo* __restrict__ scales, const double* __restrict__ terms,
                                     double* __restrict__ out) {
    const int s = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kPlanRow) return;
    const ScaleInfo sc = scales[s];
    int64_t n, m;
    if (i < kPlanLevels * kBins) { n = (int64_t)kChunkDec << (kMinFastLevel + i / kBins); m = i % kBins; }
    else if (i < kPlanLevels * kBins + kFullN) { n = kFullN; m = i - kPlanLevels * kBins; }
    else {
        const int k = i - kPlanLevels * kBins - kFullN;
        n = (int64_t)(2 * kChunkDec) << (kMinFastLevel + k / (2 * kBins)); m = k % (2 * kBins);
    }
    out[(int64_t)s * kPlanRow + i] = morse_response(m, n, sc.L, sc.k_first, sc.n_terms, terms + sc.term_off);
}

struct PlanResponses {
    std::vector<double> g;                      // [n_scales][kPlanRow]
    const double* level(int s, int lev) const { return g.data() + (size_t)s * kPlanRow + (size_t)(lev - kMinFastLevel) * kBins; }
    const double* full(int s) const { return g.data() + (size_t)s * kPlanRow + (size_t)kPlanLevels * kBins; }
    const double* wide2(int s, int lev) const {
        return g.data() + (size_t)s * kPlanRow + (size_t)kPlanLevels * kBins + kFullN + (size_t)(lev - kMinFastLevel) * 2 * kBins;
    }
};

static int compute_plan_responses(const gcwt_plan* p, PlanResponses& pr) {
    const size_t count = (size_t)p->n_scales * kPlanRow;
    double* d = nullptr;
    GCWT_CUDA_OK(cudaMalloc((void**)&d, sizeof(double) * count));
    plan_response_kernel<<<dim3((kPlanRow + 127) / 128, p->n_scales), 128>>>(p->d_scales, p->d_terms, d);
    count_launch();
    pr.g.resize(count);
    cudaError_t e = cudaMemcpy(pr.g.data(), d, sizeof(double) * count, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) { set_error(std::string("plan responses: ") + cudaGetErrorString(e)); return GCWT_ERR_CUDA; }
    return GCWT_OK;
}

static double filter_energy(const gcwt_plan* p, const ScaleInfo& sc, int64_t n) {
    const double* X = p->terms.data() + sc.term_off;
    double e = 0.0;
    for (int t = 0; t < sc.n_terms; ++t) e += X[t] * X[t];
    return e * (double)n / (double)sc.L;        // Parseval: sum_j |H(w_j)|^2 over an n-point grid, n >= L
}

// out-of-band energy test of one scale on the (1024 << level)-point grid
static bool band_fits(const gcwt_plan* p, const PlanResponses& pr, int s, int level) {
    const double* g = pr.level(s, level);
    double e_in = 0.0;
    for (int m = 0; m < kBins; ++m) e_in += g[m] * g[m];
    const double e_tot = filter_energy(p, p->scales[s], (int64_t)kChunkDec << level);
    return (1.0 - e_in / e_tot) < p->band_tol * p->band_tol;
}

// Full-spectrum kernel: how many 256-bin blocks of the 4096-point grid does the filter occupy?
// One-sided filters leave the upper blocks empty (below band_tol in energy), and the kernel's
// radix-16 pre-pass over the 16 aliases of a bin is pruned accordingly.
static int full_extent(const gcwt_plan* p, const PlanResponses& pr, int s) {
    const double* g = pr.full(s);
    const double e_tot = filter_energy(p, p->scales[s], kFullN);
    double e_in = 0.0;
    int m = 0;
    for (int nmu = 2; nmu <= 8; nmu *= 2) {
        for (; m < nmu * kBins; ++m) e_in += g[m] * g[m];
        if ((1.0 - e_in / e_tot) < p->band_tol * p->band_tol) return nmu;
    }
    return 16;
}

// Width (in bins of the level's grid) of the band that holds all but band_tol^2 of the filter's
// energy: |W|^2 of this scale is band-limited to that many bins around zero frequency.
static int band_width_bins(const gcwt_plan* p, const PlanResponses& pr, int s, int level) {
    const double* g = pr.level(s, level);
    const double e_tot = filter_energy(p, p->scales[s], (int64_t)kChunkDec << level);
    const double budget = 0.5 * p->band_tol * p->band_tol * e_tot;
    int lo = 0, hi = kBins - 1;
    double acc = 0.0;
    while (lo < hi && acc + g[lo] * g[lo] < budget) { acc += g[lo] * g[lo]; ++lo; }
    acc = 0.0;
    while (hi > lo && acc + g[hi] * g[hi] < budget) { acc += g[hi] * g[hi]; --hi; }
    return hi - lo + 1;
}

static int choose_level(const gcwt_plan* p, const PlanResponses& pr, int s) {
    const ScaleInfo& sc = p->scales[s];
    if (!(p->flags & GCWT_FLAG_FORCE_GENERIC)) {
        int lo = kMinFastLevel;
        while (lo <= kMaxFastLevel && (double)(sc.L - 1) > kMaxHaloFrac * (double)((int64_t)kChunkDec << lo)) ++lo;
        int hi = std::min(kMaxFastLevel, ilog2_ceil(sc.L) + 1);
        for (int lev = hi; lev >= lo; --lev)
            if (band_fits(p, pr, s, lev)) return lev;
        if ((double)(sc.L - 1) <= kMaxHaloFrac * kFullN) return -1;
    }
    return -2;
}

static void class_geometry(FastClass& fc) {
    const int64_t d = fc.level >= 0 ? (int64_t(1) << fc.level) : 1;
    const int64_t align = std::max<int64_t>(d, 16);
    // interpolated classes read kInterpT coarse samples around every output: keep them valid
    const int taps = fc.wide ? kWideT : kInterpT;
    const int64_t lead = fc.interp ? (int64_t)(taps / 2 - 1) << fc.log2u : 0;
    const int64_t tail = fc.interp ? (int64_t)(taps / 2 + 1) << fc.log2u : 0;
    fc.offset = ((fc.lmax / 2 + lead + align - 1) / align) * align;
    fc.hop = ((fc.nc_full - (fc.lmax - 1) / 2 - tail - fc.offset) / align) * align;
}

// Polyphase interpolator, T taps per phase: output at coarse position iota + phi/U is
// sum_t c[phi][t] * p[iota + t - (T/2 - 1)].  The interpolated signal |W|^2 is band-limited to
// |f| <= 1 / (2 os) cycles per coarse sample (os = over-sampling of the coarse grid, from the
// filters' measured band width), so each phase is the least-squares fit of a fractional delay over
// exactly that band: c = A^-1 b with A[t][t'] = sinc(2 fmax (d_t - d_t')), b[t] = sinc(2 fmax d_t),
// d_t = tap position relative to the output.  Worst-case error over ALL tones in the band (not
// just typical spectra): 8 taps 2.5e-6 at os = 4 and 4e-7 at os = 5; 12 taps 1.5e-6 at os = 2.5 --
// two orders of magnitude below a Kaiser-windowed sinc of the same length.
static long double sinc_pi(long double x) {
    const long double pi = 3.14159265358979323846264338327950288L;
    return x == 0.0L ? 1.0L : sinl(pi * x) / (pi * x);
}

static void design_interpolator(int log2u, std::vector<float>& coef, int T, double os) {
    const int U = 1 << log2u;
    const long double fmax = 0.5L / (long double)os;
    coef.resize((size_t)U * T);
    std::vector<long double> A((size_t)T * T), b(T);
    for (int t = 0; t < T; ++t) coef[t] = (t == T / 2 - 1) ? 1.f : 0.f;   // phase 0 sits on a coarse sample
    for (int phi = 1; phi < U; ++phi) {
        for (int t = 0; t < T; ++t) {
            const long double dt = (long double)(t - (T / 2 - 1)) - (long double)phi / U;
            for (int u = 0; u < T; ++u) A[(size_t)t * T + u] = sinc_pi(2.0L * fmax * (long double)(t - u));
            b[t] = sinc_pi(2.0L * fmax * dt);
        }
        // Gaussian elimination with partial pivoting in extended precision: the system is small and
        // ill-conditioned (1e13 for 8 taps), and a ridge term would buy stability with out-of-band gain
        for (int i = 0; i < T; ++i) {
            int piv = i;
            for (int r = i + 1; r < T; ++r) if (fabsl(A[(size_t)r * T + i]) > fabsl(A[(size_t)piv * T + i])) piv = r;
            if (piv != i) {
                for (int u = 0; u < T; ++u) std::swap(A[(size_t)i * T + u], A[(size_t)piv * T + u]);
                std::swap(b[i], b[piv]);
            }
            for (int r = i + 1; r < T; ++r) {
                const long double f = A[(size_t)r * T + i] / A[(size_t)i * T + i];
                for (int u = i; u < T; ++u) A[(size_t)r * T + u] -= f * A[(size_t)i * T + u];
                b[r] -= f * b[i];
            }
        }
        long double c[32], sum = 0.0L;
        for (int i = T - 1; i >= 0; --i) {
            long double v = b[i];
            for (int u = i + 1; u < T; ++u) v -= A[(size_t)i * T + u] * c[u];
            c[i] = v / A[(size_t)i * T + i];
        }
        for (int t = 0; t < T; ++t) sum += c[t];
        for (int t = 0; t < T; ++t) coef[(size_t)phi * T + t] = (float)(c[t] / sum);   // exact DC gain
    }
}

int interp_taps(int log2u, int n_taps, double os, float* out) {
    if (log2u < 0 || log2u > 20 || n_taps < 4 || n_taps > 32 || (n_taps & 1) || !(os >= 1.0) || !out) {
        set_error("interp_taps: log2_u in 0..20, n_taps even in 4..32, oversampling >= 1 required");
        return GCWT_ERR_ARG;
    }
    std::vector<float> coef;
    design_interpolator(log2u, coef, n_taps, os);
    std::copy(coef.begin(), coef.end(), out);
    return GCWT_OK;
}

static int upload_constants() {
    double odd[kHalfbandOdd];
    design_halfband(odd);
    float hb[kHalfbandOdd];
    for (int k = 0; k < kHalfbandOdd; ++k) hb[k] = (float)odd[k];
    GCWT_CUDA_OK(cudaMemcpyToSymbol(c_halfband, hb, sizeof(float) * kHalfbandOdd));
    std::vector<float> all, part;
    for (int lu = 2; lu <= 3; ++lu) {
        design_interpolator(lu, part, kInterpT, kInterpMinOs);
        all.insert(all.end(), part.begin(), part.end());
    }
    GCWT_CUDA_OK(cudaMemcpyToSymbol(c_interp_small, all.data(), sizeof(float) * kSmallCoef));
    all.clear();
    for (int lu = 2; lu <= 3; ++lu) {
        design_interpolator(lu, part, kWideT, kWideMinOs);
        all.insert(all.end(), part.begin(), part.end());
    }
    GCWT_CUDA_OK(cudaMemcpyToSymbol(c_interp_wide, all.data(), sizeof(float) * kWideCoef));
    return GCWT_OK;
}

// ---- accuracy guard: plan-time error gains -----------------------------------------------------
// For a scale served at decimation level l (D = 2^l) the fused path's response differs from the exact
// filter H only outside the kept band [0, pi / (2D)):
//   alias: a component at w = (2 pi k + theta_m) / D, k != 0, reaches bin m of the level's grid with the
//          pyramid gain g(k, m) = prod_i |hb((2 pi (k mod 2^i) + theta_m) / 2^i)|, i = 1..l, and is then
//          multiplied by the table entry T[m] = |G[m]| / Hdec[m];
//   drop:  the response H(w) itself, which the path treats as zero there (and at all negative frequencies).
// Both are reduced to one gain per octave b (|w| in (pi / 2^(b+1), pi / 2^b]) so that the execute-time
// check is  sum_b gain[b] * E_b  <=  tol^2 * (measured output energy), with E_b from the pyramid.
struct HbTaps { double odd[kHalfbandOdd]; };

__device__ __forceinline__ double hb_gain_dev(const HbTaps& h, double theta) {
    double g = 0.5;
#pragma unroll
    for (int k = 0; k < kHalfbandOdd; ++k) g += 2.0 * h.odd[k] * cos((double)(2 * k + 1) * theta);
    return g;
}

__global__ void guard_alias_kernel(int level, HbTaps h, unsigned* __restrict__ B /*[kGuardSlots][kBins] float bits*/) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int D = 1 << level;
    if (idx >= (int64_t)D * kBins) return;
    const int k = (int)(idx / kBins), m = (int)(idx % kBins);
    if (k == 0) return;                                           // k = 0 is the kept band itself
    const double two_pi = 6.283185307179586476925287;
    const double theta_m = two_pi * (double)m / (double)kChunkDec;
    double g = 1.0;
    for (int i = 1; i <= level; ++i) {
        const int r = k & ((1 << i) - 1);
        g *= fabs(hb_gain_dev(h, (two_pi * (double)r + theta_m) / (double)(1 << i)));
    }
    const int kk = min(k, D - k);                                 // |w| ~ 2 pi kk / D
    int b = 0;
    while (((int64_t)kk << (b + 2)) <= D) ++b;                    // 2 kk / D in (2^-(b+1), 2^-b]
    atomicMax(B + b * kBins + m, __float_as_uint((float)g));
}

__global__ void __launch_bounds__(256)
guard_drop_kernel(const ScaleInfo* __restrict__ scales, const double* __restrict__ terms, float* __restrict__ out) {
    __shared__ unsigned mx[kGuardSlots];
    const int s = blockIdx.x, tid = threadIdx.x;
    const ScaleInfo sc = scales[s];
    if (tid < kGuardSlots) mx[tid] = 0u;
    __syncthreads();
    const int lev = sc.level;
    if (lev >= kMinFastLevel) {
        const double* X = terms + sc.term_off;
        const double pi = 3.141592653589793238462643;
        // octave b = lev, positive side: the exact response on a 4x finer grid than the chunk's (>= 8
        // samples per side lobe), bins just above the kept band
        const int64_t n = (int64_t)(4 * kChunkDec) << lev;
        for (int i = tid; i < 4 * kBins; i += 256) {
            const double g = fabs(morse_response(4 * kBins + i, n, sc.L, sc.k_first, sc.n_terms, X));
            atomicMax(&mx[lev], __float_as_uint((float)(1.1 * g)));
        }
        // everywhere else the envelope of the side lobes, |sum_k (-1)^k X_k / sin((w - w_k) / 2)| / L, at
        // 24 log-spaced points per octave and sign; slot lev + 1 = negative frequencies below the band edge
        for (int i = tid; i < (lev + 2) * 48; i += 256) {
            const int b = i / 48, j = i % 48, t = j % 24;
            const bool neg = j >= 24;
            if (!neg && b >= lev) continue;
            double lo = pi / (double)(int64_t(1) << (b + 1)), hi = 2.0 * lo;
            if (b == lev + 1) { hi = pi / (double)(int64_t(2) << lev); lo = hi / 64.0; }
            const double w = (neg ? -1.0 : 1.0) * lo * pow(hi / lo, (double)t / 23.0);
            const double step = 2.0 * pi / (double)sc.L;
            double far = 0.0, near = 0.0;
            for (int q = 0; q < sc.n_terms; ++q) {
                const int64_t k = sc.k_first + q;
                const double d = w - step * (double)k;
                if (fabs(d) < step) near += X[q];                  // within one grid spacing: at most X_k
                else far += ((k & 1) ? -X[q] : X[q]) / sin(0.5 * d);
            }
            const double v = 1.15 * (fabs(far) / (double)sc.L + near);
            atomicMax(&mx[b], __float_as_uint((float)v));
        }
    }
    __syncthreads();
    if (tid < kGuardSlots) out[(int64_t)s * kGuardSlots + tid] = __uint_as_float(mx[tid]);
}

static int guard_plan_build(gcwt_plan* p, const PlanResponses& pr, const std::vector<double>& hb) {
    const int S = p->n_scales;
    std::vector<float> gain((size_t)S * kGuardSlots, 0.f), q(S, 0.f);
    std::vector<int32_t> cls(S, -1);
    for (size_t ci = 0; ci < p->classes.size(); ++ci)
        for (int id : p->classes[ci].scale_ids) cls[id] = (int32_t)ci;
    // side-lobe gains (device, needs the levels chosen by the planner)
    GCWT_CUDA_OK(cudaMemcpy(p->d_scales, p->scales.data(), sizeof(ScaleInfo) * S, cudaMemcpyHostToDevice));
    float* d_drop = nullptr;
    GCWT_CUDA_OK(cudaMalloc((void**)&d_drop, sizeof(float) * S * kGuardSlots));
    guard_drop_kernel<<<S, 256>>>(p->d_scales, p->d_terms, d_drop);
    count_launch();
    std::vector<float> drop((size_t)S * kGuardSlots);
    cudaError_t e = cudaMemcpy(drop.data(), d_drop, sizeof(float) * drop.size(), cudaMemcpyDeviceToHost);
    cudaFree(d_drop);
    if (e != cudaSuccess) { set_error(std::string("guard tables: ") + cudaGetErrorString(e)); return GCWT_ERR_CUDA; }
    // pyramid alias gains, one table per level in use
    HbTaps taps;
    for (int k = 0; k < kHalfbandOdd; ++k) taps.odd[k] = (double)(float)p->halfband_odd[k];
    std::map<int, std::vector<float>> alias;
    for (const FastClass& fc : p->classes) {
        if (fc.level < kMinFastLevel || alias.count(fc.level)) continue;
        unsigned* d_b = nullptr;
        GCWT_CUDA_OK(cudaMalloc((void**)&d_b, sizeof(unsigned) * kGuardSlots * kBins));
        GCWT_CUDA_OK(cudaMemset(d_b, 0, sizeof(unsigned) * kGuardSlots * kBins));
        const int64_t total = (int64_t)kBins << fc.level;
        guard_alias_kernel<<<(unsigned)((total + 255) / 256), 256>>>(fc.level, taps, d_b);
        count_launch();
        std::vector<float>& B = alias[fc.level];
        B.resize((size_t)kGuardSlots * kBins);
        e = cudaMemcpy(B.data(), d_b, sizeof(float) * B.size(), cudaMemcpyDeviceToHost);
        cudaFree(d_b);
        if (e != cudaSuccess) { set_error(std::string("guard tables: ") + cudaGetErrorString(e)); return GCWT_ERR_CUDA; }
    }
    for (int s = 0; s < S; ++s) {
        const int lev = p->scales[s].level;
        if (cls[s] < 0) continue;
        if (lev < 0) {                                             // full-spectrum class: rounding only
            const double* g = pr.full(s);
            double acc = 0.0;
            for (int m = 0; m < kFullN; ++m) acc += g[m] * g[m];
            q[s] = (float)(acc / kFullN);
            continue;
        }
        const double* g = pr.level(s, lev);
        const std::vector<float>& B = alias[lev];
        double T[kBins], acc = 0.0;
        for (int m = 0; m < kBins; ++m) {
            double t = std::fabs(g[m]);
            for (int j = 1; j <= lev; ++j) t /= hb[(size_t)j * kBins + m];
            T[m] = t;
            acc += t * t;
        }
        q[s] = (float)(acc / kChunkDec);
        for (int b = 0; b <= lev + 1 && b < kGuardSlots; ++b) {
            double al = 0.0;
            if (b < lev)
                for (int m = 0; m < kBins; ++m) al = std::max(al, (double)B[(size_t)b * kBins + m] * T[m]);
            const double tot = al + (double)drop[(size_t)s * kGuardSlots + b];
            gain[(size_t)s * kGuardSlots + b] = (float)(tot * tot);
        }
    }
    GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_gain, sizeof(float) * gain.size()));
    GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_q, sizeof(float) * S));
    GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_class, sizeof(int32_t) * S));
    GCWT_CUDA_OK(cudaMemcpy(p->d_guard_gain, gain.data(), sizeof(float) * gain.size(), cudaMemcpyHostToDevice));
    GCWT_CUDA_OK(cudaMemcpy(p->d_guard_q, q.data(), sizeof(float) * S, cudaMemcpyHostToDevice));
    GCWT_CUDA_OK(cudaMemcpy(p->d_guard_class, cls.data(), sizeof(int32_t) * S, cudaMemcpyHostToDevice));
    GCWT_CUDA_OK(cudaEventCreateWithFlags(&p->ev_guard, cudaEventDisableTiming));
    p->guard_last_flags.assign(S, 0);
    p->guard_gain_h = gain;
    p->guard_q_h = q;
    return GCWT_OK;
}

int fast_plan_build(gcwt_plan* p) {
    design_halfband(p->halfband_odd);
    {
        std::vector<float2> tw(kFullN);
        for (int k = 0; k < kFullN; ++k) {
            const double a = -2.0 * M_PI * (double)k / (double)kFullN;
            tw[k] = make_float2((float)std::cos(a), (float)std::sin(a));
        }
        GCWT_CUDA_OK(cudaMalloc((void**)&p->d_twiddle, sizeof(float2) * kFullN));
        GCWT_CUDA_OK(cudaMemcpy(p->d_twiddle, tw.data(), sizeof(float2) * kFullN, cudaMemcpyHostToDevice));
    }
    PlanResponses pr;
    { int rc = compute_plan_responses(p, pr); if (rc) return rc; }
    // half-band gains at theta = 2 pi m / (1024 * 2^j), j = 1 .. kMaxFastLevel: the decimator
    // response of a level is the product over its stages
    std::vector<double> hb((size_t)(kMaxFastLevel + 1) * kBins, 1.0);
    for (int j = 1; j <= kMaxFastLevel; ++j)
        for (int m = 0; m < kBins; ++m)
            hb[(size_t)j * kBins + m] = halfband_gain(p->halfband_odd, 2.0 * M_PI * (double)m / (double)((int64_t)kChunkDec << j));
    std::map<int, std::vector<int>> by_level;
    p->max_level = 0;
    for (int s = 0; s < p->n_scales; ++s) {
        ScaleInfo& sc = p->scales[s];
        sc.level = choose_level(p, pr, s);
        if (sc.level == -2) p->generic_ids.push_back(s);
        else by_level[sc.level].push_back(s);
        p->max_level = std::max(p->max_level, sc.level);
    }
    for (auto& kv : by_level) {
        const int level = kv.first;
        const std::vector<int>& ids = kv.second;
        const int cap = level >= 0 ? kMaxClassScales : kMaxFullScales;
        for (size_t i0 = 0; i0 < ids.size(); i0 += cap) {
            // the class enters the plan's list before its device tables are allocated, so that an error
            // return below leaves them to fast_plan_free
            p->classes.emplace_back();
            FastClass& fc = p->classes.back();
            fc.level = level;
            fc.nc_full = level >= 0 ? ((int64_t)kChunkDec << level) : kFullN;
            fc.scale_ids.assign(ids.begin() + i0, ids.begin() + std::min(ids.size(), i0 + cap));
            fc.lmax = 1;
            for (int id : fc.scale_ids) fc.lmax = std::max(fc.lmax, p->scales[id].L);
            const bool may_interp = p->out_kind != GCWT_OUT_COMPLEX && !(p->flags & GCWT_FLAG_NO_INTERP);
            fc.interp = level >= kInterpMinLevel && may_interp;
            fc.log2u = level - 1;
            // |W|^2 of a scale whose filter spans w bins of the (1024 D)-point grid reaches 2 pi w / (1024 D);
            // the coarse Nyquist frequency is pi / U: over-sampling 1024 / w on U = D/2, 512 / w on U = D
            int wmax = 1;
            if (level >= 0)
                for (int id : fc.scale_ids) wmax = std::max(wmax, band_width_bins(p, pr, id, level));
            if (may_interp && level >= 2 && level <= kWideMaxLevel) {
                // coarse spacing U = D is allowed when |W|^2 stays 2.5x over-sampled on that grid
                if (512.0 / (double)wmax >= kWideMinOs) { fc.interp = true; fc.wide = true; fc.log2u = level; }
            }
            class_geometry(fc);
            if (fc.hop <= 0) { set_error("planner: non-positive hop"); return GCWT_ERR_ARG; }
            const int ns = (int)fc.scale_ids.size();
            if (fc.wide) {                                        // same margins on the 2x longer chunk
                const int64_t d = int64_t(1) << level, align = std::max<int64_t>(d, 16), nc2 = 2 * fc.nc_full;
                const int64_t lead = (int64_t)(kWideT / 2 - 1) << fc.log2u, tail = (int64_t)(kWideT / 2 + 1) << fc.log2u;
                fc.offset2 = ((fc.lmax / 2 + lead + align - 1) / align) * align;
                fc.hop2 = ((nc2 - (fc.lmax - 1) / 2 - tail - fc.offset2) / align) * align;
                std::vector<float2> tab2((size_t)ns * 2 * kBins);
                for (int i = 0; i < ns; ++i) {
                    const ScaleInfo& sc = p->scales[fc.scale_ids[i]];
                    const double* gsrc = pr.wide2(fc.scale_ids[i], level);
                    for (int m = 0; m < 2 * kBins; ++m) {
                        double g = gsrc[m] / (double)(2 * kChunkDec);
                        // decimator: stage i of `level` runs at theta = 2 pi m 2^(i-1) / (2048 D)
                        for (int j = 1; j <= level; ++j)
                            g /= halfband_gain(p->halfband_odd, 2.0 * M_PI * (double)m / (double)((int64_t)(2 * kChunkDec) << j));
                        double re = g, im = 0.0;
                        if ((sc.L & 1) == 0) {
                            const double ph = -M_PI * (double)m / (double)nc2;
                            re = g * std::cos(ph);
                            im = g * std::sin(ph);
                        }
                        tab2[(size_t)i * 2 * kBins + m] = make_float2((float)re, (float)im);
                    }
                }
                GCWT_CUDA_OK(cudaMalloc((void**)&fc.d_table2, sizeof(float2) * tab2.size()));
                GCWT_CUDA_OK(cudaMemcpy(fc.d_table2, tab2.data(), sizeof(float2) * tab2.size(), cudaMemcpyHostToDevice));
            } else {
                const int nb = level >= 0 ? kBins : kFullN;
                std::vector<float2> tab((size_t)ns * nb);
                for (int i = 0; i < ns; ++i) {
                    const ScaleInfo& sc = p->scales[fc.scale_ids[i]];
                    const double* gsrc = level >= 0 ? pr.level(fc.scale_ids[i], level) : pr.full(fc.scale_ids[i]);
                    for (int m = 0; m < nb; ++m) {
                        double g = gsrc[m];
                        if (level >= 0) {
                            for (int j = 1; j <= level; ++j) g /= hb[(size_t)j * kBins + m];
                            g /= (double)kChunkDec;
                        } else {
                            g /= (double)kFullN;
                        }
                        double re = g, im = 0.0;
                        if ((sc.L & 1) == 0) {
                            const double ph = -M_PI * (double)m / (double)fc.nc_full;
                            re = g * std::cos(ph);
                            im = g * std::sin(ph);
                        }
                        tab[(size_t)i * nb + m] = make_float2((float)re, (float)im);
                    }
                }
                GCWT_CUDA_OK(cudaMalloc((void**)&fc.d_table, sizeof(float2) * tab.size()));
                GCWT_CUDA_OK(cudaMemcpy(fc.d_table, tab.data(), sizeof(float2) * tab.size(), cudaMemcpyHostToDevice));
                if (fc.interp) {
                    // per-class taps (spacings U >= 16): fitted to the band this class really occupies
                    std::vector<float> coef;
                    const double os = std::min(8.0, std::max(kInterpMinOs, 0.98 * 1024.0 / (double)wmax));
                    design_interpolator(fc.log2u, coef, kInterpT, os);
                    GCWT_CUDA_OK(cudaMalloc((void**)&fc.d_coef, sizeof(float) * coef.size()));
                    GCWT_CUDA_OK(cudaMemcpy(fc.d_coef, coef.data(), sizeof(float) * coef.size(), cudaMemcpyHostToDevice));
                }
            }
            if (level < 0) {
                for (int id : fc.scale_ids) fc.scale_nmu.push_back(full_extent(p, pr, id));
                GCWT_CUDA_OK(cudaMalloc((void**)&fc.d_scale_nmu, sizeof(int32_t) * ns));
                GCWT_CUDA_OK(cudaMemcpy(fc.d_scale_nmu, fc.scale_nmu.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice));
            }
            GCWT_CUDA_OK(cudaMalloc((void**)&fc.d_scale_ids, sizeof(int32_t) * ns));
            GCWT_CUDA_OK(cudaMemcpy(fc.d_scale_ids, fc.scale_ids.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice));
        }
    }
    if (p->guard && !p->classes.empty()) {
        if (p->max_level + 2 >= kGuardLevels || (int)p->classes.size() > 64) p->guard = false;   // cannot happen (kMaxFastLevel = 14)
        else { int rc = guard_plan_build(p, pr, hb); if (rc) return rc; }
    } else {
        p->guard = false;
    }
    return GCWT_OK;
}

void fast_plan_free(gcwt_plan* p) {
    if (p->d_guard_gain) cudaFree(p->d_guard_gain);
    if (p->d_guard_q) cudaFree(p->d_guard_q);
    if (p->d_guard_class) cudaFree(p->d_guard_class);
    if (p->d_guard_acc) cudaFree(p->d_guard_acc);
    if (p->d_guard_pow) cudaFree(p->d_guard_pow);
    if (p->d_guard_flags) cudaFree(p->d_guard_flags);
    if (p->h_guard_flags) cudaFreeHost(p->h_guard_flags);
    if (p->ev_guard) cudaEventDestroy(p->ev_guard);
    p->d_guard_gain = p->d_guard_q = nullptr; p->d_guard_class = nullptr; p->d_guard_acc = nullptr;
    p->d_guard_pow = nullptr; p->d_guard_flags = p->h_guard_flags = nullptr; p->ev_guard = nullptr;
    for (auto& fc : p->classes) {
        if (fc.d_table) cudaFree(fc.d_table);
        if (fc.d_table2) cudaFree(fc.d_table2);
        if (fc.d_scale_ids) cudaFree(fc.d_scale_ids);
        if (fc.d_coef) cudaFree(fc.d_coef);
        if (fc.d_scale_nmu) cudaFree(fc.d_scale_nmu);
    }
    p->classes.clear();
}

// ============================================================================ pyramid
// out[i] = 0.5 in[2i] + sum_k h[2k+1] (in[2i-(2k+1)] + in[2i+(2k+1)]), zero outside the
// readable range of `in`.  Level 1 reads the raw recording and removes the mean.
constexpr int kPyrTile = 1024;  // outputs per block: four consecutive outputs per thread

template <typename TIn, bool FIRST>
__global__ void __launch_bounds__(256)
pyramid_kernel(const TIn* __restrict__ in, int64_t in_stride, int64_t in_lo, int64_t in_hi,
               const double* __restrict__ means, float* __restrict__ out, int64_t out_stride,
               int64_t out_lo, int64_t out_len,
               double* __restrict__ acc, int acc_stride, int level, int64_t seg_in, int64_t seg_out) {
    // The tile of 2*kPyrTile + 2T inputs is kept de-interleaved: ev[i] = input(u0 + 2i),
    // od[i] = input(u0 + 2i + 1), u0 = 2 i0 - T.  With T odd the centre of output j is od[j + kMid]
    // and its taps are ev[j + kMid - k], ev[j + kMid + 1 + k].  A thread owns outputs 4 tid .. 4 tid + 3:
    // with kMid = 9 its 23 even-phase inputs start at ev[4 tid] and its four centres at od[4 tid + 9],
    // so everything arrives as 128-bit shared-memory loads (od is stored shifted by kMid + 3 to line
    // up) -- 7 loads per 4 outputs instead of 21 per output -- and leaves as one 128-bit store.
    // Guard (acc != nullptr): the energy of the owned outputs that lie inside the segment [0, seg_out) is
    // added to acc[c][level]; the first level also adds the energy of its owned inputs to acc[c][0].
    static_assert(kHalfbandT == 19, "tile indexing below assumes kMid == 9");
    constexpr int kMid = (kHalfbandT - 1) / 2;
    constexpr int kEv = kPyrTile + 2 * kMid + 2 + 4;                // 4 tid + 23 <= kEv
    constexpr int kOdShift = 12 - kMid;                             // od[i] lives at ods[i + kOdShift]: centre 4 tid + 12
    __shared__ __align__(16) float ev[kEv];
    __shared__ __align__(16) float ods[kEv + 16];
    const int c = blockIdx.y;
    const int64_t i0 = out_lo + (int64_t)blockIdx.x * kPyrTile;     // first output index of the block
    const int64_t u0 = 2 * i0 - kHalfbandT;                         // first input index needed
    const TIn* src = in + (int64_t)c * in_stride - (FIRST ? 0 : in_lo);   // level arrays start at in_lo
    // fp32 recordings: the mean is subtracted in fp32 (the rounding of the mean itself, <= 6e-8 |mean|,
    // is a constant offset the zero-DC filters ignore); fp64 recordings keep the fp64 subtraction
    typedef typename std::conditional<std::is_same<TIn, float>::value, float, double>::type TSub;
    const TSub mu = FIRST ? (TSub)means[c] : (TSub)0;
    constexpr int kIn = 2 * kPyrTile + 2 * kHalfbandT;              // inputs per tile
    constexpr int kRounds = (kIn + 255) / 256;
    TIn raw[kRounds];
#pragma unroll
    for (int it = 0; it < kRounds; ++it) {                           // all loads of the tile in flight at once
        const int k = (int)threadIdx.x + 256 * it;
        const int64_t u = u0 + k;
        raw[it] = (k < kIn && u >= in_lo && u < in_hi) ? src[u] : (TIn)0;
    }
    float e_in = 0.f;
#pragma unroll
    for (int it = 0; it < kRounds; ++it) {
        const int k = (int)threadIdx.x + 256 * it;
        const int64_t u = u0 + k;
        const float v = (u >= in_lo && u < in_hi) ? (FIRST ? (float)((TSub)raw[it] - mu) : (float)raw[it]) : 0.f;
        if (k < kIn) { if (k & 1) ods[(k >> 1) + kOdShift] = v; else ev[k >> 1] = v; }
        if (FIRST && k >= kHalfbandT && k < kHalfbandT + 2 * kPyrTile && u >= 0 && u < seg_in) e_in = fmaf(v, v, e_in);
    }
    __syncthreads();
    const int j0 = 4 * threadIdx.x;
    const bool active = i0 + j0 - out_lo < out_len;
    float e_out = 0.f;
    if (active) {
        float e[24];
#pragma unroll
        for (int v = 0; v < 6; ++v) {
            const float4 t = *(const float4*)(ev + j0 + 4 * v);
            e[4 * v] = t.x; e[4 * v + 1] = t.y; e[4 * v + 2] = t.z; e[4 * v + 3] = t.w;
        }
        const float4 ctr = *(const float4*)(ods + j0 + 12);              // od[j0 + kMid .. + 3]
        const float cv[4] = {ctr.x, ctr.y, ctr.z, ctr.w};
        float o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            // fp32 accumulation, smallest taps first (fp64 would spend the kernel on conversions)
            float a = 0.f;
#pragma unroll
            for (int k = kHalfbandOdd - 1; k >= 0; --k)
                a = fmaf(c_halfband[k], e[q + kMid - k] + e[q + kMid + 1 + k], a);
            o[q] = fmaf(0.5f, cv[q], a);
            const int64_t io = i0 + j0 + q;
            if (io >= 0 && io < seg_out) e_out = fmaf(o[q], o[q], e_out);
        }
        // rows are padded to a multiple of four floats: the last quad may spill into the padding
        *(float4*)(out + (int64_t)c * out_stride + (i0 + j0 - out_lo)) = make_float4(o[0], o[1], o[2], o[3]);
    }
    if (acc != nullptr) {                                            // block-uniform
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            e_out += __shfl_xor_sync(0xffffffffu, e_out, o);
            if (FIRST) e_in += __shfl_xor_sync(0xffffffffu, e_in, o);
        }
        __syncthreads();                                             // the tile is consumed: reuse ev as scratch
        if ((threadIdx.x & 31) == 0) { ev[threadIdx.x >> 5] = e_out; if (FIRST) ev[8 + (threadIdx.x >> 5)] = e_in; }
        __syncthreads();
        if (threadIdx.x == 0) {                                      // one atomic per block and quantity
            double* a = acc + (int64_t)c * acc_stride;
            float so = 0.f, si = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) { so += ev[w]; if (FIRST) si += ev[8 + w]; }
            if (so != 0.f) atomicAdd(a + level, (double)so);
            if (FIRST && si != 0.f) atomicAdd(a, (double)si);
        }
    }
}

// ============================================================================ fused kernels
struct FusedParams {
    const void* src;          // banded: float level array (origin src_lo); full: raw recording
    int64_t src_stride;       // elements between channels
    int64_t src_lo, src_hi;   // readable index range [lo, hi) in source index units
    const double* means;      // full only
    int log2d;                // banded: log2 of the decimation factor
    int p_cols;               // banded: P = nc_full / kBins (columns per chunk)
    int log2p;                // log2(P)
    float inv_nc;             // 1 / nc_full
    int64_t offset, hop, n_chunks, n;
    int n_scales;
    const int32_t* scale_ids;
    const float2* table;
    void* out;
    int64_t s_stride, c_stride;
    int iters;                // column blocks (16 columns each) per unit
    int units_per_chunk;      // banded: column ranges per chunk; interp: output ranges per chunk
    int log2u;                // interp: log2 of the coarse spacing U
    const float* coef;        // interp: float [U][kInterpT]
    const float2* twf;        // e^{-2 pi i k / 4096}
    const int32_t* scale_nmu; // full: occupied 256-bin blocks per scale
    // accuracy guard (all null / zero when the guard is off)
    double* acc;              // [channels][acc_stride]: e_0 .. e_(kGuardLevels-1), then one chunk energy per class
    int acc_stride;
    int class_idx;
    float ech_weight;         // chunk energy -> full-rate-equivalent energy of the segment (D * hop / chunk)
    float* pow;               // [channels][pow_stride] measured sum |W|^2 per scale
    int pow_stride;
    float pow_weight;         // measured chunks -> all chunks (the guard measures every guard_every-th chunk)
    int guard_every;
    int q_mode;               // full kernel: 0 this launch covers every chunk; 1 only chunks q = i * guard_every (measured
                              // launch); 2 all the others (n_chunks is then the number of chunks of THIS launch)
};

// e^{+2 pi i k / 4096} from the table of e^{-2 pi i k / 4096}
__device__ __forceinline__ float2 tw_pos(const float2* __restrict__ twf, int k) {
    const float2 t = __ldg(twf + (k & (kFullN - 1)));
    return make_float2(t.x, -t.y);
}

__device__ __forceinline__ float sqrt_abs_approx(float v) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fabsf(v)));  // |v| folds into the MUFU operand
    return r;
}

__device__ __forceinline__ float sqrt_approx(float v) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));       // one MUFU op, rel. error 2^-23
    return r;
}

template <int KIND> struct out_elem { typedef float type; };
template <> struct out_elem<GCWT_OUT_COMPLEX> { typedef float2 type; };

// Epilogue (kernel (3)): complex, |W| or |W|^2 of 16 register-resident outputs that lie
// `stride` elements apart; bit k of `mask` says whether output k is owned by this chunk.
__device__ __forceinline__ void st_pred(float* p, float v, unsigned on) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.f32 [%0], %1;\n\t}"
                 :: "l"(p), "f"(v), "r"(on) : "memory");
}
__device__ __forceinline__ void st_pred(float2* p, float2 v, unsigned on) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %3, 0;\n\t@q st.global.v2.f32 [%0], {%1, %2};\n\t}"
                 :: "l"(p), "f"(v.x), "f"(v.y), "r"(on) : "memory");
}

template <int KIND>
__device__ __forceinline__ void store_column(typename out_elem<KIND>::type* __restrict__ op, int64_t stride,
                                             unsigned mask, const float2* a) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const unsigned on = mask & (1u << k);                     // predicated store: no divergent branch
        if constexpr (KIND == GCWT_OUT_COMPLEX) st_pred(op + k * stride, a[k], on);
        else if constexpr (KIND == GCWT_OUT_AMPLITUDE) st_pred(op + k * stride, sqrt_approx(a[k].x * a[k].x + a[k].y * a[k].y), on);
        else st_pred(op + k * stride, a[k].x * a[k].x + a[k].y * a[k].y, on);
    }
}

// bits k in [0,16) with lo <= rel + (k << sh) < hi
__device__ __forceinline__ unsigned valid_mask(int rel, int sh, int lo, int hi) {
    const int step = 1 << sh;
    int k_lo = (lo - rel + step - 1) >> sh;
    int k_hi = (hi - rel + step - 1) >> sh;
    k_lo = max(k_lo, 0);
    k_hi = min(max(k_hi, 0), 16);
    return k_hi > k_lo ? (((1u << k_hi) - 1u) & ~((1u << k_lo) - 1u)) : 0u;
}

// Mean of the chunk a block is about to transform (NV values per thread, 256 threads).  Every filter
// has exactly zero response at bin 0 (the reference forces X[0] = 0, morseutils.py:178), so ANY constant
// may be subtracted from the whole chunk -- zero padding included -- without changing a kept output.
// Subtracting the chunk's own mean keeps the fp32 butterflies from rounding at the scale of a slow
// drift: with red (1/f^2) recordings the error of the high-frequency scales drops several-fold.
// `scratch` is 8 floats of shared memory that nobody else touches until the next barrier.
template <int NV>
__device__ __forceinline__ float chunk_mean(const float* v, float* scratch) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) s += v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = s;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += scratch[w];
    return t * (1.0f / (float)(NV * 256));
}

// Guard: sum of squares of the chunk after its mean has been removed, reduced over the block and added
// (by thread 0) to the class's chunk-energy accumulator of this channel.  `scratch` as in chunk_mean,
// but the caller must place a barrier between the two uses.
template <int NV>
__device__ __forceinline__ void chunk_energy_add(const float* v, float cm, float* scratch, double* dst, float weight) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) { const float d = v[k] - cm; s = fmaf(d, d, s); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();                                           // every thread has read the mean's partial sums
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += scratch[w];
        atomicAdd(dst, (double)(t * weight));
    }
}

// Guard: |W|^2 of the outputs a thread owns in one pass (bit k of `own`), reduced over the lanes that
// share a scale (lanes differing in bit 3 hold different scales when PAIRED) into a shared counter.
template <bool PAIRED>
__device__ __forceinline__ void guard_pow_add(const float2* a, unsigned own, float* counter) {
    float pw = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const float v = a[k].x * a[k].x + a[k].y * a[k].y;
        pw += (own >> k & 1u) ? v : 0.f;
    }
    pw += __shfl_xor_sync(0xffffffffu, pw, 16);
    if (!PAIRED) pw += __shfl_xor_sync(0xffffffffu, pw, 8);
    pw += __shfl_xor_sync(0xffffffffu, pw, 4);
    pw += __shfl_xor_sync(0xffffffffu, pw, 2);
    pw += __shfl_xor_sync(0xffffffffu, pw, 1);
    const unsigned lane = threadIdx.x & 31u;
    if ((lane & (PAIRED ? 23u : 31u)) == 0) atomicAdd(counter, pw);
}

// 1024-point forward FFT: five radix-4 Stockham passes, 256 threads, one butterfly per thread and
// pass.  Thread j handles butterfly j in every pass, so all of its 12 twiddles are fetched up
// front in one batch of independent loads (one memory latency instead of four in a chain).
// Input in `a`, scratch `b`; returns the buffer that holds the result.
__device__ __forceinline__ float2* smem_fft1024_forward(float2* a, float2* b, const float2* __restrict__ tw) {
    constexpr int M = 256;
    const int j = threadIdx.x;
    float2 w[4][3];
#pragma unroll
    for (int p = 1; p < 5; ++p) {
        const int ns = 1 << (2 * p);
        const int idx = (j & (ns - 1)) * ((kFullN / 4) / ns);
#pragma unroll
        for (int r = 0; r < 3; ++r) w[p - 1][r] = __ldg(tw + (r + 1) * idx);
    }
#pragma unroll
    for (int p = 0; p < 5; ++p) {
        const int ns = 1 << (2 * p);
        const int k = j & (ns - 1);
        float2 v0 = a[j], v1 = a[j + M], v2 = a[j + 2 * M], v3 = a[j + 3 * M];
        if (p > 0) {
            v1 = cmul(v1, w[p - 1][0]);
            v2 = cmul(v2, w[p - 1][1]);
            v3 = cmul(v3, w[p - 1][2]);
        }
        dft4<-1>(v0, v1, v2, v3);
        const int j0 = ((j - k) << 2) + k;
        b[j0] = v0; b[j0 + ns] = v1; b[j0 + 2 * ns] = v2; b[j0 + 3 * ns] = v3;
        __syncthreads();
        float2* t = a; a = b; b = t;
    }
    return a;
}

// 4096-point forward FFT as three radix-16 Stockham passes, one butterfly per thread and
// pass.  Input in `x`, result in `y`; `y` needs 256 elements of slack behind it (the first
// pass writes with a pad of one element per 16 to stay free of bank conflicts).
__device__ __forceinline__ void smem_fft4096_forward(float2* x, float2* y, const float2* __restrict__ tw) {
    const int tid = threadIdx.x;
    float2 v[16], w2[16], w3[16];
#pragma unroll
    for (int r = 1; r < 16; ++r) {                                 // both passes' twiddles, one batch of loads
        w2[r] = __ldg(tw + r * (tid & 15) * 16);
        w3[r] = __ldg(tw + r * tid);
    }
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = x[tid + 256 * r];
    dft16<-1>(v);
#pragma unroll
    for (int r = 0; r < 16; ++r) y[17 * tid + r] = v[r];                      // position 16 tid + r, padded
    __syncthreads();
    {
        const int k = tid & 15;
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = y[tid + 256 * r + (tid >> 4) + 16 * r];
#pragma unroll
        for (int r = 1; r < 16; ++r) v[r] = cmul(v[r], w2[r]);
        dft16<-1>(v);
        const int j0 = ((tid - k) << 4) + k;
#pragma unroll
        for (int r = 0; r < 16; ++r) x[j0 + 16 * r] = v[r];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = x[tid + 256 * r];
#pragma unroll
    for (int r = 1; r < 16; ++r) v[r] = cmul(v[r], w3[r]);
    dft16<-1>(v);
#pragma unroll
    for (int r = 0; r < 16; ++r) y[tid + 256 * r] = v[r];
    __syncthreads();
}

// ---------------------------------------------------------------------------- banded
// smem: ex[2][4096] | Zs[kMaxClassScales][256] | Estep[256]
constexpr size_t kBandedSmem = sizeof(float2) * (2 * 4096 + kMaxClassScales * kBins + kBins) + sizeof(int) * kMaxClassScales + 16;

template <int KIND, int LP, bool GUARD>       // LP > 0: compile-time log2(P) (store offsets become immediates)
__global__ void __launch_bounds__(256, 2)
fused_banded_kernel(const FusedParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ex = (float2*)smem_raw;
    float2* Zs = ex + 2 * 4096;
    float2* Estep = Zs + kMaxClassScales * kBins;
    int* s_ids = (int*)(Estep + kBins);
    float* s_pow = (float*)(s_ids + kMaxClassScales);            // guard: two alternating output-energy counters

    const int tid = threadIdx.x;
    if (tid < prm.n_scales) s_ids[tid] = prm.scale_ids[tid];
    if (tid < 2) s_pow[tid] = 0.f;
    const int r = tid & 15;            // column within the block of 16
    const int g = tid >> 4;            // m_lo in pass 1, n_lo in pass 2

    int64_t b = blockIdx.x;
    const int unit = (int)(b % prm.units_per_chunk); b /= prm.units_per_chunk;
    const int64_t q = b % prm.n_chunks;
    const int64_t c = b / prm.n_chunks;

    const int64_t t0 = q * prm.hop - prm.offset;                 // full-rate index of chunk sample 0
    const bool sample = GUARD && (q % prm.guard_every) == 0;     // accuracy guard: this chunk is measured (block-uniform)
    // ---- (1) forward FFT of the decimated chunk ---------------------------------
    {
        const float* src = (const float*)prm.src + c * prm.src_stride - prm.src_lo;
        const int64_t i0 = t0 >> prm.log2d;                      // exact: t0 is a multiple of D
        float raw[kChunkDec / 256];
#pragma unroll
        for (int k = 0; k < kChunkDec / 256; ++k) {
            const int64_t u = i0 + tid + 256 * k;
            raw[k] = (u >= prm.src_lo && u < prm.src_hi) ? src[u] : 0.f;
        }
        const float cm = chunk_mean<kChunkDec / 256>(raw, (float*)Zs);
        if (sample && unit == 0)
            chunk_energy_add<kChunkDec / 256>(raw, cm, (float*)Zs, prm.acc + c * prm.acc_stride + kGuardLevels + prm.class_idx,
                                              prm.ech_weight);
#pragma unroll
        for (int k = 0; k < kChunkDec / 256; ++k) ex[tid + 256 * k] = make_float2(raw[k] - cm, 0.f);
        __syncthreads();
        float2* Y = smem_fft1024_forward(ex, ex + kChunkDec, prm.twf);
        // ---- (2) multiply by every scale's response (bins 0..255) ---------------
        const float2 y = Y[tid];
        for (int s = 0; s < prm.n_scales; ++s) Zs[s * kBins + tid] = cmul(y, prm.table[s * kBins + tid]);
        Estep[tid] = expipi(2.0f * (float)(tid * 16) * prm.inv_nc);
    }
    // per-thread constants
    float2 tw[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) tw[k] = tw_pos(prm.twf, 16 * g * k);      // e^{2 pi i g k / 256}
    const int col0 = unit * prm.iters * 16;
    float2 R[16];
    if (prm.p_cols == 16) {                                      // 4096-point chunk: phases are table entries
#pragma unroll
        for (int i = 0; i < 16; ++i) R[i] = tw_pos(prm.twf, (g + 16 * i) * (col0 + r));
    } else {
        const int64_t n2 = col0 + r;
        const int64_t mask = ((int64_t)prm.p_cols * kBins) - 1;  // nc_full - 1 (power of two)
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int64_t e = ((int64_t)(g + 16 * i) * n2) & mask;
            R[i] = expipi(2.0f * (float)e * prm.inv_nc);
        }
    }
    __syncthreads();

    typedef typename out_elem<KIND>::type OutT;
    const int iters = min(prm.iters, prm.p_cols / 16 - unit * prm.iters);
    const int lp = LP > 0 ? LP : prm.log2p;
    const int own_lo = (int)prm.offset;
    const int own_hi = (int)min(prm.offset + prm.hop, prm.n - t0);       // chunk-local, <= nc_full
    const int64_t kstride = (int64_t)16 << lp;
    OutT* const out_c = (OutT*)prm.out + c * prm.c_stride + t0;
    int buf = 0;
    int pend = -1;                                                       // guard: scale whose counter is flushed after the next barrier
    float* const pow_c = sample ? prm.pow + c * prm.pow_stride : nullptr;
    for (int it = 0; it < iters; ++it) {
        const int rel = col0 + it * 16 + r + (g << lp);                  // chunk-local sample of output k = 0
        const unsigned mask = valid_mask(rel, lp + 4, own_lo, own_hi);
        for (int s = 0; s < prm.n_scales; ++s) {
            float2 a[16];
            const float2* z = Zs + s * kBins + g;
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = cmul(z[16 * i], R[i]);
            dft16<+1>(a);
            float2* e = ex + buf * 4096 + (g * 16) * 16 + r;
            e[0] = a[0];                                                  // tw[0] == 1
#pragma unroll
            for (int k = 1; k < 16; ++k) e[k * 16] = cmul(a[k], tw[k]);
            __syncthreads();
            if (pend >= 0 && tid == 0) {                                  // every add for scale `pend` came before this barrier
                atomicAdd(pow_c + s_ids[pend], s_pow[pend & 1] * (float)iters * prm.pow_weight);
                s_pow[pend & 1] = 0.f;
            }
            pend = -1;
            const float2* e2 = ex + buf * 4096 + g * 16 + r;
#pragma unroll
            for (int k = 0; k < 16; ++k) a[k] = e2[k * 256];
            dft16<+1>(a);
            store_column<KIND>(out_c + (int64_t)s_ids[s] * prm.s_stride + rel, kstride, mask, a);
            if (GUARD && pow_c != nullptr && it == 0) {                   // measured: the first column block of this unit
                guard_pow_add<false>(a, mask, s_pow + (s & 1));
                pend = s;
            }
            buf ^= 1;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) R[i] = cmul(R[i], Estep[g + 16 * i]);
    }
    if (pend >= 0) {
        __syncthreads();
        if (tid == 0) atomicAdd(pow_c + s_ids[pend], s_pow[pend & 1] * (float)iters * prm.pow_weight);
    }
}

// ---------------------------------------------------------------------------- interpolated
// Amplitude / power at level >= kInterpMinLevel.  |W_s|^2 is band-limited to +-pi/(2D), so it
// is computed on the coarse grid i = iota * U (U = D/2: 8 columns of the pruned transform,
// 2048 samples per chunk and scale, two scales per 16-lane pass) and brought to the full
// rate by a kInterpT-tap polyphase FIR: ~16 instructions per output instead of ~41, which
// moves these classes from the FP32-issue bound to the HBM bound.
// smem: ex[4096] float2 | Zs[kMaxClassScales][256] float2 | Pc[2][kPcStride] float
constexpr int kPcStride = kCoarse + 16;           // % 32 == 16: the two scales of a pair hit different banks
constexpr int kPcFloats = 2 * kPcStride;
constexpr size_t kInterpSmem = sizeof(float2) * (4096 + kMaxClassScales * kBins) + sizeof(float) * kPcFloats + sizeof(int) * kMaxClassScales + 16;

template <int KIND, int LU, int T>   // LU > 0: compile-time log2 of the coarse spacing (store offsets become immediates); T taps
__device__ __forceinline__ void interp_rows(const float* __restrict__ pc, float* __restrict__ row,
                                            const float* __restrict__ coef, const float* c0, int lu_rt,
                                            int ia, int ib, int own_hi) {
    const int lu = LU > 0 ? LU : lu_rt;
    // thread <-> phase phi; lanes of a warp hold consecutive phases of the same coarse interval,
    // so the window loads are shared-memory broadcasts and the stores are contiguous.
    const int U = 1 << lu;
    const int tid = threadIdx.x;
    int phi_step, n_phi_iter, phi, a, b;
    if (U >= 256) {
        phi = tid; phi_step = 256; n_phi_iter = U >> 8; a = ia; b = ib;
    } else {
        const int stripes = max(1, 256 >> lu), stripe = tid >> lu;
        const int len = (ib - ia + stripes - 1) / stripes;
        phi = tid & (U - 1); phi_step = U; n_phi_iter = 1;
        a = min(ib, ia + stripe * len); b = min(ib, a + len);
    }
    for (int pi = 0; pi < n_phi_iter; ++pi, phi += phi_step) {
        float c[T];
#pragma unroll
        for (int t = 0; t < T; ++t) c[t] = (n_phi_iter == 1) ? c0[t] : coef[phi * T + t];
        const int b_t = min(b, (own_hi - phi + U - 1) >> lu);     // iota with iota*U + phi < own_hi
        float w[T];
#pragma unroll
        for (int j = 0; j < T - 1; ++j) w[j] = pc[a - (T / 2 - 1) + j];
        float* op = row + ((int64_t)a << lu) + phi;
        int base = a;
        for (; base + T <= b_t; base += T) {        // full groups: no predicates
#pragma unroll
            for (int u = 0; u < T; ++u) {
                // window of iota = base + u is pc[iota-4 .. iota+5], kept in w[(u + j) % T]
                w[(u + T - 1) % T] = pc[base + u + T / 2];
                float acc = c[0] * w[u % T];
#pragma unroll
                for (int j = 1; j < T; ++j) acc = fmaf(c[j], w[(u + j) % T], acc);
                // interpolated power can undershoot zero by rounding-size amounts near nulls
                op[(int64_t)u << lu] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_abs_approx(acc) : fmaxf(acc, 0.f);
            }
            op += (int64_t)T << lu;
        }
        // tail: fewer than T intervals, leave as soon as they are done (the lanes of a warp share
        // the count except in the recording's last chunk, so the exit rarely diverges)
#pragma unroll
        for (int u = 0; u < T; ++u) {
            if (base + u >= b_t) break;
            w[(u + T - 1) % T] = pc[base + u + T / 2];
            float acc = c[0] * w[u % T];
#pragma unroll
            for (int j = 1; j < T; ++j) acc = fmaf(c[j], w[(u + j) % T], acc);
            op[(int64_t)u << lu] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_abs_approx(acc) : fmaxf(acc, 0.f);
        }
    }
}

// Smallest coarse spacing (U = 4, level 3): thread <-> coarse interval, all U phases per thread
// from one register window; taps come from the constant bank; the U consecutive outputs leave as
// one 128-bit store (the launcher guarantees 16-byte aligned rows).
template <int KIND>
__device__ __forceinline__ void interp_rows_small(const float* __restrict__ pc, float* __restrict__ row,
                                                  int ia, int ib, int own_hi) {
    constexpr int U = 4;                                          // taps: c_interp_small[0 .. 4 kInterpT)
    for (int iota = ia + (int)threadIdx.x; iota < ib; iota += 256) {
        float w[kInterpT];
#pragma unroll
        for (int j = 0; j < kInterpT; ++j) w[j] = pc[iota - (kInterpT / 2 - 1) + j];
        float o[U];
        o[0] = w[kInterpT / 2 - 1];                               // phase 0 sits on a coarse sample
#pragma unroll
        for (int phi = 1; phi < U; ++phi) {
            float acc = c_interp_small[phi * kInterpT] * w[0];
#pragma unroll
            for (int j = 1; j < kInterpT; ++j) acc = fmaf(c_interp_small[phi * kInterpT + j], w[j], acc);
            o[phi] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_abs_approx(acc) : fmaxf(acc, 0.f);
        }
        if (KIND == GCWT_OUT_AMPLITUDE) o[0] = sqrt_approx(o[0]);
        float* op = row + (int64_t)iota * U;
        if ((iota + 1) * U <= own_hi) {
            *(float4*)op = make_float4(o[0], o[1], o[2], o[3]);
        } else {
#pragma unroll
            for (int phi = 0; phi < U; ++phi) if (iota * U + phi < own_hi) op[phi] = o[phi];
        }
    }
}

// 256-bit store (sm_100: STG.E.256): eight consecutive floats, 32-byte aligned
__device__ __forceinline__ void st_v8(float* p, const float* o) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "l"(p), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]), "f"(o[4]), "f"(o[5]), "f"(o[6]), "f"(o[7]) : "memory");
}

// Wide-spacing classes (coarse spacing U = D = 4 or 8, kWideT taps from the constant bank): all U phases of a
// coarse interval from one register window, two adjacent intervals per thread.  Their windows overlap in all but
// one sample, so the 14 samples arrive as seven 64-bit shared loads (0.22 loads per output at U = 4 instead of
// 0.75 32-bit ones with one interval per thread, 42 % fewer shared-memory wavefronts) and the 2 U outputs leave
// as 256-bit stores when the rows allow it.
// `align`: 0 rows unaligned (scalar stores), 1 16-byte aligned rows, 2 32-byte aligned rows.
template <int KIND, int LU, int NI>       // NI adjacent coarse intervals per thread (ia must be a multiple of NI, NI even)
__device__ __forceinline__ void interp_rows_wide_pairs(const float* __restrict__ pc, float* __restrict__ row,
                                                       int ia, int ib, int own_hi, int align) {
    constexpr int U = 1 << LU;
    constexpr int COFF = (LU == 2) ? 0 : 4 * kWideT;
    constexpr int NW = kWideT + NI;                                             // window pc[iota - 6 .. iota + NI + 5], 64-bit aligned
    static_assert(kWideT == 12 && NI % 2 == 0 && (NI * U) % 8 == 0, "window indexing below assumes 12 taps");
    for (int iota = ia + NI * (int)threadIdx.x; iota < ib; iota += NI * 256) {
        float w[NW];
        const float2* p2 = (const float2*)(pc + iota - 6);
#pragma unroll
        for (int j = 0; j < NW / 2; ++j) { const float2 t = p2[j]; w[2 * j] = t.x; w[2 * j + 1] = t.y; }
        float o[NI * U];
#pragma unroll
        for (int h = 0; h < NI; ++h) {                                          // interval iota + h: window w[1 + h .. 12 + h]
            o[h * U] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_approx(w[6 + h]) : w[6 + h];
#pragma unroll
            for (int phi = 1; phi < U; ++phi) {
                float acc = c_interp_wide[COFF + phi * kWideT] * w[1 + h];
#pragma unroll
                for (int j = 1; j < kWideT; ++j) acc = fmaf(c_interp_wide[COFF + phi * kWideT + j], w[1 + h + j], acc);
                o[h * U + phi] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_abs_approx(acc) : fmaxf(acc, 0.f);
            }
        }
        float* op = row + (int64_t)iota * U;
        if (align && (iota + NI) * U <= own_hi) {
            if (align == 2) {
#pragma unroll
                for (int v = 0; v < NI * U / 8; ++v) st_v8(op + 8 * v, o + 8 * v);
            } else {
#pragma unroll
                for (int v = 0; v < NI * U / 4; ++v) ((float4*)op)[v] = make_float4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < NI * U; ++i) if (iota * U + i < own_hi) op[i] = o[i];
        }
    }
}

// U = 8 on the grid U = D/2 (level 4): two adjacent intervals per thread, kInterpT = 8 taps from the constant bank
// (the U <= 8 designs at over-sampling 4), the 10 window samples as five 64-bit shared loads, the 16 outputs as
// two 256-bit stores (0.31 loads and 0.125 stores per output against 1 and 1 in the sliding form).
template <int KIND>
__device__ __forceinline__ void interp_rows_pairs8(const float* __restrict__ pc, float* __restrict__ row,
                                                   int ia, int ib, int own_hi, int align) {
    constexpr int U = 8, COFF = 4 * kInterpT;                                   // behind the U = 4 taps
    static_assert(kInterpT == 8, "window indexing below assumes 8 taps");
    for (int iota = ia + 2 * (int)threadIdx.x; iota < ib; iota += 512) {        // ia is even
        float w[10];                                                            // pc[iota - 4 .. iota + 5]
        const float2* p2 = (const float2*)(pc + iota - 4);
#pragma unroll
        for (int j = 0; j < 5; ++j) { const float2 t = p2[j]; w[2 * j] = t.x; w[2 * j + 1] = t.y; }
        float o[2 * U];
#pragma unroll
        for (int h = 0; h < 2; ++h) {                                           // interval iota + h: window w[1 + h .. 8 + h]
            o[h * U] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_approx(w[4 + h]) : w[4 + h];
#pragma unroll
            for (int phi = 1; phi < U; ++phi) {
                float acc = c_interp_small[COFF + phi * kInterpT] * w[1 + h];
#pragma unroll
                for (int j = 1; j < kInterpT; ++j) acc = fmaf(c_interp_small[COFF + phi * kInterpT + j], w[1 + h + j], acc);
                o[h * U + phi] = (KIND == GCWT_OUT_AMPLITUDE) ? sqrt_abs_approx(acc) : fmaxf(acc, 0.f);
            }
        }
        float* op = row + (int64_t)iota * U;
        if (align == 2 && (iota + 2) * U <= own_hi) {
            st_v8(op, o);
            st_v8(op + 8, o + 8);
        } else {
#pragma unroll
            for (int i = 0; i < 2 * U; ++i) if (iota * U + i < own_hi) op[i] = o[i];
        }
    }
}

template <int KIND, bool GUARD>
__global__ void __launch_bounds__(256, 2)
fused_interp_kernel(const FusedParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ex = (float2*)smem_raw;
    float2* Zs = ex + 4096;
    float* Pc = (float*)(Zs + kMaxClassScales * kBins);
    int* s_ids = (int*)(Pc + kPcFloats);
    float* s_pow = (float*)(s_ids + kMaxClassScales);   // guard: output-energy counters of the two scales of a pass
    constexpr int NCOL = 8;                        // coarse columns per chunk
    constexpr int NSC = 16 / NCOL;                 // scales transformed per 16-lane pass
    constexpr int PCS = kPcStride;

    const int tid = threadIdx.x;
    if (tid < prm.n_scales) s_ids[tid] = prm.scale_ids[tid];
    if (tid < 2) s_pow[tid] = 0.f;
    const int r = tid & 15;
    const int g = tid >> 4;
    const int col = r & (NCOL - 1);    // coarse column: chunk-local sample (NCOL n1 + col) * U
    const int sidx = r / NCOL;         // which scale of the group

    int64_t bid = blockIdx.x;
    const int split = (int)(bid % prm.units_per_chunk); bid /= prm.units_per_chunk;
    const int64_t q = bid % prm.n_chunks;
    const int64_t c = bid / prm.n_chunks;
    const int64_t t0 = q * prm.hop - prm.offset;
    const bool sample = GUARD && (q % prm.guard_every) == 0;     // accuracy guard: this chunk is measured (block-uniform)

    // this block's share of the chunk's owned output window, in coarse intervals
    const int lu = prm.log2u;
    const int own_lo = (int)prm.offset;
    const int own_hi = (int)min(prm.offset + prm.hop, prm.n - t0);
    const int io_lo = own_lo >> lu, io_hi = (own_hi + (1 << lu) - 1) >> lu;
    const int len = (io_hi - io_lo + prm.units_per_chunk - 1) / prm.units_per_chunk;
    const int ia = io_lo + split * len, ib = min(io_hi, ia + len);
    if (ia >= ib) return;

    {   // (1) forward FFT of the decimated chunk, (2) multiply by every scale's response
        const float* src = (const float*)prm.src + c * prm.src_stride - prm.src_lo;
        const int64_t i0 = t0 >> prm.log2d;
        float raw[kChunkDec / 256];
#pragma unroll
        for (int k = 0; k < kChunkDec / 256; ++k) {
            const int64_t u = i0 + tid + 256 * k;
            raw[k] = (u >= prm.src_lo && u < prm.src_hi) ? src[u] : 0.f;
        }
        const float cm = chunk_mean<kChunkDec / 256>(raw, (float*)Zs);
        if (sample && split == 0)
            chunk_energy_add<kChunkDec / 256>(raw, cm, (float*)Zs, prm.acc + c * prm.acc_stride + kGuardLevels + prm.class_idx,
                                              prm.ech_weight);
#pragma unroll
        for (int k = 0; k < kChunkDec / 256; ++k) ex[tid + 256 * k] = make_float2(raw[k] - cm, 0.f);
        __syncthreads();
        float2* Y = smem_fft1024_forward(ex, ex + kChunkDec, prm.twf);
        const float2 y = Y[tid];
        for (int s = 0; s < prm.n_scales; ++s) Zs[s * kBins + tid] = cmul(y, prm.table[s * kBins + tid]);
    }
    float2 tw[16], R[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        tw[k] = tw_pos(prm.twf, 16 * g * k);                      // e^{2 pi i g k / 256}
        R[k] = tw_pos(prm.twf, (16 / NCOL) * (g + 16 * k) * col); // e^{2 pi i m col / (256 NCOL)}
    }
    __syncthreads();

    // taps of this thread's phase (one phase per thread while U <= 256): fetched once per block
    float c0[kInterpT];
    if (lu >= 3 && lu <= 8) {
        const int phi0 = tid & ((1 << lu) - 1);
#pragma unroll
        for (int t = 0; t < kInterpT; ++t) c0[t] = __ldg(prm.coef + phi0 * kInterpT + t);
    } else {
#pragma unroll
        for (int t = 0; t < kInterpT; ++t) c0[t] = 0.f;
    }
    float* const out_c = (float*)prm.out + c * prm.c_stride + t0;
    // guard: coarse samples (g + 16 k) * NCOL + col of this thread that lie in the block's own range
    unsigned own = 0;
    if (sample) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int iota = (g + 16 * k) * NCOL + col;
            own |= (unsigned)(iota >= ia && iota < ib) << k;
        }
    }
    for (int pair = 0; pair < prm.n_scales; pair += NSC) {
        const int s = min(pair + sidx, prm.n_scales - 1);
        float2 a[16];
        const float2* z = Zs + s * kBins + g;
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = cmul(z[16 * i], R[i]);
        dft16<+1>(a);
        float2* e = ex + (g * 16) * 16 + r;
        e[0] = a[0];
#pragma unroll
        for (int k = 1; k < 16; ++k) e[k * 16] = cmul(a[k], tw[k]);
        __syncthreads();
        const float2* e2 = ex + g * 16 + r;
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = e2[k * 256];
        dft16<+1>(a);
        float* pc = Pc + sidx * PCS + g * NCOL + col;             // iota = (g + 16 k) * NCOL + col
#pragma unroll
        for (int k = 0; k < 16; ++k) pc[k * 16 * NCOL] = a[k].x * a[k].x + a[k].y * a[k].y;
        if (sample) guard_pow_add<true>(a, own, s_pow + sidx);
        __syncthreads();
        // (3) polyphase interpolation + epilogue for the scales of this pass
        // (dealing the (scale, interval) pairs of a pass to the threads as one flat sequence, to save the
        // partial last round of 256 per scale, measured slower: whole idle warps cost nothing)
        const int nsc = min(NSC, prm.n_scales - pair);
        if (sample && tid < NSC) {                                 // the loop's closing barrier orders the reset
            if (tid < nsc) atomicAdd(prm.pow + c * prm.pow_stride + s_ids[pair + tid], s_pow[tid] * (float)(1 << lu) * prm.pow_weight);
            s_pow[tid] = 0.f;
        }
        for (int sl = 0; sl < nsc; ++sl) {
            const float* pcs = Pc + sl * PCS;
            float* row = out_c + (int64_t)s_ids[pair + sl] * prm.s_stride;
            if (lu == 2) {
                interp_rows_small<KIND>(pcs, row, ia, ib, own_hi);
            } else {
                switch (lu) {
                    case 3:
                        if (prm.iters == 2 && prm.units_per_chunk == 1) interp_rows_pairs8<KIND>(pcs, row, ia, ib, own_hi, 2);
                        else interp_rows<KIND, 3, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi);
                        break;
                    case 4:  interp_rows<KIND, 4, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 5:  interp_rows<KIND, 5, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 6:  interp_rows<KIND, 6, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 7:  interp_rows<KIND, 7, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 8:  interp_rows<KIND, 8, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 9:  interp_rows<KIND, 9, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    case 10: interp_rows<KIND, 10, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                    default: interp_rows<KIND, 0, kInterpT>(pcs, row, prm.coef, c0, lu, ia, ib, own_hi); break;
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------- wide classes, long chunks
// The wide classes (levels 2-3, U = D) pay most for their coarse transforms, so they use chunks of
// 2048 decimated samples with 512 bins kept: overlap-save efficiency 0.90 instead of 0.80 and half
// the per-chunk fixed cost.  The 512 useful bins of the chunk's spectrum stay in registers (two per
// thread); W on the coarse grid is a 2048-point inverse transform with 512 non-zero bins = 8 columns
// of 256-point transforms, two scales per 16-lane pass: the two alias blocks of a bin are folded
// onto the 8 columns in registers (an 8-point DFT with two inputs), then the usual 16 x 16 passes.
// |W|^2 lands in shared memory (aliasing the exchange tile) and the thread <-> interval interpolator
// of the wide classes brings it to the full rate.
// smem: B0[4096] (FFT ping, then exchange) | B1[256 x 17] (FFT pong, then alias tile / coarse rows) | ids
constexpr int kTileA = 256 * 17;   // alias tile: 16 columns per bin, rows padded to 17 (conflict-free, constant offsets)
constexpr size_t kWide2Smem = sizeof(float2) * (4096 + kTileA) + sizeof(int) * kMaxClassScales + 16;

// Bins 0 .. 511 of the 2048-point forward FFT of the real chunk in `a` (2048 float2, imaginary parts
// zero): five radix-4 Stockham passes (two butterflies per thread), then the last radix-2 pass only
// for the bins that are kept, straight into registers (y0 = bin tid, y1 = bin tid + 256).
__device__ __forceinline__ void smem_fft2048_forward_low(float2* a, float2* b, const float2* __restrict__ tw,
                                                         float2& y0, float2& y1) {
    constexpr int N = 2 * kChunkDec, M = N / 4;                     // 512 butterflies per pass
    const int tid = threadIdx.x;
#pragma unroll
    for (int p = 0; p < 5; ++p) {
        const int ns = 1 << (2 * p);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = tid + 256 * h;
            const int k = j & (ns - 1);
            float2 v0 = a[j], v1 = a[j + M], v2 = a[j + 2 * M], v3 = a[j + 3 * M];
            if (p > 0) {
                const int idx = k * ((kFullN / 4) / ns);            // e^{-2 pi i t k / (4 ns)} = tw[t k 4096 / (4 ns)]
                v1 = cmul(v1, __ldg(tw + idx));
                v2 = cmul(v2, __ldg(tw + 2 * idx));
                v3 = cmul(v3, __ldg(tw + 3 * idx));
            }
            dft4<-1>(v0, v1, v2, v3);
            const int j0 = ((j - k) << 2) + k;
            b[j0] = v0; b[j0 + ns] = v1; b[j0 + 2 * ns] = v2; b[j0 + 3 * ns] = v3;
        }
        __syncthreads();
        float2* t = a; a = b; b = t;
    }
    // radix-2: bin j = a[j] + e^{-2 pi i j / 2048} a[j + 1024], j < 1024; only j < 512 is needed
    y0 = cadd(a[tid], cmul(a[tid + N / 2], __ldg(tw + 2 * tid)));
    y1 = cadd(a[tid + 256], cmul(a[tid + 256 + N / 2], __ldg(tw + 2 * (tid + 256))));
}

template <int KIND, bool GUARD>
__global__ void __launch_bounds__(256, 2)
fused_wide2_kernel(const FusedParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* B0 = (float2*)smem_raw;
    float2* B1 = B0 + 4096;
    int* s_ids = (int*)(B1 + kTileA);
    float* s_pow = (float*)(s_ids + kMaxClassScales);

    const int tid = threadIdx.x;
    if (tid < 2) s_pow[tid] = 0.f;
    const int r = tid & 15;
    const int g = tid >> 4;
    const int64_t q = blockIdx.x % prm.n_chunks;
    const int64_t c = blockIdx.x / prm.n_chunks;
    const int64_t t0 = q * prm.hop - prm.offset;
    const int lu = prm.log2u;
    const int own_lo = (int)prm.offset;
    const int own_hi = (int)min(prm.offset + prm.hop, prm.n - t0);
    const int ia = own_lo >> lu, ib = (own_hi + (1 << lu) - 1) >> lu;
    if (tid < prm.n_scales) s_ids[tid] = prm.scale_ids[tid];
    const bool sample = GUARD && (q % prm.guard_every) == 0;     // accuracy guard: this chunk is measured (block-uniform)

    float2 y0, y1;                                                 // spectrum bins tid and tid + 256
    {
        constexpr int NV = 2 * kChunkDec / 256;
        const float* src = (const float*)prm.src + c * prm.src_stride - prm.src_lo;
        const int64_t i0 = t0 >> prm.log2d;                        // exact: t0 is a multiple of D
        float raw[NV];
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const int64_t u = i0 + tid + 256 * k;
            raw[k] = (u >= prm.src_lo && u < prm.src_hi) ? src[u] : 0.f;
        }
        const float cm = chunk_mean<NV>(raw, (float*)(B1 + 3072));
        if (sample)
            chunk_energy_add<NV>(raw, cm, (float*)(B1 + 3072), prm.acc + c * prm.acc_stride + kGuardLevels + prm.class_idx,
                                 prm.ech_weight);
#pragma unroll
        for (int k = 0; k < NV; ++k) B0[tid + 256 * k] = make_float2(raw[k] - cm, 0.f);
        __syncthreads();
        smem_fft2048_forward_low(B0, B1, prm.twf, y0, y1);
    }
    float2 tw[16], tw2k[8];
#pragma unroll
    for (int k = 0; k < 16; ++k) tw[k] = tw_pos(prm.twf, 16 * g * k);          // e^{2 pi i g k / 256}
#pragma unroll
    for (int k = 0; k < 8; ++k) tw2k[k] = tw_pos(prm.twf, 2 * tid * k);        // e^{2 pi i m' k / 2048}
    float* const out_c = (float*)prm.out + c * prm.c_stride + t0;
    const int align = prm.iters;                                   // 1: 16-byte, 2: 32-byte aligned rows (128- / 256-bit stores)
    float2* const A = B1;
    float2* const ex = B0;
    float* const Pc = (float*)B1;
    const int col = r & 7, sidx = r >> 3;
    unsigned own = 0;                                              // guard: owned coarse samples (g + 16 k) * 8 + col
    if (sample) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int iota = (g + 16 * k) * 8 + col;
            own |= (unsigned)(iota >= ia && iota < ib) << k;
        }
    }
    __syncthreads();                                               // the spectrum is in registers: both buffers are free
    for (int pair = 0; pair < prm.n_scales; pair += 2) {
        // the two alias blocks (bins m' and m' + 256) folded onto the 8 columns, both scales of the pass
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
            const int s = min(pair + sl, prm.n_scales - 1);
            const float2* tab = prm.table + (int64_t)s * (2 * kBins) + tid;
            const float2 z0 = cmul(y0, __ldg(tab));
            const float2 z1 = cmul(y1, __ldg(tab + kBins));
            const float h = 0.70710678118654752440f;
            const float2 zr = make_float2((z1.x - z1.y) * h, (z1.x + z1.y) * h);   // z1 e^{i pi/4}
            float2 v[8];
            v[0] = cadd(z0, z1);            v[4] = csub(z0, z1);
            v[2] = cadd(z0, mul_i<+1>(z1)); v[6] = csub(z0, mul_i<+1>(z1));
            v[1] = cadd(z0, zr);            v[5] = csub(z0, zr);
            v[3] = cadd(z0, mul_i<+1>(zr)); v[7] = csub(z0, mul_i<+1>(zr));
#pragma unroll
            for (int k = 0; k < 8; ++k)
                A[tid * 17 + sl * 8 + k] = k ? cmul(v[k], tw2k[k]) : v[k];
        }
        __syncthreads();
        float2 a[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = A[(g + 16 * i) * 17 + r];
        dft16<+1>(a);
        float2* e = ex + (g * 16) * 16 + r;
        e[0] = a[0];
#pragma unroll
        for (int k = 1; k < 16; ++k) e[k * 16] = cmul(a[k], tw[k]);
        __syncthreads();                                           // all reads of A are done: the coarse rows may overwrite it
        const float2* e2 = ex + g * 16 + r;
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = e2[k * 256];
        dft16<+1>(a);
        float* pc = Pc + sidx * kPcStride + g * 8 + col;           // coarse index (g + 16 k) * 8 + col
#pragma unroll
        for (int k = 0; k < 16; ++k) pc[k * 128] = a[k].x * a[k].x + a[k].y * a[k].y;
        if (sample) guard_pow_add<true>(a, own, s_pow + sidx);
        __syncthreads();
        if (sample && tid < 2) {                                    // the loop's closing barrier orders the reset
            if (pair + tid < prm.n_scales)
                atomicAdd(prm.pow + c * prm.pow_stride + s_ids[pair + tid], s_pow[tid] * (float)(1 << lu) * prm.pow_weight);
            s_pow[tid] = 0.f;
        }
        for (int sl = 0; sl < 2 && pair + sl < prm.n_scales; ++sl) {
            const float* pcs = Pc + sl * kPcStride;
            float* row = out_c + (int64_t)s_ids[pair + sl] * prm.s_stride;
            // (four intervals per thread at U = 4 measured slower: 1.99 vs 1.88 ms on level 2 of config 2)
            if (lu == 2) interp_rows_wide_pairs<KIND, 2, 2>(pcs, row, ia, ib, own_hi, align);
            else interp_rows_wide_pairs<KIND, 3, 2>(pcs, row, ia, ib, own_hi, align);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------- full spectrum
// smem: Yf[4096] | ex[4096] | A[256 x 17] | ids[64] | nmu[64]
constexpr size_t kFullSmem = sizeof(float2) * (2 * 4096 + kTileA) + sizeof(int) * 2 * kMaxFullScales + 16;

// radix-16 over the aliases m' + 256 mu of spectrum bin m' = tid, pruned to the first NMU
// aliases (the others are empty for a filter that occupies only NMU blocks of 256 bins)
// `tab` points at this thread's first table entry (global memory, stride 256).
template <int NMU>
__device__ __forceinline__ void full_prepass(const float2* __restrict__ Yf, const float2* __restrict__ tab,
                                             float2* __restrict__ A, const float2* tw4k) {
    const int tid = threadIdx.x;
    float2 a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k)
        a[k] = (k < NMU) ? cmul(Yf[tid + 256 * k], __ldg(tab + 256 * k)) : make_float2(0.f, 0.f);
    dft16<+1>(a);
#pragma unroll
    for (int k = 0; k < 16; ++k) A[tid * 17 + k] = k ? cmul(a[k], tw4k[k]) : a[k];
}

// The per-scale loop of the full-spectrum kernel.  MEASURE: also accumulate the output energy of every scale
// (accuracy guard); the flush path re-derives its pointer from the block index so that nothing extra stays live.
template <int KIND, bool MEASURE>
__device__ __forceinline__ void full_scale_loop(const FusedParams& prm, const float2* __restrict__ Yf, float2* __restrict__ ex,
                                                float2* __restrict__ A, const int* s_ids, const int* s_nmu, float* s_pow,
                                                const float2* tw, const float2* tw4k,
                                                typename out_elem<KIND>::type* out_c, int rel, unsigned mask) {
    const int tid = threadIdx.x;
    const int r = tid & 15;
    const int g = tid >> 4;
    for (int s = 0; s < prm.n_scales; ++s) {
        float2 a[16];
        const int nmu = s_nmu[s];
        // the table rows stream from L2 through L1: this kernel is co-limited by the LSU data pipe and
        // the issue slots, not by this latency -- staging the rows ahead of time changed nothing
        // measurable, neither with cp.async (a second LSU operation per entry) nor with a TMA bulk
        // copy + mbarrier one scale ahead (8.89 vs 8.92 ms on config 2)
        const float2* tab = prm.table + (int64_t)s * kFullN + tid;
        if (nmu == 2) full_prepass<2>(Yf, tab, A, tw4k);
        else if (nmu == 4) full_prepass<4>(Yf, tab, A, tw4k);
        else if (nmu == 8) full_prepass<8>(Yf, tab, A, tw4k);
        else full_prepass<16>(Yf, tab, A, tw4k);
        __syncthreads();
        if (MEASURE && s > 0 && tid == 0) {                          // every add for scale s - 1 came before this barrier
            atomicAdd(prm.pow + (blockIdx.x / prm.n_chunks) * prm.pow_stride + s_ids[s - 1], s_pow[(s - 1) & 1] * prm.pow_weight);
            s_pow[(s - 1) & 1] = 0.f;
        }
        // pass 1 of the 256-point transforms (16 columns)
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = A[(g + 16 * i) * 17 + r];
        dft16<+1>(a);
        float2* e = ex + (g * 16) * 16 + r;
        e[0] = a[0];
#pragma unroll
        for (int k = 1; k < 16; ++k) e[k * 16] = cmul(a[k], tw[k]);
        __syncthreads();
        const float2* e2 = ex + g * 16 + r;
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = e2[k * 256];
        dft16<+1>(a);
        store_column<KIND>(out_c + (int64_t)s_ids[s] * prm.s_stride + rel, 256, mask, a);
        if (MEASURE) guard_pow_add<false>(a, mask, s_pow + (s & 1));
        // no trailing barrier: the next scale's pre-pass writes A, whose readers all passed
        // the second barrier above; its pass 1 writes ex only after the next first barrier,
        // which every thread reaches after finishing the reads of ex just done.
    }
    if (MEASURE) {
        __syncthreads();
        const int s = prm.n_scales - 1;
        if (tid == 0) atomicAdd(prm.pow + (blockIdx.x / prm.n_chunks) * prm.pow_stride + s_ids[s], s_pow[s & 1] * prm.pow_weight);
    }
}

template <typename TIn, int KIND, bool GUARD>
__global__ void __launch_bounds__(256, 2)
fused_full_kernel(const FusedParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Yf = (float2*)smem_raw;      // order matters: the forward FFT's padded pass spills 2 KB into ex
    float2* ex = Yf + kFullN;
    float2* A = ex + kFullN;
    int* s_ids = (int*)(A + kTileA);
    int* s_nmu = s_ids + kMaxFullScales;
    float* s_pow = (float*)(s_nmu + kMaxFullScales);             // guard: two alternating output-energy counters

    const int tid = threadIdx.x;
    if (tid < 2) s_pow[tid] = 0.f;
    const int r = tid & 15;
    const int g = tid >> 4;
    const int64_t qi = blockIdx.x % prm.n_chunks;
    const int64_t c = blockIdx.x / prm.n_chunks;
    const int64_t q = prm.q_mode == 0 ? qi : (prm.q_mode == 1 ? qi * prm.guard_every : qi + qi / (prm.guard_every - 1) + 1);
    const int64_t t0 = q * prm.hop - prm.offset;

    {
        const TIn* src = (const TIn*)prm.src + c * prm.src_stride;
        const double mu = prm.means[c];
        TIn raw[kFullN / 256];                                    // all 16 loads in flight at once
        unsigned inside = 0;
#pragma unroll
        for (int k = 0; k < kFullN / 256; ++k) {
            const int64_t u = t0 + tid + 256 * k;
            const bool ok = u >= prm.src_lo && u < prm.src_hi;
            raw[k] = ok ? src[u] : (TIn)0;
            inside |= (unsigned)ok << k;
        }
        float val[kFullN / 256];
#pragma unroll
        for (int k = 0; k < kFullN / 256; ++k)                    // zero padding outside the readable range
            val[k] = (inside >> k & 1) ? (float)((double)raw[k] - mu) : 0.f;
        const float cm = chunk_mean<kFullN / 256>(val, (float*)ex + 2048);   // (behind the forward FFT's spill into ex)
        if (GUARD)
            chunk_energy_add<kFullN / 256>(val, cm, (float*)ex + 2048, prm.acc + c * prm.acc_stride + kGuardLevels + prm.class_idx,
                                           prm.ech_weight);
#pragma unroll
        for (int k = 0; k < kFullN / 256; ++k) A[tid + 256 * k] = make_float2(val[k] - cm, 0.f);
        __syncthreads();
        smem_fft4096_forward(A, Yf, prm.twf);
    }
    float2 tw[16], tw4k[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        tw[k] = tw_pos(prm.twf, 16 * g * k);                      // e^{2 pi i g k / 256}
        tw4k[k] = tw_pos(prm.twf, tid * k);                       // e^{2 pi i m' k / 4096}
    }
    typedef typename out_elem<KIND>::type OutT;
    const int rel = g * 16 + r;                                          // chunk-local sample of output k = 0
    const unsigned mask = valid_mask(rel, 8, (int)prm.offset, (int)min(prm.offset + prm.hop, prm.n - t0));
    OutT* const out_c = (OutT*)prm.out + c * prm.c_stride + t0;
    if (tid < prm.n_scales) { s_ids[tid] = prm.scale_ids[tid]; s_nmu[tid] = prm.scale_nmu[tid]; }
    // accuracy guard: the output energy of every scale is measured on every guard_every-th chunk; those chunks
    // run in a launch of their own (GUARD = true, q_mode 1) so that all the others run the plain kernel.
    __syncthreads();
    full_scale_loop<KIND, GUARD>(prm, Yf, ex, A, s_ids, s_nmu, s_pow, tw, tw4k, out_c, rel, mask);
}

// ============================================================================ driver
// The one place where a run-time output kind and guard flag become template arguments of the fused kernels:
// calls f(IntC<KIND>(), std::integral_constant<bool, GUARD>()).  COMPLEX = false for the interpolating
// kernels, which have no complex-output instance.
template <bool COMPLEX, typename F>
static void with_kind_guard(int kind, bool guard, const F& f) {
    with_kind<COMPLEX>(kind, [&](auto k) {
        if (guard) f(k, std::true_type());
        else f(k, std::false_type());
    });
}

struct LevelGeom { int64_t lo, hi, len, stride; float* ptr; };

template <typename TIn>
static int fast_run(gcwt_plan* p, const TIn* x, int in_type, int64_t n_channels, int64_t n,
                    int64_t x_stride, int64_t halo_l, int64_t halo_r, const double* d_means,
                    void* out, int64_t s_stride, int64_t c_stride, cudaStream_t st) {
    // ---- accuracy guard: per-execute accumulators ------------------------------------
    const bool guard = p->guard;
    const int acc_stride = kGuardLevels + (int)p->classes.size();
    if (guard) {
        if (p->guard_cap < n_channels) {               // (the previous execute has completed: it waited for its verdict)
            if (p->d_guard_acc) cudaFree(p->d_guard_acc);
            if (p->d_guard_pow) cudaFree(p->d_guard_pow);
            if (p->d_guard_flags) cudaFree(p->d_guard_flags);
            if (p->h_guard_flags) cudaFreeHost(p->h_guard_flags);
            p->d_guard_acc = nullptr; p->d_guard_pow = nullptr; p->d_guard_flags = p->h_guard_flags = nullptr; p->guard_cap = 0;
            GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_acc, sizeof(double) * acc_stride * n_channels));
            GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_pow, sizeof(float) * p->n_scales * n_channels));
            GCWT_CUDA_OK(cudaMalloc((void**)&p->d_guard_flags, (size_t)p->n_scales * n_channels));
            GCWT_CUDA_OK(cudaMallocHost((void**)&p->h_guard_flags, (size_t)p->n_scales * n_channels));
            p->guard_cap = n_channels;
        }
        GCWT_CUDA_OK(cudaMemsetAsync(p->d_guard_acc, 0, sizeof(double) * acc_stride * n_channels, st));
        GCWT_CUDA_OK(cudaMemsetAsync(p->d_guard_pow, 0, sizeof(float) * p->n_scales * n_channels, st));
    }
    // ---- pyramid geometry ---------------------------------------------------------
    // (the guard needs band energies two octaves below the deepest level in use: two more, tiny, levels)
    const int levels = std::max(p->max_level, 0) + ((guard && p->max_level > 0) ? 2 : 0);
    std::vector<LevelGeom> lv(levels + 1);
    lv[0].lo = -halo_l; lv[0].hi = n + halo_r;                    // [lo, hi)
    size_t total = 0;
    for (int j = 1; j <= levels; ++j) {
        const int64_t plo = lv[j - 1].lo, phi = lv[j - 1].hi - 1; // inclusive
        const int64_t lo = (int64_t)std::floor((double)(plo - kHalfbandT) / 2.0);
        const int64_t hi = (int64_t)std::ceil((double)(phi + kHalfbandT) / 2.0);
        lv[j].lo = lo; lv[j].hi = hi + 1; lv[j].len = hi - lo + 1;
        lv[j].stride = (lv[j].len + 3) & ~int64_t(3);
        total += (size_t)lv[j].stride * n_channels;
    }
    int rc = ensure_workspace(p, total * sizeof(float) + 256);
    if (rc) return rc;
    float* w = (float*)p->ws.ptr;
    for (int j = 1; j <= levels; ++j) { lv[j].ptr = w; w += lv[j].stride * n_channels; }

    const int sp_pyr = prof_begin(p, 0, st);
    for (int j = 1; j <= levels; ++j) {
        dim3 grid((unsigned)((lv[j].len + kPyrTile - 1) / kPyrTile), (unsigned)n_channels);
        double* acc = guard ? p->d_guard_acc : nullptr;
        const int64_t seg_in = (n + (int64_t(1) << (j - 1)) - 1) >> (j - 1), seg_out = (n + (int64_t(1) << j) - 1) >> j;
        if (j == 1)
            pyramid_kernel<TIn, true><<<grid, 256, 0, st>>>(x, x_stride, lv[0].lo, lv[0].hi, d_means, lv[1].ptr,
                                                            lv[1].stride, lv[1].lo, lv[1].len, acc, acc_stride, j,
                                                            seg_in, seg_out);
        else
            pyramid_kernel<float, false><<<grid, 256, 0, st>>>(lv[j - 1].ptr, lv[j - 1].stride, lv[j - 1].lo,
                                                               lv[j - 1].hi, nullptr, lv[j].ptr, lv[j].stride,
                                                               lv[j].lo, lv[j].len, acc, acc_stride, j, seg_in, seg_out);
        count_launch();
    }
    prof_end(p, sp_pyr, st);
    GCWT_CUDA_OK(cudaGetLastError());

    // ---- fused kernels ---------------------------------------------------------------
    // the thread <-> interval interpolator of fused_interp_kernel at U = 4 writes 128-bit vectors:
    // rows must be 16-byte aligned, else the class falls back to the direct kernel
    const bool rows_aligned = ((uintptr_t)out % 16 == 0) && (s_stride % 4 == 0) && (c_stride % 4 == 0);
    const bool rows_aligned32 = ((uintptr_t)out % 32 == 0) && (s_stride % 8 == 0) && (c_stride % 8 == 0);
    auto uses_interp = [&](const FastClass& fc) {
        if (fc.level < 0 || !fc.interp) return false;
        if (fc.wide) return true;                                 // fused_wide2_kernel stores scalars when it must
        return fc.log2u >= 3 || rows_aligned;
    };
    cudaStream_t full_meas_stream = nullptr;      // guard: where the measured chunks of the full-spectrum class run
    auto launch_class = [&](const FastClass& fc, cudaStream_t cs, bool own_span) -> int {
        const int sp = own_span ? prof_begin(p, fc.level < 0 ? 1 : (fc.interp ? 4 : 2), cs, fc.level + 2) : -1;
        // (an interpolated class that falls back to the direct kernel is still booked as [4])
        FusedParams prm;
        prm.means = d_means;
        prm.offset = fc.offset; prm.hop = fc.hop; prm.n = n;
        prm.n_chunks = (n + fc.hop - 1) / fc.hop;
        prm.n_scales = (int)fc.scale_ids.size();
        prm.scale_ids = fc.d_scale_ids;
        prm.table = fc.d_table;
        prm.out = out; prm.s_stride = s_stride; prm.c_stride = c_stride;
        prm.inv_nc = 1.0f / (float)fc.nc_full;
        prm.log2u = fc.log2u; prm.coef = fc.d_coef; prm.twf = p->d_twiddle; prm.scale_nmu = fc.d_scale_nmu;
        prm.q_mode = 0;
        prm.acc = guard ? p->d_guard_acc : nullptr; prm.acc_stride = acc_stride;
        prm.class_idx = (int)(&fc - p->classes.data());
        prm.pow = guard ? p->d_guard_pow : nullptr; prm.pow_stride = p->n_scales;
        // the guard measures every guard_every-th chunk of a long segment (block-uniform choice in the kernels)
        auto set_guard_sampling = [&](int64_t n_chunks, int every, double chunk_to_rate) {
            prm.guard_every = n_chunks >= 512 ? 2 * every : (n_chunks >= 256 ? every : (n_chunks >= 64 ? every / 2 : 1));
            const double w = (double)n_chunks / (double)((n_chunks + prm.guard_every - 1) / prm.guard_every);
            prm.pow_weight = (float)w;
            // chunk energy -> energy of the segment at the full rate: D samples per decimated one, chunks overlap
            prm.ech_weight = (float)(w * chunk_to_rate);
        };
        set_guard_sampling(prm.n_chunks, fc.level >= 0 ? 8 : 16,
                           (double)(fc.level >= 0 ? (int64_t(1) << fc.level) : 1) * (double)fc.hop / (double)fc.nc_full);
        if (fc.wide) {
            const LevelGeom& g = lv[fc.level];
            prm.src = g.ptr; prm.src_stride = g.stride; prm.src_lo = g.lo; prm.src_hi = g.hi;
            prm.log2d = fc.level;
            prm.offset = fc.offset2; prm.hop = fc.hop2;
            prm.n_chunks = (n + fc.hop2 - 1) / fc.hop2;
            prm.table = fc.d_table2;
            set_guard_sampling(prm.n_chunks, 8, (double)(int64_t(1) << fc.level) * (double)fc.hop2 / (double)(2 * fc.nc_full));
            prm.p_cols = 8; prm.log2p = 3; prm.units_per_chunk = 1;
            prm.iters = rows_aligned32 ? 2 : (rows_aligned ? 1 : 0);   // 256-bit / 128-bit stores allowed
            const int64_t nblk = n_channels * prm.n_chunks;
            if (nblk > 0x7fffffffLL) { set_error("fast path: grid too large"); return GCWT_ERR_UNSUPPORTED; }
            with_kind_guard<false>(p->out_kind, guard, [&](auto K, auto G) {
                fused_wide2_kernel<K, G><<<(unsigned)nblk, 256, kWide2Smem, cs>>>(prm);
            });
        } else if (uses_interp(fc)) {
            const LevelGeom& g = lv[fc.level];
            prm.src = g.ptr; prm.src_stride = g.stride; prm.src_lo = g.lo; prm.src_hi = g.hi;
            prm.log2d = fc.level;
            prm.p_cols = (int)(fc.nc_full / kBins);
            prm.log2p = ilog2_ceil(prm.p_cols);
            prm.iters = rows_aligned32 ? 2 : 1;                    // 2: rows 32-byte aligned (256-bit stores allowed)
            // enough blocks for ~6 waves of 2 x 148, but at least ~64 coarse intervals per block
            const int64_t chunks = n_channels * prm.n_chunks;
            int64_t splits = (1776 + chunks - 1) / chunks;
            // every block repeats the chunk's forward FFT and coarse transforms: only split
            // when the interpolation work per block stays several times larger
            splits = std::max<int64_t>(1, std::min<int64_t>(splits, std::max<int64_t>(1, (int64_t(1) << fc.level) / 32)));
            splits = std::min<int64_t>(splits, 24);
            prm.units_per_chunk = (int)splits;
            const int64_t nblk = chunks * splits;
            if (nblk > 0x7fffffffLL) { set_error("fast path: grid too large"); return GCWT_ERR_UNSUPPORTED; }
            with_kind_guard<false>(p->out_kind, guard, [&](auto K, auto G) {
                fused_interp_kernel<K, G><<<(unsigned)nblk, 256, kInterpSmem, cs>>>(prm);
            });
        } else if (fc.level >= 0) {
            const LevelGeom& g = lv[fc.level];
            prm.src = g.ptr; prm.src_stride = g.stride; prm.src_lo = g.lo; prm.src_hi = g.hi;
            prm.log2d = fc.level;
            prm.p_cols = (int)(fc.nc_full / kBins);
            prm.log2p = ilog2_ceil(prm.p_cols);
            const int blocks = prm.p_cols / 16;
            prm.iters = std::min(blocks, 16);
            prm.units_per_chunk = (blocks + prm.iters - 1) / prm.iters;
            const int64_t nblk = n_channels * prm.n_chunks * prm.units_per_chunk;
            if (nblk > 0x7fffffffLL) { set_error("fast path: grid too large"); return GCWT_ERR_UNSUPPORTED; }
            with_kind_guard<true>(p->out_kind, guard, [&](auto K, auto G) {
                if (prm.log2p == 4) fused_banded_kernel<K, 4, G><<<(unsigned)nblk, 256, kBandedSmem, cs>>>(prm);
                else fused_banded_kernel<K, 0, G><<<(unsigned)nblk, 256, kBandedSmem, cs>>>(prm);
            });
        } else {
            prm.src = x; prm.src_stride = x_stride; prm.src_lo = -halo_l; prm.src_hi = n + halo_r;
            prm.log2d = 0; prm.p_cols = 16; prm.log2p = 4; prm.iters = 1; prm.units_per_chunk = 1;
            const int64_t nblk = n_channels * prm.n_chunks;
            if (nblk > 0x7fffffffLL) { set_error("fast path: grid too large"); return GCWT_ERR_UNSUPPORTED; }
            const auto launch_full = [&](cudaStream_t fs, bool measure) {
                with_kind_guard<true>(p->out_kind, measure, [&](auto K, auto G) {
                    fused_full_kernel<TIn, K, G><<<(unsigned)(n_channels * prm.n_chunks), 256, kFullSmem, fs>>>(prm);
                });
            };
            if (!guard) {
                launch_full(cs, false);
            } else {
                // measured chunks (every guard_every-th) and the others in two launches of two kernels
                const int64_t n_all = prm.n_chunks, n_meas = (n_all + prm.guard_every - 1) / prm.guard_every;
                if (n_all > n_meas) {
                    prm.q_mode = 2; prm.n_chunks = n_all - n_meas;
                    launch_full(cs, false);
                    count_launch();
                }
                prm.q_mode = prm.guard_every > 1 ? 1 : 0; prm.n_chunks = n_meas;
                launch_full(full_meas_stream ? full_meas_stream : cs, true);
            }
        }
        count_launch();
        prof_end(p, sp, cs);
        return GCWT_OK;
    };

    // full-spectrum and direct classes: one after the other on the caller's stream.  With the guard on, the
    // (few) measured chunks of the full-spectrum class run as a launch of their own on a forked stream, so that
    // its partial last wave overlaps the main launch instead of extending it (serial when profiling per family).
    bool side0_pending = false;
    if (guard && !p->profile && getenv("GCWT_STREAMS") == nullptr) {
        if (!p->side_stream[0]) {
            GCWT_CUDA_OK(cudaStreamCreateWithFlags(&p->side_stream[0], cudaStreamNonBlocking));
            GCWT_CUDA_OK(cudaEventCreateWithFlags(&p->ev_join[0], cudaEventDisableTiming));
        }
        if (!p->ev_fork) GCWT_CUDA_OK(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
        GCWT_CUDA_OK(cudaEventRecord(p->ev_fork, st));
        GCWT_CUDA_OK(cudaStreamWaitEvent(p->side_stream[0], p->ev_fork, 0));
        full_meas_stream = p->side_stream[0];
        side0_pending = true;
    }
    int n_group = 0;
    for (const FastClass& fc : p->classes) {
        if (uses_interp(fc)) { ++n_group; continue; }
        rc = launch_class(fc, st, true);
        if (rc) return rc;
    }
    // interpolated classes: independent launches (disjoint output rows, read-only inputs) of 5-20 waves
    // each.  They are dealt to two streams that fork from and join `st`, so that the tail of one launch
    // overlaps the head of the next (+1 % on config 2, +2.4 % on config 3 with its 8 tiles); the
    // profiling span covers the whole group.  GCWT_STREAMS=1 (or per-class timing) serialises them.
    if (n_group > 0) {
        int n_streams = 2;
        if (const char* e = getenv("GCWT_STREAMS")) n_streams = std::max(1, std::min(1 + gcwt_plan::kSideStreams, atoi(e)));
        const bool per_class = p->profile && getenv("GCWT_CLASS_TIMES") != nullptr;
        if (per_class || n_group < 2) n_streams = 1;
        const int n_side = n_streams - 1;
        for (int k = 0; k < n_side; ++k) {
            if (!p->side_stream[k]) {
                GCWT_CUDA_OK(cudaStreamCreateWithFlags(&p->side_stream[k], cudaStreamNonBlocking));
                GCWT_CUDA_OK(cudaEventCreateWithFlags(&p->ev_join[k], cudaEventDisableTiming));
            }
        }
        if (n_side > 0 && !p->ev_fork) GCWT_CUDA_OK(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
        const int sp = per_class ? -1 : prof_begin(p, 4, st, 63);
        if (n_side > 0) {
            GCWT_CUDA_OK(cudaEventRecord(p->ev_fork, st));
            for (int k = 0; k < n_side; ++k) GCWT_CUDA_OK(cudaStreamWaitEvent(p->side_stream[k], p->ev_fork, 0));
        }
        int ci = 0;
        for (const FastClass& fc : p->classes) {
            if (!uses_interp(fc)) continue;
            const int slot = ci++ % n_streams;
            rc = launch_class(fc, slot ? p->side_stream[slot - 1] : st, per_class);
            if (rc) return rc;
        }
        for (int k = 0; k < n_side; ++k) {
            GCWT_CUDA_OK(cudaEventRecord(p->ev_join[k], p->side_stream[k]));
            GCWT_CUDA_OK(cudaStreamWaitEvent(st, p->ev_join[k], 0));
            if (k == 0) side0_pending = false;
        }
        prof_end(p, sp, st);
    }
    if (side0_pending) {
        GCWT_CUDA_OK(cudaEventRecord(p->ev_join[0], p->side_stream[0]));
        GCWT_CUDA_OK(cudaStreamWaitEvent(st, p->ev_join[0], 0));
    }
    GCWT_CUDA_OK(cudaGetLastError());
    return GCWT_OK;
}

// ---- accuracy guard: verdict per (channel, scale) -----------------------------------------------
__global__ void guard_eval_kernel(int n_scales, const ScaleInfo* __restrict__ scales, const float* __restrict__ gain,
                                  const float* __restrict__ q, const int32_t* __restrict__ cls,
                                  const double* __restrict__ acc, int acc_stride, const float* __restrict__ pow,
                                  double tol2, unsigned char* __restrict__ flags) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (s >= n_scales) return;
    unsigned char flag = 0;
    const int ci = cls[s];
    if (ci >= 0) {
        const double* a = acc + (int64_t)c * acc_stride;
        const int lev = scales[s].level;
        const double eps = 5.9604644775390625e-08;                // 2^-24
        const double qs = (double)q[s];
        // rounding of the chunk transform against the (mean-removed) energy of the chunks
        double bound = (kGuardKRound * eps) * (kGuardKRound * eps) * qs * a[kGuardLevels + ci];
        if (lev >= 0) {
            // a[j] is the plain sum of squares of level j: its energy at the full rate is 2^j times that
            const float* gs = gain + (int64_t)s * kGuardSlots;
            for (int b = 0; b <= lev; ++b) {
                const double e_lo = b + 2 < kGuardLevels ? ldexp(a[b + 2], b + 2) : 0.0;
                const double eb = fmax(ldexp(a[b], b) - e_lo, 0.0);  // octave b (two octaves wide: the transition bands smear)
                bound += (double)gs[b] * eb;
            }
            if (lev + 1 < kGuardLevels) bound += (double)gs[lev + 1] * ldexp(a[lev + 1], lev + 1);
            double stage = 0.0;                                    // storage rounding of the pyramid's stages
            for (int j = 1; j <= lev; ++j) stage += ldexp(a[j], j + j - lev);
            bound += (kGuardKStage * eps) * (kGuardKStage * eps) * qs * stage / 3.0;
        }
        flag = bound > tol2 * (double)pow[(int64_t)c * n_scales + s];
    }
    flags[(int64_t)c * n_scales + s] = flag;
}

int guard_resolve(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                  int64_t x_stride, int64_t halo_l, int64_t halo_r, const double* d_means,
                  void* out, int64_t s_stride, int64_t c_stride, cudaStream_t st) {
    if (!p->guard) return GCWT_OK;
    const int S = p->n_scales;
    const int acc_stride = kGuardLevels + (int)p->classes.size();
    guard_eval_kernel<<<dim3((S + 127) / 128, (unsigned)n_channels), 128, 0, st>>>(
        S, p->d_scales, p->d_guard_gain, p->d_guard_q, p->d_guard_class, p->d_guard_acc, acc_stride, p->d_guard_pow,
        p->guard_tol * p->guard_tol, p->d_guard_flags);
    count_launch();
    GCWT_CUDA_OK(cudaMemcpyAsync(p->h_guard_flags, p->d_guard_flags, (size_t)S * n_channels, cudaMemcpyDeviceToHost, st));
    GCWT_CUDA_OK(cudaEventRecord(p->ev_guard, st));
    GCWT_CUDA_OK(cudaEventSynchronize(p->ev_guard));
    p->guard_last = 0;
    p->guard_checked += (int64_t)S * n_channels;
    std::fill(p->guard_last_flags.begin(), p->guard_last_flags.end(), 0);
    const size_t in_el = in_type == GCWT_F32 ? 4 : 8;
    const size_t out_el = p->out_kind == GCWT_OUT_COMPLEX ? 8 : 4;
    if (getenv("GCWT_GUARD_DUMP")) {       // developer aid: what made the guard fire, per flagged pair (first 12)
        std::vector<double> a((size_t)acc_stride * n_channels);
        std::vector<float> pw((size_t)S * n_channels);
        cudaMemcpy(a.data(), p->d_guard_acc, sizeof(double) * a.size(), cudaMemcpyDeviceToHost);
        cudaMemcpy(pw.data(), p->d_guard_pow, sizeof(float) * pw.size(), cudaMemcpyDeviceToHost);
        int shown = 0;
        const double eps = 5.9604644775390625e-08;
        for (int64_t c = 0; c < n_channels && shown < 12; ++c)
            for (int s2 = 0; s2 < S && shown < 12; ++s2) {
                if (!p->h_guard_flags[c * S + s2]) continue;
                ++shown;
                const double* ac = a.data() + c * acc_stride;
                const int lev = p->scales[s2].level, ci = [&] { for (size_t k = 0; k < p->classes.size(); ++k) for (int id : p->classes[k].scale_ids) if (id == s2) return (int)k; return 0; }();
                const double P = pw[c * S + s2], qs = p->guard_q_h[s2];
                fprintf(stderr, "gcwt guard: n=%lld ch %lld scale %d level %d L %lld: P %.3e  round %.2e", (long long)n_samples, (long long)c, s2, lev,
                        (long long)p->scales[s2].L, P, std::sqrt(kGuardKRound * eps * kGuardKRound * eps * qs * ac[kGuardLevels + ci] / P));
                if (lev >= 0) {
                    double stage = 0.0;
                    for (int j = 1; j <= lev; ++j) stage += std::ldexp(ac[j], j + j - lev);
                    fprintf(stderr, "  stage %.2e  band:", std::sqrt(kGuardKStage * eps * kGuardKStage * eps * qs * stage / 3.0 / P));
                    for (int b = 0; b <= lev + 1; ++b) {
                        const double e_lo = (b <= lev && b + 2 < kGuardLevels) ? std::ldexp(ac[b + 2], b + 2) : 0.0;
                        const double eb = std::max(std::ldexp(ac[b], b) - e_lo, 0.0);
                        fprintf(stderr, " %.1e", std::sqrt(p->guard_gain_h[(size_t)s2 * kGuardSlots + b] * eb / P));
                    }
                }
                fprintf(stderr, "\n");
            }
    }
    // runs of consecutive channels with the same failing scales are re-computed together
    std::vector<int> ids, run_ids;
    int64_t run_start = 0;
    for (int64_t c = 0; c <= n_channels; ++c) {
        ids.clear();
        if (c < n_channels)
            for (int s2 = 0; s2 < S; ++s2)
                if (p->h_guard_flags[c * S + s2]) { ids.push_back(s2); p->guard_last_flags[s2] = 1; }
        p->guard_last += (int64_t)ids.size();
        if (c < n_channels && c > run_start && ids == run_ids) continue;
        if (c > run_start && !run_ids.empty()) {
            const int sp = prof_begin(p, 3, st);
            int rc = generic_execute(p, run_ids, (const char*)x + in_el * run_start * x_stride, in_type, c - run_start, n_samples,
                                     x_stride, halo_l, halo_r, d_means + run_start, (char*)out + out_el * run_start * c_stride,
                                     s_stride, c_stride, st);
            prof_end(p, sp, st);
            if (rc) return rc;
        }
        run_start = c;
        run_ids = ids;
    }
    p->guard_total += p->guard_last;
    return GCWT_OK;
}

static std::atomic<bool> g_device_ready[64];

int prepare_device(int device) {
    if (g_device_ready[device & 63]) return GCWT_OK;
    std::vector<SmemKernel> big = fourstep_kernels();
    for (int kind = GCWT_OUT_COMPLEX; kind <= GCWT_OUT_POWER; ++kind)
        for (bool guard : {false, true})
            with_kind_guard<true>(kind, guard, [&](auto K, auto G) {
                big.push_back({(const void*)fused_banded_kernel<K, 0, G>, kBandedSmem});
                big.push_back({(const void*)fused_banded_kernel<K, 4, G>, kBandedSmem});
                big.push_back({(const void*)fused_full_kernel<float, K, G>, kFullSmem});
                big.push_back({(const void*)fused_full_kernel<double, K, G>, kFullSmem});
                if constexpr (K != GCWT_OUT_COMPLEX) {
                    big.push_back({(const void*)fused_interp_kernel<K, G>, kInterpSmem});
                    big.push_back({(const void*)fused_wide2_kernel<K, G>, kWide2Smem});
                }
            });
    for (const SmemKernel& k : big) {
        const cudaError_t e = cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.bytes);
        if (e != cudaSuccess) { set_error(std::string("shared-memory limit of a kernel: ") + cudaGetErrorString(e)); return GCWT_ERR_CUDA; }
    }
    int rc = upload_constants();
    if (rc) return rc;
    g_device_ready[device & 63] = true;
    return GCWT_OK;
}

int fast_execute(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                 int64_t x_stride, int64_t halo_l, int64_t halo_r, const double* d_means, void* out,
                 int64_t s_stride, int64_t c_stride, cudaStream_t st) {
    if (in_type == GCWT_F32)
        return fast_run<float>(p, (const float*)x, in_type, n_channels, n_samples, x_stride, halo_l, halo_r,
                               d_means, out, s_stride, c_stride, st);
    return fast_run<double>(p, (const double*)x, in_type, n_channels, n_samples, x_stride, halo_l, halo_r,
                            d_means, out, s_stride, c_stride, st);
}

}  // namespace gcwt
