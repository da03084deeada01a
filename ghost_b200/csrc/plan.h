// Internal plan representation shared by the path drivers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>
#include "../../include/ghost_cwt.h"

namespace gcwt {

constexpr int kBins = 256;          // spectrum bins kept per chunk by the band-limited path
constexpr int kChunkDec = 1024;     // chunk length in decimated samples (forward FFT size)
constexpr int kFullN = 4096;        // chunk length of the full-spectrum fused kernel
constexpr int kMaxClassScales = 16; // scales handled by one fused launch (shared-memory table)
constexpr int kMinFastLevel = 2;    // P = kChunkDec * 2^level / kBins must be >= 16
constexpr int kInterpT = 8;         // taps of the polyphase interpolator (amplitude / power output)
constexpr int kInterpMinLevel = 3;  // interpolated classes: coarse spacing U = 2^(level-1) >= 4
constexpr int kCoarse = 2048;       // coarse |W|^2 samples per chunk and scale (8 columns x 256)
constexpr int kWideT = 12;          // taps of the interpolator of the wide-spacing classes (U = D)
constexpr int kWideMaxLevel = 3;    // levels 2 and 3 use U = D when their bands allow it
constexpr double kInterpMinOs = 4.0; // |W|^2 over-sampling guaranteed on the grid U = D/2 (band <= kBins bins)
constexpr double kWideMinOs = 2.5;   // over-sampling required of a class before it may use U = D
constexpr int kHalfbandT = 19;      // half-band taps run from -T..T
constexpr int kHalfbandOdd = (kHalfbandT + 1) / 2;

struct ScaleInfo {                  // mirrored on the device (generic path)
    int64_t L;
    int32_t k_first;
    int32_t n_terms;
    int32_t term_off;
    int32_t level;                  // >=0 fast level, -1 full fused, -2 generic
};

struct FastClass {
    int level = 0;                  // -1: full-spectrum kernel at full rate
    int64_t nc_full = 0;            // chunk length in full-rate samples
    int64_t lmax = 0;
    int64_t offset = 0;             // first owned chunk-local sample
    int64_t hop = 0;                // owned samples per chunk
    std::vector<int> scale_ids;     // global scale indices, <= kMaxClassScales
    // banded: float2 [n][kBins] (response / decimator, incl. 1/kChunkDec)
    // full:   float2 [n][kFullN] (response incl. 1/kFullN)
    // (null for wide classes, which read d_table2)
    float2* d_table = nullptr;
    int32_t* d_scale_ids = nullptr;
    // amplitude / power at level >= kInterpMinLevel: |W|^2 on a grid of spacing U = 2^log2u,
    // then a kInterpT-tap polyphase interpolator; d_coef is float [U][kInterpT] (not wide classes)
    std::vector<int> scale_nmu;     // full-spectrum kernel: occupied 256-bin blocks per scale (2, 4, 8, 16)
    int32_t* d_scale_nmu = nullptr;
    bool interp = false;
    bool wide = false;              // coarse spacing U = D (4 columns), kWideT taps; else U = D/2, kInterpT taps
    // wide classes run on chunks of 2 * kChunkDec decimated samples with 2 * kBins bins kept
    // (fused_wide2_kernel): own table [n][2 kBins] and overlap-save geometry
    float2* d_table2 = nullptr;
    int64_t offset2 = 0, hop2 = 0;
    int log2u = 0;
    float* d_coef = nullptr;
};

// ---- execute-time accuracy guard (fp32 plans) -------------------------------------------------
// The band-limited classes drop each filter's response outside the kept band (band_tol) and rely on a
// decimator with a finite stop band, and every fp32 class rounds against the energy of the chunk it
// transforms; all three are harmless unless the recording holds far more energy outside a scale's band
// than inside it.  Per (channel, scale) the guard compares a bound on that error, built from measured
// octave-band energies, with the measured output energy, and re-computes the pairs that fail in fp64.
constexpr int kGuardSlots = 18;     // octave slots b = 0 .. level + 1 of the per-scale error gains
constexpr int kGuardLevels = 20;    // pyramid energies e_0 .. e_(max_level + 2)
constexpr double kGuardKRound = 6.0;   // chunk-transform rounding: err^2 <= (k eps)^2 q E_chunk   (measured 1 .. 4.7)
constexpr double kGuardKStage = 2.0;   // pyramid storage rounding: err^2 <= (k eps)^2 q sum_j E_j 2^(j-l) / 3 (measured ~1)

struct Workspace {
    void* ptr = nullptr;
    size_t bytes = 0;
};

// ---- scale-averaged band power (gcwt_band_reduce, gcwt_execute_host_bands) ---------------------
// Band b sums rows first[b] .. first[b] + count[b] - 1 with weights w[off[b] + k].  The table is passed to
// the kernel by value (__grid_constant__), so a call needs no allocation and no host-to-device copy.
constexpr int kMaxBands = 64;
constexpr int kMaxBandEntries = 1024;   // sum of count[b]
struct BandTable {
    int32_t n_bands;
    int32_t rows;                       // max(first[b] + count[b]): rows of a channel the bands read
    int32_t first[kMaxBands], count[kMaxBands], off[kMaxBands];
    double w[kMaxBandEntries];
};

}  // namespace gcwt

struct gcwt_plan {
    int n_scales = 0;
    int compute_type = GCWT_F32;
    int out_kind = GCWT_OUT_AMPLITUDE;
    int device = 0;
    int flags = 0;
    double band_tol = 1e-7;
    std::vector<gcwt::ScaleInfo> scales;
    std::vector<double> terms;
    gcwt::ScaleInfo* d_scales = nullptr;
    double* d_terms = nullptr;
    std::vector<gcwt::FastClass> classes;   // fp32 fused-kernel groups
    std::vector<int> generic_ids;           // scales served by the generic path
    int max_level = 0;
    double halfband_odd[gcwt::kHalfbandOdd];  // h[1], h[3], ... (h[0] = 0.5)
    gcwt::Workspace ws;
    bool profile = false;
    struct Span { cudaEvent_t a, b; int kind; int launches; int tag; };
    std::vector<Span> spans;
    double prof_ms[GCWT_PROFILE_KINDS] = {0, 0, 0, 0, 0};
    double class_ms[64] = {0};              // per scale class (level + 2), printed when GCWT_CLASS_TIMES is set
    int64_t prof_launches[GCWT_PROFILE_KINDS] = {0, 0, 0, 0, 0};
    float2* d_twiddle = nullptr;            // e^{-2 pi i k / 4096}, k < 4096 (forward FFTs of the fused kernels)
    double* d_means = nullptr;              // internal per-channel means
    size_t means_bytes = 0;
    static constexpr int kSideStreams = 3;
    cudaStream_t side_stream[kSideStreams] = {nullptr, nullptr, nullptr};   // forked streams of the interpolated classes
    cudaEvent_t ev_fork = nullptr, ev_join[kSideStreams] = {nullptr, nullptr, nullptr};
    double* d_partial = nullptr;            // scratch of the mean reduction
    size_t partial_bytes = 0;
    // accuracy guard: plan-time tables (per scale) and per-execute accumulators (per channel)
    bool guard = false;
    double guard_tol = 5e-6;
    float* d_guard_gain = nullptr;          // [n_scales][kGuardSlots] squared error gain per octave slot
    float* d_guard_q = nullptr;             // [n_scales] mean |H|^2 over the chunk grid
    int32_t* d_guard_class = nullptr;       // [n_scales] index into classes (-1: not guarded)
    double* d_guard_acc = nullptr;          // [channels][kGuardLevels + n_classes] band and chunk energies
    float* d_guard_pow = nullptr;           // [channels][n_scales] measured output energy
    unsigned char* d_guard_flags = nullptr; // [channels][n_scales]
    unsigned char* h_guard_flags = nullptr; // pinned copy
    int64_t guard_cap = 0;                  // channels the accumulators are sized for
    cudaEvent_t ev_guard = nullptr;
    int64_t guard_last = 0, guard_total = 0, guard_checked = 0;   // re-computed (channel, scale) pairs
    std::vector<unsigned char> guard_last_flags;                  // any-channel flag per scale of the last call
    std::vector<float> guard_gain_h, guard_q_h;                   // host copies of the tables (diagnostics)
    // fp64 four-step path: twiddle tables and the cache of filter responses (transposed order) for one nfft
    double2* d_tw1k = nullptr;              // e^{-2 pi i j / 1024}
    double2* d_tw_fine = nullptr;           // e^{-2 pi i j / nfft}, j < 1024
    int64_t tw_fine_n = 0;
    double2* d_hcache = nullptr;            // [n_scales][nfft]
    int64_t hcache_n = 0;
    // host-buffer path (gcwt_execute_host*): persistent staging, grown on demand
    struct HostStage {
        void* d_in = nullptr; size_t in_bytes = 0;                            // the channel group's samples
        void* d_out[2] = {nullptr, nullptr}; size_t out_bytes[2] = {0, 0};    // double-buffered full-rate tiles
        void* d_red[2] = {nullptr, nullptr}; size_t red_bytes[2] = {0, 0};    // reduced tiles: pooled bins or band rows
        void* h_ring[2] = {nullptr, nullptr}; size_t ring_bytes[2] = {0, 0};  // pinned ring (pageable destinations only)
        double* d_means = nullptr; size_t means_bytes = 0;
        double* d_acc = nullptr; size_t acc_bytes = 0;                         // event sums of a channel group
        int64_t* d_events = nullptr; size_t events_bytes = 0;                  // the event samples of a call
        cudaStream_t st_compute = nullptr, st_copy = nullptr;
        cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
        double last_ms[4] = {0, 0, 0, 0};                   // wall, h2d, tiles, bytes out (diagnostics)
    } host;
};

namespace gcwt {
int ensure_workspace(gcwt_plan* p, size_t bytes);
// grow-on-demand buffers: when *have < need, free *ptr and allocate `need` bytes (the contents are not kept);
// `who` prefixes the error text
int grow_device(void** ptr, size_t* have, size_t need, const char* who);
int grow_pinned(void** ptr, size_t* have, size_t need, const char* who);
void count_launch(int n = 1);
int64_t launches_so_far();
// RAII-less profiling span: begin returns an index (or -1 when profiling is off)
int prof_begin(gcwt_plan* p, int kind, cudaStream_t st, int tag = 0);
void prof_end(gcwt_plan* p, int idx, cudaStream_t st);

// a kernel launched with more dynamic shared memory than the 48 KB default, and the bytes it is launched with
struct SmemKernel { const void* fn; size_t bytes; };
std::vector<SmemKernel> fourstep_kernels();   // the four-step FFT kernels of the generic path
// Once per device, from gcwt_plan_create: the shared-memory limit of every such kernel of both paths, and the
// fused kernels' filter taps in constant memory.  Both are per device and do not depend on the plan.
int prepare_device(int device);

// path drivers (each returns a GCWT_* code)
int generic_execute(gcwt_plan* p, const std::vector<int>& ids, const void* x, int in_type,
                    int64_t n_channels, int64_t n_samples, int64_t x_stride,
                    int64_t halo_l, int64_t halo_r, const double* d_means,
                    void* out, int64_t s_stride, int64_t c_stride, cudaStream_t st);
int guard_resolve(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                  int64_t x_stride, int64_t halo_l, int64_t halo_r, const double* d_means,
                  void* out, int64_t s_stride, int64_t c_stride, cudaStream_t st);
int fast_execute(gcwt_plan* p, const void* x, int in_type,
                 int64_t n_channels, int64_t n_samples, int64_t x_stride,
                 int64_t halo_l, int64_t halo_r, const double* d_means,
                 void* out, int64_t s_stride, int64_t c_stride, cudaStream_t st);
int interp_taps(int log2u, int n_taps, double os, float* out);   // host: the interpolator design
int fast_plan_build(gcwt_plan* p);       // classify scales + upload tables (fp32 plans)
void fast_plan_free(gcwt_plan* p);
int means_blocks(int64_t n_samples);
int means_launch(const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                 int64_t x_stride, double* d_means, double* partial, cudaStream_t st);
int host_execute(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n_samples, int64_t x_stride,
                 const int64_t* epochs, int n_epochs, const double* means_host, void* out, int64_t s_stride,
                 int64_t c_stride, int64_t pool_width = 0, int pool_mode = 0, const BandTable* bands = nullptr);
int pool_rows_launch(const void* x_dev, int type, int64_t n_rows, int64_t n_cols, int64_t row_stride, int64_t width,
                     int mode, int square, double* out_dev, int64_t out_stride, cudaStream_t st);
// host-side checks of a band table (NULL pointers, 1..kMaxBands bands, count >= 1, first >= 0, at most
// kMaxBandEntries entries); `who` prefixes the error text.  Ranges against the scale count are the caller's.
int band_table_build(int n_bands, const int32_t* first, const int32_t* count, const double* weights, BandTable* tab,
                     const char* who);
// out[c, b, n] = sum_k w[off_b + k] |x[c, first_b + k, n]|^2 in fp64, written as `type`; x holds elements of
// `type` (float2 / double2 for kind GCWT_OUT_COMPLEX), strides in elements, out strides in real elements
int band_reduce_launch(const void* x_dev, int type, int kind, int64_t n_channels, int64_t n_samples, int64_t s_stride,
                       int64_t c_stride, const BandTable& tab, void* out_dev, int64_t out_b_stride, int64_t out_c_stride,
                       cudaStream_t st);
// acc_power[c, s, l] += sum_e |x[c, s, events[e] + lag_first + l - sample0]|^2 and, when acc_phase is not NULL
// (complex kinds only), acc_phase[c, s, l] += sum_e W / |W|, in fp64, over the events whose sample lies inside
// [0, n_samples); x strides in elements of `type` (float2 / double2 for complex), acc strides in elements
int event_reduce_launch(const void* x_dev, int type, int kind, int64_t n_channels, int n_scales, int64_t n_samples,
                        int64_t s_stride, int64_t c_stride, int64_t sample0, const int64_t* events_dev, int64_t n_events,
                        int64_t lag_first, int64_t n_lags, double* acc_power, double2* acc_phase, int64_t as_stride,
                        int64_t ac_stride, cudaStream_t st);
// host-side checks of gcwt_execute_host_events, run before any device work: the epochs as gcwt_execute_host checks
// them, events ascending, and every window [e + lag_first, e + lag_first + n_lags) inside one epoch
int check_event_args(int64_t n_samples, const int64_t* epochs, int n_epochs, const int64_t* events, int64_t n_events,
                     int64_t lag_first, int64_t n_lags);
// the events' arguments have passed check_event_args
int host_execute_events(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n_samples,
                        int64_t x_stride, const int64_t* epochs, int n_epochs, const double* means_host,
                        const int64_t* events, int64_t n_events, int64_t lag_first, int64_t n_lags, double* power_out,
                        double* phase_out, int64_t out_s_stride, int64_t out_c_stride);
void host_stage_free(gcwt_plan* p);
}  // namespace gcwt
