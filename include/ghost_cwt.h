/* ghost_cwt.h -- C ABI of the B200-native Morse-wavelet CWT hot path.
 *
 * The reference (nelpy/ghost) has no FFI: its boundary for this path is the Python
 * class ghost.wave.ContinuousWaveletTransform.  Inside transform() there are exactly
 * two seams, and this ABI replaces what sits behind them:
 *
 *   kernel, _ = wv(length)                       ghost/wave/transforms.py:197
 *       -> Morse.__call__                        ghost/wave/morse.py:53-91
 *       -> morsewave / _morsewave                ghost/wave/morseutils.py:22-151
 *   res = convfun(x[start:stop], kernel)         ghost/wave/transforms.py:203
 *       -> fastconv_scipy / fastconv_fftw        ghost/sigtools/convolution.py:16-216
 *   out_array[idx, start:stop] = np.abs(res)     ghost/wave/transforms.py:204
 *
 * plus the mean removal (transforms.py:142-143).  The frequency grid and the per-scale
 * tap counts L stay on the host in float64 with the reference's operation order
 * (transforms.py:147-182, morse.py:93-122) because they must be bit-identical; they are
 * passed in through gcwt_plan_desc together with the non-zero samples X[k] of each
 * scale's L-point Morse spectrum (morseutils.py:129-133,178).
 *
 * Threading: a plan owns its workspace, per-call accumulators, side streams and staging buffers, so it
 * serves ONE gcwt_execute / gcwt_execute_host at a time (calls on one plan from several threads or
 * streams must be serialised by the caller; different plans are independent).  Every entry point
 * selects the plan's device and restores the caller's current device before returning.
 *
 * All functions return 0 on success or a negative GCWT_ERR_* code; the message for the
 * last failure on the calling thread is available from gcwt_last_error().  There is no
 * CPU fallback: every entry point that computes needs a CUDA device.
 */
#ifndef GHOST_CWT_H
#define GHOST_CWT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCWT_VERSION 200

/* error codes */
#define GCWT_OK            0
#define GCWT_ERR_ARG      -1
#define GCWT_ERR_CUDA     -2
#define GCWT_ERR_NOMEM    -3
#define GCWT_ERR_UNSUPPORTED -4

/* element types */
#define GCWT_F32 0
#define GCWT_F64 1

/* what the epilogue writes (kernel (3) of the design): the reference stores |W|
 * (transforms.py:204); power is amplitude**2 (transforms.py:507-510); complex is the
 * value before np.abs. */
#define GCWT_OUT_COMPLEX   0
#define GCWT_OUT_AMPLITUDE 1
#define GCWT_OUT_POWER     2

/* plan flags */
#define GCWT_FLAG_FORCE_GENERIC 1   /* fp32 only: skip the band-limited fast path */
#define GCWT_FLAG_NO_INTERP     2   /* fp32 amplitude/power: compute every output sample with the pruned
                                       inverse FFT instead of coarse grid + polyphase interpolation */

#define GCWT_FLAG_NO_GUARD      4   /* fp32 only: skip the execute-time accuracy guard (see gcwt_guard_stats) */

typedef struct gcwt_plan gcwt_plan;

typedef struct gcwt_plan_desc {
    int32_t        n_scales;
    const int64_t *lengths;      /* [n_scales] tap count L per scale (morse.py:108-122)          */
    const int32_t *k_first;      /* [n_scales] first L-grid bin with a non-zero spectrum sample   */
    const int32_t *n_terms;      /* [n_scales] number of consecutive non-zero samples             */
    const double  *terms;        /* concatenated X[k] values, sum(n_terms) doubles                */
    int32_t        compute_type; /* GCWT_F32 or GCWT_F64: arithmetic and output element type      */
    int32_t        out_kind;     /* GCWT_OUT_*                                                    */
    int32_t        device;       /* CUDA device ordinal                                           */
    int32_t        flags;        /* GCWT_FLAG_*                                                   */
    double         band_tol;     /* fp32 fast path: allowed out-of-band filter energy (amplitude
                                    ratio); 0 selects the default 1e-7                            */
    double         guard_tol;    /* fp32 accuracy guard: largest tolerated bound on a scale's relative
                                    L2 error before it is re-computed in fp64; 0 selects 5e-6      */
} gcwt_plan_desc;

/* Build device tables for a set of scales.  Replaces the per-scale kernel synthesis
 * Morse.__call__ (morse.py:53-91). */
int gcwt_plan_create(gcwt_plan **out, const gcwt_plan_desc *desc);
int gcwt_plan_destroy(gcwt_plan *plan);

/* Introspection: per scale, the decimation level the planner chose (>= 0: band-limited
 * fast path at 2**level; -1: full-spectrum fused kernel; -2: generic global-memory path). */
int gcwt_plan_levels(const gcwt_plan *plan, int32_t *levels_out);

/* Introspection: the scale classes of an fp32 plan's fused kernels (one fused launch each; the guard
 * splits the full-spectrum launch in two on long segments).  The planner forms classes from band widths
 * it measures on the device, so this is the only way to see them.  kernel is the kernel as planned: at
 * execute time an interpolated class with log2u == 2 falls back to the banded kernel when the output rows
 * are not 16-byte aligned.  chunk, offset and hop describe the chunk that kernel transforms (full-rate
 * samples): a wide-interpolation class runs on chunks of twice its level's 1024 << level samples.
 *   n_classes       number of classes (0 for fp64 plans and plans of generic scales only)
 *   info            optional [*n_classes] records
 *   class_of_scale  optional [n_scales]: index into info, -1 for a scale of the generic path */
#define GCWT_KERNEL_FULL   0   /* fused_full_kernel: full spectrum at the full rate (level -1)      */
#define GCWT_KERNEL_BANDED 1   /* fused_banded_kernel: pruned inverse FFT of every output sample   */
#define GCWT_KERNEL_INTERP 2   /* fused_interp_kernel: |W|^2 on a grid of 2**log2u + interpolator  */
#define GCWT_KERNEL_WIDE2  3   /* fused_wide2_kernel: levels 2-3, spacing U = 2**level, 2x chunks  */
typedef struct gcwt_class_info {
    int32_t level;      /* >= 2: band-limited at decimation 2**level; -1: full spectrum              */
    int32_t kernel;     /* GCWT_KERNEL_*                                                             */
    int32_t log2u;      /* coarse spacing of the interpolated kernels (0 for full and banded)         */
    int32_t n_scales;   /* scales of the class (<= 16; <= 64 for the full-spectrum class)             */
    int64_t chunk;      /* chunk length in full-rate samples                                          */
    int64_t offset;     /* first chunk-local sample a chunk owns                                      */
    int64_t hop;        /* samples owned per chunk: chunk q owns [q hop, (q + 1) hop) of the segment  */
} gcwt_class_info;
int gcwt_plan_classes(const gcwt_plan *plan, int32_t *n_classes, gcwt_class_info *info,
                      int32_t *class_of_scale);

/* Transform one contiguous segment (an epoch, or one rank's time shard) of n_channels
 * channels.  Replaces, for every scale, convfun(x[start:stop], kernel) followed by
 * np.abs (transforms.py:202-204), i.e. a zero-padded 'same' linear convolution.
 *
 *   x            device pointer to sample 0 of channel 0 of the segment; element type in_type
 *   x_stride     elements between channels
 *   halo_left / halo_right
 *                number of REAL samples readable before x[0] / after x[n_samples-1] in each
 *                channel (0 at true signal or epoch edges, where the reference zero-pads;
 *                > 0 for time shards so that shard seams carry no edge effect)
 *   means        device pointer to one double per channel that is subtracted from every
 *                sample (the reference removes the GLOBAL mean, transforms.py:143), or NULL
 *                to use the mean of the segment itself
 *   out          device pointer; coefficient (c, s, n) is written at
 *                out[c * out_channel_stride + s * out_scale_stride + n] in units of the
 *                output element (float/double, or float2/double2 for GCWT_OUT_COMPLEX)
 *   stream       cudaStream_t (may be NULL for the default stream)
 */
int gcwt_execute(gcwt_plan *plan, const void *x, int32_t in_type,
                 int64_t n_channels, int64_t n_samples, int64_t x_stride,
                 int64_t halo_left, int64_t halo_right, const double *means,
                 void *out, int64_t out_scale_stride, int64_t out_channel_stride,
                 void *stream);

/* The whole transform body for HOST buffers: what transform() does between `input_asarray -= mean`
 * and `self._amplitude = out_array` (ghost/wave/transforms.py:142-143, 185, 202-204, 231).
 *
 *   x             host pointer, n_channels rows of n_samples (x_stride elements apart); never written
 *   epoch_bounds  n_epochs pairs [start, stop) of sample indices, ascending; every epoch is convolved on
 *                 its own with zero padding (transforms.py:202-204) and samples outside all epochs are
 *                 zero in the result.  NULL / 0: one epoch [0, n_samples)
 *   means_host    one double per channel, or NULL for each channel's mean over all n_samples
 *                 (transforms.py:143 subtracts the mean of the WHOLE array, not of an epoch)
 *   out           host pointer, coefficient (c, s, t) at out[c * out_channel_stride + s * out_scale_stride + t]
 *
 * The result is streamed: tiles of (channel group x scales x time stretch) alternate between two
 * plan-owned device buffers and travel to the host while the next tile is computed, so results larger
 * than device memory work and device memory holds one channel group's samples plus two tiles.  A pinned
 * `out` (cudaHostAlloc, cudaHostRegister, torch pin_memory) is written by DMA directly; a pageable one is
 * filled from a plan-owned pinned ring by a few host threads.  Synchronous: returns when `out` is complete.
 * One call at a time per plan. */
int gcwt_execute_host(gcwt_plan *plan, const void *x, int32_t in_type,
                      int64_t n_channels, int64_t n_samples, int64_t x_stride,
                      const int64_t *epoch_bounds, int32_t n_epochs,
                      const double *means_host,
                      void *out, int64_t out_scale_stride, int64_t out_channel_stride);

/* Pooling for display.  plot() draws the whole (scales, samples) array (ghost/wave/transforms.py:356-367,
 * 395-396) although a display has a few thousand columns: these reduce every run of pool_width consecutive
 * samples of a row to its mean (GCWT_POOL_MEAN) or maximum (GCWT_POOL_MAX), in fp64, on the device.
 *
 * gcwt_pool_rows: device array of n_rows rows (row_stride elements apart) of n_cols samples ->
 *   out_dev[row * out_stride + bin], ceil(n_cols / pool_width) float64 bins per row; square != 0 pools x^2
 *   (power from an amplitude array).
 * gcwt_execute_host_pooled: gcwt_execute_host (one epoch, amplitude or power plans) whose tiles are pooled
 *   on the device, so that only ceil(n_samples / pool_width) float64 bins per (channel, scale) cross the
 *   link instead of every coefficient: out[c * out_channel_stride + s * out_scale_stride + bin].  The bins
 *   reach `out` as gcwt_execute_host's rows do: by DMA when `out` is pinned, through the pinned ring and host
 *   threads when it is pageable. */
#define GCWT_POOL_MEAN 0
#define GCWT_POOL_MAX  1
int gcwt_pool_rows(const void *x_dev, int32_t type, int64_t n_rows, int64_t n_cols, int64_t row_stride,
                   int64_t pool_width, int32_t pool_mode, int32_t square, double *out_dev, int64_t out_stride,
                   int32_t device, void *stream);
int gcwt_execute_host_pooled(gcwt_plan *plan, const void *x, int32_t in_type,
                             int64_t n_channels, int64_t n_samples, int64_t x_stride,
                             const double *means_host, int64_t pool_width, int32_t pool_mode,
                             double *out, int64_t out_scale_stride, int64_t out_channel_stride);

/* Scale-averaged band power: band power over time (theta, gamma, ripple envelopes) without the full
 * (channels, scales, samples) result crossing the link.  Band b sums the count[b] adjacent scales starting at
 * first[b]; its weights are weights[off_b .. off_b + count[b]) with off_b = count[0] + ... + count[b-1]
 * (1 / count[b] for a mean).  Bands may overlap.  At most 64 bands and 1024 (band, scale) entries.
 *
 * gcwt_band_reduce: out[c, b, n] = sum_{k < count[b]} weights[off_b + k] * |W[c, first[b] + k, n]|^2 with fp64
 *   accumulation, on a device array of kind coef_kind (GCWT_OUT_*: |W|^2 is the square of an amplitude, a
 *   power as it is, re^2 + im^2 of a complex value); W[c, s, n] at coef_dev[c * channel_stride +
 *   s * scale_stride + n] in elements of coef_type (float2 / double2 for complex) -> out_dev[c *
 *   out_channel_stride + b * out_band_stride + n], real elements of coef_type.  Asynchronous on `stream`. */
int gcwt_band_reduce(const void *coef_dev, int32_t coef_type, int32_t coef_kind,
                     int64_t n_channels, int64_t n_samples, int64_t scale_stride, int64_t channel_stride,
                     int32_t n_bands, const int32_t *band_first, const int32_t *band_count, const double *weights,
                     void *out_dev, int64_t out_band_stride, int64_t out_channel_stride,
                     int32_t device, void *stream);
/* gcwt_execute_host, but every tile is band-reduced on the device and only (channels x bands x samples)
 * travels to `out` (host, plan dtype).  Epochs as gcwt_execute_host.
 *   out[c * out_channel_stride + b * out_band_stride + t]: float for fp32 plans, double for fp64 plans, whatever
 *   the plan's out_kind; samples outside all epochs are zero.  The coefficients summed are those
 *   gcwt_execute_host would have written, accuracy-guard re-computations included. */
int gcwt_execute_host_bands(gcwt_plan *plan, const void *x, int32_t in_type,
                            int64_t n_channels, int64_t n_samples, int64_t x_stride,
                            const int64_t *epoch_bounds, int32_t n_epochs, const double *means_host,
                            int32_t n_bands, const int32_t *band_first, const int32_t *band_count,
                            const double *weights,
                            void *out, int64_t out_band_stride, int64_t out_channel_stride);

/* Event-locked averages: the mean spectrogram around a set of events (stimuli, ripple peaks, spikes, trial starts)
 * and the inter-trial phase coherence, without the full (channels, scales, samples) result crossing the link.
 * Events are sample indices; event e covers the n_lags samples e + lag_first + l, l = 0 .. n_lags - 1 (lag_first
 * may be negative).  |W|^2 follows the kind as in gcwt_band_reduce; the phase term is W / |W| (0 where |W| = 0, and
 * still counted).  Sums are fp64 and in one fixed order: the same bits on every run.
 *
 * gcwt_event_reduce: ADDS, for every event whose sample e + lag_first + l lies in the tile
 *   [sample0, sample0 + n_samples), |W[c, s, e + lag_first + l - sample0]|^2 to acc_power_dev[c * acc_channel_stride +
 *   s * acc_scale_stride + l] (double) and, when acc_phase_dev is not NULL (complex coefficients only), W / |W| to
 *   acc_phase_dev at the same index (double2, 16-byte aligned); W[c, s, t] at coef_dev[c * channel_stride +
 *   s * scale_stride + t] in elements of coef_type (float2 / double2 for complex).  Events in any order, duplicates
 *   count twice.  A caller can drive a result tile by tile into one accumulator; the means are sums / n_events.
 *   Asynchronous on `stream`; at most 65535 scales.
 * gcwt_execute_host_events: gcwt_execute_host (epochs, means) whose tiles are reduced on the device; writes MEANS over
 *   the n_events events: power_out[c * out_channel_stride + s * out_scale_stride + l] (host double) and, for complex
 *   plans, phase_out at the same index (host complex double, re/im interleaved; NULL skips the phase).  Events must
 *   ascend and each window must lie inside one epoch; otherwise GCWT_ERR_ARG names the event, before any device work.
 *   The coefficients summed are those gcwt_execute_host would have written, accuracy-guard re-computations included.
 *   gcwt_host_stats reports bytes_out = the bytes of the means, and 0 for a pinned destination (they arrive through
 *   the plan's pinned ring). */
int gcwt_event_reduce(const void *coef_dev, int32_t coef_type, int32_t coef_kind,
                      int64_t n_channels, int32_t n_scales, int64_t n_samples,
                      int64_t scale_stride, int64_t channel_stride, int64_t sample0,
                      const int64_t *events_dev, int64_t n_events, int64_t lag_first, int64_t n_lags,
                      double *acc_power_dev, double *acc_phase_dev,
                      int64_t acc_scale_stride, int64_t acc_channel_stride,
                      int32_t device, void *stream);
int gcwt_execute_host_events(gcwt_plan *plan, const void *x, int32_t in_type,
                             int64_t n_channels, int64_t n_samples, int64_t x_stride,
                             const int64_t *epoch_bounds, int32_t n_epochs, const double *means_host,
                             const int64_t *events_host, int64_t n_events, int64_t lag_first, int64_t n_lags,
                             double *power_out, double *phase_out,
                             int64_t out_scale_stride, int64_t out_channel_stride);

/* Diagnostics of the last gcwt_execute_host: out4 = {wall ms, 1 if `out` was pinned (direct DMA) else 0,
 * tiles, bytes copied to the host}. */
int gcwt_host_stats(const gcwt_plan *plan, double *out4);

/* Per-channel mean in float64 (transforms.py:143): means[c] = mean(x[c, 0:n_samples]). */
int gcwt_channel_means(const void *x, int32_t in_type, int64_t n_channels,
                       int64_t n_samples, int64_t x_stride, double *means_dev,
                       int32_t device, void *stream);

/* Exact transfer function of one scale's reference kernel on an n_fft-point DFT grid
 * (device evaluation of the closed form; used by tests and by INTEGRATION examples).
 * Writes n_bins complex doubles (re, im interleaved) for bins first_bin.. to host memory. */
int gcwt_filter_response(int64_t length, int32_t k_first, int32_t n_terms,
                         const double *terms, int64_t n_fft, int64_t first_bin,
                         int64_t n_bins, double *out_host, int32_t device);

/* The L-tap time-domain kernel psi_L itself (what Morse.__call__ returns first,
 * ghost/wave/morse.py:84-91 -> morseutils.py:145-149), synthesised on the device as the
 * sum of its n_terms complex exponentials.  Writes `length` complex doubles to host. */
int gcwt_morse_kernel(int64_t length, int32_t k_first, int32_t n_terms, const double *terms,
                      double *out_host, int32_t device);

/* Taps of the polyphase interpolator that brings |W|^2 from the coarse grid (spacing U = 2^log2_u
 * samples) to the full rate on the amplitude / power paths: least-squares fractional-delay fit over
 * the band |f| <= 1 / (2 * oversampling) cycles per coarse sample.  Host-only (no device needed).
 * Writes U * n_taps floats, phase-major: output at coarse position iota + phi / U is
 * sum_t taps[phi][t] * p[iota + t - (n_taps / 2 - 1)].  n_taps even, 4 .. 32. */
int gcwt_interp_taps(int32_t log2_u, int32_t n_taps, double oversampling, float *out_host);

/* ---- sigtools helpers (SURVEY.md section 8(f)); host pointers, complex128 like the reference ----
 *
 * gcwt_fastconv: full linear convolution, n + m - 1 complex outputs (interleaved re, im).  Replaces
 *   fastconv_scipy / fastconv_fftw (ghost/sigtools/convolution.py:16-216); the 'same' / 'valid'
 *   slices (convolution.py:79-87) are views of this result.  *_is_complex: 0 = real doubles.
 * gcwt_dft: DFT of any length (Bluestein chirp-z for non powers of two), sign -1 forward, +1
 *   backward (unscaled).  Replaces chirpz_dft (ghost/sigtools/fourier.py:9-48).
 * gcwt_analytic_signal: x + i Hilbert(x) for a real signal of any length.  Replaces
 *   analytic_signal_scipy / analytic_signal_fftw (ghost/sigtools/analytic.py:15-112). */
int gcwt_fastconv(const double *signal, int32_t signal_is_complex, int64_t n,
                  const double *kernel, int32_t kernel_is_complex, int64_t m,
                  double *out_full, int32_t device);
int gcwt_dft(const double *x_complex, int64_t n, int32_t sign, double *out_complex, int32_t device);
int gcwt_analytic_signal(const double *x, int64_t n, double *out_complex, int32_t device);

/* Global mean and (population) standard deviation, in fp64, of n device elements x (or of x^2 when
 * square != 0: power from an amplitude array).  What plot(standardize=True) computes on the host
 * over the whole (S, N) array (ghost/wave/transforms.py:360-366).  out_host[0] = mean, [1] = std. */
int gcwt_moments(const void *x_dev, int32_t type, int64_t n, int32_t square, double *out_host,
                 int32_t device, void *stream);

/* Execute-time accuracy guard of the fp32 paths.  The reference convolves with an exact L-tap FIR for
 * any input spectrum (ghost/sigtools/convolution.py:72-87).  The fp32 fused kernels are exact only up
 * to (a) the filter response dropped outside the band they keep (band_tol), (b) the stop band of the
 * decimation pyramid and (c) fp32 rounding against the energy of the chunk being transformed.  All
 * three are far below the 1e-5 bar unless a scale's true output is orders of magnitude weaker than
 * what the recording holds elsewhere in the spectrum (blue or high-passed recordings, a weak tone
 * beside a strong one).  During gcwt_execute the kernels therefore measure octave-band energies of
 * every channel and the output energy of every (channel, scale); a bound on the three errors is
 * compared with guard_tol, and the pairs that fail are re-computed with the fp64 generic path (cast
 * to the plan's fp32 output).  gcwt_execute waits for the verdict, i.e. it synchronises `stream`
 * once per call unless the plan was created with GCWT_FLAG_NO_GUARD.
 *   last_pairs   (channel, scale) pairs re-computed by the last gcwt_execute
 *   total_pairs  same, accumulated since plan creation;  checked_pairs: pairs examined so far
 *   scale_flags  optional [n_scales] bytes: 1 where the last call re-computed that scale for any channel */
int gcwt_guard_stats(const gcwt_plan *plan, int64_t *last_pairs, int64_t *total_pairs,
                     int64_t *checked_pairs, unsigned char *scale_flags);

/* Bytes of device workspace the plan currently holds (grows on demand in execute). */
size_t gcwt_plan_workspace_bytes(const gcwt_plan *plan);

/* Per-kernel-family device timing for the roofline report.  With profiling enabled,
 * gcwt_execute brackets every launch group with CUDA events on the launch stream.
 * gcwt_profile_read synchronises those events and returns accumulated milliseconds and
 * launch counts for: [0] mean + decimation pyramid, [1] fused full-spectrum kernel,
 * [2] fused band-limited kernel, [3] generic global-memory path, [4] fused band-limited
 * kernel with coarse grid + polyphase interpolation. */
#define GCWT_PROFILE_KINDS 5
int gcwt_profile_enable(gcwt_plan *plan, int32_t on);
int gcwt_profile_read(gcwt_plan *plan, double *ms_out, int64_t *launches_out, int32_t reset);

/* Number of kernel launches issued by this library on the calling thread since the
 * last call with reset != 0 (bench.py reports it as gpu_launches). */
int64_t gcwt_launch_count(int32_t reset);

const char *gcwt_last_error(void);
int gcwt_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GHOST_CWT_H */
