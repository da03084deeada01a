// extern "C" boundary (include/ghost_cwt.h): plan management and dispatch.
#include "plan.h"
#include "common.cuh"
#include <cstring>
#include <cstdio>
#include <cstdlib>
#include <new>

namespace gcwt {

static thread_local std::string g_last_error;
static thread_local int64_t g_launches = 0;

void set_error(const std::string& msg) { g_last_error = msg; }
void count_launch(int n) { g_launches += n; }
int64_t launches_so_far() { return g_launches; }

int prof_begin(gcwt_plan* p, int kind, cudaStream_t st, int tag) {
    if (!p->profile) return -1;
    gcwt_plan::Span sp;
    sp.kind = kind;
    sp.tag = tag;
    sp.launches = (int)g_launches;
    if (cudaEventCreate(&sp.a) != cudaSuccess || cudaEventCreate(&sp.b) != cudaSuccess) return -1;
    cudaEventRecord(sp.a, st);
    p->spans.push_back(sp);
    return (int)p->spans.size() - 1;
}

void prof_end(gcwt_plan* p, int idx, cudaStream_t st) {
    if (idx < 0) return;
    gcwt_plan::Span& sp = p->spans[idx];
    sp.launches = (int)g_launches - sp.launches;
    cudaEventRecord(sp.b, st);
}

static void prof_collect(gcwt_plan* p) {
    for (auto& sp : p->spans) {
        float ms = 0.f;
        if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
            p->prof_ms[sp.kind] += ms;
            p->class_ms[sp.tag & 63] += ms;
            p->prof_launches[sp.kind] += sp.launches;
        }
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    p->spans.clear();
}

int ensure_workspace(gcwt_plan* p, size_t bytes) {
    if (p->ws.bytes >= bytes) return GCWT_OK;
    if (p->ws.ptr) { cudaFree(p->ws.ptr); p->ws.ptr = nullptr; p->ws.bytes = 0; }
    size_t want = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&p->ws.ptr, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = bytes;
        e = cudaMalloc(&p->ws.ptr, want);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("workspace allocation of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
        return GCWT_ERR_NOMEM;
    }
    p->ws.bytes = want;
    return GCWT_OK;
}

static int grow(void** ptr, size_t* have, size_t need, bool pinned, const char* who) {
    if (*have >= need) return GCWT_OK;
    if (*ptr) pinned ? cudaFreeHost(*ptr) : cudaFree(*ptr);
    *ptr = nullptr; *have = 0;
    const cudaError_t e = pinned ? cudaMallocHost(ptr, need) : cudaMalloc(ptr, need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error(std::string(who) + (pinned ? ": pinned" : ": device") + " allocation of " + std::to_string(need) +
                  " bytes: " + cudaGetErrorString(e));
        return GCWT_ERR_NOMEM;
    }
    *have = need;
    return GCWT_OK;
}

int grow_device(void** ptr, size_t* have, size_t need, const char* who) { return grow(ptr, have, need, false, who); }
int grow_pinned(void** ptr, size_t* have, size_t need, const char* who) { return grow(ptr, have, need, true, who); }

int filter_response_device(int64_t L, int k_first, int n_terms, const double* terms_host, int64_t nfft,
                           int64_t first_bin, int64_t n_bins, double* out_host);

int morse_kernel_device(int64_t L, int k_first, int n_terms, const double* terms_host, double* out_host);

int sig_dft_host(const double* x_host, int64_t n, int sign, double* out_host);
int sig_analytic_host(const double* x_host, int64_t n, double* out_host);
int sig_fastconv_host(const double* sig_host, int sig_complex, int64_t n, const double* ker_host, int ker_complex,
                      int64_t m, double* out_host);

int sig_moments(const void* x_dev, int type, int64_t n, int square, double* out_host, cudaStream_t st);

// Every entry point selects the plan's device; the caller's current device is restored on return.
struct DeviceScope {
    int prev = -1;
    explicit DeviceScope(int dev) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};

static int check_exec_args(const gcwt_plan* plan, const void* x, int in_type, int64_t n_channels,
                           int64_t n_samples, int64_t x_stride, const void* out) {
    if (!plan) { set_error("plan is NULL"); return GCWT_ERR_ARG; }
    if (!x || !out) { set_error("x/out is NULL"); return GCWT_ERR_ARG; }
    if (in_type != GCWT_F32 && in_type != GCWT_F64) { set_error("in_type must be GCWT_F32 or GCWT_F64"); return GCWT_ERR_ARG; }
    if (n_channels <= 0 || n_samples <= 0) { set_error("n_channels and n_samples must be positive"); return GCWT_ERR_ARG; }
    if (n_channels > 65535) { set_error("at most 65535 channels per call"); return GCWT_ERR_ARG; }
    if (x_stride < n_samples && n_channels > 1) { set_error("x_stride smaller than n_samples"); return GCWT_ERR_ARG; }
    return GCWT_OK;
}

// the checks both device reductions make on their coefficients: non-NULL pointers, type, kind and positive sizes;
// the error texts name the entry point (`who`), its pointers (`ptrs`) and its sizes (`sizes`)
static int check_coef_args(const char* who, bool ptrs_ok, const char* ptrs, int type, int kind, bool sizes_ok, const char* sizes) {
    const std::string msg = !ptrs_ok ? std::string(ptrs) + " is NULL"
                          : type != GCWT_F32 && type != GCWT_F64 ? "coef_type must be GCWT_F32 or GCWT_F64"
                          : kind < GCWT_OUT_COMPLEX || kind > GCWT_OUT_POWER ? "bad coef_kind"
                          : !sizes_ok ? std::string(sizes) + " must be positive" : "";
    if (msg.empty()) return GCWT_OK;
    set_error(std::string(who) + ": " + msg);
    return GCWT_ERR_ARG;
}

}  // namespace gcwt

using namespace gcwt;

extern "C" {

int gcwt_version(void) { return GCWT_VERSION; }

const char* gcwt_last_error(void) { return g_last_error.c_str(); }

int64_t gcwt_launch_count(int32_t reset) {
    const int64_t v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

int gcwt_plan_create(gcwt_plan** out, const gcwt_plan_desc* d) {
    if (!out || !d) { set_error("plan_create: NULL argument"); return GCWT_ERR_ARG; }
    *out = nullptr;
    if (d->n_scales <= 0 || !d->lengths || !d->k_first || !d->n_terms || !d->terms) {
        set_error("plan_create: empty or NULL scale tables"); return GCWT_ERR_ARG;
    }
    if (d->compute_type != GCWT_F32 && d->compute_type != GCWT_F64) { set_error("plan_create: bad compute_type"); return GCWT_ERR_ARG; }
    if (d->out_kind < GCWT_OUT_COMPLEX || d->out_kind > GCWT_OUT_POWER) { set_error("plan_create: bad out_kind"); return GCWT_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (this library has no CPU fallback)");
        return GCWT_ERR_CUDA;
    }
    if (d->device < 0 || d->device >= ndev) { set_error("plan_create: bad device ordinal"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(d->device);
    int rc = prepare_device(d->device);
    if (rc) return rc;

    gcwt_plan* p = new (std::nothrow) gcwt_plan();
    if (!p) { set_error("out of host memory"); return GCWT_ERR_NOMEM; }
    p->n_scales = d->n_scales;
    p->compute_type = d->compute_type;
    p->out_kind = d->out_kind;
    p->device = d->device;
    p->flags = d->flags;
    p->band_tol = d->band_tol > 0 ? d->band_tol : 1e-7;
    p->guard_tol = d->guard_tol > 0 ? d->guard_tol : 5e-6;
    p->guard = d->compute_type == GCWT_F32 && !(d->flags & (GCWT_FLAG_NO_GUARD | GCWT_FLAG_FORCE_GENERIC));
    int off = 0;
    for (int s = 0; s < d->n_scales; ++s) {
        ScaleInfo sc;
        sc.L = d->lengths[s];
        sc.k_first = d->k_first[s];
        sc.n_terms = d->n_terms[s];
        sc.term_off = off;
        sc.level = -2;
        if (sc.L < 1 || sc.n_terms < 1 || sc.k_first < 0 || sc.k_first + sc.n_terms > sc.L) {
            set_error("plan_create: inconsistent scale " + std::to_string(s));
            delete p;
            return GCWT_ERR_ARG;
        }
        off += sc.n_terms;
        p->scales.push_back(sc);
    }
    p->terms.assign(d->terms, d->terms + off);

    {
        cudaError_t e = cudaMalloc((void**)&p->d_scales, sizeof(ScaleInfo) * p->n_scales);
        if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_terms, sizeof(double) * p->terms.size());
        if (e == cudaSuccess) e = cudaMemcpy(p->d_scales, p->scales.data(), sizeof(ScaleInfo) * p->n_scales, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(p->d_terms, p->terms.data(), sizeof(double) * p->terms.size(), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { set_error(std::string("plan_create: ") + cudaGetErrorString(e)); rc = GCWT_ERR_CUDA; }
    }
    if (rc == GCWT_OK) {
        if (p->compute_type == GCWT_F32) rc = fast_plan_build(p);
        else for (int s = 0; s < p->n_scales; ++s) p->generic_ids.push_back(s);
    }
    if (rc == GCWT_OK && p->compute_type == GCWT_F32) {      // levels were chosen by the planner: refresh the device copy
        cudaError_t e = cudaMemcpy(p->d_scales, p->scales.data(), sizeof(ScaleInfo) * p->n_scales, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { set_error(std::string("plan_create: ") + cudaGetErrorString(e)); rc = GCWT_ERR_CUDA; }
    }
    if (rc != GCWT_OK) { gcwt_plan_destroy(p); return rc; }
    *out = p;
    return GCWT_OK;
}

int gcwt_plan_destroy(gcwt_plan* p) {
    if (!p) return GCWT_OK;
    DeviceScope dev_scope(p->device);
    prof_collect(p);
    host_stage_free(p);
    fast_plan_free(p);
    if (p->d_scales) cudaFree(p->d_scales);
    if (p->d_terms) cudaFree(p->d_terms);
    if (p->ws.ptr) cudaFree(p->ws.ptr);
    if (p->d_means) cudaFree(p->d_means);
    if (p->d_partial) cudaFree(p->d_partial);
    if (p->d_twiddle) cudaFree(p->d_twiddle);
    if (p->d_tw1k) cudaFree(p->d_tw1k);
    if (p->d_tw_fine) cudaFree(p->d_tw_fine);
    if (p->d_hcache) cudaFree(p->d_hcache);
    for (int k = 0; k < gcwt_plan::kSideStreams; ++k) {
        if (p->side_stream[k]) { cudaStreamSynchronize(p->side_stream[k]); cudaStreamDestroy(p->side_stream[k]); }
        if (p->ev_join[k]) cudaEventDestroy(p->ev_join[k]);
    }
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    delete p;
    return GCWT_OK;
}

int gcwt_profile_enable(gcwt_plan* p, int32_t on) {
    if (!p) { set_error("profile_enable: NULL plan"); return GCWT_ERR_ARG; }
    p->profile = on != 0;
    return GCWT_OK;
}

int gcwt_profile_read(gcwt_plan* p, double* ms_out, int64_t* launches_out, int32_t reset) {
    if (!p || !ms_out || !launches_out) { set_error("profile_read: NULL argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(p->device);
    prof_collect(p);
    if (getenv("GCWT_CLASS_TIMES")) {                  // developer aid: per-class milliseconds since the last reset
        for (int t = 0; t < 64; ++t)
            if (p->class_ms[t] > 0) fprintf(stderr, "gcwt class level %d: %.4f ms\n", t - 2, p->class_ms[t]);
    }
    if (reset) for (int t = 0; t < 64; ++t) p->class_ms[t] = 0;
    for (int k = 0; k < GCWT_PROFILE_KINDS; ++k) {
        ms_out[k] = p->prof_ms[k];
        launches_out[k] = p->prof_launches[k];
        if (reset) { p->prof_ms[k] = 0; p->prof_launches[k] = 0; }
    }
    return GCWT_OK;
}

int gcwt_plan_levels(const gcwt_plan* p, int32_t* levels_out) {
    if (!p || !levels_out) { set_error("plan_levels: NULL argument"); return GCWT_ERR_ARG; }
    for (int s = 0; s < p->n_scales; ++s) levels_out[s] = p->scales[s].level;
    return GCWT_OK;
}

int gcwt_plan_classes(const gcwt_plan* p, int32_t* n_classes, gcwt_class_info* info, int32_t* class_of_scale) {
    if (!p || !n_classes) { set_error("plan_classes: NULL argument"); return GCWT_ERR_ARG; }
    const int nc = (int)p->classes.size();
    *n_classes = nc;
    if (class_of_scale)
        for (int s = 0; s < p->n_scales; ++s) class_of_scale[s] = -1;
    for (int i = 0; i < nc; ++i) {
        const gcwt::FastClass& fc = p->classes[i];
        if (info) {
            gcwt_class_info& ci = info[i];
            ci.level = fc.level;
            ci.kernel = fc.level < 0 ? GCWT_KERNEL_FULL
                      : fc.wide ? GCWT_KERNEL_WIDE2 : (fc.interp ? GCWT_KERNEL_INTERP : GCWT_KERNEL_BANDED);
            ci.log2u = fc.interp ? fc.log2u : 0;
            ci.n_scales = (int32_t)fc.scale_ids.size();
            ci.chunk = fc.wide ? 2 * fc.nc_full : fc.nc_full;
            ci.offset = fc.wide ? fc.offset2 : fc.offset;
            ci.hop = fc.wide ? fc.hop2 : fc.hop;
        }
        if (class_of_scale)
            for (int id : fc.scale_ids) class_of_scale[id] = i;
    }
    return GCWT_OK;
}

size_t gcwt_plan_workspace_bytes(const gcwt_plan* p) { return p ? p->ws.bytes : 0; }

int gcwt_guard_stats(const gcwt_plan* p, int64_t* last_pairs, int64_t* total_pairs, int64_t* checked_pairs,
                     unsigned char* scale_flags) {
    if (!p) { set_error("guard_stats: NULL plan"); return GCWT_ERR_ARG; }
    if (last_pairs) *last_pairs = p->guard_last;
    if (total_pairs) *total_pairs = p->guard_total;
    if (checked_pairs) *checked_pairs = p->guard_checked;
    if (scale_flags)
        for (int s = 0; s < p->n_scales; ++s) scale_flags[s] = (size_t)s < p->guard_last_flags.size() ? p->guard_last_flags[s] : 0;
    return GCWT_OK;
}

int gcwt_channel_means(const void* x, int32_t in_type, int64_t n_channels, int64_t n_samples,
                       int64_t x_stride, double* means_dev, int32_t device, void* stream) {
    if (!x || !means_dev) { set_error("channel_means: NULL argument"); return GCWT_ERR_ARG; }
    if (in_type != GCWT_F32 && in_type != GCWT_F64) { set_error("channel_means: bad in_type"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    // stand-alone call: scratch is allocated and freed here (synchronous; not on the transform path)
    double* partial = nullptr;
    GCWT_CUDA_OK(cudaMalloc((void**)&partial, sizeof(double) * means_blocks(n_samples) * n_channels));
    int rc = means_launch(x, in_type, n_channels, n_samples, x_stride, means_dev, partial, (cudaStream_t)stream);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(partial);
    return rc;
}

int gcwt_execute(gcwt_plan* p, const void* x, int32_t in_type, int64_t n_channels, int64_t n_samples,
                 int64_t x_stride, int64_t halo_left, int64_t halo_right, const double* means,
                 void* out, int64_t out_scale_stride, int64_t out_channel_stride, void* stream) {
    int rc = check_exec_args(p, x, in_type, n_channels, n_samples, x_stride, out);
    if (rc) return rc;
    if (halo_left < 0 || halo_right < 0) { set_error("execute: negative halo"); return GCWT_ERR_ARG; }
    if (n_channels > 1 && x_stride < n_samples + halo_left + halo_right) {
        set_error("execute: x_stride smaller than n_samples plus the halos (channels would overlap)"); return GCWT_ERR_ARG;
    }
    if (out_scale_stride < n_samples) { set_error("execute: out_scale_stride smaller than n_samples"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    const double* d_means = means;
    if (!d_means) {
        rc = grow_device((void**)&p->d_means, &p->means_bytes, sizeof(double) * n_channels, "execute");
        if (rc == GCWT_OK)
            rc = grow_device((void**)&p->d_partial, &p->partial_bytes, sizeof(double) * means_blocks(n_samples) * n_channels, "execute");
        if (rc) return rc;
        const int sp = prof_begin(p, 0, st);
        rc = means_launch(x, in_type, n_channels, n_samples, x_stride, p->d_means, p->d_partial, st);
        prof_end(p, sp, st);
        if (rc) return rc;
        d_means = p->d_means;
    }
    // The fused kernels keep their pyramid in the plan's workspace, and the guard's fp64 re-computation lays out its
    // own buffers there.  The generic scales reuse the workspace too, and ensure_workspace may free it to grow it, so
    // the generic part starts only once the work queued on `st` (side streams joined) is done with it.
    if (p->compute_type == GCWT_F32 && !p->classes.empty()) {
        rc = fast_execute(p, x, in_type, n_channels, n_samples, x_stride, halo_left, halo_right, d_means,
                          out, out_scale_stride, out_channel_stride, st);
        if (rc) return rc;
        // accuracy guard: waits for the verdict of this call and re-computes the failing pairs in fp64
        rc = guard_resolve(p, x, in_type, n_channels, n_samples, x_stride, halo_left, halo_right, d_means,
                           out, out_scale_stride, out_channel_stride, st);
        if (rc) return rc;
        if (!p->generic_ids.empty()) GCWT_CUDA_OK(cudaStreamSynchronize(st));
    }
    if (!p->generic_ids.empty()) {
        const int sp = prof_begin(p, 3, st);
        rc = generic_execute(p, p->generic_ids, x, in_type, n_channels, n_samples, x_stride, halo_left,
                             halo_right, d_means, out, out_scale_stride, out_channel_stride, st);
        prof_end(p, sp, st);
        if (rc) return rc;
    }
    return GCWT_OK;
}

int gcwt_execute_host(gcwt_plan* p, const void* x, int32_t in_type, int64_t n_channels,
                      int64_t n_samples, int64_t x_stride, const int64_t* epoch_bounds, int32_t n_epochs,
                      const double* means_host, void* out, int64_t out_scale_stride, int64_t out_channel_stride) {
    int rc = check_exec_args(p, x, in_type, n_channels, n_samples, x_stride, out);
    if (rc) return rc;
    if (out_scale_stride < n_samples) { set_error("execute_host: out_scale_stride smaller than n_samples"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(p->device);
    return host_execute(p, x, in_type, n_channels, n_samples, x_stride, epoch_bounds, n_epochs, means_host, out,
                        out_scale_stride, out_channel_stride);
}

int gcwt_execute_host_pooled(gcwt_plan* p, const void* x, int32_t in_type, int64_t n_channels, int64_t n_samples,
                             int64_t x_stride, const double* means_host, int64_t pool_width, int32_t pool_mode,
                             double* out, int64_t out_scale_stride, int64_t out_channel_stride) {
    int rc = check_exec_args(p, x, in_type, n_channels, n_samples, x_stride, out);
    if (rc) return rc;
    if (pool_width < 1 || (pool_mode != GCWT_POOL_MEAN && pool_mode != GCWT_POOL_MAX)) { set_error("execute_host_pooled: bad pool_width / pool_mode"); return GCWT_ERR_ARG; }
    if (out_scale_stride < (n_samples + pool_width - 1) / pool_width) { set_error("execute_host_pooled: out_scale_stride smaller than the bin count"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(p->device);
    return host_execute(p, x, in_type, n_channels, n_samples, x_stride, nullptr, 0, means_host, out, out_scale_stride,
                        out_channel_stride, pool_width, pool_mode);
}

int gcwt_pool_rows(const void* x_dev, int32_t type, int64_t n_rows, int64_t n_cols, int64_t row_stride, int64_t pool_width,
                   int32_t pool_mode, int32_t square, double* out_dev, int64_t out_stride, int32_t device, void* stream) {
    if (!x_dev || !out_dev || (type != GCWT_F32 && type != GCWT_F64)) { set_error("pool_rows: bad argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return pool_rows_launch(x_dev, type, n_rows, n_cols, row_stride, pool_width, pool_mode, square, out_dev, out_stride,
                            (cudaStream_t)stream);
}

int gcwt_band_reduce(const void* coef_dev, int32_t coef_type, int32_t coef_kind, int64_t n_channels, int64_t n_samples,
                     int64_t scale_stride, int64_t channel_stride, int32_t n_bands, const int32_t* band_first,
                     const int32_t* band_count, const double* weights, void* out_dev, int64_t out_band_stride,
                     int64_t out_channel_stride, int32_t device, void* stream) {
    BandTable tab;
    int rc = check_coef_args("band_reduce", coef_dev && out_dev, "coef/out", coef_type, coef_kind,
                             n_channels > 0 && n_samples > 0, "n_channels and n_samples");
    if (rc == GCWT_OK) rc = band_table_build(n_bands, band_first, band_count, weights, &tab, "band_reduce");
    if (rc) return rc;
    if (scale_stride < n_samples || (n_channels > 1 && channel_stride < (int64_t)tab.rows * scale_stride)) {
        set_error("band_reduce: scale_stride below n_samples, or channel_stride below the rows the bands read"); return GCWT_ERR_ARG;
    }
    if (out_band_stride < n_samples || (n_channels > 1 && out_channel_stride < (int64_t)n_bands * out_band_stride)) {
        set_error("band_reduce: out_band_stride below n_samples, or out_channel_stride below n_bands rows"); return GCWT_ERR_ARG;
    }
    DeviceScope dev_scope(device);
    return band_reduce_launch(coef_dev, coef_type, coef_kind, n_channels, n_samples, scale_stride, channel_stride, tab,
                              out_dev, out_band_stride, out_channel_stride, (cudaStream_t)stream);
}

int gcwt_execute_host_bands(gcwt_plan* p, const void* x, int32_t in_type, int64_t n_channels, int64_t n_samples,
                            int64_t x_stride, const int64_t* epoch_bounds, int32_t n_epochs, const double* means_host,
                            int32_t n_bands, const int32_t* band_first, const int32_t* band_count, const double* weights,
                            void* out, int64_t out_band_stride, int64_t out_channel_stride) {
    BandTable tab;
    int rc = band_table_build(n_bands, band_first, band_count, weights, &tab, "execute_host_bands");
    if (rc) return rc;
    rc = check_exec_args(p, x, in_type, n_channels, n_samples, x_stride, out);
    if (rc) return rc;
    if (tab.rows > p->n_scales) {
        set_error("execute_host_bands: a band reaches scale " + std::to_string(tab.rows - 1) + " of a plan with " +
                  std::to_string(p->n_scales) + " scales");
        return GCWT_ERR_ARG;
    }
    if (out_band_stride < n_samples || (n_channels > 1 && out_channel_stride < (int64_t)n_bands * out_band_stride)) {
        set_error("execute_host_bands: out_band_stride below n_samples, or out_channel_stride below n_bands rows"); return GCWT_ERR_ARG;
    }
    DeviceScope dev_scope(p->device);
    return host_execute(p, x, in_type, n_channels, n_samples, x_stride, epoch_bounds, n_epochs, means_host, out,
                        out_band_stride, out_channel_stride, 0, 0, &tab);
}

int gcwt_event_reduce(const void* coef_dev, int32_t coef_type, int32_t coef_kind, int64_t n_channels, int32_t n_scales,
                      int64_t n_samples, int64_t scale_stride, int64_t channel_stride, int64_t sample0,
                      const int64_t* events_dev, int64_t n_events, int64_t lag_first, int64_t n_lags,
                      double* acc_power_dev, double* acc_phase_dev, int64_t acc_scale_stride,
                      int64_t acc_channel_stride, int32_t device, void* stream) {
    const int rc = check_coef_args("event_reduce", coef_dev && events_dev && acc_power_dev, "coef/events/acc_power", coef_type,
                                   coef_kind, n_channels > 0 && n_scales > 0 && n_samples > 0 && n_events > 0 && n_lags > 0,
                                   "n_channels, n_scales, n_samples, n_events and n_lags");
    if (rc) return rc;
    if (acc_phase_dev && coef_kind != GCWT_OUT_COMPLEX) { set_error("event_reduce: a phase accumulator needs complex coefficients"); return GCWT_ERR_ARG; }
    if (n_scales > 65535) { set_error("event_reduce: at most 65535 scales"); return GCWT_ERR_ARG; }
    if (scale_stride < n_samples || (n_channels > 1 && channel_stride < (int64_t)n_scales * scale_stride)) {
        set_error("event_reduce: scale_stride below n_samples, or channel_stride below n_scales rows"); return GCWT_ERR_ARG;
    }
    if (acc_scale_stride < n_lags || (n_channels > 1 && acc_channel_stride < (int64_t)n_scales * acc_scale_stride)) {
        set_error("event_reduce: acc_scale_stride below n_lags, or acc_channel_stride below n_scales rows"); return GCWT_ERR_ARG;
    }
    if (acc_phase_dev && (uintptr_t)acc_phase_dev % 16) { set_error("event_reduce: acc_phase must be 16-byte aligned"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return event_reduce_launch(coef_dev, coef_type, coef_kind, n_channels, n_scales, n_samples, scale_stride, channel_stride,
                               sample0, events_dev, n_events, lag_first, n_lags, acc_power_dev, (double2*)acc_phase_dev,
                               acc_scale_stride, acc_channel_stride, (cudaStream_t)stream);
}

int gcwt_execute_host_events(gcwt_plan* p, const void* x, int32_t in_type, int64_t n_channels, int64_t n_samples,
                             int64_t x_stride, const int64_t* epoch_bounds, int32_t n_epochs, const double* means_host,
                             const int64_t* events, int64_t n_events, int64_t lag_first, int64_t n_lags, double* power_out,
                             double* phase_out, int64_t out_scale_stride, int64_t out_channel_stride) {
    if (!events) { set_error("execute_host_events: events is NULL"); return GCWT_ERR_ARG; }
    if (n_events <= 0 || n_lags <= 0) { set_error("execute_host_events: n_events and n_lags must be positive"); return GCWT_ERR_ARG; }
    int rc = check_event_args(n_samples, epoch_bounds, n_epochs, events, n_events, lag_first, n_lags);
    if (rc) return rc;
    rc = check_exec_args(p, x, in_type, n_channels, n_samples, x_stride, power_out);
    if (rc) return rc;
    if (phase_out && p->out_kind != GCWT_OUT_COMPLEX) { set_error("execute_host_events: phase_out needs a complex plan"); return GCWT_ERR_ARG; }
    if (out_scale_stride < n_lags || (n_channels > 1 && out_channel_stride < (int64_t)p->n_scales * out_scale_stride)) {
        set_error("execute_host_events: out_scale_stride below n_lags, or out_channel_stride below n_scales rows"); return GCWT_ERR_ARG;
    }
    DeviceScope dev_scope(p->device);
    return host_execute_events(p, x, in_type, n_channels, n_samples, x_stride, epoch_bounds, n_epochs, means_host, events,
                               n_events, lag_first, n_lags, power_out, phase_out, out_scale_stride, out_channel_stride);
}

int gcwt_host_stats(const gcwt_plan* p, double* out4) {
    if (!p || !out4) { set_error("host_stats: NULL argument"); return GCWT_ERR_ARG; }
    for (int k = 0; k < 4; ++k) out4[k] = p->host.last_ms[k];
    return GCWT_OK;
}

int gcwt_interp_taps(int32_t log2_u, int32_t n_taps, double oversampling, float* out_host) {
    return interp_taps(log2_u, n_taps, oversampling, out_host);
}

int gcwt_filter_response(int64_t length, int32_t k_first, int32_t n_terms, const double* terms,
                         int64_t n_fft, int64_t first_bin, int64_t n_bins, double* out_host,
                         int32_t device) {
    if (!terms || !out_host || length < 1 || n_terms < 1 || n_fft < length || n_bins < 1 || first_bin < 0) {
        set_error("filter_response: bad argument"); return GCWT_ERR_ARG;
    }
    DeviceScope dev_scope(device);
    return filter_response_device(length, k_first, n_terms, terms, n_fft, first_bin, n_bins, out_host);
}

int gcwt_morse_kernel(int64_t length, int32_t k_first, int32_t n_terms, const double* terms,
                      double* out_host, int32_t device) {
    if (!terms || !out_host || length < 1 || n_terms < 1 || k_first < 0) {
        set_error("morse_kernel: bad argument"); return GCWT_ERR_ARG;
    }
    DeviceScope dev_scope(device);
    return morse_kernel_device(length, k_first, n_terms, terms, out_host);
}

int gcwt_fastconv(const double* signal, int32_t signal_is_complex, int64_t n, const double* kernel,
                  int32_t kernel_is_complex, int64_t m, double* out_full, int32_t device) {
    if (!signal || !kernel || !out_full || n < 1 || m < 1) { set_error("fastconv: bad argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return sig_fastconv_host(signal, signal_is_complex, n, kernel, kernel_is_complex, m, out_full);
}

int gcwt_dft(const double* x_complex, int64_t n, int32_t sign, double* out_complex, int32_t device) {
    if (!x_complex || !out_complex || n < 1 || (sign != 1 && sign != -1)) { set_error("dft: bad argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return sig_dft_host(x_complex, n, sign, out_complex);
}

int gcwt_moments(const void* x_dev, int32_t type, int64_t n, int32_t square, double* out_host, int32_t device,
                 void* stream) {
    if (!x_dev || !out_host || n < 1 || (type != GCWT_F32 && type != GCWT_F64)) { set_error("moments: bad argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return sig_moments(x_dev, type, n, square, out_host, (cudaStream_t)stream);
}

int gcwt_analytic_signal(const double* x, int64_t n, double* out_complex, int32_t device) {
    if (!x || !out_complex || n < 1) { set_error("analytic_signal: bad argument"); return GCWT_ERR_ARG; }
    DeviceScope dev_scope(device);
    return sig_analytic_host(x, n, out_complex);
}

}  // extern "C"
