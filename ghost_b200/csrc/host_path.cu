// Host-buffer entry point: numpy in, numpy out, through a streamed, double-buffered pipeline.
//
// The reference returns a complete host array of shape (scales, samples) per channel
// (ghost/wave/transforms.py:185,231).  Here the caller's host buffers are the only full-size storage:
// the result is produced in tiles (a group of channels x all scales x a stretch of samples) that
// alternate between two device buffers, and tile k travels to the host while tile k + 1 is computed.
// Results larger than device memory (config 3: 295 GB per GPU) therefore work, the device holds one
// channel group's samples plus two tiles, and the link -- not the kernels -- sets the pace.
//
// One walk (walk_tiles) computes the tiles of every host call; its output decides what happens to each tile.
// What travels is the tile itself (full rate) or its reduction on the device (pooled bins or band power), and
// every such output takes the same route (Streamed):
//   pinned destination (cudaHostAlloc / cudaHostRegister / torch pin_memory): rows are written by DMA,
//     one cudaMemcpy2DAsync per channel of a tile;
//   pageable destination (a plain numpy array): tiles land in a plan-owned pinned ring by DMA and a few
//     host threads copy the rows out (which also first-touches the caller's pages in parallel).
// Event-locked averages (EventSums) send nothing per tile: each tile is added into a device accumulator of
// (channels x scales x lags) and only that crosses the link, once per channel group.
//
// Epochs (transforms.py:202-204): every epoch is a zero-padded convolution of its own; samples outside
// all epochs are zero.  The mean is the channel's mean over ALL samples (transforms.py:142-143).
#include "plan.h"
#include "common.cuh"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace gcwt {

void host_stage_free(gcwt_plan* p) {
    gcwt_plan::HostStage& h = p->host;
    if (h.st_compute) cudaStreamSynchronize(h.st_compute);
    if (h.st_copy) cudaStreamSynchronize(h.st_copy);
    if (h.d_in) cudaFree(h.d_in);
    for (int b = 0; b < 2; ++b) {
        if (h.d_out[b]) cudaFree(h.d_out[b]);
        if (h.d_red[b]) cudaFree(h.d_red[b]);
        if (h.h_ring[b]) cudaFreeHost(h.h_ring[b]);
        if (h.ev_done[b]) cudaEventDestroy(h.ev_done[b]);
        if (h.ev_out[b]) cudaEventDestroy(h.ev_out[b]);
    }
    if (h.d_means) cudaFree(h.d_means);
    if (h.d_acc) cudaFree(h.d_acc);
    if (h.d_events) cudaFree(h.d_events);
    if (h.st_compute) cudaStreamDestroy(h.st_compute);
    if (h.st_copy) cudaStreamDestroy(h.st_copy);
    h = gcwt_plan::HostStage();
}

static bool is_pinned(const void* ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// rows [r0, r1) of a tile: row r = (channel, scale or band) -> width bytes from the ring to the caller's array
struct RowCopy {
    const char* src; size_t src_pitch;          // ring: rows as staged on the device
    char* dst; int64_t s_stride_b, c_stride_b;  // caller strides in bytes
    int rows_per_channel; size_t width; int64_t n_rows;
};

static void copy_rows(const RowCopy& rc, int n_threads) {
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t r = next.fetch_add(1);
            if (r >= rc.n_rows) break;
            const int64_t c = r / rc.rows_per_channel, s = r % rc.rows_per_channel;
            memcpy(rc.dst + c * rc.c_stride_b + s * rc.s_stride_b, rc.src + (size_t)r * rc.src_pitch, rc.width);
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < n_threads; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}

static int check_epochs(const int64_t* epochs, int n_epochs, int64_t n) {
    for (int e = 0; e < n_epochs; ++e)
        if (epochs[2 * e] < 0 || epochs[2 * e + 1] > n || epochs[2 * e] >= epochs[2 * e + 1] ||
            (e > 0 && epochs[2 * e] < epochs[2 * e - 1])) {
            set_error("execute_host: epoch bounds must be ascending, non-empty and inside [0, n_samples)");
            return GCWT_ERR_ARG;
        }
    return GCWT_OK;
}

// a tile is a group of g channels x all scales x a stretch of `tile` samples, computed with `halo` real samples
// on each side where its epoch has them; on the device its rows lie `alloc` elements apart
struct TileGeometry { int64_t g, tile, halo, alloc; };

static TileGeometry tile_geometry(const gcwt_plan* p, int64_t n_channels, int64_t n, size_t out_el, int64_t pool_width) {
    const int S = p->n_scales;
    int64_t lmax = 1;
    for (const ScaleInfo& sc : p->scales) lmax = std::max<int64_t>(lmax, sc.L);
    const size_t budget = (size_t)1 << 30;                        // bytes per result tile (two on the device)
    const size_t per_channel = (size_t)S * (size_t)n * out_el;
    TileGeometry t;
    t.halo = lmax - 1;
    t.g = std::max<int64_t>(1, std::min<int64_t>(n_channels, (int64_t)(budget / std::max<size_t>(per_channel, 1))));
    t.tile = n;
    if (per_channel > budget) {
        t.tile = std::max<int64_t>((int64_t)(budget / ((size_t)S * out_el)), std::min<int64_t>(n, 4 * lmax));
        t.tile = std::min<int64_t>(n, (t.tile + 1023) / 1024 * 1024);
    }
    if (const char* e = getenv("GCWT_HOST_TILE")) {               // developer aid: force the time tile
        const int64_t hint = atoll(e);
        if (hint > 0) t.tile = std::min<int64_t>(n, std::max<int64_t>(hint, 1024));
    }
    if (pool_width > 0 && t.tile < n)                             // tiles end on bin boundaries
        t.tile = std::max<int64_t>(pool_width, t.tile / pool_width * pool_width);
    t.alloc = (t.tile + 3) & ~int64_t(3);                         // rows of a tile stay 16-byte aligned
    return t;
}

// the compute and copy streams and the two slots' events, created on a plan's first host call
static int ensure_streams(gcwt_plan::HostStage& h) {
    if (h.st_compute) return GCWT_OK;
    GCWT_CUDA_OK(cudaStreamCreateWithFlags(&h.st_compute, cudaStreamNonBlocking));
    GCWT_CUDA_OK(cudaStreamCreateWithFlags(&h.st_copy, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
        GCWT_CUDA_OK(cudaEventCreateWithFlags(&h.ev_done[b], cudaEventDisableTiming));
        GCWT_CUDA_OK(cudaEventCreateWithFlags(&h.ev_out[b], cudaEventDisableTiming));
    }
    return GCWT_OK;
}

// upload channels [c0, c0 + gc) of x into d_in and put their means into d_means, on the compute stream
static int load_group(gcwt_plan* p, const void* x, int in_type, int64_t n, int64_t x_stride, const double* means_host,
                      int64_t c0, int64_t gc) {
    gcwt_plan::HostStage& h = p->host;
    const size_t in_el = in_type == GCWT_F32 ? 4 : 8;
    // the previous group's tiles may still be copying out, but nothing reads d_in any more: every execute of
    // that group has completed (gcwt_execute waits, or we wait here)
    GCWT_CUDA_OK(cudaStreamSynchronize(h.st_compute));
    GCWT_CUDA_OK(cudaMemcpy2DAsync(h.d_in, (size_t)n * in_el, (const char*)x + (size_t)c0 * x_stride * in_el, (size_t)x_stride * in_el,
                                   (size_t)n * in_el, (size_t)gc, cudaMemcpyHostToDevice, h.st_compute));
    if (means_host) {
        GCWT_CUDA_OK(cudaMemcpyAsync(h.d_means, means_host + c0, sizeof(double) * gc, cudaMemcpyHostToDevice, h.st_compute));
        return GCWT_OK;
    }
    const size_t need = sizeof(double) * means_blocks(n) * gc;
    if (p->partial_bytes < need) {
        GCWT_CUDA_OK(cudaStreamSynchronize(h.st_compute));
        const int r = grow_device((void**)&p->d_partial, &p->partial_bytes, need, "execute_host");
        if (r) return r;
    }
    return means_launch(h.d_in, in_type, gc, n, n, h.d_means, p->d_partial, h.st_compute);
}

// zero the columns outside the epochs (the reference starts from np.zeros, transforms.py:185)
static void zero_gaps(char* out, const int64_t* epochs, int n_epochs, int64_t n, int64_t n_channels, int R,
                      int64_t s_stride, int64_t c_stride, size_t el) {
    int64_t pos = 0;
    for (int e = 0; e <= n_epochs; ++e) {
        const int64_t gap_end = e < n_epochs ? epochs[2 * e] : n;
        if (gap_end > pos)
            for (int64_t c = 0; c < n_channels; ++c)
                for (int s = 0; s < R; ++s)
                    memset(out + ((size_t)c * c_stride + (size_t)s * s_stride + pos) * el, 0, (size_t)(gap_end - pos) * el);
        if (e < n_epochs) pos = epochs[2 * e + 1];
    }
}

// The tiles of one host call: channel groups of geo.g channels, each epoch of a group, tiles of geo.tile samples in
// an epoch, alternating between the slots d_out[0] and d_out[1].  Out says what the call makes of them: prepare(geo,
// epochs, n_epochs) sets up its buffers; slot_free(b) does what must happen before d_out[b] is overwritten;
// group_begin / group_end(c0, gc) frame the tiles of channels [c0, c0 + gc); tile(b, c0, gc, a, len) works on the
// tile of samples [a, a + len) in d_out[b], on the copy stream; pinned and bytes_out go to host_stats.
template <class Out>
static int walk_tiles(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n, int64_t x_stride,
                      const int64_t* epochs, int n_epochs, const double* means_host, int64_t pool_width, Out& out) {
    gcwt_plan::HostStage& h = p->host;
    const auto t_begin = std::chrono::steady_clock::now();
    const int S = p->n_scales;
    const size_t in_el = in_type == GCWT_F32 ? 4 : 8;
    const size_t real_el = p->compute_type == GCWT_F32 ? 4 : 8;
    const size_t out_el = p->out_kind == GCWT_OUT_COMPLEX ? 2 * real_el : real_el;
    int64_t one_epoch[2] = {0, n};
    if (!epochs || n_epochs <= 0) { epochs = one_epoch; n_epochs = 1; }
    int rc = check_epochs(epochs, n_epochs, n);
    if (rc == GCWT_OK) rc = ensure_streams(h);
    if (rc) return rc;
    const TileGeometry geo = tile_geometry(p, n_channels, n, out_el, pool_width);
    rc = grow_device(&h.d_in, &h.in_bytes, (size_t)geo.g * n * in_el, "execute_host");
    for (int b = 0; b < 2 && rc == GCWT_OK; ++b)
        rc = grow_device(&h.d_out[b], &h.out_bytes[b], (size_t)geo.g * S * geo.alloc * out_el, "execute_host");
    if (rc == GCWT_OK) rc = grow_device((void**)&h.d_means, &h.means_bytes, sizeof(double) * geo.g, "execute_host");
    if (rc == GCWT_OK) rc = out.prepare(geo, epochs, n_epochs);
    if (rc) return rc;

    auto run_tile = [&](int b, int64_t c0, int64_t gc, int64_t a, int64_t len, int64_t halo_l, int64_t halo_r) -> int {
        int r = out.slot_free(b);
        if (r) return r;
        r = gcwt_execute(p, (const char*)h.d_in + (size_t)a * in_el, in_type, gc, len, n, halo_l, halo_r, h.d_means,
                         h.d_out[b], geo.alloc, (int64_t)S * geo.alloc, h.st_compute);
        if (r) return r;
        // ev_done follows the whole of gcwt_execute in stream order, including the accuracy guard's fp64 re-computation
        // of the failing (channel, scale) pairs (guard_resolve), so the reductions on the copy stream read the corrected
        // coefficients.  For the same reason band power and event sums are passes of their own and not part of the
        // fused kernels' epilogue: there they would sum values the guard then replaces.
        GCWT_CUDA_OK(cudaEventRecord(h.ev_done[b], h.st_compute));
        GCWT_CUDA_OK(cudaStreamWaitEvent(h.st_copy, h.ev_done[b], 0));
        return out.tile(b, c0, gc, a, len);
    };

    int slot = 0;
    int64_t n_tiles = 0;
    for (int64_t c0 = 0; c0 < n_channels && rc == GCWT_OK; c0 += geo.g) {
        const int64_t gc = std::min<int64_t>(geo.g, n_channels - c0);
        rc = load_group(p, x, in_type, n, x_stride, means_host, c0, gc);
        if (rc == GCWT_OK) rc = out.group_begin(c0, gc);
        for (int e = 0; e < n_epochs && rc == GCWT_OK; ++e) {
            const int64_t e0 = epochs[2 * e], e1 = epochs[2 * e + 1];
            for (int64_t a = e0; a < e1 && rc == GCWT_OK; a += geo.tile) {
                const int64_t len = std::min(e1, a + geo.tile) - a;
                rc = run_tile(slot, c0, gc, a, len, std::min(geo.halo, a - e0), std::min(geo.halo, e1 - a - len));
                if (rc) break;
                ++n_tiles;
                slot ^= 1;
            }
        }
        if (rc == GCWT_OK) rc = out.group_end(c0, gc);
    }
    for (int b = 0; b < 2; ++b) {                                  // the last tiles have left both slots
        const int r = out.slot_free(b);
        if (rc == GCWT_OK) rc = r;
    }
    cudaStreamSynchronize(h.st_copy);
    cudaStreamSynchronize(h.st_compute);
    h.last_ms[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    h.last_ms[1] = out.pinned ? 1.0 : 0.0;
    h.last_ms[2] = (double)n_tiles;
    h.last_ms[3] = out.bytes_out;
    return rc;
}

// Full-rate, pooled or band-power tiles, sent to the caller's array `out`.
// pool_width > 0: `out` is a float64 array of ceil(n / pool_width) bins per row; every tile is reduced on the device
// (mean or max over pool_width consecutive samples) and only the bins travel to the host.
// bands: `out` holds (channels x bands x samples) of the plan's real type (s_stride is the band stride); every tile
// is band-reduced on the device and only the band rows travel.  The tile geometry stays that of the full-rate path,
// so every coefficient summed is the one gcwt_execute_host would have written.
struct Streamed {
    gcwt_plan* p; int64_t n_channels, n; char* out; int64_t s_stride, c_stride, pool_width; int pool_mode;
    const BandTable* bands;
    gcwt_plan::HostStage& h = p->host;
    const int S = p->n_scales;
    const bool reduced = pool_width > 0 || bands;
    const bool pinned = is_pinned(out);
    double bytes_out = 0;
    // What reaches `out`: R rows per channel of `el`-byte elements.  A tile of `len` samples that starts at sample
    // a fills width(len) columns of them from column col(a); on the device its rows are staged `pitch` elements apart.
    const int R = bands ? bands->n_bands : S;
    const size_t real_el = p->compute_type == GCWT_F32 ? 4 : 8;
    const size_t el = bands ? real_el : pool_width > 0 ? sizeof(double) : p->out_kind == GCWT_OUT_COMPLEX ? 2 * real_el : real_el;
    int64_t pitch = 0, alloc = 0;
    int n_threads = 1;
    bool live[2] = {false, false};
    std::thread copier[2];

    // the copiers are joined on every return path: an early error return must not destroy a running thread
    ~Streamed() { for (auto& t : copier) if (t.joinable()) t.join(); }
    int64_t col(int64_t a) const { return pool_width > 0 ? a / pool_width : a; }
    int64_t width(int64_t len) const { return pool_width > 0 ? (len + pool_width - 1) / pool_width : len; }

    int prepare(const TileGeometry& geo, const int64_t* epochs, int n_epochs) {
        alloc = geo.alloc;
        pitch = pool_width > 0 ? (geo.tile + pool_width - 1) / pool_width : geo.alloc;
        const size_t stage_bytes = (size_t)geo.g * R * pitch * el;
        int rc = GCWT_OK;
        for (int b = 0; b < 2 && rc == GCWT_OK; ++b) {
            rc = grow_device(&h.d_red[b], &h.red_bytes[b], reduced ? stage_bytes : 0, "execute_host");
            if (rc == GCWT_OK) rc = grow_pinned(&h.h_ring[b], &h.ring_bytes[b], pinned ? 0 : stage_bytes, "execute_host");
        }
        if (rc) return rc;
        // copier threads of the pageable path (measured on a 16-core host, 6.9 GB per call: 8 threads 34 GB/s, see DESIGN.md)
        n_threads = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency() > 2 ? std::thread::hardware_concurrency() - 2 : 1u));
        if (const char* e = getenv("GCWT_HOST_THREADS")) n_threads = std::max(1, atoi(e));
        zero_gaps(out, epochs, n_epochs, n, n_channels, R, s_stride, c_stride, el);
        return GCWT_OK;
    }
    int slot_free(int b) {                                         // tile in slot b has reached the caller's array
        if (!live[b]) return GCWT_OK;
        if (pinned) GCWT_CUDA_OK(cudaEventSynchronize(h.ev_out[b]));
        else if (copier[b].joinable()) copier[b].join();
        live[b] = false;
        return GCWT_OK;
    }
    int group_begin(int64_t, int64_t) { return GCWT_OK; }
    int group_end(int64_t, int64_t) { return GCWT_OK; }
    // reduce the tile if this call asks for a reduction, and send its rows to `out`
    int tile(int b, int64_t c0, int64_t gc, int64_t a, int64_t len) {
        int r = GCWT_OK;
        if (pool_width > 0)
            r = pool_rows_launch(h.d_out[b], p->compute_type, gc * S, len, alloc, pool_width, pool_mode, 0,
                                 (double*)h.d_red[b], pitch, h.st_copy);
        else if (bands)
            r = band_reduce_launch(h.d_out[b], p->compute_type, p->out_kind, gc, len, alloc, (int64_t)S * alloc, *bands,
                                   h.d_red[b], pitch, (int64_t)R * pitch, h.st_copy);
        if (r) return r;
        const char* src = (const char*)(reduced ? h.d_red[b] : h.d_out[b]);
        char* dst = out + ((size_t)c0 * c_stride + (size_t)col(a)) * el;
        const size_t row_bytes = (size_t)width(len) * el;
        if (pinned) {
            for (int64_t c = 0; c < gc; ++c)
                GCWT_CUDA_OK(cudaMemcpy2DAsync(dst + (size_t)c * c_stride * el, (size_t)s_stride * el,
                                               src + (size_t)c * R * pitch * el, (size_t)pitch * el, row_bytes, (size_t)R,
                                               cudaMemcpyDeviceToHost, h.st_copy));
            GCWT_CUDA_OK(cudaEventRecord(h.ev_out[b], h.st_copy));
        } else {
            GCWT_CUDA_OK(cudaMemcpyAsync(h.h_ring[b], src, (size_t)gc * R * pitch * el, cudaMemcpyDeviceToHost, h.st_copy));
            GCWT_CUDA_OK(cudaEventRecord(h.ev_out[b], h.st_copy));
            const RowCopy rcp{(const char*)h.h_ring[b], (size_t)pitch * el, dst, s_stride * (int64_t)el,
                              c_stride * (int64_t)el, R, row_bytes, gc * R};
            cudaEvent_t ev = h.ev_out[b];
            const int dev = p->device, nt = n_threads;
            copier[b] = std::thread([rcp, ev, dev, nt]() {
                cudaSetDevice(dev);
                cudaEventSynchronize(ev);
                copy_rows(rcp, nt);
            });
        }
        live[b] = true;
        bytes_out += (double)gc * R * row_bytes;
        return GCWT_OK;
    }
};

int host_execute(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n, int64_t x_stride,
                 const int64_t* epochs, int n_epochs, const double* means_host, void* out, int64_t s_stride,
                 int64_t c_stride, int64_t pool_width, int pool_mode, const BandTable* bands) {
    if (pool_width > 0) {
        if (p->out_kind == GCWT_OUT_COMPLEX) { set_error("execute_host: pooling needs amplitude or power output"); return GCWT_ERR_ARG; }
        if (epochs && n_epochs > 0 && (n_epochs != 1 || epochs[0] != 0 || epochs[1] != n)) {
            set_error("execute_host: pooling across epoch gaps is not supported (pool the full-rate result instead)");
            return GCWT_ERR_UNSUPPORTED;
        }
    }
    Streamed s{p, n_channels, n, (char*)out, s_stride, c_stride, pool_width, pool_mode, bands};
    return walk_tiles(p, x, in_type, n_channels, n, x_stride, epochs, n_epochs, means_host, pool_width, s);
}

int check_event_args(int64_t n, const int64_t* epochs, int n_epochs, const int64_t* events, int64_t n_events,
                     int64_t lag_first, int64_t n_lags) {
    int64_t one_epoch[2] = {0, n};
    if (!epochs || n_epochs <= 0) { epochs = one_epoch; n_epochs = 1; }
    const int rc = check_epochs(epochs, n_epochs, n);
    if (rc) return rc;
    for (int64_t i = 0; i < n_events; ++i) {
        if (i > 0 && events[i] < events[i - 1]) {
            set_error("execute_host_events: events must be ascending (event " + std::to_string(i) + " at sample " +
                      std::to_string(events[i]) + " follows sample " + std::to_string(events[i - 1]) + ")");
            return GCWT_ERR_ARG;
        }
        int64_t w0 = 0, w1 = 0;
        bool inside = !__builtin_add_overflow(events[i], lag_first, &w0) && !__builtin_add_overflow(w0, n_lags, &w1);
        if (inside) {                                              // the last epoch that starts at or before w0
            int lo = 0, hi = n_epochs;
            while (lo < hi) {
                const int mid = (lo + hi) / 2;
                if (epochs[2 * mid] <= w0) lo = mid + 1; else hi = mid;
            }
            inside = lo > 0 && w1 <= epochs[2 * (lo - 1) + 1];
        }
        if (!inside) {
            set_error("execute_host_events: the window of event " + std::to_string(i) + " (sample " +
                      std::to_string(events[i]) + ") does not lie inside one epoch");
            return GCWT_ERR_ARG;
        }
    }
    return GCWT_OK;
}

// Event-locked sums: no tile travels.  After a tile's ev_done the copy stream adds the tile's part of every window that
// meets it into a per-group fp64 accumulator (event_reduce_kernel), and ev_out[b] keeps the next tile of slot b from
// overwriting d_out[b] before that reduction has read it.  After the group's last tile the accumulator travels once,
// through the pinned ring, and the host divides by n_events.  The events have passed check_event_args.
struct EventSums {
    gcwt_plan* p; const int64_t* events; int64_t n_events, lag_first, n_lags; double* power_out; double* phase_out;
    int64_t os_stride, oc_stride;
    gcwt_plan::HostStage& h = p->host;
    const int S = p->n_scales;
    static constexpr bool pinned = false;                          // the means reach the caller from the pinned ring
    double bytes_out = 0;
    int64_t alloc = 0;

    // a group's accumulator: gc x S x n_lags power sums, then as many double2 phase sums on a 16-byte boundary
    int64_t power_cells(int64_t gc) const { return (gc * S * n_lags + 1) & ~int64_t(1); }
    size_t acc_bytes(int64_t gc) const {
        return sizeof(double) * (size_t)power_cells(gc) + (phase_out ? sizeof(double2) * (size_t)(gc * S * n_lags) : 0);
    }

    int prepare(const TileGeometry& geo, const int64_t*, int) {
        alloc = geo.alloc;
        int rc = grow_device((void**)&h.d_acc, &h.acc_bytes, acc_bytes(geo.g), "execute_host_events");
        if (rc == GCWT_OK) rc = grow_device((void**)&h.d_events, &h.events_bytes, sizeof(int64_t) * n_events, "execute_host_events");
        if (rc == GCWT_OK) rc = grow_pinned(&h.h_ring[0], &h.ring_bytes[0], acc_bytes(geo.g), "execute_host_events");
        if (rc) return rc;
        GCWT_CUDA_OK(cudaMemcpyAsync(h.d_events, events, sizeof(int64_t) * n_events, cudaMemcpyHostToDevice, h.st_copy));
        return GCWT_OK;
    }
    int slot_free(int b) {                                         // on the device: the host never waits per tile
        GCWT_CUDA_OK(cudaStreamWaitEvent(h.st_compute, h.ev_out[b], 0));
        return GCWT_OK;
    }
    int group_begin(int64_t, int64_t gc) {
        const cudaError_t e = cudaMemsetAsync(h.d_acc, 0, acc_bytes(gc), h.st_copy);
        if (e != cudaSuccess) { set_error(std::string("execute_host_events: ") + cudaGetErrorString(e)); return GCWT_ERR_CUDA; }
        return GCWT_OK;
    }
    // add the tile's part of every window that meets it
    int tile(int b, int64_t, int64_t gc, int64_t a, int64_t len) {
        // the events whose windows start in (a - n_lags, a + len): a host-side binary search over ascending events
        const int64_t* lo = std::partition_point(events, events + n_events,
                                                 [&](int64_t e) { return e + lag_first <= a - n_lags; });
        const int64_t* hi = std::partition_point(lo, events + n_events, [&](int64_t e) { return e + lag_first < a + len; });
        const int r = event_reduce_launch(h.d_out[b], p->compute_type, p->out_kind, gc, S, len, alloc, (int64_t)S * alloc,
                                          a, h.d_events + (lo - events), hi - lo, lag_first, n_lags, h.d_acc,
                                          phase_out ? (double2*)(h.d_acc + power_cells(gc)) : nullptr, n_lags,
                                          (int64_t)S * n_lags, h.st_copy);
        if (r) return r;
        GCWT_CUDA_OK(cudaEventRecord(h.ev_out[b], h.st_copy));
        return GCWT_OK;
    }
    // the group's means: one D2H of its accumulator, then sum / n_events into the caller's arrays
    int group_end(int64_t c0, int64_t gc) {
        GCWT_CUDA_OK(cudaMemcpyAsync(h.h_ring[0], h.d_acc, acc_bytes(gc), cudaMemcpyDeviceToHost, h.st_copy));
        GCWT_CUDA_OK(cudaStreamSynchronize(h.st_copy));
        const double* sums = (const double*)h.h_ring[0];
        const double* phase_sums = sums + power_cells(gc);
        const double cnt = (double)n_events;
        for (int64_t c = 0; c < gc; ++c)
            for (int s = 0; s < S; ++s) {
                const int64_t row = c * S + s, o = (c0 + c) * oc_stride + (int64_t)s * os_stride;
                for (int64_t l = 0; l < n_lags; ++l) power_out[o + l] = sums[row * n_lags + l] / cnt;
                if (phase_out)
                    for (int64_t l = 0; l < 2 * n_lags; ++l) phase_out[2 * o + l] = phase_sums[2 * row * n_lags + l] / cnt;
            }
        bytes_out += (double)gc * S * n_lags * (sizeof(double) + (phase_out ? sizeof(double2) : 0));
        return GCWT_OK;
    }
};

int host_execute_events(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n, int64_t x_stride,
                        const int64_t* epochs, int n_epochs, const double* means_host, const int64_t* events,
                        int64_t n_events, int64_t lag_first, int64_t n_lags, double* power_out, double* phase_out,
                        int64_t os_stride, int64_t oc_stride) {
    EventSums s{p, events, n_events, lag_first, n_lags, power_out, phase_out, os_stride, oc_stride};
    return walk_tiles(p, x, in_type, n_channels, n, x_stride, epochs, n_epochs, means_host, 0, s);
}

}  // namespace gcwt
