// Host-buffer entry point: numpy in, numpy out, through a streamed, double-buffered pipeline.
//
// The reference returns a complete host array of shape (scales, samples) per channel
// (ghost/wave/transforms.py:185,231).  Here the caller's host buffers are the only full-size storage:
// the result is produced in tiles (a group of channels x all scales x a stretch of samples) that
// alternate between two device buffers, and tile k travels to the host while tile k + 1 is computed.
// Results larger than device memory (config 3: 295 GB per GPU) therefore work, the device holds one
// channel group's samples plus two tiles, and the link -- not the kernels -- sets the pace.
//
//   pinned destination (cudaHostAlloc / cudaHostRegister / torch pin_memory): rows are written by DMA,
//     one cudaMemcpy2DAsync per channel of a tile;
//   pageable destination (a plain numpy array): tiles land in a plan-owned pinned ring by DMA and a few
//     host threads copy the rows out (which also first-touches the caller's pages in parallel).
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

static int grow_device(void** ptr, size_t* have, size_t need) {
    if (*have >= need) return GCWT_OK;
    if (*ptr) { cudaFree(*ptr); *ptr = nullptr; *have = 0; }
    cudaError_t e = cudaMalloc(ptr, need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("execute_host: device staging of " + std::to_string(need) + " bytes: " + cudaGetErrorString(e));
        return GCWT_ERR_NOMEM;
    }
    *have = need;
    return GCWT_OK;
}

void host_stage_free(gcwt_plan* p) {
    gcwt_plan::HostStage& h = p->host;
    if (h.st_compute) cudaStreamSynchronize(h.st_compute);
    if (h.st_copy) cudaStreamSynchronize(h.st_copy);
    if (h.d_in) cudaFree(h.d_in);
    for (int b = 0; b < 2; ++b) {
        if (h.d_out[b]) cudaFree(h.d_out[b]);
        if (h.h_ring[b]) cudaFreeHost(h.h_ring[b]);
        if (h.d_pool[b]) cudaFree(h.d_pool[b]);
        if (h.h_pool[b]) cudaFreeHost(h.h_pool[b]);
        if (h.ev_done[b]) cudaEventDestroy(h.ev_done[b]);
        if (h.ev_out[b]) cudaEventDestroy(h.ev_out[b]);
    }
    if (h.d_means) cudaFree(h.d_means);
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
    const char* src; size_t src_pitch;          // ring: rows are dense (tile_alloc elements apart)
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

int host_execute(gcwt_plan* p, const void* x, int in_type, int64_t n_channels, int64_t n, int64_t x_stride,
                 const int64_t* epochs, int n_epochs, const double* means_host, void* out, int64_t s_stride,
                 int64_t c_stride, int64_t tile_hint, int64_t pool_width, int pool_mode, const BandTable* bands) {
    // pool_width > 0: `out` is a float64 array of ceil(n / pool_width) bins per row; every tile is reduced on the
    // device (mean or max over pool_width consecutive samples) and only the bins travel to the host.
    // bands: `out` holds (channels x bands x samples) of the plan's real type (s_stride is the band stride); every
    // tile is band-reduced on the device into d_pool and only the band rows travel, by the same pinned-DMA /
    // ring-and-copier routes as full-rate tiles (h_pool is the ring).  The tile geometry stays that of the
    // full-rate path, so every coefficient summed is the one gcwt_execute_host would have written.
    gcwt_plan::HostStage& h = p->host;
    const auto t_begin = std::chrono::steady_clock::now();
    const int S = p->n_scales;
    const size_t in_el = in_type == GCWT_F32 ? 4 : 8;
    size_t out_el = p->compute_type == GCWT_F32 ? 4 : 8;
    if (p->out_kind == GCWT_OUT_COMPLEX) out_el *= 2;
    const bool pooled = pool_width > 0, banded = bands != nullptr;
    const int R = banded ? bands->n_bands : S;                    // rows per channel that reach `out`
    const size_t xfer_el = banded ? (p->compute_type == GCWT_F32 ? 4 : 8) : out_el;
    int64_t one_epoch[2] = {0, n};
    if (!epochs || n_epochs <= 0) { epochs = one_epoch; n_epochs = 1; }
    for (int e = 0; e < n_epochs; ++e)
        if (epochs[2 * e] < 0 || epochs[2 * e + 1] > n || epochs[2 * e] >= epochs[2 * e + 1] ||
            (e > 0 && epochs[2 * e] < epochs[2 * e - 1])) {
            set_error("execute_host: epoch bounds must be ascending, non-empty and inside [0, n_samples)");
            return GCWT_ERR_ARG;
        }
    if (!h.st_compute) {
        GCWT_CUDA_OK(cudaStreamCreateWithFlags(&h.st_compute, cudaStreamNonBlocking));
        GCWT_CUDA_OK(cudaStreamCreateWithFlags(&h.st_copy, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            GCWT_CUDA_OK(cudaEventCreateWithFlags(&h.ev_done[b], cudaEventDisableTiming));
            GCWT_CUDA_OK(cudaEventCreateWithFlags(&h.ev_out[b], cudaEventDisableTiming));
        }
    }
    // ---- tile geometry: a group of g channels x all scales x a stretch of `tile` samples ----------
    int64_t lmax = 1;
    for (const ScaleInfo& sc : p->scales) lmax = std::max<int64_t>(lmax, sc.L);
    const int64_t halo = lmax - 1;
    const size_t budget = (size_t)1 << 30;                        // bytes per result tile (two on the device)
    const size_t per_channel = (size_t)S * (size_t)n * out_el;
    int64_t g = std::max<int64_t>(1, std::min<int64_t>(n_channels, (int64_t)(budget / std::max<size_t>(per_channel, 1))));
    int64_t tile = n;
    if (per_channel > budget) {
        tile = std::max<int64_t>((int64_t)(budget / ((size_t)S * out_el)), std::min<int64_t>(n, 4 * lmax));
        tile = std::min<int64_t>(n, (tile + 1023) / 1024 * 1024);
    }
    if (tile_hint > 0) tile = std::min<int64_t>(n, std::max<int64_t>(tile_hint, 1024));
    if (pooled) {
        if (p->out_kind == GCWT_OUT_COMPLEX) { set_error("execute_host: pooling needs amplitude or power output"); return GCWT_ERR_ARG; }
        if (n_epochs != 1 || epochs[0] != 0 || epochs[1] != n) {
            set_error("execute_host: pooling across epoch gaps is not supported (pool the full-rate result instead)");
            return GCWT_ERR_UNSUPPORTED;
        }
        if (tile < n) tile = std::max<int64_t>(pool_width, tile / pool_width * pool_width);   // tiles end on bin boundaries
    }
    const int64_t bins_per_tile = pooled ? (tile + pool_width - 1) / pool_width : 0;
    const int64_t tile_alloc = (tile + 3) & ~int64_t(3);          // rows of a tile stay 16-byte aligned
    const size_t tile_bytes = (size_t)g * S * tile_alloc * out_el;
    int rc = grow_device(&h.d_in, &h.in_bytes, (size_t)g * n * in_el);
    if (rc) return rc;
    for (int b = 0; b < 2; ++b) {
        size_t have = h.out_bytes;
        rc = grow_device(&h.d_out[b], &have, tile_bytes);
        if (rc) return rc;
        if (b == 1) h.out_bytes = have;
    }
    if (h.means_cap < g) {
        if (h.d_means) cudaFree(h.d_means);
        h.d_means = nullptr; h.means_cap = 0;
        GCWT_CUDA_OK(cudaMalloc((void**)&h.d_means, sizeof(double) * g));
        h.means_cap = g;
    }
    const size_t reduced_bytes = pooled ? (size_t)g * S * bins_per_tile * sizeof(double)
                                        : banded ? (size_t)g * R * tile_alloc * xfer_el : 0;
    if (h.pool_bytes < reduced_bytes) {
        for (int b = 0; b < 2; ++b) {
            if (h.d_pool[b]) { cudaFree(h.d_pool[b]); h.d_pool[b] = nullptr; }
            if (h.h_pool[b]) { cudaFreeHost(h.h_pool[b]); h.h_pool[b] = nullptr; }
        }
        h.pool_bytes = 0;
        for (int b = 0; b < 2; ++b) {
            GCWT_CUDA_OK(cudaMalloc(&h.d_pool[b], reduced_bytes));
            GCWT_CUDA_OK(cudaMallocHost(&h.h_pool[b], reduced_bytes));
        }
        h.pool_bytes = reduced_bytes;
    }
    const bool direct = pooled || is_pinned(out);
    if (!direct && !banded && h.ring_bytes < tile_bytes) {
        for (int b = 0; b < 2; ++b) {
            if (h.h_ring[b]) { cudaFreeHost(h.h_ring[b]); h.h_ring[b] = nullptr; }
            cudaError_t e = cudaMallocHost(&h.h_ring[b], tile_bytes);
            if (e != cudaSuccess) {
                cudaGetLastError(); h.ring_bytes = 0;
                set_error(std::string("execute_host: pinned staging: ") + cudaGetErrorString(e));
                return GCWT_ERR_NOMEM;
            }
        }
        h.ring_bytes = tile_bytes;
    }
    // copier threads of the pageable path (measured on a 16-core host, 6.9 GB per call: 8 threads 34 GB/s, see DESIGN.md)
    int n_threads = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency() > 2 ? std::thread::hardware_concurrency() - 2 : 1u));
    if (const char* e = getenv("GCWT_HOST_THREADS")) n_threads = std::max(1, atoi(e));

    // zero rows outside the epochs (the reference starts from np.zeros, transforms.py:185)
    if (!pooled) {
        int64_t pos = 0;
        for (int e = 0; e <= n_epochs; ++e) {
            const int64_t gap_end = e < n_epochs ? epochs[2 * e] : n;
            if (gap_end > pos)
                for (int64_t c = 0; c < n_channels; ++c)
                    for (int s = 0; s < R; ++s)
                        memset((char*)out + ((size_t)c * c_stride + (size_t)s * s_stride + pos) * xfer_el, 0, (size_t)(gap_end - pos) * xfer_el);
            if (e < n_epochs) pos = epochs[2 * e + 1];
        }
    }

    struct Pending { bool live = false; int64_t c0 = 0, gc = 0, a = 0, len = 0; };
    auto drain_pool = [&](int b, const Pending& pd) {              // pooled tile: pinned staging -> the caller's float64 rows
        const int64_t nb = (pd.len + pool_width - 1) / pool_width, b0 = pd.a / pool_width;
        for (int64_t c = 0; c < pd.gc; ++c)
            for (int s = 0; s < S; ++s)
                memcpy((double*)out + (size_t)(pd.c0 + c) * c_stride + (size_t)s * s_stride + b0,
                       (const double*)h.h_pool[b] + ((size_t)c * S + s) * bins_per_tile, (size_t)nb * sizeof(double));
    };
    Pending pend[2];
    struct Copiers {                                               // joined on every return path (an early error return
        std::thread t[2];                                          // must not destroy a running thread)
        ~Copiers() { for (auto& th : t) if (th.joinable()) th.join(); }
        std::thread& operator[](int i) { return t[i]; }
    } copier;
    auto finish = [&](int b) -> int {                              // tile in slot b has reached the caller's array
        if (!pend[b].live) return GCWT_OK;
        if (pooled) {
            GCWT_CUDA_OK(cudaEventSynchronize(h.ev_out[b]));
            drain_pool(b, pend[b]);
        } else if (direct) {
            GCWT_CUDA_OK(cudaEventSynchronize(h.ev_out[b]));
        } else if (copier[b].joinable()) {
            copier[b].join();
        }
        pend[b].live = false;
        return GCWT_OK;
    };
    int slot = 0;
    int64_t n_tiles = 0;
    double bytes_out = 0;
    for (int64_t c0 = 0; c0 < n_channels && rc == GCWT_OK; c0 += g) {
        const int64_t gc = std::min<int64_t>(g, n_channels - c0);
        // the group's samples and means; the previous group's tiles may still be copying out, but nothing reads
        // d_in any more: every execute of that group has completed (gcwt_execute waits, or we wait below)
        GCWT_CUDA_OK(cudaStreamSynchronize(h.st_compute));
        GCWT_CUDA_OK(cudaMemcpy2DAsync(h.d_in, (size_t)n * in_el, (const char*)x + (size_t)c0 * x_stride * in_el, (size_t)x_stride * in_el,
                                       (size_t)n * in_el, (size_t)gc, cudaMemcpyHostToDevice, h.st_compute));
        if (means_host) {
            GCWT_CUDA_OK(cudaMemcpyAsync(h.d_means, means_host + c0, sizeof(double) * gc, cudaMemcpyHostToDevice, h.st_compute));
        } else {
            const int64_t need = (int64_t)means_blocks(n) * gc;
            if (p->partial_cap < need) {
                GCWT_CUDA_OK(cudaStreamSynchronize(h.st_compute));
                if (p->d_partial) cudaFree(p->d_partial);
                p->d_partial = nullptr; p->partial_cap = 0;
                GCWT_CUDA_OK(cudaMalloc((void**)&p->d_partial, sizeof(double) * need));
                p->partial_cap = need;
            }
            rc = means_launch(h.d_in, in_type, gc, n, n, h.d_means, p->d_partial, h.st_compute);
            if (rc) break;
        }
        for (int e = 0; e < n_epochs && rc == GCWT_OK; ++e) {
            const int64_t e0 = epochs[2 * e], e1 = epochs[2 * e + 1];
            for (int64_t a = e0; a < e1 && rc == GCWT_OK; a += tile) {
                const int64_t b_end = std::min(e1, a + tile), len = b_end - a;
                rc = finish(slot);                                 // the slot's previous tile has left the device buffer / ring
                if (rc) break;
                rc = gcwt_execute(p, (const char*)h.d_in + (size_t)a * in_el, in_type, gc, len, n, std::min(halo, a - e0),
                                  std::min(halo, e1 - b_end), h.d_means, h.d_out[slot], tile_alloc, (int64_t)S * tile_alloc,
                                  h.st_compute);
                if (rc) break;
                // ev_done follows the whole of gcwt_execute in stream order, including the accuracy guard's fp64
                // re-computation of the failing (channel, scale) pairs (guard_resolve), so the reductions below read
                // the corrected coefficients.  For the same reason band power is a pass of its own and not part of
                // the fused kernels' epilogue: there it would sum values the guard then replaces.
                GCWT_CUDA_OK(cudaEventRecord(h.ev_done[slot], h.st_compute));
                GCWT_CUDA_OK(cudaStreamWaitEvent(h.st_copy, h.ev_done[slot], 0));
                char* dst = (char*)out + ((size_t)c0 * c_stride + (size_t)a) * xfer_el;
                const void* src = h.d_out[slot];                   // what travels: the tile, or its band rows
                void* ring = h.h_ring[slot];
                if (banded) {
                    rc = band_reduce_launch(h.d_out[slot], p->compute_type, p->out_kind, gc, len, tile_alloc, (int64_t)S * tile_alloc,
                                            *bands, h.d_pool[slot], tile_alloc, (int64_t)R * tile_alloc, h.st_copy);
                    if (rc) break;
                    src = h.d_pool[slot];
                    ring = h.h_pool[slot];
                }
                if (pooled) {
                    rc = pool_rows_launch(h.d_out[slot], p->compute_type, gc * S, len, tile_alloc, pool_width, pool_mode, 0,
                                          (double*)h.d_pool[slot], bins_per_tile, h.st_copy);
                    if (rc) break;
                    GCWT_CUDA_OK(cudaMemcpyAsync(h.h_pool[slot], h.d_pool[slot], (size_t)gc * S * bins_per_tile * sizeof(double),
                                                 cudaMemcpyDeviceToHost, h.st_copy));
                    GCWT_CUDA_OK(cudaEventRecord(h.ev_out[slot], h.st_copy));
                } else if (direct) {
                    for (int64_t c = 0; c < gc; ++c)
                        GCWT_CUDA_OK(cudaMemcpy2DAsync(dst + (size_t)c * c_stride * xfer_el, (size_t)s_stride * xfer_el,
                                                       (const char*)src + (size_t)c * R * tile_alloc * xfer_el,
                                                       (size_t)tile_alloc * xfer_el, (size_t)len * xfer_el, (size_t)R,
                                                       cudaMemcpyDeviceToHost, h.st_copy));
                    GCWT_CUDA_OK(cudaEventRecord(h.ev_out[slot], h.st_copy));
                } else {
                    GCWT_CUDA_OK(cudaMemcpyAsync(ring, src, (size_t)gc * R * tile_alloc * xfer_el,
                                                 cudaMemcpyDeviceToHost, h.st_copy));
                    GCWT_CUDA_OK(cudaEventRecord(h.ev_out[slot], h.st_copy));
                    RowCopy rcp;
                    rcp.src = (const char*)ring; rcp.src_pitch = (size_t)tile_alloc * xfer_el;
                    rcp.dst = dst; rcp.s_stride_b = s_stride * (int64_t)xfer_el; rcp.c_stride_b = c_stride * (int64_t)xfer_el;
                    rcp.rows_per_channel = R; rcp.width = (size_t)len * xfer_el; rcp.n_rows = gc * R;
                    cudaEvent_t ev = h.ev_out[slot];
                    const int dev = p->device;
                    copier[slot] = std::thread([rcp, ev, dev, n_threads]() {
                        cudaSetDevice(dev);
                        cudaEventSynchronize(ev);
                        copy_rows(rcp, n_threads);
                    });
                }
                pend[slot].live = true; pend[slot].c0 = c0; pend[slot].gc = gc; pend[slot].a = a; pend[slot].len = len;
                bytes_out += pooled ? (double)gc * S * ((len + pool_width - 1) / pool_width) * sizeof(double) : (double)gc * R * len * xfer_el;
                ++n_tiles;
                slot ^= 1;
            }
        }
    }
    for (int b = 0; b < 2; ++b) {
        const int r2 = finish(b);
        if (rc == GCWT_OK) rc = r2;
        if (copier[b].joinable()) copier[b].join();
    }
    cudaStreamSynchronize(h.st_copy);
    cudaStreamSynchronize(h.st_compute);
    h.last_ms[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    h.last_ms[1] = direct ? 1.0 : 0.0;
    h.last_ms[2] = (double)n_tiles;
    h.last_ms[3] = bytes_out;
    return rc;
}

}  // namespace gcwt
