"""Thin Python handle on a device plan (ctypes over include/ghost_cwt.h).

PyTorch supplies device buffers and streams only; all arithmetic happens in
libghostcwt.so.  A plan is built from the host planner's per-scale tables and is
independent of the recording length.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

__all__ = ["CwtPlan", "scale_tables", "band_tables", "event_windows", "OUT_KINDS"]

OUT_KINDS = {"complex": _lib.OUT_COMPLEX, "amplitude": _lib.OUT_AMPLITUDE, "power": _lib.OUT_POWER}
BAND_REDUCE = ("mean", "sum")


def band_tables(frequencies, bands, reduce="mean"):
    """Map frequency bands in Hz to the scale rows of a grid: ``(first, count, weights)`` for
    gcwt_band_reduce / gcwt_execute_host_bands.

    Band ``(lo, hi)`` holds every scale whose grid frequency f satisfies ``lo <= f <= hi``; on a monotone grid
    that is one contiguous run of rows ``first .. first + count - 1``.  Bands keep the caller's order and may
    overlap.  ``reduce='mean'`` weights each scale 1 / count, ``'sum'`` weights it 1."""
    if reduce not in BAND_REDUCE:
        raise ValueError("'band_reduce' must be 'mean' or 'sum' but got {}".format(reduce))
    f = np.asarray(frequencies, dtype=np.float64).ravel()
    try:
        bands = [(float(lo), float(hi)) for lo, hi in bands]
    except (TypeError, ValueError):
        raise ValueError("'bands' must be a sequence of (low, high) pairs in Hz") from None
    if not bands:
        raise ValueError("'bands' must hold at least one (low, high) pair")
    first, count = [], []
    for lo, hi in bands:
        if not (lo > 0 and hi > 0):
            raise ValueError("band ({}, {}) Hz: limits must be positive".format(lo, hi))
        if lo > hi:
            raise ValueError("band ({}, {}) Hz: low limit above high limit".format(lo, hi))
        idx = np.nonzero((f >= lo) & (f <= hi))[0]
        if idx.size == 0:
            grid = "the grid is empty" if f.size == 0 else "the grid spans {:.6g} .. {:.6g} Hz".format(f.min(), f.max())
            raise ValueError("band ({}, {}) Hz holds no scale: {}".format(lo, hi, grid))
        if idx[-1] - idx[0] + 1 != idx.size:
            raise ValueError("band ({}, {}) Hz: the frequency grid is not monotone".format(lo, hi))
        first.append(int(idx[0]))
        count.append(int(idx.size))
    count = np.asarray(count, dtype=np.int32)
    weights = np.concatenate([np.full(c, 1.0 / c if reduce == "mean" else 1.0) for c in count])
    return np.asarray(first, dtype=np.int32), count, np.ascontiguousarray(weights, dtype=np.float64)


def event_windows(time, events_s, window_s, epoch_bounds, fs):
    """Map events in seconds to sample indices for gcwt_execute_host_events / gcwt_event_reduce: ``(samples,
    kept_mask, lag_first, n_lags)``.

    Each event goes to its nearest timestamp of ``time``; one more than half a sample period from every timestamp
    (inside a gap) is dropped.  ``window_s = (t_pre, t_post)`` gives ``lag_first = round(t_pre * fs)`` and ``n_lags =
    round(t_post * fs) - lag_first + 1``.  An event whose window ``[sample + lag_first, sample + lag_first + n_lags)``
    leaves its epoch (``epoch_bounds``: (E, 2) [start, stop) sample indices) is dropped as well.  ``samples`` holds
    the kept events' indices in the caller's order, ``kept_mask`` one flag per given event."""
    try:
        t_pre, t_post = (float(v) for v in window_s)
    except (TypeError, ValueError):
        raise ValueError("'event_window' must be a (t_pre, t_post) pair in seconds") from None
    fs = float(fs)
    lag_first = int(round(t_pre * fs))
    n_lags = int(round(t_post * fs)) - lag_first + 1
    if n_lags < 1:
        raise ValueError("event window ({}, {}) s holds no sample at {} Hz".format(t_pre, t_post, fs))
    t = np.asarray(time, dtype=np.float64).ravel()
    ev = np.asarray(events_s, dtype=np.float64).ravel()
    if ev.size == 0:
        raise ValueError("'events' is empty")
    if not np.all(np.isfinite(ev)):
        raise ValueError("'events' must be finite times in seconds")
    # nearest timestamp: the one at or after the event, or the one before it
    hi = np.clip(np.searchsorted(t, ev), 0, t.size - 1)
    lo = np.clip(hi - 1, 0, t.size - 1)
    idx = np.where(np.abs(t[lo] - ev) <= np.abs(t[hi] - ev), lo, hi)
    kept = np.abs(t[idx] - ev) <= 0.5 / fs * (1 + 1e-9)        # an event midway between two samples is kept
    bounds = np.asarray(epoch_bounds, dtype=np.int64).reshape(-1, 2)
    w0 = idx + lag_first
    ep = np.clip(np.searchsorted(bounds[:, 0], w0, side="right") - 1, 0, None)
    kept &= (w0 >= bounds[ep, 0]) & (w0 + n_lags <= bounds[ep, 1])
    if not kept.any():
        raise ValueError("no event has its whole window ({}, {}) s inside one epoch of the recording".format(
            t_pre, t_post))
    return idx[kept].astype(np.int64), kept, lag_first, n_lags


def _band_args(first, count, weights):
    first = np.ascontiguousarray(first, dtype=np.int32)
    count = np.ascontiguousarray(count, dtype=np.int32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    if first.ndim != 1 or first.shape != count.shape or weights.shape != (int(count.sum()),):
        raise ValueError("first and count need one entry per band and weights one per (band, scale) entry")
    return first, count, weights


def scale_tables(wavelet, norm_radian_freqs, lengths):
    """Per-scale (k_first, n_terms, concatenated X[k]) for the C plan descriptor."""
    k_first, n_terms, terms = [], [], []
    for w, L in zip(np.atleast_1d(norm_radian_freqs), np.atleast_1d(lengths)):
        k0, X = wavelet.spectrum_terms(int(L), float(w))
        k_first.append(k0)
        n_terms.append(len(X))
        terms.append(X)
    return (np.asarray(k_first, dtype=np.int32), np.asarray(n_terms, dtype=np.int32),
            np.ascontiguousarray(np.concatenate(terms), dtype=np.float64))


def _torch():
    import torch
    return torch


class CwtPlan:
    """Device tables for one set of scales."""

    def __init__(self, lengths, k_first, n_terms, terms, *, dtype=np.float32, output="amplitude",
                 device=0, force_generic=False, no_interp=False, band_tol=0.0, guard=True, guard_tol=0.0):
        dtype = np.dtype(dtype)
        if dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise ValueError("dtype must be float32 or float64 but got {}".format(dtype))
        if output not in OUT_KINDS:
            raise ValueError("output must be 'amplitude', 'power' or 'complex' but got {}".format(output))
        self.lib = _lib.load()
        self.dtype = dtype
        self.output = output
        self.device = int(device)
        self.lengths = np.ascontiguousarray(lengths, dtype=np.int64)
        self.n_scales = int(self.lengths.size)
        self._k_first = np.ascontiguousarray(k_first, dtype=np.int32)
        self._n_terms = np.ascontiguousarray(n_terms, dtype=np.int32)
        self._terms = np.ascontiguousarray(terms, dtype=np.float64)
        desc = _lib.PlanDesc()
        desc.n_scales = self.n_scales
        desc.lengths = self.lengths.ctypes.data_as(C.POINTER(C.c_int64))
        desc.k_first = self._k_first.ctypes.data_as(C.POINTER(C.c_int32))
        desc.n_terms = self._n_terms.ctypes.data_as(C.POINTER(C.c_int32))
        desc.terms = self._terms.ctypes.data_as(C.POINTER(C.c_double))
        desc.compute_type = _lib.F32 if dtype == np.float32 else _lib.F64
        desc.out_kind = OUT_KINDS[output]
        desc.device = self.device
        desc.flags = (_lib.FLAG_FORCE_GENERIC if force_generic else 0) | (_lib.FLAG_NO_INTERP if no_interp else 0) \
            | (0 if guard else _lib.FLAG_NO_GUARD)
        desc.band_tol = float(band_tol)
        desc.guard_tol = float(guard_tol)
        handle = C.c_void_p()
        _lib.check(self.lib.gcwt_plan_create(C.byref(handle), C.byref(desc)))
        self._h = handle

    # ------------------------------------------------------------------ info
    @property
    def max_length(self):
        return int(self.lengths.max())

    def levels(self):
        out = np.empty(self.n_scales, dtype=np.int32)
        _lib.check(self.lib.gcwt_plan_levels(self._h, out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def classes(self):
        """Scale classes of the fp32 fused kernels (include/ghost_cwt.h, gcwt_plan_classes): a list of dicts
        (level, kernel as planned: 'full' / 'banded' / 'interp' / 'wide2', log2u, n_scales, and the chunk,
        offset and hop of the chunk that kernel transforms), and per scale its class index (-1: generic path)."""
        n = C.c_int32()
        _lib.check(self.lib.gcwt_plan_classes(self._h, C.byref(n), None, None))
        info = (_lib.ClassInfo * max(1, n.value))()
        of_scale = np.empty(self.n_scales, dtype=np.int32)
        _lib.check(self.lib.gcwt_plan_classes(self._h, C.byref(n), info, of_scale.ctypes.data_as(C.POINTER(C.c_int32))))
        names = {_lib.KERNEL_FULL: "full", _lib.KERNEL_BANDED: "banded", _lib.KERNEL_INTERP: "interp",
                 _lib.KERNEL_WIDE2: "wide2"}
        out = [{"level": c.level, "kernel": names[c.kernel], "log2u": c.log2u, "n_scales": c.n_scales,
                "chunk": c.chunk, "offset": c.offset, "hop": c.hop} for c in info[:n.value]]
        return out, of_scale

    def guard_stats(self):
        """Accuracy guard of the fp32 paths (include/ghost_cwt.h, gcwt_guard_stats): dict with the
        (channel, scale) pairs re-computed in fp64 by the last execute, in total, the pairs examined
        so far, and a per-scale flag array of the last execute."""
        last, total, checked = C.c_int64(), C.c_int64(), C.c_int64()
        flags = np.zeros(self.n_scales, dtype=np.uint8)
        _lib.check(self.lib.gcwt_guard_stats(self._h, C.byref(last), C.byref(total), C.byref(checked),
                                             flags.ctypes.data_as(C.POINTER(C.c_ubyte))))
        return {"last": int(last.value), "total": int(total.value), "checked": int(checked.value),
                "scales": flags.astype(bool)}

    def workspace_bytes(self):
        return int(self.lib.gcwt_plan_workspace_bytes(self._h))

    @property
    def torch_out_dtype(self):
        torch = _torch()
        if self.output == "complex":
            return torch.complex64 if self.dtype == np.float32 else torch.complex128
        return torch.float32 if self.dtype == np.float32 else torch.float64

    # ------------------------------------------------------------------ run
    def alloc_out(self, n_channels, n_samples):
        torch = _torch()
        return torch.empty((n_channels, self.n_scales, n_samples), dtype=self.torch_out_dtype,
                           device="cuda:%d" % self.device)

    def channel_means(self, x, n_samples=None):
        """float64 mean per channel of a (C, N) device tensor (reference transforms.py:143)."""
        torch = _torch()
        n = x.shape[1] if n_samples is None else int(n_samples)
        means = torch.empty(x.shape[0], dtype=torch.float64, device=x.device)
        in_type = _lib.F32 if x.dtype == torch.float32 else _lib.F64
        st = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self.lib.gcwt_channel_means(x.data_ptr(), in_type, x.shape[0], n, x.stride(0),
                                               means.data_ptr(), self.device, st))
        return means

    def execute(self, x, out=None, *, means=None, start=0, stop=None, halo_left=0, halo_right=0,
                out_start=None):
        """Transform samples ``[start, stop)`` of every channel of ``x`` (C, N) into
        ``out[:, :, out_start : out_start + stop - start]`` (``out_start`` defaults to
        ``start``).  ``x`` and ``out`` are CUDA tensors; ``out`` is (C, S, >= needed)."""
        torch = _torch()
        if x.dim() != 2 or not x.is_cuda or x.stride(1) != 1:
            raise ValueError("x must be a (channels, samples) CUDA tensor with unit sample stride")
        if x.dtype not in (torch.float32, torch.float64):
            raise ValueError("x must be float32 or float64")
        n_ch, n_all = x.shape
        stop = n_all if stop is None else int(stop)
        start = int(start)
        if not (0 <= start < stop <= n_all):
            raise ValueError("bad segment [{}, {})".format(start, stop))
        if halo_left > start or halo_right > n_all - stop:
            raise ValueError("halo reaches outside the tensor")
        out_start = start if out_start is None else int(out_start)
        if out is None:
            out = self.alloc_out(n_ch, out_start + stop - start)
        if out.dtype != self.torch_out_dtype or out.dim() != 3 or out.stride(2) != 1 \
                or out.shape[0] != n_ch or out.shape[1] != self.n_scales \
                or out_start < 0 or out.shape[2] < out_start + stop - start:
            raise ValueError("out must be (channels, scales, samples) of dtype %s" % self.torch_out_dtype)
        esz = x.element_size()
        osz = out.element_size()
        mptr = None
        if means is not None:
            if means.dtype != torch.float64 or means.numel() != n_ch or not means.is_cuda:
                raise ValueError("means must be a float64 CUDA tensor with one entry per channel")
            mptr = means.data_ptr()
        st = torch.cuda.current_stream(x.device).cuda_stream
        in_type = _lib.F32 if x.dtype == torch.float32 else _lib.F64
        _lib.check(self.lib.gcwt_execute(
            self._h, x.data_ptr() + start * esz, in_type, n_ch, stop - start, x.stride(0),
            int(halo_left), int(halo_right), mptr,
            out.data_ptr() + out_start * osz, out.stride(1), out.stride(0), st))
        return out

    def execute_tiled(self, x, tile, out=None, consumer=None, means=None):
        """Transform a recording whose result does not fit in device memory.

        The samples are cut into tiles of ``tile`` samples; each tile is transformed with
        real-sample halos on both sides (exact: the filters are FIR, see DESIGN.md) into
        the same reused ``out`` buffer (C, S, tile) and handed to ``consumer(out, start,
        stop)`` -- which must be done with the buffer when it returns (same stream).
        Returns the number of coefficients produced."""
        torch = _torch()
        n_ch, n = x.shape
        tile = int(min(tile, n))
        if out is None:
            out = self.alloc_out(n_ch, tile)
        if means is None:
            means = self.channel_means(x)
        halo = self.max_length - 1
        done = 0
        for a in range(0, n, tile):
            b = min(n, a + tile)
            self.execute(x, out, means=means, start=a, stop=b, halo_left=min(halo, a),
                         halo_right=min(halo, n - b), out_start=0)
            if consumer is not None:
                consumer(out, a, b)
            done += (b - a) * n_ch * self.n_scales
        return done

    def _host_args(self, x, means, epochs):
        """Leading ctypes arguments of the gcwt_execute_host* entry points: ``x`` (channels, samples) or (samples,),
        promoted to float64 unless it and the plan are float32, with unit sample stride; ``means`` one float64 per
        channel; ``epochs`` (E, 2) int64 [start, stop) bounds.  Returns ``(n_channels, n_samples, x_args,
        epoch_args, means_ptr)``; every pointer keeps its array alive."""
        x = np.asarray(x)
        if x.ndim == 1:
            x = x[None, :]
        if x.ndim != 2:
            raise ValueError("x must be (channels, samples)")
        if x.dtype not in (np.float32, np.float64) or (self.dtype == np.float64 and x.dtype != np.float64):
            x = x.astype(np.float64)
        if x.strides[1] != x.itemsize:
            x = np.ascontiguousarray(x)
        n_ch, n = x.shape
        if means is not None:
            means = np.ascontiguousarray(means, dtype=np.float64)
            if means.size != n_ch:
                raise ValueError("means must hold one value per channel")
        if epochs is not None:
            epochs = np.ascontiguousarray(epochs, dtype=np.int64).reshape(-1, 2)

        def ptr(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)
        in_type = _lib.F32 if x.dtype == np.float32 else _lib.F64
        return (n_ch, n, (ptr(x), in_type, n_ch, n, x.strides[0] // x.itemsize),
                (ptr(epochs), 0 if epochs is None else int(epochs.shape[0])), ptr(means))

    def execute_host(self, x, out=None, means=None, epochs=None):
        """Host-buffer entry point (numpy in, numpy out) through gcwt_execute_host: the whole transform
        body of the reference (global mean removal, one zero-padded convolution per epoch, zeros outside
        the epochs; transforms.py:142-143,185,202-204) as one streamed, double-buffered call.

        ``x`` (channels, samples) or (samples,); ``out`` optional (channels, scales, samples) array of the
        plan's output dtype with unit sample stride -- pass a pinned one (e.g. the numpy view of a
        ``torch.empty(..., pin_memory=True)``) to let the device write it by DMA; ``epochs`` optional
        (E, 2) array of [start, stop) sample bounds.  Results larger than device memory are fine."""
        n_ch, n, xa, ea, mp = self._host_args(x, means, epochs)
        if self.output == "complex":
            odt = np.dtype(np.complex64 if self.dtype == np.float32 else np.complex128)
        else:
            odt = self.dtype
        if out is None:
            out = np.empty((n_ch, self.n_scales, n), dtype=odt)
        if out.dtype != odt or out.shape != (n_ch, self.n_scales, n) or out.strides[2] != out.itemsize \
                or out.strides[0] % out.itemsize or out.strides[1] % out.itemsize:
            raise ValueError("out must be (channels, scales, samples) of dtype %s with unit sample stride" % odt)
        _lib.check(self.lib.gcwt_execute_host(self._h, *xa, *ea, mp, out.ctypes.data, out.strides[1] // out.itemsize,
                                              out.strides[0] // out.itemsize))
        return out

    def execute_host_pooled(self, x, pool_width, pool="mean", means=None):
        """As :meth:`execute_host` (one epoch, amplitude or power plans), but every tile is pooled on the
        device: runs of ``pool_width`` consecutive samples are reduced to their mean (``pool='mean'``) or
        maximum (``'max'``) and only those float64 bins cross the link.  Returns (channels, scales,
        ceil(samples / pool_width)) float64 -- what a display of a few thousand columns needs
        (reference plot: transforms.py:356-367,395-396)."""
        if pool not in ("mean", "max"):
            raise ValueError("pool must be 'mean' or 'max' but got {}".format(pool))
        pool_width = int(pool_width)
        if pool_width < 1:
            raise ValueError("pool_width must be a positive integer")
        n_ch, n, xa, _, mp = self._host_args(x, means, None)
        n_bins = -(-n // pool_width)
        out = np.empty((n_ch, self.n_scales, n_bins), dtype=np.float64)
        _lib.check(self.lib.gcwt_execute_host_pooled(
            self._h, *xa, mp, pool_width, _lib.POOL_MEAN if pool == "mean" else _lib.POOL_MAX, out.ctypes.data,
            n_bins, n_bins * self.n_scales))
        return out

    def pool_rows(self, res, pool_width, pool="mean", square=False):
        """Pool the last axis of a contiguous CUDA tensor (a device-resident result) in runs of ``pool_width``
        samples: float64 CUDA tensor with ceil(n / pool_width) bins per row.  ``square`` pools the squares."""
        torch = _torch()
        if not res.is_cuda or res.is_complex() or res.dtype not in (torch.float32, torch.float64) or res.stride(-1) != 1:
            raise ValueError("pool_rows needs a real float32 / float64 CUDA tensor with unit stride along the last axis")
        if pool not in ("mean", "max"):
            raise ValueError("pool must be 'mean' or 'max' but got {}".format(pool))
        flat = res.reshape(-1, res.shape[-1]) if res.is_contiguous() else None
        if flat is None:
            if res.dim() != 2:
                raise ValueError("pool_rows needs a contiguous tensor (or a 2-D one with a row stride)")
            flat = res
        n_rows, n = flat.shape
        n_bins = -(-n // int(pool_width))
        out = torch.empty((n_rows, n_bins), dtype=torch.float64, device=res.device)
        st = torch.cuda.current_stream(res.device).cuda_stream
        _lib.check(self.lib.gcwt_pool_rows(flat.data_ptr(), _lib.F32 if res.dtype == torch.float32 else _lib.F64, n_rows, n,
                                           flat.stride(0), int(pool_width), _lib.POOL_MEAN if pool == "mean" else _lib.POOL_MAX,
                                           1 if square else 0, out.data_ptr(), n_bins, self.device, st))
        return out.reshape(tuple(res.shape[:-1]) + (n_bins,))

    def execute_host_bands(self, x, first, count, weights, epochs=None, means=None):
        """As :meth:`execute_host`, but every tile is reduced to scale-averaged band power on the device
        (gcwt_execute_host_bands) and only (channels, bands, samples) of the plan's real dtype crosses the link.
        Band b is ``sum_k weights[off_b + k] * |W[:, first[b] + k, :]|**2`` (see :func:`band_tables`); samples
        outside the ``epochs`` are zero."""
        first, count, weights = _band_args(first, count, weights)
        n_ch, n, xa, ea, mp = self._host_args(x, means, epochs)
        n_b = int(first.size)
        out = np.empty((n_ch, n_b, n), dtype=self.dtype)
        _lib.check(self.lib.gcwt_execute_host_bands(
            self._h, *xa, *ea, mp, n_b, first.ctypes.data, count.ctypes.data, weights.ctypes.data, out.ctypes.data,
            n, n_b * n))
        return out

    def _device_coef_args(self, res, who):
        """Checks a device-resident (channels, scales, samples) result; returns its real dtype, type code, kind (a
        real ``res`` holds this plan's ``output``) and the current stream of its device."""
        torch = _torch()
        if not res.is_cuda or res.dim() != 3 or res.stride(2) != 1 or \
                res.dtype not in (torch.float32, torch.float64, torch.complex64, torch.complex128):
            raise ValueError(who + " needs a (channels, scales, samples) float / complex CUDA tensor with unit "
                             "sample stride")
        rdt = {torch.complex64: torch.float32, torch.complex128: torch.float64}.get(res.dtype, res.dtype)
        kind = _lib.OUT_COMPLEX if res.is_complex() else (_lib.OUT_POWER if self.output == "power" else _lib.OUT_AMPLITUDE)
        return rdt, _lib.F32 if rdt == torch.float32 else _lib.F64, kind, torch.cuda.current_stream(res.device).cuda_stream

    def band_reduce(self, res, first, count, weights):
        """Scale-averaged band power of a device-resident (channels, scales, samples) result ``res`` (a CUDA
        tensor with unit sample stride; a window of a larger result is fine): a (channels, bands, samples) CUDA
        tensor of ``res``'s real dtype, through gcwt_band_reduce on the current stream.  |W|^2 is re^2 + im^2
        for a complex tensor, and for a real one the square of an amplitude or the power itself, as this
        plan's ``output`` says."""
        torch = _torch()
        first, count, weights = _band_args(first, count, weights)
        rdt, code, kind, st = self._device_coef_args(res, "band_reduce")
        if int((first + count).max()) > res.shape[1]:
            raise ValueError("a band reaches past the {} scales of the result".format(res.shape[1]))
        n_ch, _, n = res.shape
        out = torch.empty((n_ch, first.size, n), dtype=rdt, device=res.device)
        _lib.check(self.lib.gcwt_band_reduce(
            res.data_ptr(), code, kind, n_ch, n, res.stride(1), res.stride(0), int(first.size), first.ctypes.data,
            count.ctypes.data, weights.ctypes.data, out.data_ptr(), n, first.size * n, res.device.index, st))
        return out

    def execute_host_events(self, x, events, lag_first, n_lags, epochs=None, means=None):
        """As :meth:`execute_host`, but every tile is reduced on the device to event-locked sums
        (gcwt_execute_host_events) and only the means cross the link: ``(power, phase)``, power (channels, scales,
        n_lags) float64 = mean over events of |W(c, s, e + lag_first + l)|**2, phase the same shape complex128 = mean
        of W / |W| for complex plans (its modulus is the inter-trial phase coherence), else None.  ``events`` are
        ascending sample indices whose windows each lie inside one epoch."""
        n_ch, n, xa, ea, mp = self._host_args(x, means, epochs)
        ev = np.ascontiguousarray(events, dtype=np.int64).ravel()
        L = int(n_lags)
        power = np.empty((n_ch, self.n_scales, L), dtype=np.float64)
        phase = np.empty((n_ch, self.n_scales, L), dtype=np.complex128) if self.output == "complex" else None
        _lib.check(self.lib.gcwt_execute_host_events(
            self._h, *xa, *ea, mp, ev.ctypes.data, ev.size, int(lag_first), L, power.ctypes.data,
            None if phase is None else phase.ctypes.data, L, self.n_scales * L))
        return power, phase

    def event_reduce(self, res, events, lag_first, n_lags, *, sample0=0, power=None, phase=None):
        """Event-locked sums of a device-resident (channels, scales, samples) result ``res`` (a CUDA tensor with unit
        sample stride, possibly one tile of a longer result starting at sample ``sample0``), through
        gcwt_event_reduce on the current stream: adds |W(c, s, e + lag_first + l)|**2 into ``power`` (float64) and,
        for a complex ``res``, W / |W| into ``phase`` (complex128), both (channels, scales, n_lags) CUDA tensors,
        allocated as zeros when not given.  Only the event samples inside the tile contribute, so tiles can be added
        into the same accumulators one after another.  Returns ``(power, phase or None)``: sums, not means."""
        torch = _torch()
        _, code, kind, st = self._device_coef_args(res, "event_reduce")
        n_ch, S, n = res.shape
        L = int(n_lags)
        cx = res.is_complex()
        if isinstance(events, torch.Tensor):
            ev = events.to(device=res.device, dtype=torch.int64).contiguous().view(-1)
        else:
            ev = torch.from_numpy(np.ascontiguousarray(events, dtype=np.int64).ravel()).to(res.device)
        if power is None:
            power = torch.zeros((n_ch, S, L), dtype=torch.float64, device=res.device)
        if cx and phase is None:
            phase = torch.zeros((n_ch, S, L), dtype=torch.complex128, device=res.device)
        if power.dtype != torch.float64 or power.shape != (n_ch, S, L) or power.stride(2) != 1 or not power.is_cuda:
            raise ValueError("power must be a float64 (channels, scales, n_lags) CUDA tensor with unit lag stride")
        if phase is not None:
            if not cx:
                raise ValueError("phase needs a complex result")
            if phase.dtype != torch.complex128 or phase.shape != (n_ch, S, L) or phase.stride() != power.stride() \
                    or not phase.is_cuda:
                raise ValueError("phase must be a complex128 CUDA tensor of power's shape and strides")
        _lib.check(self.lib.gcwt_event_reduce(
            res.data_ptr(), code, kind, n_ch, S, n, res.stride(1), res.stride(0), int(sample0), ev.data_ptr(),
            ev.numel(), int(lag_first), L, power.data_ptr(), None if phase is None else phase.data_ptr(),
            power.stride(1), power.stride(0), res.device.index, st))
        return power, phase

    def host_stats(self):
        """{wall_ms, pinned_destination, tiles, bytes_out} of the last execute_host."""
        v = (C.c_double * 4)()
        _lib.check(self.lib.gcwt_host_stats(self._h, v))
        return {"wall_ms": float(v[0]), "pinned_destination": bool(v[1]), "tiles": int(v[2]), "bytes_out": int(v[3])}

    PROFILE_KINDS = ("mean+pyramid", "fused_full", "fused_banded", "generic", "fused_interp")

    def profile(self, on=True):
        _lib.check(self.lib.gcwt_profile_enable(self._h, 1 if on else 0))

    def profile_read(self, reset=True):
        """{family: (milliseconds, launches)} accumulated since the last reset."""
        ms = (C.c_double * 5)()
        ln = (C.c_int64 * 5)()
        _lib.check(self.lib.gcwt_profile_read(self._h, ms, ln, 1 if reset else 0))
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(self.PROFILE_KINDS)}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.gcwt_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
