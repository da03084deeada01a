"""Continuous wavelet transform on the GPU behind the reference's class interface.

Drop-in for ``ghost.wave.ContinuousWaveletTransform`` (reference
ghost/wave/transforms.py:34-527): same constructor, same ``transform`` keywords, same
validation errors, same read-only properties (``fs``, ``frequencies``, ``wavelet``,
``amplitude``, ``power``, ``time``) and ``plot``.  The per-scale loop
(transforms.py:187-224) -- kernel synthesis, FFT convolution, ``np.abs`` -- is one call
into libghostcwt.so.

Extensions (keyword-only, all optional): ``dtype`` (float64 reproduces the reference to
1e-10; float32 is the HBM-roofline path), ``output`` ('amplitude' | 'power' | 'complex'),
``device``, ``multichannel`` (rows of a 2-D array are channels) and ``keep_on_device``; ``bands`` keeps
only scale-averaged band power (``band_power``), reduced on the device; ``events`` / ``event_window`` keep only
event-locked power and inter-trial phase coherence (``event_power``, ``itc``), reduced on the device.
"""
from __future__ import annotations

import logging
import time as _time
from abc import ABC

import numpy as np

from . import morse
from . import wavelet as wavedef
from ..formats.preprocessing import standardize_input, is_analog_signal_array

__all__ = ["ContinuousWaveletTransform"]


class WaveletTransform(ABC):

    def __init__(self):
        pass

    def __repr__(self):
        return self.__class__.__name__


def _as_float(dtype):
    dt = np.dtype(np.float64 if dtype is None else dtype)
    if dt not in (np.dtype(np.float32), np.dtype(np.float64)):
        raise ValueError("'dtype' must be float32 or float64 but got {}".format(dt))
    return dt


class ContinuousWaveletTransform(WaveletTransform):
    """Continuous wavelet transform with a Morse wavelet.

    Parameters
    ----------
    wavelet : ghost_b200.wave.Wavelet, optional
        Default ``Morse()`` (gamma=3, beta=20), as the reference (transforms.py:42-46).
    dtype : float32 or float64, optional
        Arithmetic and result type on the device.  Default float64.
    output : 'amplitude', 'power' or 'complex', optional
        What the device epilogue writes.  Default 'amplitude' (what the reference stores).
    device : int, optional
        CUDA device ordinal.  Default 0.
    band_tol : float, optional
        float32 only: out-of-band filter energy (amplitude ratio) the band-limited kernels may drop.
        Default 1e-7.
    guard : bool, optional
        float32 only: measure, per call, whether the recording's spectrum lets the float32 kernels hold
        the 1e-5 bar for every (channel, scale) and re-compute the ones that cannot in float64
        (``guard_tol``: the bound that triggers it, default 5e-6).  Default True.
    """

    _PLAN_CACHE_SIZE = 4

    def __init__(self, *, wavelet=None, dtype=None, output=None, device=None, band_tol=None, guard=None,
                 guard_tol=None):
        if wavelet is None:
            wavelet = morse.Morse()
        self._wavelet = wavelet
        self._dtype = _as_float(dtype)
        if output is None:
            output = "amplitude"
        if output not in ("amplitude", "power", "complex"):
            raise ValueError("'output' must be 'amplitude', 'power' or 'complex' but got {}".format(output))
        self._output = output
        self._device = 0 if device is None else int(device)
        self._band_tol = 0.0 if band_tol is None else float(band_tol)
        if self._band_tol < 0:
            raise ValueError("'band_tol' must be positive")
        self._guard = True if guard is None else bool(guard)
        self._guard_tol = 0.0 if guard_tol is None else float(guard_tol)

        self._frequencies = None
        self._fs = None
        self._amplitude = None
        self._power = None
        self._time = None
        self._result = None          # torch tensor (C, S, N) on the device, or None
        self._host = None            # numpy view of the result, filled lazily
        self._band_power = None      # (B, N) or (C, B, N) after transform(bands=...): the only result kept
        self._band_frequencies = None
        self._event_power = None     # (S, L) or (C, S, L) after transform(events=...): the only result kept
        self._event_phase = None
        self._event_lags = None
        self._events_used = None
        self._epoch_bounds = None
        self._pooled = False         # the result was pooled over time (pool_width)
        self._multichannel = False
        self._time_auto = None       # (n, fs) when self._time is the implicit arange(n) / fs
        self._plans = {}
        self.last_plan = None

    # ------------------------------------------------------------------ planning
    def plan_frequencies(self, n_min, *, freq_limits=None, freqs=None, voices_per_octave=10):
        """Frequency grid in Hz for a shortest segment of ``n_min`` samples
        (transforms.py:147-175).  ``self.fs`` must be set."""
        freq_bounds_ref = self._norm_radians_to_hz(self.wavelet.compute_freq_bounds(n_min))
        if freqs is not None:
            # The reference takes freqs[1] as the upper bound and so keeps two values
            # (SURVEY.md quirk Q1); the intended bound freqs[-1] is used here.
            freqs = np.sort(np.asarray(freqs, dtype=np.float64))
            lb, ub = self._check_freq_bounds([freqs[0], freqs[-1]], freq_bounds_ref)
            return freqs[np.logical_and(freqs >= lb, freqs <= ub)]
        if freq_limits is not None:
            freq_limits = np.sort(freq_limits)
            f_low, f_high = self._check_freq_bounds([freq_limits[0], freq_limits[1]], freq_bounds_ref)
        else:
            f_low, f_high = freq_bounds_ref[0], freq_bounds_ref[1]
        n_octaves = np.log2(f_high / f_low)
        J = np.floor(n_octaves * voices_per_octave)
        j = np.arange(J + 1)
        return f_high / 2 ** (j / voices_per_octave)

    def _get_plan(self, frequencies):
        from ..engine import CwtPlan, scale_tables
        omegas = self._hz_to_norm_radians(frequencies)
        lengths = self.wavelet.compute_lengths(omegas)
        key = (float(self.wavelet.gamma), float(self.wavelet.beta), float(self._fs), self._dtype.str,
               self._output, self._device, self._band_tol, self._guard, self._guard_tol, frequencies.tobytes())
        plan = self._plans.get(key)
        if plan is None:
            k_first, n_terms, terms = scale_tables(self.wavelet, omegas, lengths)
            plan = CwtPlan(lengths, k_first, n_terms, terms, dtype=self._dtype, output=self._output,
                           device=self._device, band_tol=self._band_tol, guard=self._guard,
                           guard_tol=self._guard_tol)
            if len(self._plans) >= self._PLAN_CACHE_SIZE:
                old = next(iter(self._plans))
                self._plans.pop(old).close()
            self._plans[key] = plan
        self.last_plan = plan
        return plan

    # ------------------------------------------------------------------ transform
    def transform(self, data, *, timestamps=None, fs=None, freq_limits=None, freqs=None,
                  voices_per_octave=None, parallel=None, verbose=None, multichannel=None,
                  keep_on_device=None, out=None, pool_width=None, pool=None, bands=None, band_reduce=None,
                  events=None, event_window=None, **kwargs):
        """Continuous wavelet transform of one recording.

        Parameters as the reference (transforms.py:59-106): ``data`` is an ndarray with
        one non-singleton dimension or a single-signal nelpy
        RegularlySampledAnalogSignalArray; ``fs`` in Hz (required for ndarrays);
        ``timestamps`` in seconds (gaps of two or more sample periods split the data into
        epochs that are convolved separately); ``freq_limits`` = [low, high] in Hz, or
        explicit ``freqs``; ``voices_per_octave`` even, 4..48, default 10; ``parallel`` and
        ``verbose`` are accepted and validated (``parallel`` has no effect: the device
        always processes all scales at once).

        ``multichannel=True`` accepts a (channels, samples) ndarray; results then have
        shape (channels, scales, samples).  ``out`` is an optional preallocated result array
        ((scales, samples), or (channels, scales, samples) with ``multichannel``) of the output dtype;
        a pinned one is written by DMA.  ``keep_on_device=True`` leaves the result on the GPU instead
        (``device_result``; it must then fit in device memory).  ``pool_width=w`` (with ``pool='mean'`` or
        ``'max'``) is for displays: the result is reduced on the device over runs of ``w`` samples, the
        arrays read back have ceil(samples / w) columns (float64) and ``time`` holds the bin centres --
        the link then carries kilobytes instead of every coefficient.

        ``bands=[(lo, hi), ...]`` (Hz) keeps only scale-averaged band power: for every band, the mean
        (``band_reduce='mean'``) or sum (``'sum'``) of |W|^2 over the scales whose frequency lies in
        [lo, hi], at every sample, reduced on the device tile by tile so that only (bands x samples) per
        channel crosses the link.  The result is ``band_power``, shaped (B, N), or (C, B, N) with
        ``multichannel``, in the plan's dtype; ``band_frequencies`` lists each band's grid frequencies.
        ``amplitude``, ``power`` and ``coefficients`` are then not available.

        ``events=[t, ...]`` (seconds on the ``time`` axis) with ``event_window=(t_pre, t_post)`` (seconds, t_pre may
        be negative) keeps only event-locked averages, reduced on the device tile by tile so that only (scales x lags)
        per channel crosses the link: ``event_power`` = mean over events of |W|^2 at every lag, ``event_phase`` = mean
        of W / |W| (output='complex' only, else None) and ``itc`` = its modulus, the inter-trial phase coherence;
        shaped (S, L), or (C, S, L) with ``multichannel``, float64 / complex128; ``event_lags`` holds the lags in
        seconds.  Each event is taken at its nearest sample; events in a gap, and events whose window leaves their
        epoch, are dropped (with a warning), and ``events_used`` lists the event times averaged.  ``amplitude``,
        ``power`` and ``coefficients`` are then not available.

        Returns None; results are read from the properties.
        """
        if (events is None) != (event_window is None):
            raise ValueError("'events' and 'event_window' go together")
        if events is not None and (bands is not None or pool_width is not None or out is not None or keep_on_device):
            raise ValueError("'events' cannot be combined with 'bands', 'pool_width', 'out' or 'keep_on_device'")
        if bands is None:
            if band_reduce is not None:
                raise ValueError("'band_reduce' needs 'bands'")
        elif out is not None or pool_width is not None or keep_on_device:
            raise ValueError("'bands' cannot be combined with 'out', 'pool_width' or 'keep_on_device'")
        if multichannel is None:
            multichannel = False
        if multichannel:
            if is_analog_signal_array(data):
                samples, fs, timestamps, epoch_bounds = standardize_input(
                    data, fs=fs, timestamps=timestamps, n_signals=None)
                x_host = np.ascontiguousarray(samples.T)
            else:
                if not isinstance(data, np.ndarray) or data.ndim != 2:
                    raise TypeError("multichannel input must be a (channels, samples) ndarray")
                if fs is None:
                    raise TypeError("transform() missing 1 required keyword argument: 'fs'")
                if timestamps is None and self._time_auto == (data.shape[1], fs):
                    # same implicit time base as the previous call (batches of channels of one recording)
                    timestamps, epoch_bounds = self._time, np.array([[0, data.shape[1]]], dtype=int)
                else:
                    auto = timestamps is None
                    _, fs, timestamps, epoch_bounds = standardize_input(
                        data[0], fs=fs, timestamps=timestamps, n_signals=1)
                    self._time_auto = (data.shape[1], fs) if auto else None
                x_host = data
        else:
            samples, fs, timestamps, epoch_bounds = standardize_input(
                data, fs=fs, timestamps=timestamps, n_signals=1)
            self._time_auto = None
            x_host = samples.squeeze()[None, :]

        self.fs = fs                       # validates (transforms.py:109, :457-462)
        self._time = timestamps

        if freqs is not None and freq_limits is not None:
            raise ValueError("freq_limits and freqs cannot both be used at the same time. Either"
                             " specify one or the either, or leave both as unspecified")
        if voices_per_octave is None:
            voices_per_octave = 10
        if voices_per_octave not in np.arange(4, 50, step=2):
            raise ValueError("'voices_per_octave' must be an even number between 4 and 48, inclusive")
        if parallel is None:
            parallel = False
        if parallel not in (True, False):
            raise ValueError("'parallel' must be either True or False")
        if verbose is None:
            verbose = False
        if verbose not in (True, False):
            raise ValueError("'verbose' must be either True or False")

        epoch_bounds = np.asarray(kwargs.pop("epoch_bounds", epoch_bounds))
        lengths = np.diff(epoch_bounds, axis=1).astype(int)
        self._wavelet.fs = self._fs        # transforms.py:179
        frequencies = np.asarray(self.plan_frequencies(int(np.min(lengths)), freq_limits=freq_limits,
                                                       freqs=freqs, voices_per_octave=voices_per_octave),
                                 dtype=np.float64)
        self._frequencies = frequencies
        self._band_power = self._band_frequencies = None
        self._event_power = self._event_phase = self._event_lags = self._events_used = None
        self._epoch_bounds = epoch_bounds
        self._pooled = pool_width is not None
        if bands is not None:
            from ..engine import band_tables
            b_first, b_count, b_weights = band_tables(frequencies, bands, "mean" if band_reduce is None else band_reduce)
        if events is not None:
            from ..engine import event_windows
            ev_samples, ev_kept, lag_first, n_lags = event_windows(self._time, events, event_window, epoch_bounds, fs)
            if not ev_kept.all():
                logging.warning("events: kept {} of {}; the others lie in a gap or their window leaves the "
                                "recording's epoch".format(int(ev_kept.sum()), ev_kept.size))
        if frequencies.size == 0:
            # data too short for any scale: the reference ends up with a (0, N) array
            self._multichannel = bool(multichannel)
            self._result = None
            cdt = np.dtype(self._dtype)
            if self._output == "complex":
                cdt = np.dtype(np.complex64 if self._dtype == np.float32 else np.complex128)
            shape = (x_host.shape[0], 0, x_host.shape[1]) if multichannel else (0, x_host.shape[1])
            self._host = np.zeros(shape, dtype=cdt)
            return
        plan = self._get_plan(frequencies)

        in_dtype = np.float32 if (x_host.dtype == np.float32 and self._dtype == np.float32) else np.float64
        self._multichannel = bool(multichannel)
        self._host = None
        self._result = None
        start_time = _time.time()
        x_in = x_host if x_host.dtype == in_dtype else x_host.astype(in_dtype)
        if events is not None:
            # event-locked averages only: every tile is added into (scales x lags) sums per channel on the device
            # and only those cross the link, once per channel group
            power, phase = plan.execute_host_events(x_in, np.sort(ev_samples), lag_first, n_lags, epochs=epoch_bounds)
            self._event_power = power if multichannel else power[0]
            if phase is not None:
                self._event_phase = phase if multichannel else phase[0]
            self._event_lags = (lag_first + np.arange(n_lags)) / float(fs)
            self._events_used = np.asarray(events, dtype=np.float64).ravel()[ev_kept]
        elif bands is not None:
            # band power only: every tile is reduced over scales on the device and (bands x samples) per channel
            # travels to the host, epochs and zeros between them as for the full result
            res = plan.execute_host_bands(x_in, b_first, b_count, b_weights, epochs=epoch_bounds)
            self._band_power = res if multichannel else res[0]
            self._band_frequencies = [frequencies[a:a + c] for a, c in zip(b_first, b_count)]
        elif pool_width is not None:
            if keep_on_device or out is not None:
                raise ValueError("'pool_width' cannot be combined with 'keep_on_device' or 'out'")
            if self._output == "complex":
                raise ValueError("'pool_width' needs output='amplitude' or 'power'")
            if len(epoch_bounds) != 1:
                raise ValueError("'pool_width' needs gap-free timestamps (one epoch)")
            res = plan.execute_host_pooled(x_in, pool_width, "mean" if pool is None else pool)
            self._host = res if multichannel else res[0]
            w = int(pool_width)
            n_all = x_host.shape[1]
            edges = np.minimum(np.arange(0, n_all + w, w), n_all)
            ts = np.asarray(self._time, dtype=np.float64)
            self._time = np.array([ts[a:b].mean() for a, b in zip(edges[:-1], edges[1:]) if b > a])
            self._time_auto = None
        elif not keep_on_device:
            # host arrays in, host arrays out (what the reference returns, transforms.py:185,231): one
            # streamed call into the library -- tiles of the result travel to the host while the next is
            # computed, so results larger than device memory work
            if out is not None:
                res = out if multichannel else out[None]
            else:
                res = None
            res = plan.execute_host(x_in, out=res, epochs=epoch_bounds)
            self._host = res if multichannel else res[0]
        else:
            import torch
            dev = torch.device("cuda", self._device)
            x_dev = torch.from_numpy(np.ascontiguousarray(x_in)).to(dev)
            means = plan.channel_means(x_dev)                  # global mean, transforms.py:142-143
            res = plan.alloc_out(x_dev.shape[0], x_dev.shape[1])
            covered = 0
            for start, stop in epoch_bounds:                   # transforms.py:202-204
                plan.execute(x_dev, res, means=means, start=int(start), stop=int(stop))
                covered += int(stop) - int(start)
            if covered != x_dev.shape[1]:
                out_mask = torch.ones(x_dev.shape[1], dtype=torch.bool, device=dev)
                for start, stop in epoch_bounds:
                    out_mask[int(start):int(stop)] = False
                res[:, :, out_mask] = 0
            torch.cuda.synchronize(dev)
            self._result = res
        if verbose:
            print("Elapsed time (only wavelet convolution): {} seconds to analyze {} frequencies".format(
                _time.time() - start_time, frequencies.size))

    # ------------------------------------------------------------------ results
    def _check_full_rate(self):
        if self._band_power is not None:
            raise ValueError("transform(bands=...) kept only band_power; run transform without 'bands' for the "
                             "full-rate amplitude, power or coefficients")
        if self._event_power is not None:
            raise ValueError("transform(events=...) kept only the event-locked averages; run transform without "
                             "'events' for the full-rate amplitude, power or coefficients")

    def _check_full_rate_result(self, needs):
        self._check_full_rate()
        if self._frequencies is None or (self._result is None and self._host is None):
            raise ValueError("no full-rate result: call transform() first")
        if self._pooled:
            raise ValueError("the result was pooled over time (pool_width): {} the full-rate result".format(needs))

    def _host_power(self, block):
        """|W|^2 in float64 of a block of the host-resident result by output kind, as mag2 in sigtools.cu reads it."""
        if self._output == "complex":
            block = block.astype(np.complex128)
            return np.square(block.real) + np.square(block.imag)
        block = block.astype(np.float64)
        return block if self._output == "power" else np.square(block)

    def _materialise(self):
        self._check_full_rate()
        if self._host is None:
            if self._result is None:
                return None
            host = self._result.cpu().numpy()
            self._host = host if self._multichannel else host[0]
        return self._host

    @property
    def device_result(self):
        """The (channels, scales, samples) CUDA tensor when ``keep_on_device=True``."""
        return self._result

    @property
    def coefficients(self):
        """Complex coefficients (only for ``output='complex'``)."""
        self._check_full_rate()
        if self._output != "complex":
            raise ValueError("complex coefficients need output='complex'")
        return self._materialise()

    @property
    def amplitude(self):
        res = self._materialise()
        if res is None:
            return None
        if self._output == "amplitude":
            return res
        if self._output == "power":
            return np.sqrt(res)
        return np.abs(res)

    @amplitude.setter
    def amplitude(self, val):
        raise ValueError("Overriding the amplitude attribute is not allowed")

    @property
    def power(self):
        res = self._materialise()
        if res is None:
            return None
        if self._output == "power":
            return res
        return np.square(self.amplitude)                  # transforms.py:507-510

    @power.setter
    def power(self, val):
        raise ValueError("Overriding the power attribute is not allowed")

    @property
    def _amplitude(self):
        return self.amplitude

    @_amplitude.setter
    def _amplitude(self, val):
        pass

    @property
    def band_power(self):
        """Scale-averaged band power of the last ``transform(bands=...)``: (B, N), or (C, B, N) with
        ``multichannel``; None after a full-rate transform."""
        return self._band_power

    @property
    def band_frequencies(self):
        """The grid frequencies (Hz) of each band of ``band_power``, one array per band."""
        return self._band_frequencies

    def scale_averaged_power(self, bands, reduce="mean"):
        """Band power of the existing full-rate result: for every band ``(lo, hi)`` (Hz), the mean
        (``reduce='mean'``) or sum (``'sum'``) of |W|^2 over the scales whose frequency lies in [lo, hi], at
        every sample -- what ``transform(bands=...)`` returns.  Shape (B, N), or (C, B, N) with
        ``multichannel``.  A device-resident result (``keep_on_device=True``) is reduced on the GPU and only the
        bands are copied back (plan dtype); a host-resident one is reduced in numpy in float64."""
        from ..engine import band_tables
        self._check_full_rate_result("band power needs")
        first, count, weights = band_tables(self._frequencies, bands, reduce)
        if self._result is not None and self._host is None:
            res = self.last_plan.band_reduce(self._result, first, count, weights).cpu().numpy()
        else:
            data = self._host if self._multichannel else self._host[None]
            res = np.empty((data.shape[0], first.size, data.shape[2]), dtype=np.float64)
            off = 0
            for b, (a, c) in enumerate(zip(first, count)):
                res[:, b] = np.tensordot(weights[off:off + c], self._host_power(data[:, a:a + c]), axes=(0, 1))
                off += c
        return res if self._multichannel else res[0]

    @property
    def event_power(self):
        """Mean |W|^2 over the events of the last ``transform(events=...)`` at every (scale, lag): (S, L), or
        (C, S, L) with ``multichannel``, float64; None after any other transform."""
        return self._event_power

    @property
    def event_phase(self):
        """Mean of W / |W| over the events (complex128, shaped as ``event_power``); output='complex' only."""
        return self._event_phase

    @property
    def itc(self):
        """Inter-trial phase coherence |mean W / |W||: 1 where the phase is locked to the events, about
        1 / sqrt(n_events) where it is not.  Needs output='complex'; None otherwise."""
        return None if self._event_phase is None else np.abs(self._event_phase)

    @property
    def event_lags(self):
        """The lags of ``event_power``'s last axis, in seconds relative to the events."""
        return self._event_lags

    @property
    def events_used(self):
        """The event times (seconds, as given) that ``event_power`` averages."""
        return self._events_used

    def event_average(self, events, event_window):
        """Event-locked averages of the existing full-rate result: ``(power, phase)`` as ``transform(events=...,
        event_window=...)`` computes them (``phase`` None unless output='complex'), shaped (S, L), or (C, S, L) with
        ``multichannel``.  Events map to samples as there (engine.event_windows).  A device-resident result
        (``keep_on_device=True``) is reduced on the GPU and only the means are copied back; a host-resident one is
        reduced in numpy in float64."""
        from ..engine import event_windows
        self._check_full_rate_result("event averages need")
        samples, _, lag_first, n_lags = event_windows(self._time, events, event_window, self._epoch_bounds, self._fs)
        cx = self._output == "complex"
        if self._result is not None and self._host is None:
            power, phase = self.last_plan.event_reduce(self._result, samples, lag_first, n_lags)
            power = (power / samples.size).cpu().numpy()
            phase = None if phase is None else (phase / samples.size).cpu().numpy()
        else:
            data = self._host if self._multichannel else self._host[None]
            power = np.zeros(data.shape[:2] + (n_lags,))
            phase = np.zeros(power.shape, dtype=np.complex128) if cx else None
            for s in samples:
                w = data[:, :, s + lag_first:s + lag_first + n_lags]
                power += self._host_power(w)
                if cx:
                    w = w.astype(np.complex128)
                    m = np.abs(w)
                    phase += np.where(m > 0, w / np.where(m > 0, m, 1.0), 0.0)
            power /= samples.size
            if cx:
                phase /= samples.size
        if self._multichannel:
            return power, phase
        return power[0], None if phase is None else phase[0]

    @property
    def time(self):
        return self._time

    @time.setter
    def time(self, val):
        raise ValueError("Overriding the time attribute is not allowed")

    @property
    def fs(self):
        return self._fs

    @fs.setter
    def fs(self, samplerate):
        if samplerate <= 0:
            raise ValueError("Sampling rate must be positive")
        self._fs = samplerate

    @property
    def frequencies(self):
        """The frequencies this transform analyzes, in Hz"""
        return self._frequencies

    @frequencies.setter
    def frequencies(self, val):
        raise ValueError("Setting frequencies outside of cwt() is disallowed. Please use the cwt()"
                         " interface if you want to use a different set of frequencies for the cwt")

    @property
    def wavelet(self):
        return self._wavelet

    @wavelet.setter
    def wavelet(self, wav):
        if wav.fs != self._fs:
            raise ValueError("Wavelet must have same sampling rate as input data")
        if not isinstance(wav, wavedef.Wavelet):
            raise TypeError("The wavelet must be of type ghost.Wavelet")
        self._wavelet = wav

    # ------------------------------------------------------------------ helpers
    def _norm_radians_to_hz(self, val):
        return np.array(val) / np.pi * self._fs / 2.0          # transforms.py:404-406

    def _hz_to_norm_radians(self, val):
        return np.array(val) / (self._fs / 2.0) * np.pi        # transforms.py:408-410

    def _check_freq_bounds(self, freq_bounds, freq_bounds_ref):
        """Clip [lb, ub] (Hz) into the reference bounds with a warning (transforms.py:412-434)."""
        lb, ub = freq_bounds[0], freq_bounds[1]
        lb_ref, ub_ref = freq_bounds_ref[0], freq_bounds_ref[1]
        if lb < lb_ref:
            logging.warning("Specified lower bound was {:.3f} Hz but lower bound computed on shortest"
                            " segment was determined to be {:.3f} Hz. The lower bound will be adjusted"
                            " upward to {:.3f} Hz accordingly".format(lb, lb_ref, lb_ref))
            lb = lb_ref
        if ub > ub_ref:
            logging.warning("Specified upper bound was {:.3f} Hz but upper bound was determined to be"
                            " {:.3f} Hz. The upper bound will be adjusted downward to {:.3f} Hz"
                            " accordingly".format(ub, ub_ref, ub_ref))
            ub = ub_ref
        return lb, ub

    def _restrict_plot_time(self, limits):
        limits = np.atleast_1d(np.asarray(limits).squeeze())
        tstart, tstop = np.searchsorted(self._time, limits)
        return slice(tstart, tstop)

    def _restrict_plot_freq(self, limits):
        f0, f1 = np.searchsorted(self._frequencies[::-1], limits)
        n = len(self._frequencies)
        return slice(n - f1, n - f0)

    # ------------------------------------------------------------------ plot
    def spectrogram_data(self, *, kind=None, standardize=None, time_limits=None, freq_limits=None, max_points=None,
                         pool=None):
        """The arrays ``plot`` draws: (time, frequencies, data) after the same selection and
        optional global standardisation as the reference (transforms.py:356-367).

        ``max_points``: at most that many columns -- the selected window is pooled over runs of
        ceil(columns / max_points) samples (``pool='mean'`` or ``'max'``; on the device when the result is
        still there, so that only the pooled window is copied to the host) and the time axis holds the
        bin centres.  Standardisation uses the statistics of the full-rate array, as the reference does."""
        if pool is None:
            pool = "mean"
        if pool not in ("mean", "max"):
            raise ValueError("'pool' must be 'mean' or 'max' but got {}".format(pool))
        if max_points is not None and int(max_points) < 1:
            raise ValueError("'max_points' must be a positive integer")
        if kind is None:
            kind = "amplitude"
        if kind not in ("amplitude", "power"):
            raise ValueError("'kind' must be 'amplitude' or 'power', but got {}".format(kind))
        if standardize is None:
            standardize = False
        if standardize not in (True, False):
            raise ValueError("'standardize' must be True or False but got {}".format(standardize))
        if self._multichannel:
            raise ValueError("plotting needs a single-channel transform")
        time_slice = slice(None) if time_limits is None else self._restrict_plot_time(np.array(time_limits))
        freq_slice = slice(None) if freq_limits is None else self._restrict_plot_freq(freq_limits)
        tvec = np.asarray(self._time)[time_slice]
        width = 1 if max_points is None else max(1, -(-len(tvec) // int(max_points)))

        def pooled_time():
            edges = np.minimum(np.arange(0, len(tvec) + width, width), len(tvec))
            return np.array([tvec[a:b].mean() for a, b in zip(edges[:-1], edges[1:]) if b > a])

        if self._result is not None and self._host is None and self._output in ("amplitude", "power") \
                and (self._output == kind or (self._output == "amplitude" and kind == "power")):
            # result still on the device (keep_on_device=True): global moments there, and only the
            # requested (pooled) window is copied to the host
            sq = kind == "power" and self._output == "amplitude"
            if width > 1:
                dev_win = self._result[0][freq_slice, time_slice]
                win = self.last_plan.pool_rows(dev_win, width, pool, square=sq).cpu().numpy()
                tvec = pooled_time()
            else:
                win = self._result[0][freq_slice, time_slice].cpu().numpy()
                if sq:
                    win = np.square(win)
            if standardize:
                mean, std = self.device_moments(square=sq)
                win = (win - mean) / std
            return tvec, self._frequencies[freq_slice], win
        data = self.amplitude if kind == "amplitude" else self.power
        mean, std = (data.mean(), data.std()) if standardize else (0.0, 1.0)
        win = data[freq_slice, time_slice]
        if width > 1:
            nb = -(-win.shape[1] // width)
            pad = nb * width - win.shape[1]
            fill = np.nan if pool == "mean" else -np.inf
            wp = np.concatenate([win.astype(np.float64), np.full((win.shape[0], pad), fill)], axis=1).reshape(win.shape[0], nb, width)
            win = np.nanmean(wp, axis=2) if pool == "mean" else wp.max(axis=2)
            tvec = pooled_time()
        if standardize:
            win = (win - mean) / std
        return tvec, self._frequencies[freq_slice], win

    def device_moments(self, square=False):
        """(mean, std) in float64 over the whole device-resident result (of its square when
        ``square``), reduced on the GPU: the statistics ``plot(standardize=True)`` uses
        (reference transforms.py:360-366)."""
        import ctypes as C
        import torch
        from .. import _lib
        if self._result is None:
            raise ValueError("no device-resident result: call transform(..., keep_on_device=True)")
        res = self._result
        if res.is_complex() or not res.is_contiguous():
            raise ValueError("moments need a contiguous real result")
        out = (C.c_double * 2)()
        st = torch.cuda.current_stream(res.device).cuda_stream
        _lib.check(_lib.load().gcwt_moments(res.data_ptr(), _lib.F32 if res.dtype == torch.float32 else _lib.F64,
                                            res.numel(), 1 if square else 0, out, self._device, st))
        return float(out[0]), float(out[1])

    def plot(self, *, kind=None, timescale=None, logscale=None, standardize=None, relative_time=None,
             center_time=None, time_limits=None, freq_limits=None, ax=None, max_points=None, pool=None, **kwargs):
        """Filled-contour spectrogram (transforms.py:233-402).  Needs matplotlib.  ``max_points`` / ``pool``:
        see :meth:`spectrogram_data` (pooling to the display's resolution, on the device when possible)."""
        if timescale is None:
            timescale = "seconds"
        if timescale not in ("milliseconds", "seconds", "minutes", "hours"):
            raise ValueError("timescale must be 'milliseconds', seconds', 'minutes', or 'hours' but"
                             " got {}".format(timescale))
        if logscale is None:
            logscale = True
        if logscale not in (True, False):
            raise ValueError("'logscale' must be True or False but got {}".format(logscale))
        if relative_time is None:
            relative_time = False
        if relative_time not in (True, False):
            raise ValueError("'relative_time' must be True or False but got {}".format(relative_time))
        if center_time is None:
            center_time = False
        if center_time not in (True, False):
            raise ValueError("'center_time' must be True or False but got {}".format(center_time))
        if center_time and not relative_time:
            raise ValueError("'relative_time' must be True to use option 'center_time'")
        if time_limits is not None:
            if hasattr(time_limits, "data") and not isinstance(time_limits, np.ndarray):
                time_limits = np.asarray(time_limits.data)          # nelpy EpochArray
                if time_limits.shape[0] != 1:
                    raise ValueError("Detected {} epochs but can only restrict spectrogram plot to 1"
                                     " epoch".format(time_limits.shape[0]))
            elif isinstance(time_limits, (np.ndarray, list)):
                time_limits = np.array(time_limits)
            else:
                raise TypeError("'time_limits' must be of type nelpy.EpochArray or np.ndarray but got"
                                " {}".format(type(time_limits)))
        timevec, freqvec, data = self.spectrogram_data(kind=kind, standardize=standardize, time_limits=time_limits,
                                                       freq_limits=freq_limits, max_points=max_points, pool=pool)
        kind = "amplitude" if kind is None else kind
        title = "Wavelet Amplitude Spectrogram" if kind == "amplitude" else "Wavelet Power Spectrogram"
        scale, xlabel = {"milliseconds": (1000.0, "Time (msec)"), "seconds": (1.0, "Time (sec)"),
                         "minutes": (1 / 60.0, "Time (min)"), "hours": (1 / 3600.0, "Time (hr)")}[timescale]
        timevec = timevec * scale
        if relative_time:
            if center_time:
                half = len(timevec) // 2
                center_val = timevec[half] if len(timevec) & 1 else (timevec[half - 1] + timevec[half]) / 2
                timevec = timevec - center_val
            else:
                timevec = timevec - timevec[0]
        if ax is None:
            import matplotlib.pyplot as plt
            ax = plt.gca()
        tt, ff = np.meshgrid(timevec, freqvec)
        ax.contourf(tt, ff, data, **kwargs)
        if logscale:
            ax.set_yscale("log")
        ax.set_title(title)
        ax.set_xlabel(xlabel)
        ax.set_ylabel("Frequency (Hz)")
        return ax
