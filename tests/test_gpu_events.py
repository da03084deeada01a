"""Event-locked power and inter-trial phase coherence on the device (gcwt_event_reduce, gcwt_execute_host_events,
transform(events=...)): checked against numpy averages of windows of the full-rate result and of the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, Morse, _lib, synth  # noqa: E402
from ghost_b200.engine import CwtPlan, event_windows, scale_tables       # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402


def _plan(fs, freqs, **kw):
    m = Morse(fs=fs)
    om = np.asarray(freqs) / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    return CwtPlan(L, k0, nt, terms, **kw)


def _np_sums(full, events, lag_first, n_lags, kind, sample0=0):
    """float64 numpy sums over events of |W|^2 and W / |W| of a (C, S, N) array holding samples [sample0, sample0 + N);
    samples outside it are skipped, as gcwt_event_reduce skips them."""
    full = np.asarray(full)
    n = full.shape[2]
    power = np.zeros(full.shape[:2] + (n_lags,))
    phase = np.zeros(power.shape, dtype=np.complex128)
    for e in events:
        t = e + lag_first + np.arange(n_lags) - sample0
        ok = (t >= 0) & (t < n)
        w = full[:, :, t[ok]]
        if kind == "complex":
            w = w.astype(np.complex128)
            power[:, :, ok] += w.real ** 2 + w.imag ** 2
            m = np.abs(w)
            phase[:, :, ok] += np.where(m > 0, w / np.where(m > 0, m, 1.0), 0.0)
        else:
            w = w.astype(np.float64)
            power[:, :, ok] += w if kind == "power" else w ** 2
    return power, phase


def _np_means(full, events, lag_first, n_lags, kind):
    p, ph = _np_sums(full, events, lag_first, n_lags, kind)
    return p / len(events), ph / len(events)


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


# ------------------------------------------------------------------ the kernel on random device arrays
@pytest.mark.parametrize("output", ["amplitude", "power"])
def test_event_reduce_matches_numpy(output):
    plan = _plan(1000.0, np.array([100.0, 50.0]), dtype=np.float32, output=output)
    rng = np.random.default_rng(3)
    # any order, a duplicate, windows cut by both ends of the array
    events = np.array([700, 100, 2500, 100, 3990, 650, 20, 1990, 2010], dtype=np.int64)
    lag_first, L = -30, 50
    for dt in (np.float32, np.float64, np.complex64, np.complex128):
        a = rng.standard_normal((3, 5, 4000))
        if np.iscomplexobj(np.zeros(1, dt)):
            a = a + 1j * rng.standard_normal(a.shape)
            a[0, 0, 700 - 30] = 0                                    # |W| = 0: counted, adds nothing to the phase
        elif output == "power":
            a = np.abs(a)
        a = a.astype(dt)
        kind = "complex" if np.iscomplexobj(a) else output
        d = torch.from_numpy(a).cuda()
        power, phase = plan.event_reduce(d, events, lag_first, L)
        assert power.dtype == torch.float64 and power.shape == (3, 5, L)
        assert (phase is not None) == (kind == "complex")
        want_p, want_ph = _np_sums(a, events, lag_first, L, kind)
        np.testing.assert_allclose(power.cpu().numpy(), want_p, rtol=1e-12, atol=0)
        if phase is not None:
            np.testing.assert_allclose(phase.cpu().numpy(), want_ph, rtol=0, atol=1e-12 * events.size)
        # the same result in tiles, added into one accumulator in turn: windows lie wholly, partly or not at all in
        # a tile (sample0 = the tile's first sample)
        acc_p = torch.zeros_like(power)
        acc_ph = None if phase is None else torch.zeros_like(phase)
        for t0, t1 in ((0, 1000), (1000, 2000), (2000, 2600), (2600, 4000)):
            tile = d[:, :, t0:t1]
            got_p, got_ph = plan.event_reduce(tile, events, lag_first, L, sample0=t0)
            wp, wph = _np_sums(a[:, :, t0:t1], events, lag_first, L, kind, sample0=t0)
            np.testing.assert_allclose(got_p.cpu().numpy(), wp, rtol=1e-12, atol=0)
            if got_ph is not None:
                np.testing.assert_allclose(got_ph.cpu().numpy(), wph, rtol=0, atol=1e-12 * events.size)
            plan.event_reduce(tile, events, lag_first, L, sample0=t0, power=acc_p, phase=acc_ph)
        assert _rel(acc_p.cpu().numpy(), power.cpu().numpy()) <= 1e-14
        if phase is not None:
            assert _rel(acc_ph.cpu().numpy(), phase.cpu().numpy()) <= 1e-14
        # a strided window of a larger result (rows not 16-byte aligned), events as a device tensor
        view = d[:, 1:4, 7:3907]
        ev_dev = torch.from_numpy(events).cuda()
        got_p, _ = plan.event_reduce(view, ev_dev, -3, 11, sample0=7)
        want_p, _ = _np_sums(a[:, 1:4, 7:3907], events, -3, 11, kind, sample0=7)
        np.testing.assert_allclose(got_p.cpu().numpy(), want_p, rtol=1e-12, atol=0)
        # run to run, the same bits
        again, _ = plan.event_reduce(d, events, lag_first, L)
        assert torch.equal(again, power)


# ------------------------------------------------------------------ transform(events=...) against the oracle
def test_fp64_event_power_against_the_oracle():
    fs, n = 1000.0, 60000                                            # config 1
    x = synth.chirp_pink(n, fs, 0, np.float64)
    amp, f, _ = orc.cwt_amplitude(x, fs, parallel=True)
    ev_s = np.arange(1.0, 58.5, 0.5) + 0.0003
    cwt = ContinuousWaveletTransform(dtype=np.float64)
    cwt.transform(x, fs=fs, events=ev_s, event_window=(-0.3, 0.6))
    assert cwt.frequencies.tolist() == f.tolist()
    samples, kept, lag_first, n_lags = event_windows(cwt.time, ev_s, (-0.3, 0.6), [[0, n]], fs)
    assert kept.all() and (lag_first, n_lags) == (-300, 901)
    assert np.array_equal(cwt.events_used, ev_s)
    np.testing.assert_allclose(cwt.event_lags, (np.arange(901) - 300) / fs, rtol=0, atol=1e-15)
    want, _ = _np_means(amp[None], samples, lag_first, n_lags, "amplitude")
    got = cwt.event_power
    assert got.shape == (f.size, 901) and got.dtype == np.float64
    assert cwt.event_phase is None and cwt.itc is None
    err = np.abs(got - want[0]).max(axis=1) / np.abs(want[0]).max(axis=1)
    assert err.max() <= 1e-10, err.max()
    for attr in ("amplitude", "power", "coefficients"):
        with pytest.raises(ValueError, match="only the event-locked averages"):
            getattr(cwt, attr)


@pytest.mark.parametrize("tile", [None, "7000"])
@pytest.mark.parametrize("output", ["amplitude", "complex"])
def test_fp32_events_against_the_full_result(output, tile, monkeypatch):
    """Event means of the host path equal numpy means over the same plan's execute_host result, untiled and with
    forced time tiles (windows straddle tiles)."""
    fs, n = 1000.0, 50000
    X = synth.recording(2, n, fs, np.float32)
    rng = np.random.default_rng(7)
    ev_s = np.sort(np.concatenate([rng.uniform(0.0, n / fs, 120), [0.1, n / fs - 0.1]]))
    if tile:
        monkeypatch.setenv("GCWT_HOST_TILE", tile)
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=output)
    cwt.transform(X, fs=fs, multichannel=True, events=ev_s, event_window=(-0.2, 0.3))
    plan = cwt.last_plan
    samples, kept, lag_first, n_lags = event_windows(cwt.time, ev_s, (-0.2, 0.3), [[0, n]], fs)
    assert 0 < kept.sum() < ev_s.size                                # events near both ends are dropped
    assert np.array_equal(cwt.events_used, ev_s[kept])
    S = cwt.frequencies.size
    st = plan.host_stats()
    assert st["tiles"] == (1 if tile is None else 8)
    assert st["bytes_out"] == 2 * S * n_lags * (24 if output == "complex" else 8)
    power = cwt.event_power
    assert power.shape == (2, S, n_lags)
    if tile:                                                         # some windows straddle a tile boundary
        assert any((s + lag_first) // 7000 != (s + lag_first + n_lags - 1) // 7000 for s in samples)
    full = plan.execute_host(X)                                      # the same tiles, full rate
    want_p, want_ph = _np_means(full, samples, lag_first, n_lags, output)
    assert _rel(power, want_p) <= 1e-12
    if output == "complex":
        np.testing.assert_allclose(cwt.event_phase, want_ph, rtol=0, atol=1e-12)
        np.testing.assert_allclose(cwt.itc, np.abs(want_ph), rtol=0, atol=1e-12)
        assert cwt.itc.max() <= 1.0 + 1e-12
    else:
        assert cwt.event_phase is None


def test_events_across_epochs_and_gaps():
    fs, n = 1000.0, 40000
    x = synth.chirp_pink(n, fs, 2, np.float32)
    ts = np.arange(n) / fs
    ts[20000:] += 0.5
    ts[32000:] += 0.3                                                # epochs [0, 20000), [20000, 32000), [32000, 40000)
    ev_s = np.array([1.0, 19.95, 20.2, 20.55, 25.0, 32.0, 32.85, 32.6, 39.0])
    cwt = ContinuousWaveletTransform(dtype=np.float32, output="complex")
    cwt.transform(x, fs=fs, timestamps=ts, freq_limits=[5.0, 300.0], events=ev_s, event_window=(-0.1, 0.2))
    # 19.95 s: the window ends past sample 20000; 20.2 s: in the first gap; 20.55 s = t[20050]: the window starts
    # before 20000; 32.85 s = t[32050]: it crosses 32000; 32.6 s: in the second gap
    assert np.array_equal(cwt.events_used, [1.0, 25.0, 32.0, 39.0])
    plan = cwt.last_plan
    epochs = np.array([[0, 20000], [20000, 32000], [32000, 40000]])
    samples = np.array([1000, 24500, 31500, 38200])
    full = plan.execute_host(x, epochs=epochs)
    want_p, want_ph = _np_means(full, samples, -100, 301, "complex")
    assert _rel(cwt.event_power, want_p[0]) <= 1e-12
    np.testing.assert_allclose(cwt.event_phase, want_ph[0], rtol=0, atol=1e-12)
    # the C entry rejects an event whose window crosses a gap, and events out of order
    with pytest.raises(_lib.GcwtError, match="event 1 .sample 19950. does not lie inside one epoch"):
        plan.execute_host_events(x, [1000, 19950], -100, 301, epochs=epochs)
    with pytest.raises(_lib.GcwtError, match="ascending"):
        plan.execute_host_events(x, [24500, 1000], -100, 301, epochs=epochs)
    # a phase output needs a complex plan
    amp_plan = _plan(fs, cwt.frequencies, dtype=np.float32)
    with pytest.raises(_lib.GcwtError, match="complex plan"):
        _lib.check(amp_plan.lib.gcwt_execute_host_events(
            amp_plan._h, x.ctypes.data, _lib.F32, 1, n, n, None, 0, None, samples.ctypes.data, 4, -100, 301,
            want_p.ctypes.data, want_ph.ctypes.data, 301, 301 * amp_plan.n_scales))


def test_itc_of_a_phase_locked_tone_and_of_noise():
    fs, n = 1000.0, 120000
    rng = np.random.default_rng(11)
    t = np.arange(n) / fs
    x = np.sin(2 * np.pi * 10.0 * t) + 0.5 * rng.standard_normal(n)
    locked = np.arange(2.0, 118.0, 1.0)                              # whole seconds: the same 10 Hz phase
    cwt = ContinuousWaveletTransform(dtype=np.float32, output="complex")
    cwt.transform(x, fs=fs, freq_limits=[2.0, 100.0], events=locked, event_window=(-0.5, 0.5))
    s10 = int(np.argmin(np.abs(cwt.frequencies - 10.0)))
    assert cwt.itc[s10].min() >= 0.95, cwt.itc[s10].min()
    noise = rng.standard_normal(n)
    random_ev = np.sort(rng.uniform(1.0, 119.0, 200))
    # scales of 8 Hz and up: their coherence time is below the mean spacing of the events, so the events'
    # phases are close to independent
    cwt.transform(noise, fs=fs, freq_limits=[8.0, 300.0], events=random_ev, event_window=(-0.25, 0.25))
    k = cwt.events_used.size
    assert k == 200
    itc = cwt.itc
    assert np.median(itc) <= 1.2 / np.sqrt(k), np.median(itc)
    assert np.mean(itc > 3.0 / np.sqrt(k)) <= 1e-3, np.mean(itc > 3.0 / np.sqrt(k))


def _hostile_tones(n, fs, seed=5):
    """A weak in-band tone beside an out-of-band tone 1e4 times stronger (test_gpu_guard's recipe): the fp32 bar
    holds there only with the accuracy guard's fp64 re-computation."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / fs
    return 1e-4 * np.sin(2 * np.pi * 0.003 * fs * t) + np.sin(2 * np.pi * 0.1234 * fs * t) + 1e-4 * rng.standard_normal(n)


def test_event_power_reads_the_guard_corrected_coefficients():
    fs, n = 1000.0, 60000
    x = _hostile_tones(n, fs).astype(np.float32)
    ev_s = np.arange(2.0, 58.0, 0.7)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(x, fs=fs, events=ev_s, event_window=(-0.4, 0.4))
    plan = cwt.last_plan
    assert plan.guard_stats()["last"] > 0
    samples, _, lag_first, n_lags = event_windows(cwt.time, ev_s, (-0.4, 0.4), [[0, n]], fs)
    full = plan.execute_host(x)                                      # corrected by the guard as well
    assert plan.guard_stats()["last"] > 0
    want, _ = _np_means(full, samples, lag_first, n_lags, "amplitude")
    assert _rel(cwt.event_power, want[0]) <= 1e-12
    sel = plan.guard_stats()["scales"]                               # the re-computed scales on their own
    got, wnt = cwt.event_power[sel], want[0][sel]
    assert np.max(np.abs(got - wnt) / np.abs(wnt).max(axis=1, keepdims=True)) <= 1e-12


# ------------------------------------------------------------------ event_average on a full-rate result
@pytest.mark.parametrize("output", ["amplitude", "complex"])
def test_event_average_device_and_host(output):
    fs, n = 1250.0, 100000
    X = synth.recording(2, n, fs, np.float32)
    ev_s = np.sort(np.random.default_rng(2).uniform(0.0, n / fs, 60))
    win = (-0.25, 0.5)
    kw = dict(fs=fs, multichannel=True, freq_limits=[2.0, 300.0])
    locked = ContinuousWaveletTransform(dtype=np.float32, output=output)
    locked.transform(X, events=ev_s, event_window=win, **kw)
    dev = ContinuousWaveletTransform(dtype=np.float32, output=output)
    dev.transform(X, keep_on_device=True, **kw)
    p, ph = dev.event_average(ev_s, win)
    assert p.shape == locked.event_power.shape and p.dtype == np.float64
    assert _rel(p, locked.event_power) <= 1e-12
    host = ContinuousWaveletTransform(dtype=np.float32, output=output)
    host.transform(X, **kw)
    hp, hph = host.event_average(ev_s, win)
    assert _rel(hp, locked.event_power) <= 1e-12
    if output == "complex":
        np.testing.assert_allclose(ph, locked.event_phase, rtol=0, atol=1e-12)
        np.testing.assert_allclose(hph, locked.event_phase, rtol=0, atol=1e-12)
    else:
        assert ph is None and hph is None
    one = ContinuousWaveletTransform(dtype=np.float32, output=output)
    one.transform(X[1], fs=fs, freq_limits=[2.0, 300.0], keep_on_device=True)
    p1, _ = one.event_average(ev_s, win)
    assert p1.shape == locked.event_power.shape[1:]
    assert _rel(p1, locked.event_power[1]) <= 3e-6                   # one channel per call: fp32 rounding differs
    with pytest.raises(ValueError, match="only the event-locked averages"):
        locked.event_average(ev_s, win)
    # a full-rate transform after an event-locked one keeps the full result again
    locked.transform(X, **kw)
    assert locked.event_power is None and locked.power.shape == (2, locked.frequencies.size, n)
