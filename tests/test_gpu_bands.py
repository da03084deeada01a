"""Scale-averaged band power on the device (gcwt_band_reduce, gcwt_execute_host_bands, transform(bands=...)):
band power over time is what users most often derive from a CWT; these check it against numpy reductions of
the full-rate result and against the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, Morse, _lib, synth  # noqa: E402
from ghost_b200.engine import CwtPlan, band_tables, scale_tables         # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402

FP32_BAR = 1e-5


def _plan(fs, freqs, **kw):
    m = Morse(fs=fs)
    om = np.asarray(freqs) / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    return CwtPlan(L, k0, nt, terms, **kw)


def _np_bands(full, first, count, weights, kind):
    """float64 numpy reduction of a (C, S, N) result of kind 'amplitude' | 'power' | 'complex'."""
    full = np.asarray(full)
    out = np.empty((full.shape[0], len(first), full.shape[2]), dtype=np.float64)
    off = 0
    for b, (a, c) in enumerate(zip(first, count)):
        rows = full[:, a:a + c]
        if kind == "complex":
            rows = rows.astype(np.complex128)
            p = rows.real ** 2 + rows.imag ** 2
        else:
            rows = rows.astype(np.float64)
            p = rows if kind == "power" else rows ** 2
        out[:, b] = np.tensordot(weights[off:off + c], p, axes=(0, 1))
        off += c
    return out


def _l2rel(a, b):
    return np.linalg.norm(a - b, axis=-1) / np.linalg.norm(b, axis=-1)


def _shaped_noise(rng, n, fs, power=0.0, f_hp=None):
    spec = np.fft.rfft(rng.standard_normal(n))
    f = np.fft.rfftfreq(n, 1.0 / fs)
    g = (f / f[-1]) ** power if power else np.ones_like(f)
    if f_hp:
        g = g * (f >= f_hp)
    x = np.fft.irfft(spec * g, n=n)
    return x / x.std()


def _hostile(name, n, fs, seed=5):
    """The recipe of test_gpu_guard._hostile: spectra on which only the accuracy guard holds the fp32 bar."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / fs
    if name == "violet":                      # amplitude ~ f^2
        return _shaped_noise(rng, n, fs, power=2.0)
    if name == "tones":                       # weak in-band tone + an out-of-band tone 1e4 times stronger
        return 1e-4 * np.sin(2 * np.pi * 0.003 * fs * t) + np.sin(2 * np.pi * 0.1234 * fs * t) \
            + 1e-4 * rng.standard_normal(n)
    raise KeyError(name)


# theta, gamma, ripple, a band overlapping theta and gamma, and (added per grid) a one-scale band
EPHYS_BANDS = [(6.0, 12.0), (30.0, 80.0), (150.0, 250.0), (8.0, 40.0)]


# ------------------------------------------------------------------ the kernel on random device arrays
@pytest.mark.parametrize("output", ["amplitude", "power"])
def test_band_reduce_matches_numpy(output):
    plan = _plan(1000.0, np.array([100.0, 50.0]), dtype=np.float32, output=output)
    rng = np.random.default_rng(1)
    first = np.array([0, 2, 8, 1], dtype=np.int32)
    count = np.array([3, 5, 1, 7], dtype=np.int32)                # overlapping bands and a one-scale band
    weights = rng.uniform(0.1, 2.0, int(count.sum()))
    for dt in (np.float32, np.float64, np.complex64, np.complex128):
        a = rng.standard_normal((3, 9, 10016))
        if np.iscomplexobj(np.zeros(1, dt)):
            a = a + 1j * rng.standard_normal(a.shape)
        elif output == "power":
            a = np.abs(a)                                           # a power is never negative
        a = a.astype(dt)
        kind = "complex" if np.iscomplexobj(a) else output
        rdt = np.float32 if dt in (np.float32, np.complex64) else np.float64
        rtol = 1e-6 if rdt == np.float32 else 1e-12
        d = torch.from_numpy(a).cuda()
        got = plan.band_reduce(d[:, :, :10007], first, count, weights).cpu().numpy()   # aligned rows, partial last vector
        assert got.shape == (3, 4, 10007) and got.dtype == rdt
        np.testing.assert_allclose(got, _np_bands(a[:, :, :10007], first, count, weights, kind), rtol=rtol, atol=0)
        # a strided window of a larger result: 16-byte aligned rows (vector loads) and misaligned ones
        f2, c2 = np.array([0, 3], dtype=np.int32), np.array([4, 5], dtype=np.int32)
        w2 = weights[:9]
        for lo in (100, 101):
            view = d[:, 1:, lo:9001]
            got = plan.band_reduce(view, f2, c2, w2).cpu().numpy()
            want = _np_bands(a[:, 1:, lo:9001], f2, c2, w2, kind)
            np.testing.assert_allclose(got, want, rtol=rtol, atol=0)
    with pytest.raises(ValueError, match="past the 9 scales"):
        plan.band_reduce(d, np.array([5], dtype=np.int32), np.array([5], dtype=np.int32), np.ones(5))


# ------------------------------------------------------------------ transform(bands=...) against the oracle
def test_fp64_bands_against_the_oracle():
    fs, n = 1000.0, 60000
    x = synth.chirp_pink(n, fs, 0, np.float64)
    amp, f, _ = orc.cwt_amplitude(x, fs, parallel=True)
    bands = EPHYS_BANDS + [(1.5, 4.0), (f[40], f[40])]
    cwt = ContinuousWaveletTransform(dtype=np.float64)
    cwt.transform(x, fs=fs, bands=bands)
    assert cwt.frequencies.tolist() == f.tolist()
    first, count, w = band_tables(f, bands)
    want = _np_bands(amp[None], first, count, w, "amplitude")[0]
    got = cwt.band_power
    assert got.shape == (len(bands), n) and got.dtype == np.float64
    err = np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)
    assert err.max() <= 1e-10, err


@pytest.fixture(scope="module")
def recording_2ch():
    fs, n = 1250.0, 300000
    X = synth.recording(2, n, fs, np.float32)
    amp = [orc.cwt_amplitude(X[c].astype(np.float64), fs, freq_limits=[2.0, 300.0], parallel=True) for c in range(2)]
    return fs, X, np.stack([a[0] for a in amp]), amp[0][1]


@pytest.mark.parametrize("output", ["amplitude", "power", "complex"])
def test_fp32_multichannel_bands(output, recording_2ch):
    fs, X, amp, f = recording_2ch
    bands = EPHYS_BANDS + [(f[20], f[20])]
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=output)
    cwt.transform(X, fs=fs, multichannel=True, freq_limits=[2.0, 300.0], bands=bands)
    plan = cwt.last_plan
    bp = cwt.band_power
    assert bp.shape == (2, len(bands), X.shape[1]) and bp.dtype == np.float32
    assert plan.host_stats()["bytes_out"] == bp.nbytes
    assert cwt.frequencies.tolist() == f.tolist()
    first, count, w = band_tables(f, bands)
    assert [list(b) for b in cwt.band_frequencies] == [f[a:a + c].tolist() for a, c in zip(first, count)]
    assert count[-1] == 1
    # the same plan's full-rate result, reduced in numpy
    full = plan.execute_host(X)
    np.testing.assert_allclose(bp, _np_bands(full, first, count, w, output), rtol=1e-6, atol=0)
    # the oracle
    err = _l2rel(bp.astype(np.float64), _np_bands(amp, first, count, w, "amplitude"))
    assert err.max() <= FP32_BAR, (output, err.max())


def test_bands_across_epochs_and_gaps():
    fs, n = 1000.0, 40000
    x = synth.chirp_pink(n, fs, 2, np.float32)
    ts = np.arange(n) / fs
    ts[20000:] += 0.5
    ts[32000:] += 0.3                                             # three epochs
    bands = [(12.0, 20.0), (30.0, 80.0), (150.0, 250.0), (20.0, 60.0)]
    a = ContinuousWaveletTransform(dtype=np.float32, output="power")
    a.transform(x, fs=fs, timestamps=ts, freq_limits=[5.0, 300.0], bands=bands)
    assert a.last_plan.host_stats()["tiles"] == 3                 # one tile per epoch
    b = ContinuousWaveletTransform(dtype=np.float32, output="power")
    b.transform(x, fs=fs, timestamps=ts, freq_limits=[5.0, 300.0])
    np.testing.assert_allclose(a.band_power, b.scale_averaged_power(bands), rtol=1e-6, atol=0)
    # samples outside every epoch are zero, the rest is the reduction of the full multi-epoch result
    plan = a.last_plan
    first, count, w = band_tables(a.frequencies, bands)
    epochs = np.array([[100, 12000], [12500, 21500], [21500, 30000]])
    got = plan.execute_host_bands(x, first, count, w, epochs=epochs)
    assert np.all(got[0][:, :100] == 0) and np.all(got[0][:, 12000:12500] == 0) and np.all(got[0][:, 30000:] == 0)
    want = _np_bands(plan.execute_host(x, epochs=epochs), first, count, w, "power")
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=0)


def test_bands_with_forced_time_tiles(monkeypatch):
    fs, n = 1000.0, 50000
    X = synth.recording(2, n, fs, np.float32)
    bands = EPHYS_BANDS + [(1.5, 4.0)]
    whole = ContinuousWaveletTransform(dtype=np.float32, output="power")
    whole.transform(X, fs=fs, multichannel=True, bands=bands)
    assert whole.last_plan.host_stats()["tiles"] == 1
    monkeypatch.setenv("GCWT_HOST_TILE", "7000")
    tiled = ContinuousWaveletTransform(dtype=np.float32, output="power")
    tiled.transform(X, fs=fs, multichannel=True, bands=bands)
    assert tiled.last_plan.host_stats()["tiles"] == 8
    err = _l2rel(tiled.band_power.astype(np.float64), whole.band_power.astype(np.float64))
    assert err.max() <= 3e-6, err.max()
    first, count, w = band_tables(tiled.frequencies, bands)
    full = tiled.last_plan.execute_host(X)                        # the same forced tiles, full rate
    np.testing.assert_allclose(tiled.band_power, _np_bands(full, first, count, w, "power"), rtol=1e-6, atol=0)


@pytest.mark.parametrize("tile", [None, "7000"])
@pytest.mark.parametrize("dest", ["pinned", "strided"])
def test_bands_into_pinned_and_strided_destinations(dest, tile, monkeypatch):
    """Band rows reach a pinned array by DMA and a strided pageable one through the copier threads, as
    band_reduce of the device path's full result has them; the padding behind every row stays untouched."""
    fs, n = 1000.0, 50000
    X = synth.recording(2, n, fs, np.float32)
    f = orc.frequency_grid(fs, n)
    plan = _plan(fs, f, dtype=np.float32, output="power")
    first, count, w = band_tables(f, EPHYS_BANDS + [(1.5, 4.0)])
    B = first.size
    want = plan.band_reduce(plan.execute(torch.from_numpy(X).cuda()), first, count, w).cpu().numpy()
    if tile:
        monkeypatch.setenv("GCWT_HOST_TILE", tile)
    if dest == "pinned":
        keep = torch.full((2, B, n + 5), -1.0, dtype=torch.float32).pin_memory()
        big = keep.numpy()
    else:
        big = np.full((2, B + 1, n + 5), -1.0, dtype=np.float32)
    got = big[:, :B, :n]
    _lib.check(plan.lib.gcwt_execute_host_bands(plan._h, X.ctypes.data, _lib.F32, 2, n, n, None, 0, None, B,
                                                first.ctypes.data, count.ctypes.data, w.ctypes.data, got.ctypes.data,
                                                got.strides[1] // 4, got.strides[0] // 4))
    st = plan.host_stats()
    assert st["pinned_destination"] == (dest == "pinned") and st["tiles"] == (1 if tile is None else 8)
    assert st["bytes_out"] == got.nbytes
    assert np.all(big[:, :, n:] == -1.0) and np.all(big[:, B:] == -1.0)
    if tile is None:
        assert np.array_equal(got, want)
    else:
        err = _l2rel(got.astype(np.float64), want.astype(np.float64))
        assert err.max() <= 3e-6, err.max()


@pytest.mark.parametrize("name", ["tones", "violet"])
def test_bands_read_the_guard_corrected_coefficients(name):
    """The reduction starts after the guard's fp64 re-computation: the bands over the re-computed scales hold
    the bar, which the same bands miss without the guard."""
    fs, n = 1000.0, 60000
    x = _hostile(name, n, fs).astype(np.float32)
    amp, f, _ = orc.cwt_amplitude(x.astype(np.float64), fs, parallel=True)
    probe = ContinuousWaveletTransform(dtype=np.float32)
    probe.transform(x, fs=fs)
    sel = np.nonzero(probe.last_plan.guard_stats()["scales"])[0][:63]
    assert sel.size > 0
    bands = [(f[s], f[s]) for s in sel] + [(f[sel].min(), f[sel].max())]
    first, count, w = band_tables(f, bands)
    want = _np_bands(amp[None], first, count, w, "amplitude")[0]
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(x, fs=fs, bands=bands)
    assert cwt.last_plan.guard_stats()["last"] > 0
    err = _l2rel(cwt.band_power.astype(np.float64), want)
    assert err.max() <= FP32_BAR, (name, int(np.argmax(err)), err.max())
    raw = ContinuousWaveletTransform(dtype=np.float32, guard=False)
    raw.transform(x, fs=fs, bands=bands)
    raw_err = _l2rel(raw.band_power.astype(np.float64), want)
    assert raw_err.max() > 3 * err.max(), (name, raw_err.max(), err.max())


# ------------------------------------------------------------------ scale_averaged_power on a full-rate result
@pytest.mark.parametrize("output", ["amplitude", "complex"])
def test_scale_averaged_power_device_and_host(output):
    fs, n = 1250.0, 100000
    X = synth.recording(2, n, fs, np.float32)
    bands = EPHYS_BANDS + [(2.0, 4.0)]
    kw = dict(fs=fs, multichannel=True, freq_limits=[2.0, 300.0])
    banded = ContinuousWaveletTransform(dtype=np.float32, output=output)
    banded.transform(X, bands=bands, **kw)
    dev = ContinuousWaveletTransform(dtype=np.float32, output=output)
    dev.transform(X, keep_on_device=True, **kw)
    got = dev.scale_averaged_power(bands)
    assert got.dtype == np.float32 and got.shape == banded.band_power.shape
    np.testing.assert_allclose(got, banded.band_power, rtol=1e-6, atol=0)
    host = ContinuousWaveletTransform(dtype=np.float32, output=output)
    host.transform(X, **kw)
    got = host.scale_averaged_power(bands)
    assert got.dtype == np.float64
    np.testing.assert_allclose(got, banded.band_power, rtol=1e-6, atol=0)
    np.testing.assert_allclose(dev.scale_averaged_power(bands, "sum"), host.scale_averaged_power(bands, "sum"),
                               rtol=1e-6, atol=0)
    one = ContinuousWaveletTransform(dtype=np.float32, output=output)
    one.transform(X[1], fs=fs, freq_limits=[2.0, 300.0], keep_on_device=True)
    assert _l2rel(one.scale_averaged_power(bands).astype(np.float64), banded.band_power[1].astype(np.float64)).max() <= 3e-6
    # after transform(bands=...) only band_power is kept
    for attr in ("amplitude", "power", "coefficients"):
        with pytest.raises(ValueError, match="only band_power"):
            getattr(banded, attr)
    with pytest.raises(ValueError, match="only band_power"):
        banded.scale_averaged_power(bands)
    # a full-rate transform after a banded one keeps the full result again
    banded.transform(X, **kw)
    assert banded.band_power is None and banded.power.shape == (2, 73, n)
    for kw2 in (dict(out=np.empty((2, 73, n), dtype=np.float32)), dict(pool_width=16), dict(keep_on_device=True)):
        with pytest.raises(ValueError, match="'bands' cannot be combined"):
            banded.transform(X, bands=bands, **kw, **kw2)
