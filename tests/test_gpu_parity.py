"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden
fixtures produced by the reference.  Bars (BASELINE.md section 5):

* fp64: per scale  max|a - b| / max|b| <= 1e-10  (complex coefficients and amplitude)
* fp32: per scale  ||a - b||_2 / ||b||_2 <= 1e-5  (amplitude and power)
"""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, Morse, synth, _lib   # noqa: E402
from ghost_b200.engine import CwtPlan, scale_tables                      # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402

FP64_BAR = 1e-10
FP32_BAR = 1e-5


def _maxrel(a, b):
    return np.max(np.abs(a - b), axis=-1) / np.max(np.abs(b), axis=-1)


def _l2rel(a, b):
    return np.linalg.norm(a - b, axis=-1) / np.linalg.norm(b, axis=-1)


def _plan_for(gamma, beta, fs, freqs, **kw):
    m = Morse(gamma=gamma, beta=beta, fs=fs)
    om = np.asarray(freqs) / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    return CwtPlan(L, k0, nt, terms, **kw), L


# ------------------------------------------------------------------ building blocks
def test_filter_response_matches_fft_of_reference_kernel(golden_dir):
    z = np.load(os.path.join(golden_dir, "kernels.npz"))
    lib = _lib.load()
    for i, (g, b, om, L) in enumerate(z["meta"]):
        L = int(L)
        psi = z[f"psi_{i}"]
        nfft = 1 << int(np.ceil(np.log2(4 * L)))
        buf = np.zeros(nfft, dtype=complex)
        adv = (L - 1) // 2
        idx = (np.arange(L) - adv) % nfft
        buf[idx] = psi                                   # kernel advanced like the 'same' slice
        want = np.fft.fft(buf)
        k0, X = Morse(gamma=g, beta=b).spectrum_terms(L, om)
        got = np.empty(nfft, dtype=np.complex128)
        _lib.check(lib.gcwt_filter_response(L, k0, len(X), X.ctypes.data_as(C.POINTER(C.c_double)), nfft, 0,
                                            nfft, got.ctypes.data_as(C.POINTER(C.c_double)), 0))
        assert np.max(np.abs(got - want)) <= 1e-13 * np.max(np.abs(want)), (g, b, L)


def test_morse_kernel_synthesis(golden_dir):
    z = np.load(os.path.join(golden_dir, "kernels.npz"))
    for i, (g, b, om, L) in enumerate(z["meta"]):
        m = Morse(gamma=g, beta=b)
        m.norm_radian_freq = om
        psi, psif = m(int(L))
        assert np.max(np.abs(psi - z[f"psi_{i}"])) <= 1e-13 * np.max(np.abs(z[f"psi_{i}"]))
        assert np.max(np.abs(psif - z[f"psif_{i}"])) <= 1e-15 * np.max(z[f"psif_{i}"])


# ------------------------------------------------------------------ golden fixtures (reference outputs)
def test_golden_default_transform_fp64(golden_dir):
    z = np.load(os.path.join(golden_dir, "cwt_small.npz"))
    cwt = ContinuousWaveletTransform()
    cwt.transform(z["a_x"], fs=float(z["a_fs"]))
    assert cwt.frequencies.tolist() == z["a_f"].tolist()
    assert cwt.amplitude.dtype == np.float64 and cwt.amplitude.shape == (len(z["a_f"]), len(z["a_x"]))
    assert _maxrel(cwt.amplitude[:, z["a_cols"]], z["a_amp"]).max() <= FP64_BAR
    assert np.array_equal(cwt.power, np.square(cwt.amplitude))
    assert np.allclose(cwt.time, np.arange(len(z["a_x"])) / float(z["a_fs"]))


def test_golden_two_epochs_nonzero_mean_fp64(golden_dir):
    z = np.load(os.path.join(golden_dir, "cwt_small.npz"))
    cwt = ContinuousWaveletTransform(wavelet=Morse(gamma=6, beta=10))
    cwt.transform(z["b_x"], fs=float(z["b_fs"]), timestamps=z["b_ts"], freq_limits=[20, 300],
                  voices_per_octave=6)
    assert cwt.frequencies.tolist() == z["b_f"].tolist()
    assert cwt.amplitude.shape == (len(z["b_f"]), len(z["b_x"]))
    assert _maxrel(cwt.amplitude[:, z["b_cols"]], z["b_amp"]).max() <= FP64_BAR


def test_golden_float32_input_row_vector(golden_dir):
    z = np.load(os.path.join(golden_dir, "cwt_small.npz"))
    cwt = ContinuousWaveletTransform()
    cwt.transform(z["c_x"][None, :], fs=float(z["c_fs"]), parallel=True)
    assert cwt.amplitude.dtype == np.float64 and cwt.amplitude.shape == (len(z["c_f"]), len(z["c_x"]))
    assert _maxrel(cwt.amplitude[:, z["c_cols"]], z["c_amp"]).max() <= FP64_BAR


def test_golden_complex_coefficients_fp64(golden_dir):
    """Reference inner loop (Morse kernel + fastconv_scipy, no abs) at hand-picked
    frequencies, some outside the range transform() would allow: go through the plan."""
    z = np.load(os.path.join(golden_dir, "cwt_small.npz"))
    fs = float(z["d_fs"])
    plan, L = _plan_for(3, 20, fs, z["d_f"], dtype=np.float64, output="complex")
    assert L.tolist() == z["d_L"].tolist()
    got = plan.execute(torch.from_numpy(z["d_x"][None, :]).cuda())[0].cpu().numpy()
    cols = z["d_cols"]                                          # the columns stored of the reference's output
    assert got.shape == (len(z["d_f"]), len(z["d_x"]))
    assert _maxrel(got[:, cols], z["d_W"]).max() <= FP64_BAR
    cwt = ContinuousWaveletTransform(output="complex")
    cwt.transform(z["d_x"], fs=fs, freqs=z["d_f"])
    keep = np.sort(z["d_f"][z["d_f"] >= 17.1])               # freqs= clips to the usable range, ascending
    assert cwt.frequencies.tolist() == keep.tolist()
    idx = [int(np.flatnonzero(z["d_f"] == f)[0]) for f in keep]
    assert cwt.coefficients.shape == (len(keep), len(z["d_x"]))
    assert _maxrel(cwt.coefficients[:, cols], z["d_W"][idx]).max() <= FP64_BAR
    assert _maxrel(cwt.amplitude[:, cols], np.abs(z["d_W"][idx])).max() <= FP64_BAR


def test_golden_cfg1_samples_fp32_and_fp64(golden_dir):
    z = np.load(os.path.join(golden_dir, "cfg1_samples.npz"))
    x = synth.chirp_pink(60000, 1000.0, 0, np.float32)
    for dtype, bar in ((np.float64, 1e-10), (np.float32, 2e-5)):
        cwt = ContinuousWaveletTransform(dtype=dtype)
        cwt.transform(x, fs=1000.0)
        assert cwt.frequencies.tolist() == z["f"].tolist()
        amp = cwt.amplitude
        assert amp.shape == (84, 60000) and amp.dtype == dtype
        got = amp[:, z["cols"]].astype(np.float64)
        assert (np.max(np.abs(got - z["amp"]), axis=1) / np.max(z["amp"], axis=1)).max() <= bar
        l2 = np.sqrt((amp.astype(np.float64) ** 2).sum(axis=1))
        assert np.max(np.abs(l2 - z["row_l2"]) / z["row_l2"]) <= (1e-11 if dtype == np.float64 else 1e-6)


# ------------------------------------------------------------------ oracle comparisons
@pytest.mark.parametrize("gamma,beta,vpo,n", [(3, 20, 10, 16384), (1, 1, 4, 8192), (2, 10, 8, 10000),
                                              (3, 80, 16, 12000), (6, 3, 6, 9000), (9, 40, 12, 20000),
                                              (3, 20, 48, 6000), (3, 20, 48, 262144), (1, 20, 6, 30000),
                                              (2, 5, 10, 262144), (9, 80, 8, 40000), (6, 40, 20, 50000),
                                              (3, 1, 4, 16000), (1, 80, 4, 25000)])
def test_fp64_complex_sweep(gamma, beta, vpo, n):
    """Config 5: fp64 complex coefficients over gamma/beta and voices-per-octave."""
    fs = 2000.0
    x = synth.chirp_pink(n, fs, 11, np.float64) + 0.25
    f = orc.frequency_grid(fs, n, gamma, beta, None, vpo)
    W, _, _ = orc.cwt_complex(x, fs, gamma=gamma, beta=beta, frequencies=f, parallel=True)
    cwt = ContinuousWaveletTransform(wavelet=Morse(gamma=gamma, beta=beta), output="complex")
    cwt.transform(x, fs=fs, voices_per_octave=vpo)
    assert cwt.frequencies.tolist() == f.tolist()
    if (vpo, n) == (48, 262144):
        assert len(f) >= 500                                   # config 5's upper scale count
    err = _maxrel(cwt.coefficients, W)
    assert err.max() <= FP64_BAR, (int(np.argmax(err)), err.max())


@pytest.mark.parametrize("output", ["amplitude", "power", "complex"])
def test_fp32_fast_path_cfg1(output):
    fs, n = 1000.0, 60000
    x = synth.chirp_pink(n, fs, 0, np.float32)
    W, f, _ = orc.cwt_complex(x, fs, parallel=True)
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=output)
    cwt.transform(x, fs=fs)
    levels = cwt.last_plan.levels()
    assert levels.min() == -1 and levels.max() >= 5          # full-spectrum and band-limited kernels both ran
    if output == "complex":
        got, want = cwt.coefficients, W
        assert got.dtype == np.complex64
    elif output == "power":
        got, want = cwt.power, np.abs(W) ** 2
        assert got.dtype == np.float32
    else:
        got, want = cwt.amplitude, np.abs(W)
    err = _l2rel(got.astype(want.dtype), want)
    assert err.max() <= FP32_BAR, (int(np.argmax(err)), err.max())


@pytest.mark.parametrize("gamma,beta,vpo", [(3, 20, 10), (1, 1, 4), (2, 10, 8), (3, 80, 6), (9, 3, 8), (6, 40, 12)])
def test_fp32_gamma_beta_grid(gamma, beta, vpo):
    fs, n = 2000.0, 40000
    x = synth.chirp_pink(n, fs, 3, np.float32)
    amp, f, _ = orc.cwt_amplitude(x, fs, gamma=gamma, beta=beta, voices_per_octave=vpo, parallel=True)
    cwt = ContinuousWaveletTransform(wavelet=Morse(gamma=gamma, beta=beta), dtype=np.float32)
    cwt.transform(x, fs=fs, voices_per_octave=vpo)
    err = _l2rel(cwt.amplitude.astype(np.float64), amp)
    assert err.max() <= FP32_BAR, (gamma, beta, int(np.argmax(err)), err.max(), cwt.last_plan.levels().tolist())


def test_fp32_long_kernels_high_levels():
    """Config 3/4 territory: 30 kHz, kernels of 4 k ... 236 k taps (decimation levels 5 ... 11,
    coarse spacings up to 1024) against the oracle, at hand-picked frequencies."""
    fs, n = 30000.0, 1500000
    x = synth.chirp_pink(n, fs, 21, np.float32)
    freqs = np.array([120.0, 61.0, 30.0, 13.0, 7.0, 4.0, 2.5, 1.7673])
    W, _, L = orc.cwt_complex(x, fs, frequencies=freqs, parallel=True)
    assert int(L.max()) == 236760 or int(L.max()) > 230000
    xd = torch.from_numpy(x[None, :]).cuda()
    for output, want in (("amplitude", np.abs(W)), ("power", np.abs(W) ** 2), ("complex", W)):
        plan, _ = _plan_for(3, 20, fs, freqs, dtype=np.float32, output=output)
        lev = plan.levels()
        assert lev.min() >= 5 and lev.max() >= 11
        got = plan.execute(xd)[0].cpu().numpy()
        err = _l2rel(got.astype(want.dtype), want)
        assert err.max() <= FP32_BAR, (output, err)


def test_fp32_generic_fallback_matches():
    fs, n = 1000.0, 30000
    x = synth.chirp_pink(n, fs, 2, np.float32)
    f = orc.frequency_grid(fs, n)
    amp, _, _ = orc.cwt_amplitude(x, fs, frequencies=f, parallel=True)
    plan, _ = _plan_for(3, 20, fs, f, dtype=np.float32, force_generic=True)
    assert set(plan.levels().tolist()) == {-2}
    out = plan.execute(torch.from_numpy(x[None, :]).cuda())
    err = _l2rel(out[0].cpu().numpy().astype(np.float64), amp)
    assert err.max() <= FP32_BAR


def test_edge_samples_zero_padding_fp32_and_fp64():
    """The first and last L/2 samples see the zero padding of the 'same' convolution."""
    fs, n = 500.0, 5003                                       # odd, not a multiple of anything
    x = synth.chirp_pink(n, fs, 4, np.float64) + 10.0         # big mean: edges depend on its removal
    amp, f, L = orc.cwt_amplitude(x, fs)
    for dtype, bar in ((np.float64, 1e-10), (np.float32, 2e-5)):
        cwt = ContinuousWaveletTransform(dtype=dtype)
        cwt.transform(x, fs=fs)
        got = cwt.amplitude.astype(np.float64)
        edge = np.r_[0:200, n - 200:n]
        err = np.max(np.abs(got[:, edge] - amp[:, edge]), axis=1) / np.max(amp, axis=1)
        assert err.max() <= bar, (dtype, err.max())


def test_short_and_ragged_lengths():
    for n in (64, 257, 1000, 4097):
        fs = 200.0
        x = synth.chirp_pink(n, fs, n, np.float64)
        amp, f, _ = orc.cwt_amplitude(x, fs)
        for dtype, bar in ((np.float64, 1e-10), (np.float32, 1e-5)):
            cwt = ContinuousWaveletTransform(dtype=dtype)
            cwt.transform(x, fs=fs)
            assert cwt.amplitude.shape == amp.shape
            if amp.shape[0] == 0:                          # too short for any scale, like the reference
                assert n == 64
                continue
            if dtype == np.float64:
                assert _maxrel(cwt.amplitude, amp).max() <= bar
            else:
                assert _l2rel(cwt.amplitude.astype(np.float64), amp).max() <= bar


def test_multichannel_equals_channel_loop():
    fs, n, nch = 1250.0, 20000, 5
    X = synth.recording(nch, n, fs, np.float32)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(X, fs=fs, multichannel=True, freq_limits=[2, 300])
    A = cwt.amplitude
    assert A.shape == (nch, len(cwt.frequencies), n)
    one = ContinuousWaveletTransform(dtype=np.float32)
    for c in (0, 3, 4):
        one.transform(X[c], fs=fs, freq_limits=[2, 300])
        assert np.array_equal(one.amplitude, A[c])            # same kernels, same chunk grid: bit-identical
    amp, _, _ = orc.cwt_amplitude(X[1], fs, freq_limits=[2, 300], parallel=True)
    assert _l2rel(A[1].astype(np.float64), amp).max() <= FP32_BAR


def test_multiple_epochs_fp32():
    fs, n = 1000.0, 30000
    x = synth.chirp_pink(n, fs, 6, np.float32) - 2.0
    ts = np.arange(n) / fs
    ts[9000:] += 1.0
    ts[21000:] += 0.01
    amp, f, _ = orc.cwt_amplitude(x, fs, timestamps=ts, parallel=True)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(x, fs=fs, timestamps=ts)
    assert cwt.frequencies.tolist() == f.tolist()
    assert _l2rel(cwt.amplitude.astype(np.float64), amp).max() <= FP32_BAR


def test_analog_signal_array_input():
    class FakeASA:
        def __init__(self, data, fs):
            self._data_colsig = data.reshape(-1, 1)
            self.n_signals, self.fs = 1, fs
            self.lengths = np.array([len(data)])
            self.abscissa_vals = 100.0 + np.arange(len(data)) / fs
    fs, n = 1000.0, 8000
    x = synth.chirp_pink(n, fs, 8, np.float64)
    cwt = ContinuousWaveletTransform()
    cwt.transform(FakeASA(x, fs))
    amp, f, _ = orc.cwt_amplitude(x, fs)
    assert cwt.fs == fs and cwt.time[0] == 100.0
    assert _maxrel(cwt.amplitude, amp).max() <= FP64_BAR


def test_plot_inputs_and_device_standardisation():
    """The arrays plot() draws (reference transforms.py:356-367): amplitude or power, optional
    global standardisation, time / frequency windows -- from a device-resident result without a
    full host copy, against the same selection done with numpy on the oracle's output."""
    fs, n = 1000.0, 30000
    x = synth.chirp_pink(n, fs, 12, np.float32)
    amp, f, _ = orc.cwt_amplitude(x, fs, parallel=True)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(x, fs=fs, keep_on_device=True)
    assert cwt.device_result is not None and cwt.device_result.is_cuda
    for kind, ref in (("amplitude", amp), ("power", amp ** 2)):
        want = (ref - ref.mean()) / ref.std()
        mean, std = cwt.device_moments(square=(kind == "power"))
        assert abs(mean - ref.mean()) <= 1e-5 * abs(ref.mean()) and abs(std - ref.std()) <= 1e-5 * ref.std()
        t, fr, data = cwt.spectrogram_data(kind=kind, standardize=True, time_limits=[5.0, 12.5], freq_limits=[10.0, 100.0])
        ts, fsl = slice(5000, 12500), slice(len(f) - np.searchsorted(f[::-1], 100.0), len(f) - np.searchsorted(f[::-1], 10.0))
        assert data.shape == want[fsl, ts].shape and len(t) == 7500 and np.array_equal(fr, f[fsl])
        assert np.max(np.abs(data - want[fsl, ts])) <= 2e-4 * np.max(np.abs(want))
    host = ContinuousWaveletTransform(dtype=np.float32)
    host.transform(x, fs=fs)
    _, _, d_host = host.spectrogram_data(kind="power", standardize=True, time_limits=[5.0, 12.5], freq_limits=[10.0, 100.0])
    assert np.allclose(d_host, data, rtol=0, atol=2e-4 * np.max(np.abs(d_host)))


# ------------------------------------------------------------------ time shards (halo semantics)
@pytest.mark.parametrize("dtype,bar", [(np.float64, 1e-11), (np.float32, 3e-6)])
def test_time_shards_with_halos_equal_whole(dtype, bar):
    fs, n = 1000.0, 120000
    x = synth.chirp_pink(n, fs, 9, np.float32)
    f = orc.frequency_grid(fs, 60000)
    plan, L = _plan_for(3, 20, fs, f, dtype=dtype)
    xd = torch.from_numpy(x[None, :]).cuda()
    means = plan.channel_means(xd)
    whole = plan.execute(xd, means=means).cpu().numpy()[0]
    halo = int(L.max()) - 1
    parts = plan.alloc_out(1, n)
    cuts = [0, 41000, 77777, n]
    for a, b in zip(cuts[:-1], cuts[1:]):
        plan.execute(xd, parts, means=means, start=a, stop=b, halo_left=min(halo, a), halo_right=min(halo, n - b))
    parts = parts.cpu().numpy()[0]
    # shards use their own chunk / coarse-grid alignment, so fp32 results differ by rounding and
    # by the interpolation error: compare in the norm of the parity bar (pointwise, sqrt of a
    # nearly-zero power amplifies tiny differences)
    err = np.linalg.norm(parts - whole, axis=1) / np.linalg.norm(whole, axis=1)
    assert err.max() <= bar, err.max()
    assert (np.max(np.abs(parts - whole), axis=1) / np.max(np.abs(whole), axis=1)).max() <= 30 * bar
    # without halos the seams are wrong: the halo is what makes sharding exact
    bad = plan.alloc_out(1, n)
    for a, b in zip(cuts[:-1], cuts[1:]):
        plan.execute(xd, bad, means=means, start=a, stop=b)
    bad = bad.cpu().numpy()[0]
    assert (np.max(np.abs(bad - whole), axis=1) / np.max(np.abs(whole), axis=1)).max() > 1e-3


def test_tiled_execution_equals_whole():
    """Results larger than HBM are produced in time tiles with real-sample halos
    (CwtPlan.execute_tiled): every tile must equal the same columns of the whole transform."""
    fs, n, tile = 1000.0, 100000, 30000
    X = synth.recording(2, n, fs, np.float32) + 1.5
    f = orc.frequency_grid(fs, 50000)
    plan, L = _plan_for(3, 20, fs, f, dtype=np.float32, output="power")
    xd = torch.from_numpy(X).cuda()
    whole = plan.execute(xd)
    seen = []

    def consumer(out, a, b):
        num = torch.linalg.vector_norm(out[:, :, :b - a] - whole[:, :, a:b], dim=2)
        den = torch.linalg.vector_norm(whole[:, :, a:b], dim=2)
        seen.append((a, b, float((num / den).max())))

    count = plan.execute_tiled(xd, tile, consumer=consumer)
    assert count == 2 * len(f) * n
    assert [(a, b) for a, b, _ in seen] == [(0, 30000), (30000, 60000), (60000, 90000), (90000, 100000)]
    assert max(e for _, _, e in seen) <= 4e-6, seen


# ------------------------------------------------------------------ host-pointer ABI
def test_execute_host_entry_point():
    fs, n = 1000.0, 12000
    X = synth.recording(2, n, fs, np.float32)
    f = orc.frequency_grid(fs, n)
    plan, _ = _plan_for(3, 20, fs, f, dtype=np.float32, output="power")
    got = plan.execute_host(X)
    dev = plan.execute(torch.from_numpy(X).cuda()).cpu().numpy()
    assert got.shape == (2, len(f), n) and np.array_equal(got, dev)
    amp, _, _ = orc.cwt_amplitude(X[1], fs, frequencies=f, parallel=True)
    assert _l2rel(got[1].astype(np.float64), amp ** 2).max() <= 2 * FP32_BAR


# ------------------------------------------------------------------ full-size properties (config 2 shape)
def test_cfg2_shape_properties():
    """One channel of config 2 (1.25 kHz, 30 min, 96 scales): the oracle would need
    minutes, so check size-independent properties: fp32 fast path against the fp64
    device path (itself pinned to the oracle above) on windows, power == amplitude**2,
    and linearity."""
    fs, n = 1250.0, 2250000
    x = synth.chirp_pink(n, fs, 0, np.float32)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.fs = fs
    cwt.wavelet.fs = fs
    f = cwt.plan_frequencies(n, freq_limits=[0.40, 300], voices_per_octave=10)
    assert len(f) == 96
    p32, L = _plan_for(3, 20, fs, f, dtype=np.float32)
    assert int(L.max()) == 42080
    xd = torch.from_numpy(x[None, :]).cuda()
    a32 = p32.execute(xd)[0]
    p64, _ = _plan_for(3, 20, fs, f, dtype=np.float64)
    a64 = p64.execute(xd)[0]
    num = torch.linalg.vector_norm(a32.double() - a64, dim=1)
    den = torch.linalg.vector_norm(a64, dim=1)
    err = (num / den).cpu().numpy()
    assert err.max() <= FP32_BAR, (int(np.argmax(err)), err.max())
    del a64, p64
    ppow, _ = _plan_for(3, 20, fs, f, dtype=np.float32, output="power")
    pw = ppow.execute(xd)[0]
    rel = (torch.linalg.vector_norm(pw - a32 * a32, dim=1) / torch.linalg.vector_norm(pw, dim=1)).max().item()
    assert rel <= 1e-6
    # linearity of the complex transform: W(2x + y) = 2 W(x) + W(y) on a 200k window
    pc, _ = _plan_for(3, 20, fs, f, dtype=np.float32, output="complex")
    y = torch.from_numpy(synth.chirp_pink(200000, fs, 1, np.float32)[None, :]).cuda()
    xs = xd[:, :200000].contiguous()
    zero = torch.zeros(1, dtype=torch.float64, device="cuda")
    lhs = pc.execute(2 * xs + y, means=zero)[0]
    rhs = 2 * pc.execute(xs, means=zero)[0] + pc.execute(y, means=zero)[0]
    rel = (torch.linalg.vector_norm(lhs - rhs, dim=1) / torch.linalg.vector_norm(rhs, dim=1)).max().item()
    assert rel <= 5e-6


def test_fp32_red_noise_recording():
    """A random walk plus an offset (1/f^2 spectrum, like a drifting LFP baseline): the drift inside a
    chunk is what fp32 FFT butterflies round against, so every fused kernel subtracts the chunk's own
    mean first (exact: all filters have zero DC response).  Odd length: rows are not 16-byte aligned."""
    fs, n = 1250.0, 150001
    rng = np.random.default_rng(7)
    x = (np.cumsum(rng.standard_normal(n)) * 0.05 + rng.standard_normal(n) + 2.5).astype(np.float32)
    amp, f, _ = orc.cwt_amplitude(x.astype(np.float64), fs, freq_limits=[1.0, 400.0], parallel=True)
    for nn in (n, n - 1):                                       # unaligned and aligned output rows
        cwt = ContinuousWaveletTransform(dtype=np.float32)
        cwt.transform(x[:nn], fs=fs, freq_limits=[1.0, 400.0])
        if nn != n:
            amp, f, _ = orc.cwt_amplitude(x[:nn].astype(np.float64), fs, freq_limits=[1.0, 400.0], parallel=True)
        lev = cwt.last_plan.levels()
        assert lev.min() == -1 and lev.max() >= 5
        err = _l2rel(cwt.amplitude.astype(np.float64), amp)
        assert err.max() <= FP32_BAR, (nn, int(np.argmax(err)), err.max(), lev.tolist())
        assert err.max() <= 5e-6, (nn, err.max())              # what the chunk-mean removal leaves


def test_multi_stream_class_launches_are_bit_identical(monkeypatch):
    """GCWT_STREAMS = k deals the independent scale-class launches to k forked streams: same kernels,
    same data, bit-identical results."""
    fs, n, nch = 1250.0, 60000, 3
    X = synth.recording(nch, n, fs, np.float32)
    outs = []
    for k in ("1", "3"):
        monkeypatch.setenv("GCWT_STREAMS", k)
        cwt = ContinuousWaveletTransform(dtype=np.float32, output="power")
        cwt.transform(X, fs=fs, multichannel=True, freq_limits=[1, 400])
        outs.append(cwt.power.copy())
    assert np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("n", [700, 1000, 1500, 2047, 3000])
def test_fp64_small_transform_sizes(n):
    """Transform sizes around the lower limit of the four-step path (2048 points: below it the older
    global-memory passes run).  Found by tools/fuzz_fp64_vs_oracle.py: 1024 points once had an empty grid."""
    fs = 200.0
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n) + 0.3
    W, f, _ = orc.cwt_complex(x, fs, voices_per_octave=8, parallel=True)
    cwt = ContinuousWaveletTransform(output="complex")
    cwt.transform(x, fs=fs, voices_per_octave=8)
    assert cwt.frequencies.tolist() == f.tolist() and len(f) > 0
    assert _maxrel(cwt.coefficients, W).max() <= FP64_BAR
