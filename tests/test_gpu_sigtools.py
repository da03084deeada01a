"""Device sigtools helpers, modelled on the reference's own tests
(tests/test_convolution.py, tests/test_fourier.py, tests/test_hilbert.py): random input, a
trusted implementation, np.allclose -- plus tighter relative bounds."""
import numpy as np
import pytest
from scipy.signal import convolve, hilbert

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import sigtools   # noqa: E402


def _rel(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def test_fastconv_time_domain():
    # reference tests/test_convolution.py:6-21
    rng = np.random.default_rng(0)
    x, y = rng.random(10000), rng.random(1000)
    for mode in ("full", "same", "valid"):
        conv = convolve(x, y, mode=mode)
        got_a = sigtools.fastconv_fftw(x, y, mode=mode, fft_length=2048)
        got_b = sigtools.fastconv_scipy(x, y, mode=mode, fft_length=2048)
        assert got_a.shape == conv.shape and got_a.dtype == np.complex128
        assert np.allclose(got_b, conv) and np.allclose(got_a, conv) and np.allclose(got_a, got_b)
        assert _rel(got_a, conv) <= 1e-13


def test_fastconv_complex_kernel_same_offset(golden_dir):
    # the reference's own outputs for fastconv_scipy (oracle/gen_golden.py), even and odd kernels
    import os
    z = np.load(os.path.join(golden_dir, "conv.npz"))
    i = 0
    while f"s_{i}" in z:
        got = sigtools.fastconv(z[f"s_{i}"], z[f"k_{i}"])
        assert got.shape == z[f"s_{i}"].shape
        assert _rel(got[z[f"cols_{i}"]], z[f"y_{i}"]) <= 1e-13      # at the columns stored of the reference's output
        i += 1
    assert i == 6


def test_fastconv_freq_domain():
    # reference tests/test_convolution.py:23-42
    rng = np.random.default_rng(1)
    x, y = rng.random(10000), rng.random(1000)
    Y = np.fft.fft(y, n=3000)
    for mode in ("full", "same", "valid"):
        conv = convolve(x, y, mode=mode)
        got = sigtools.fastconv_freq_scipy(x, Y, len(y), mode=mode)
        assert np.allclose(got, conv) and np.allclose(sigtools.fastconv_freq_fftw(x, Y, len(y), mode=mode), conv)


def test_chirpz_dft():
    # reference tests/test_fourier.py:4-16 (odd prime and even lengths) + a power of two
    rng = np.random.default_rng(2)
    for n in (1009, 1010, 4096, 1, 2, 3, 100003):
        x = rng.random(n)
        want = np.fft.fft(x)
        got = sigtools.chirpz_dft(x)
        assert np.allclose(want, got)
        assert _rel(got, want) <= 1e-12
    z = rng.random(777) + 1j * rng.random(777)
    assert _rel(sigtools.dft(np.fft.fft(z), inverse=True), z) <= 1e-12


def test_hilbert():
    # reference tests/test_hilbert.py:4-12, same length (30 kHz x 60 s)
    rng = np.random.default_rng(3)
    x = rng.random(30000 * 60)
    want = hilbert(x)
    got = sigtools.analytic_signal_fftw(x)
    assert np.allclose(got, want) and np.allclose(sigtools.analytic_signal_scipy(x), want)
    assert _rel(got, want) <= 1e-11
    for n in (1001, 4096, 50):
        x = rng.standard_normal(n)
        assert _rel(sigtools.analytic_signal(x), hilbert(x)) <= 1e-12


def test_argument_errors():
    with pytest.raises(ValueError):
        sigtools.fastconv(np.zeros((2, 5)), np.zeros(3))
    with pytest.raises(ValueError):
        sigtools.fastconv(np.zeros(5), np.zeros(3), mode="circular")
    with pytest.raises(ValueError):
        sigtools.fastconv(np.zeros(3), np.zeros(5), mode="valid")
    with pytest.raises(ValueError):
        sigtools.chirpz_dft(np.zeros((3, 3)))


def test_fastconv_freq_keeps_the_reference_wraparound():
    """ADVICE r1: the reference multiplies every block's spectrum by kernel_fd as it is
    (ghost/sigtools/convolution.py:263-273), i.e. convolves circularly with the WHOLE inverse DFT of
    kernel_fd; taps beyond kernel_len therefore wrap around.  Same here (numpy restatement of that loop)."""
    rng = np.random.default_rng(4)
    x = rng.standard_normal(5000)
    taps = rng.standard_normal(700) * np.hanning(700)              # 700 real taps, but the caller claims 400
    nfd, m = 1500, 400
    Y = np.fft.fft(taps, nfd)
    res = np.zeros(len(x) + m - 1, dtype=complex)
    chunk = min(nfd - m + 1, len(x))
    for start in range(0, len(x), chunk):
        length = min(chunk, len(x) - start)
        conv = np.fft.ifft(np.fft.fft(x[start:start + length], n=nfd) * Y)[:length + m - 1]
        res[start:start + len(conv)] += conv
    for mode, sl in (("full", slice(None)), ("same", slice((m - 1) // 2, (m - 1) // 2 + len(x)))):
        got = sigtools.fastconv_freq_fftw(x, Y, m, mode=mode, n_threads=4)
        assert np.allclose(got, res[sl], rtol=1e-10, atol=1e-10)
    assert not np.allclose(res[(m - 1) // 2:(m - 1) // 2 + len(x)], np.convolve(x, taps[:m])[(m - 1) // 2:(m - 1) // 2 + len(x)])
