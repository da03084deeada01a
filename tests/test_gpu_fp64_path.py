"""The fp64 generic path on its two FFT routes, and on more than one device in one process.

* Kernels longer than 2^18 taps on a long recording need chunks of 2^21 points, above the four-step FFT's 2^20:
  they run the Stockham passes through global memory.  Bar as in test_gpu_parity.py: per scale
  max|a - b| / max|b| <= 1e-10 against the oracle.
* Kernel attributes and constant memory are per device: a plan on a second device must give the same bits
  as the same plan on the first, for the four-step route and for the fp32 guard's fp64 re-computation.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, Morse, synth        # noqa: E402
from ghost_b200.engine import CwtPlan, scale_tables                      # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402
from test_gpu_guard import _hostile                                      # noqa: E402

FP64_BAR = 1e-10


def _maxrel(a, b):
    return np.max(np.abs(a - b), axis=-1) / np.max(np.abs(b), axis=-1)


def test_stockham_route_2p21_points_fp64():
    fs, n = 30000.0, 1_200_000
    freqs = np.array([2.0, 1.5])
    m = Morse(gamma=3, beta=20, fs=fs)
    om = freqs / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    assert L.max() > (1 << 18)                    # nfft = max(2^17, pow2(4 L_max)) = 2^21 > 2^20: not the four-step FFT
    x = synth.chirp_pink(n, fs, 0, np.float64)
    W, _, L_ref = orc.cwt_complex(x, fs, frequencies=freqs, parallel=True)
    assert np.array_equal(np.asarray(L_ref), L)
    plan = CwtPlan(L, *scale_tables(m, om, L), dtype=np.float64, output="complex")
    got = plan.execute(torch.from_numpy(x)[None].cuda())[0].cpu().numpy()
    err = _maxrel(got, W)
    assert err.max() <= FP64_BAR, err


def test_second_device_gives_the_same_bits():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    fs = 1000.0
    x = synth.chirp_pink(200_000, fs, 0, np.float64)           # nfft <= 2^20: the four-step FFT
    got = []
    for dev in (0, 1):
        cwt = ContinuousWaveletTransform(dtype=np.float64, output="complex", device=dev)
        cwt.transform(x, fs=fs)
        got.append(cwt.coefficients)
    assert np.array_equal(got[0], got[1])

    v = _hostile("violet", 60000, fs).astype(np.float32)        # the guard re-computes pairs in fp64
    got, pairs = [], []
    for dev in (0, 1):
        cwt = ContinuousWaveletTransform(dtype=np.float32, output="amplitude", device=dev)
        cwt.transform(v, fs=fs)
        got.append(cwt.amplitude)
        pairs.append(cwt.last_plan.guard_stats()["last"])
    assert pairs[0] > 0 and pairs[0] == pairs[1]
    assert np.array_equal(got[0], got[1])
