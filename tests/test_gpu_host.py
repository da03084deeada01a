"""The streamed host-buffer path (gcwt_execute_host): what ContinuousWaveletTransform.transform calls
when the caller wants host arrays back, as the reference returns them (ghost/wave/transforms.py:185,231)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, Morse, synth        # noqa: E402
from ghost_b200.engine import CwtPlan, scale_tables                      # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402


def _plan(fs, freqs, **kw):
    m = Morse(fs=fs)
    om = np.asarray(freqs) / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    return CwtPlan(L, k0, nt, terms, **kw)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_host_path_equals_device_path_bitwise(dtype):
    fs, n, nch = 1250.0, 70001, 3
    X = synth.recording(nch, n, fs, np.float32)
    f = orc.frequency_grid(fs, n, freq_limits=[2.0, 400.0])
    plan = _plan(fs, f, dtype=dtype, output="amplitude")
    xd = torch.from_numpy(X).cuda()
    want = plan.execute(xd).cpu().numpy()
    got = plan.execute_host(X)
    assert got.dtype == dtype and np.array_equal(got, want)
    st = plan.host_stats()
    assert st["tiles"] >= 1 and st["bytes_out"] == got.nbytes and not st["pinned_destination"]


def test_host_path_time_tiles_and_channel_groups(monkeypatch):
    """Forced small time tiles (the config-3 situation: the result does not fit on the device) give the
    same coefficients as one tile up to fp32 rounding, for every tile boundary."""
    fs, n, nch = 1000.0, 50000, 2
    X = synth.recording(nch, n, fs, np.float32)
    f = orc.frequency_grid(fs, n)
    plan = _plan(fs, f, dtype=np.float32, output="power")
    whole = plan.execute_host(X)
    monkeypatch.setenv("GCWT_HOST_TILE", "7000")
    tiled = plan.execute_host(X)
    assert plan.host_stats()["tiles"] == 8
    rel = np.linalg.norm(tiled - whole, axis=2) / np.linalg.norm(whole, axis=2)
    assert rel.max() <= 3e-6, rel.max()
    amp = np.stack([orc.cwt_amplitude(X[c].astype(np.float64), fs, frequencies=f, parallel=True)[0] for c in range(nch)])
    rel = np.linalg.norm(tiled - amp ** 2, axis=2) / np.linalg.norm(amp ** 2, axis=2)
    assert rel.max() <= 1e-5, rel.max()


def test_host_path_pinned_strided_destination_and_epochs():
    fs, n = 1000.0, 30000
    x = synth.chirp_pink(n, fs, 5, np.float32) + 1.5
    f = orc.frequency_grid(fs, 9000, freq_limits=[5.0, 300.0])
    plan = _plan(fs, f, dtype=np.float32, output="amplitude")
    S = len(f)
    epochs = np.array([[100, 12000], [12500, 21500], [21500, 30000]])
    big = torch.zeros((1, S, n + 64), dtype=torch.float32).pin_memory()     # rows 64 elements longer than needed
    view = big.numpy()[:, :, :n]
    view[:] = -1.0
    out = plan.execute_host(x, out=view, epochs=epochs)
    assert out is view and plan.host_stats()["pinned_destination"]
    assert np.all(big.numpy()[:, :, n:] == 0.0)                  # the padding behind every row is untouched
    want, _, _ = orc.cwt_amplitude(x.astype(np.float64), fs, frequencies=f, epoch_bounds=epochs, parallel=True)
    assert np.all(out[0][:, :100] == 0.0) and np.all(out[0][:, 12000:12500] == 0.0)
    for a, b in epochs:
        rel = np.linalg.norm(out[0][:, a:b] - want[:, a:b], axis=1) / np.linalg.norm(want[:, a:b], axis=1)
        assert rel.max() <= 1e-5, (a, b, rel.max())


def test_transform_default_path_is_the_host_path():
    fs, n = 1000.0, 40000
    x = synth.chirp_pink(n, fs, 2, np.float32)
    ts = np.arange(n) / fs
    ts[25000:] += 0.5                                             # a gap: two epochs
    a = ContinuousWaveletTransform(dtype=np.float32, output="power")
    a.transform(x, fs=fs, timestamps=ts)
    assert a.last_plan.host_stats()["tiles"] == 2                 # one tile per epoch
    b = ContinuousWaveletTransform(dtype=np.float32, output="power")
    b.transform(x, fs=fs, timestamps=ts, keep_on_device=True)
    assert b.device_result is not None and np.array_equal(a.power, b.power)
    out = np.empty_like(a.power)
    c = ContinuousWaveletTransform(dtype=np.float32, output="power")
    c.transform(x, fs=fs, timestamps=ts, out=out)
    assert np.shares_memory(c.power, out) and np.array_equal(out, a.power)


def test_host_path_argument_errors():
    fs = 1000.0
    f = np.array([100.0, 50.0])
    plan = _plan(fs, f, dtype=np.float32)
    x = np.zeros(5000, dtype=np.float32)
    with pytest.raises(ValueError):
        plan.execute_host(x, out=np.empty((1, 2, 4999), dtype=np.float32))
    from ghost_b200 import _lib
    with pytest.raises(_lib.GcwtError, match="epoch"):
        plan.execute_host(x, epochs=np.array([[10, 5]]))
    with pytest.raises(_lib.GcwtError, match="epoch"):
        plan.execute_host(x, epochs=np.array([[0, 3000], [2000, 5000]]))
    x2 = np.zeros((2, 5000), dtype=np.float32)
    with pytest.raises(ValueError, match="one value per channel"):
        plan.execute_host_pooled(x2, 16, means=np.zeros(1))
