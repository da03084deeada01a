"""Pooling for display (SURVEY.md section 8(f1)): plot() draws the whole (scales, samples) array
(ghost/wave/transforms.py:356-367,395-396); these reduce it to a display's resolution on the device."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import ContinuousWaveletTransform, _lib, synth  # noqa: E402
from oracle import cwt_oracle as orc                             # noqa: E402


def _np_pool(a, width, mode):
    nb = -(-a.shape[-1] // width)
    pad = nb * width - a.shape[-1]
    fill = np.nan if mode == "mean" else -np.inf
    ap = np.concatenate([a.astype(np.float64), np.full(a.shape[:-1] + (pad,), fill)], axis=-1)
    ap = ap.reshape(a.shape[:-1] + (nb, width))
    return np.nanmean(ap, axis=-1) if mode == "mean" else ap.max(axis=-1)


def test_pool_rows_matches_numpy():
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(synth.chirp_pink(5000, 1000.0, 0, np.float32), fs=1000.0, keep_on_device=True)
    plan = cwt.last_plan
    rng = np.random.default_rng(0)
    for dtype in (np.float32, np.float64):
        a = rng.standard_normal((3, 7, 10007)).astype(dtype)
        d = torch.from_numpy(a).cuda()
        for width in (1, 7, 64, 1000, 20000):
            for mode in ("mean", "max"):
                got = plan.pool_rows(d, width, mode).cpu().numpy()
                want = _np_pool(a, width, mode)
                assert got.shape == want.shape and got.dtype == np.float64
                assert np.allclose(got, want, rtol=1e-12, atol=1e-12), (dtype, width, mode)
        got = plan.pool_rows(d, 50, "mean", square=True).cpu().numpy()
        assert np.allclose(got, _np_pool(a.astype(np.float64) ** 2, 50, "mean"), rtol=1e-12)
        view = d[1][2:6, 100:9000]                                   # a window: rows with a stride
        got = plan.pool_rows(view, 33, "max").cpu().numpy()
        assert np.array_equal(got, _np_pool(a[1][2:6, 100:9000], 33, "max"))


def test_spectrogram_data_max_points_device_host_and_oracle():
    fs, n = 1000.0, 60000
    x = synth.chirp_pink(n, fs, 3, np.float32)
    amp, f, _ = orc.cwt_amplitude(x.astype(np.float64), fs, parallel=True)
    dev = ContinuousWaveletTransform(dtype=np.float32)
    dev.transform(x, fs=fs, keep_on_device=True)
    host = ContinuousWaveletTransform(dtype=np.float32)
    host.transform(x, fs=fs)
    for kind, ref in (("amplitude", amp), ("power", amp ** 2)):
        for pool in ("mean", "max"):
            t_d, f_d, w_d = dev.spectrogram_data(kind=kind, max_points=800, pool=pool, time_limits=[5.0, 50.0])
            t_h, f_h, w_h = host.spectrogram_data(kind=kind, max_points=800, pool=pool, time_limits=[5.0, 50.0])
            assert w_d.shape == w_h.shape and w_d.shape[1] <= 800 and w_d.shape[0] == len(f)
            assert np.allclose(t_d, t_h) and np.array_equal(f_d, f_h)
            assert np.allclose(w_d, w_h, rtol=1e-6, atol=0)
            width = -(-45000 // 800)
            want = _np_pool(ref[:, 5000:50000], width, pool)       # numpy pooling of the oracle's array
            rel = np.linalg.norm(w_d - want, axis=1) / np.linalg.norm(want, axis=1)
            assert rel.max() <= 2e-5, (kind, pool, rel.max())
    # standardisation uses the moments of the full-rate array, like the reference (transforms.py:365-366)
    _, _, w = dev.spectrogram_data(kind="amplitude", standardize=True, max_points=500)
    a32 = host.amplitude
    want = (_np_pool(a32, -(-n // 500), "mean") - a32.mean()) / a32.std()
    assert np.allclose(w, want, rtol=1e-4, atol=1e-5)


def test_transform_pool_width_streams_only_the_bins():
    fs, n = 1250.0, 300000
    X = synth.recording(2, n, fs, np.float32)
    full = ContinuousWaveletTransform(dtype=np.float32, output="power")
    full.transform(X, fs=fs, multichannel=True, freq_limits=[2.0, 300.0])
    for pool in ("mean", "max"):
        cwt = ContinuousWaveletTransform(dtype=np.float32, output="power")
        cwt.transform(X, fs=fs, multichannel=True, freq_limits=[2.0, 300.0], pool_width=512, pool=pool)
        got = cwt.power
        want = _np_pool(full.power, 512, pool)
        assert got.shape == want.shape == (2, full.frequencies.size, -(-n // 512)) and got.dtype == np.float64
        assert np.allclose(got, want, rtol=1e-6)
        st = cwt.last_plan.host_stats()
        assert st["bytes_out"] == got.nbytes and st["bytes_out"] * 250 < full.power.nbytes
        assert not st["pinned_destination"]
        assert len(cwt.time) == got.shape[2] and abs(cwt.time[0] - 255.5 / fs) < 1e-12
    with pytest.raises(ValueError):
        ContinuousWaveletTransform(dtype=np.float32, output="complex").transform(X[0], fs=fs, pool_width=16)


def test_pooled_host_path_with_forced_time_tiles(monkeypatch):
    """Tiles of the pooled host path end on bin boundaries, whatever tile length is asked for."""
    fs, n = 1000.0, 50001
    x = synth.chirp_pink(n, fs, 7, np.float32)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.transform(x, fs=fs)
    want = _np_pool(cwt.amplitude, 300, "mean")
    monkeypatch.setenv("GCWT_HOST_TILE", "7000")
    pooled = ContinuousWaveletTransform(dtype=np.float32)
    pooled.transform(x, fs=fs, pool_width=300)
    assert pooled.last_plan.host_stats()["tiles"] == -(-n // 6900)
    rel = np.linalg.norm(pooled.amplitude - want, axis=1) / np.linalg.norm(want, axis=1)
    assert pooled.amplitude.shape == want.shape and rel.max() <= 3e-6, rel.max()


@pytest.mark.parametrize("tile", [None, "7000"])
@pytest.mark.parametrize("dest", ["pinned", "strided"])
def test_pooled_host_path_into_pinned_and_strided_destinations(dest, tile, monkeypatch):
    """Pooled bins reach a pinned array by DMA and a strided pageable one through the copier threads, as the
    device path's pooling of the full result has them; the padding behind every row stays untouched."""
    fs, n, width = 1000.0, 50001, 300
    X = synth.recording(2, n, fs, np.float32)
    cwt = ContinuousWaveletTransform(dtype=np.float32, output="power")
    cwt.transform(X, fs=fs, multichannel=True, freq_limits=[2.0, 300.0], keep_on_device=True)
    plan, S, nb = cwt.last_plan, cwt.frequencies.size, -(-n // width)
    full = plan.execute(torch.from_numpy(X).cuda())
    if tile:
        monkeypatch.setenv("GCWT_HOST_TILE", tile)
    for pool, mode in (("mean", _lib.POOL_MEAN), ("max", _lib.POOL_MAX)):
        want = plan.pool_rows(full, width, pool).cpu().numpy()
        if dest == "pinned":
            keep = torch.full((2, S, nb + 5), -1.0, dtype=torch.float64).pin_memory()
            big = keep.numpy()
        else:
            big = np.full((2, S + 1, nb + 5), -1.0)
        got = big[:, :S, :nb]
        _lib.check(plan.lib.gcwt_execute_host_pooled(plan._h, X.ctypes.data, _lib.F32, 2, n, n, None, width, mode,
                                                     got.ctypes.data, got.strides[1] // 8, got.strides[0] // 8))
        st = plan.host_stats()
        assert st["pinned_destination"] == (dest == "pinned") and st["tiles"] == (1 if tile is None else -(-n // 6900))
        assert np.all(big[:, :, nb:] == -1.0) and np.all(big[:, S:] == -1.0)
        if tile is None:
            assert np.array_equal(got, want), pool
        else:
            rel = np.linalg.norm(got - want, axis=2) / np.linalg.norm(want, axis=2)
            assert rel.max() <= 3e-6, (pool, rel.max())
