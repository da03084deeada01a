"""Scale-averaged band power: the Hz-band -> scale-row mapping, argument checks of the two C entry points and
of transform(bands=...) that need no device."""
import ctypes as C

import numpy as np
import pytest

from ghost_b200 import ContinuousWaveletTransform, _lib
from ghost_b200.engine import band_tables
from oracle import cwt_oracle as orc

GRID = orc.frequency_grid(1250.0, 300000, freq_limits=[2.0, 300.0])       # descending, 10 voices per octave


def test_band_tables_inclusive_edges_on_a_descending_grid():
    assert GRID[0] > GRID[-1]
    lo, hi = GRID[12], GRID[5]                                  # band edges exactly on grid frequencies
    first, count, w = band_tables(GRID, [(lo, hi)])
    assert first.tolist() == [5] and count.tolist() == [8]
    assert first.dtype == np.int32 and count.dtype == np.int32 and w.dtype == np.float64
    assert np.array_equal(w, np.full(8, 1.0 / 8))
    first, count, _ = band_tables(GRID, [(np.nextafter(lo, np.inf), np.nextafter(hi, 0))])
    assert first.tolist() == [6] and count.tolist() == [6]    # just inside the edges: both edge scales drop out
    _, _, w = band_tables(GRID, [(lo, hi)], "sum")
    assert np.array_equal(w, np.ones(8))


def test_band_tables_overlap_one_scale_and_caller_order():
    bands = [(150.0, 250.0), (6.0, 12.0), (30.0, 80.0), (GRID[20], GRID[20]), (8.0, 40.0)]
    first, count, w = band_tables(GRID, bands)
    for (lo, hi), a, c in zip(bands, first, count):
        want = np.nonzero((GRID >= lo) & (GRID <= hi))[0]
        assert (a, c) == (want[0], want.size), (lo, hi)
    assert count[3] == 1 and first[3] == 20
    rows = [set(range(a, a + c)) for a, c in zip(first, count)]
    assert rows[1] & rows[4] and rows[2] & rows[4]              # overlapping bands share scales
    assert w.size == count.sum()
    off = np.concatenate([[0], np.cumsum(count)])
    for b, c in enumerate(count):
        assert np.allclose(w[off[b]:off[b + 1]].sum(), 1.0)
    # the order of the bands is the caller's
    f2, c2, _ = band_tables(GRID, bands[::-1])
    assert f2.tolist() == first[::-1].tolist() and c2.tolist() == count[::-1].tolist()


def test_band_tables_on_an_ascending_grid():
    first, count, _ = band_tables(GRID[::-1], [(6.0, 12.0)])
    want = np.nonzero((GRID[::-1] >= 6.0) & (GRID[::-1] <= 12.0))[0]
    assert first[0] == want[0] and count[0] == want.size


def test_band_tables_errors():
    with pytest.raises(ValueError, match=r"\(400.0, 500.0\) Hz holds no scale: the grid spans 2\.04\d* \.\. 300 Hz"):
        band_tables(GRID, [(6.0, 12.0), (400.0, 500.0)])
    with pytest.raises(ValueError, match="holds no scale"):
        band_tables(GRID, [(GRID[3] * 1.001, GRID[2] * 0.999)])    # between two grid frequencies
    with pytest.raises(ValueError, match="low limit above high limit"):
        band_tables(GRID, [(12.0, 6.0)])
    for bad in ((0.0, 10.0), (-5.0, 10.0), (5.0, -1.0)):
        with pytest.raises(ValueError, match="positive"):
            band_tables(GRID, [bad])
    with pytest.raises(ValueError, match="'mean' or 'sum'"):
        band_tables(GRID, [(6.0, 12.0)], "max")
    with pytest.raises(ValueError):
        band_tables(GRID, [])
    with pytest.raises(ValueError):
        band_tables(GRID, [6.0, 12.0])
    with pytest.raises(ValueError, match="empty"):
        band_tables(np.array([]), [(6.0, 12.0)])


def _i32(*v):
    return np.array(v, dtype=np.int32)


def test_band_reduce_abi_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = C.c_void_p(16)                                      # never dereferenced: every call fails its checks
    first, count, w = _i32(0, 2), _i32(2, 1), np.ones(3)
    F = (first.ctypes.data, count.ctypes.data, w.ctypes.data)

    def call(coef=dummy, ctype=_lib.F32, kind=_lib.OUT_AMPLITUDE, n_ch=2, n=100, s_str=100, c_str=300,
             n_bands=2, tables=F, out=dummy, ob=100, oc=200):
        return lib.gcwt_band_reduce(coef, ctype, kind, n_ch, n, s_str, c_str, n_bands, *tables, out, ob, oc, 0, None)

    assert call(coef=None) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(out=None) == -1
    assert call(tables=(None, F[1], F[2])) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(ctype=7) == -1
    assert call(kind=3) == -1
    assert call(n=0) == -1
    assert call(n_bands=0) == -1 and b"n_bands" in lib.gcwt_last_error()
    assert call(n_bands=65) == -1
    bad = _i32(0, -1)
    assert call(tables=(bad.ctypes.data, F[1], F[2])) == -1 and b"band 1" in lib.gcwt_last_error()
    bad = _i32(2, 0)
    assert call(tables=(F[0], bad.ctypes.data, F[2])) == -1 and b"count" in lib.gcwt_last_error()
    big = _i32(600, 600)
    wbig = np.ones(1200)
    assert call(tables=(first.ctypes.data, big.ctypes.data, wbig.ctypes.data)) == -1 and b"1024" in lib.gcwt_last_error()
    assert call(s_str=99) == -1 and b"stride" in lib.gcwt_last_error()
    assert call(c_str=299) == -1                               # rows 0..2 of a channel need 3 x 100 elements
    assert call(ob=99) == -1
    assert call(oc=199) == -1


def test_execute_host_bands_abi_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    x = np.zeros(1000, dtype=np.float32)
    out = np.zeros((2, 1000), dtype=np.float32)
    first, count, w = _i32(0, 2), _i32(2, 1), np.ones(3)

    def call(plan=None, tables=(first.ctypes.data, count.ctypes.data, w.ctypes.data), n_bands=2):
        return lib.gcwt_execute_host_bands(plan, x.ctypes.data, _lib.F32, 1, 1000, 1000, None, 0, None,
                                           n_bands, *tables, out.ctypes.data, 1000, 2000)

    assert call() == -1 and b"plan is NULL" in lib.gcwt_last_error()
    assert call(tables=(None, count.ctypes.data, w.ctypes.data)) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(n_bands=100) == -1 and b"n_bands" in lib.gcwt_last_error()
    bad = _i32(-3, 2)
    assert call(tables=(bad.ctypes.data, count.ctypes.data, w.ctypes.data)) == -1
    assert b"first >= 0" in lib.gcwt_last_error()


def test_transform_bands_argument_combinations_fail_before_any_device_work():
    x = np.zeros(20000)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    for kw in (dict(out=np.empty((1, 1))), dict(pool_width=64), dict(keep_on_device=True)):
        with pytest.raises(ValueError, match="'bands' cannot be combined"):
            cwt.transform(x, fs=1000.0, bands=[(6.0, 12.0)], **kw)
    with pytest.raises(ValueError, match="holds no scale"):
        cwt.transform(x, fs=1000.0, bands=[(6.0, 12.0), (1000.0, 2000.0)])
    with pytest.raises(ValueError, match="'mean' or 'sum'"):
        cwt.transform(x, fs=1000.0, bands=[(6.0, 12.0)], band_reduce="median")
    with pytest.raises(ValueError, match="'band_reduce' needs 'bands'"):
        cwt.transform(x, fs=1000.0, band_reduce="sum")
