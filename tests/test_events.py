"""Event-locked averages: the seconds -> samples mapping, argument checks of the two C entry points and of
transform(events=...) that need no device."""
import ctypes as C

import numpy as np
import pytest

from ghost_b200 import ContinuousWaveletTransform, _lib
from ghost_b200.engine import event_windows

FS = 1000.0


def _gapped_time():
    """Three epochs of 1000, 500 and 1500 samples at 1 kHz with gaps of 0.5 s and 0.25 s."""
    t = np.arange(3000) / FS
    t[1000:] += 0.5
    t[1500:] += 0.25
    return t, np.array([[0, 1000], [1000, 1500], [1500, 3000]])


def test_event_windows_nearest_sample_across_gaps():
    t, bounds = _gapped_time()
    ev = np.array([0.2003, 0.2006, 1.7, 1.2, 2.5004, 0.0496])
    samples, kept, lag_first, n_lags = event_windows(t, ev, (-0.01, 0.02), bounds, FS)
    assert (lag_first, n_lags) == (-10, 31)
    # 0.2003 -> sample 200, 0.2006 -> 201, 1.7 s is t[1200] (1.2 + 0.5 gap), 1.2 s lies in the first gap,
    # 2.5004 s -> t[1750] (2.5 - 0.75), 0.0496 -> 50
    assert kept.tolist() == [True, True, True, False, True, True]
    assert samples.tolist() == [200, 201, 1200, 1750, 50] and samples.dtype == np.int64
    # an event within half a sample period of a timestamp is kept, beyond it (inside the gap) dropped
    s, k, _, _ = event_windows(t, [t[999] + 0.4 / FS, t[999] + 0.6 / FS, t[1000] - 0.4 / FS], (0.0, 0.0), bounds, FS)
    assert k.tolist() == [True, False, True] and s.tolist() == [999, 1000]
    # exactly midway between two samples (at 1250 Hz, 0.4 ms from both, whatever the float rounding): the earlier
    t2 = np.arange(2250000) / 1250.0
    mid = 0.5 + 0.999 * np.arange(1800)                             # half of them fall midway
    s, k, _, _ = event_windows(t2, mid, (0.0, 0.0), [[0, t2.size]], 1250.0)
    assert k.all() and np.all(np.abs(t2[s] - mid) <= 0.4e-3 + 1e-12)
    assert event_windows(t2, [0.0004], (0.0, 0.0), [[0, t2.size]], 1250.0)[0].tolist() == [0]


def test_event_windows_drop_windows_that_leave_their_epoch():
    t, bounds = _gapped_time()
    win = (-0.05, 0.1)                                              # lags -50 .. +100
    idx = np.array([49, 50, 899, 900, 1049, 1050, 1399, 1400, 1500 + 50, 2899, 2900])
    samples, kept, lag_first, n_lags = event_windows(t, t[idx], win, bounds, FS)
    assert (lag_first, n_lags) == (-50, 151)
    assert kept.tolist() == [False, True, True, False, False, True, True, False, True, True, False]
    assert samples.tolist() == idx[kept].tolist()
    for s in samples:                                               # every kept window lies inside one epoch
        w0, w1 = s + lag_first, s + lag_first + n_lags
        assert any(a <= w0 and w1 <= b for a, b in bounds)
    with pytest.raises(ValueError, match="no event has its whole window"):
        event_windows(t, t[[10, 990]], win, bounds, FS)


def test_event_windows_rounding():
    t = np.arange(10000) / 1250.0
    b = np.array([[0, 10000]])
    assert event_windows(t, [4.0], (-0.5, 1.0), b, 1250.0)[2:] == (-625, 1876)
    assert event_windows(t, [4.0], (0.0, 0.0), b, 1250.0)[2:] == (0, 1)
    assert event_windows(t, [4.0], (0.1, 0.2), b, 1250.0)[2:] == (125, 126)          # a window after the event
    assert event_windows(t, [4.0], (-0.0011, 0.0013), b, 1250.0)[2:] == (-1, 4)      # -1.375 -> -1, 1.625 -> 2
    assert event_windows(t, [4.0], (-0.0013, 0.0011), b, 1250.0)[2:] == (-2, 4)      # -1.625 -> -2, 1.375 -> 1
    with pytest.raises(ValueError, match="holds no sample"):
        event_windows(t, [4.0], (0.01, 0.0), b, 1250.0)
    with pytest.raises(ValueError, match="pair"):
        event_windows(t, [4.0], 0.5, b, 1250.0)
    with pytest.raises(ValueError, match="empty"):
        event_windows(t, [], (-0.1, 0.1), b, 1250.0)
    with pytest.raises(ValueError, match="finite"):
        event_windows(t, [np.nan], (-0.1, 0.1), b, 1250.0)


def test_event_reduce_abi_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = C.c_void_p(16)                                          # never dereferenced: every call fails its checks

    def call(coef=dummy, ctype=_lib.F32, kind=_lib.OUT_AMPLITUDE, n_ch=2, S=3, n=100, s_str=100, c_str=300,
             events=dummy, n_ev=4, lag_first=-5, L=20, power=dummy, phase=None, a_s=20, a_c=60):
        return lib.gcwt_event_reduce(coef, ctype, kind, n_ch, S, n, s_str, c_str, 0, events, n_ev, lag_first, L,
                                     power, phase, a_s, a_c, 0, None)

    assert call(coef=None) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(events=None) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(power=None) == -1 and b"NULL" in lib.gcwt_last_error()
    assert call(ctype=7) == -1 and b"coef_type" in lib.gcwt_last_error()
    assert call(kind=3) == -1 and b"coef_kind" in lib.gcwt_last_error()
    for kind in (_lib.OUT_AMPLITUDE, _lib.OUT_POWER):
        assert call(kind=kind, phase=C.c_void_p(32)) == -1 and b"complex" in lib.gcwt_last_error()
    for kw in (dict(n_ch=0), dict(S=0), dict(n=0), dict(n_ev=0), dict(L=0), dict(L=-1)):
        assert call(**kw) == -1 and b"positive" in lib.gcwt_last_error(), kw
    assert call(S=70000, c_str=7000000) == -1 and b"65535" in lib.gcwt_last_error()
    assert call(s_str=99) == -1 and b"scale_stride" in lib.gcwt_last_error()
    assert call(c_str=299) == -1 and b"channel_stride" in lib.gcwt_last_error()
    assert call(a_s=19) == -1 and b"acc_scale_stride" in lib.gcwt_last_error()
    assert call(a_c=59) == -1 and b"acc_channel_stride" in lib.gcwt_last_error()
    assert call(kind=_lib.OUT_COMPLEX, phase=C.c_void_p(40)) == -1 and b"16-byte" in lib.gcwt_last_error()


def test_execute_host_events_abi_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    x = np.zeros(1000, dtype=np.float32)
    power = np.zeros((4, 20))
    two = np.array([[0, 400], [500, 1000]], dtype=np.int64)

    def call(plan=None, events=(100, 200, 600), lag_first=-10, L=20, epochs=None, n_events=None):
        ev = None if events is None else np.ascontiguousarray(events, dtype=np.int64)
        ep = None if epochs is None else np.ascontiguousarray(epochs, dtype=np.int64)
        n_ev = (0 if ev is None else ev.size) if n_events is None else n_events
        return lib.gcwt_execute_host_events(plan, x.ctypes.data, _lib.F32, 1, 1000, 1000,
                                            None if ep is None else ep.ctypes.data, 0 if ep is None else ep.shape[0],
                                            None, None if ev is None else ev.ctypes.data, n_ev, lag_first, L,
                                            power.ctypes.data, None, 20, 80)

    assert call(events=None) == -1 and b"events is NULL" in lib.gcwt_last_error()
    assert call(n_events=0) == -1 and b"positive" in lib.gcwt_last_error()
    assert call(L=0) == -1 and b"positive" in lib.gcwt_last_error()
    assert call(events=(100, 600, 200)) == -1
    assert b"ascending (event 2" in lib.gcwt_last_error()
    assert call(events=(5, 100)) == -1                                # window starts at sample -5
    assert b"event 0 (sample 5)" in lib.gcwt_last_error()
    assert call(events=(100, 991)) == -1 and b"event 1 (sample 991)" in lib.gcwt_last_error()   # ends at 1001
    assert call(events=(100, 395, 600), epochs=two) == -1             # crosses the gap at 400 .. 500
    assert b"event 1 (sample 395)" in lib.gcwt_last_error()
    assert call(events=(100, 505, 600), epochs=two) == -1             # starts inside the gap
    assert b"event 1" in lib.gcwt_last_error()
    assert call(lag_first=2 ** 62, events=(2 ** 62,)) == -1           # no overflow: outside every epoch
    assert b"event 0" in lib.gcwt_last_error()
    assert call(epochs=[[0, 400], [300, 1000]]) == -1 and b"epoch bounds" in lib.gcwt_last_error()
    # every window inside an epoch: the next check is the plan
    assert call(events=(10, 100, 100, 380, 510, 980), epochs=two) == -1 and b"plan is NULL" in lib.gcwt_last_error()
    assert call(events=(10, 980), L=11) == -1 and b"plan is NULL" in lib.gcwt_last_error()


def test_transform_events_argument_combinations_fail_before_any_device_work():
    x = np.zeros(20000)
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    with pytest.raises(ValueError, match="go together"):
        cwt.transform(x, fs=1000.0, events=[5.0])
    with pytest.raises(ValueError, match="go together"):
        cwt.transform(x, fs=1000.0, event_window=(-0.5, 1.0))
    for kw in (dict(bands=[(6.0, 12.0)]), dict(out=np.empty((1, 1))), dict(pool_width=64), dict(keep_on_device=True)):
        with pytest.raises(ValueError, match="'events' cannot be combined"):
            cwt.transform(x, fs=1000.0, events=[5.0], event_window=(-0.5, 1.0), **kw)
    with pytest.raises(ValueError, match="no event has its whole window"):
        cwt.transform(x, fs=1000.0, events=[0.1, 19.5, 30.0], event_window=(-0.5, 1.0))
    with pytest.raises(ValueError, match="holds no sample"):
        cwt.transform(x, fs=1000.0, events=[5.0], event_window=(1.0, -0.5))
