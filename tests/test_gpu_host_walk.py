"""The streamed host path (csrc/host_path.cu, walk_tiles) against per-tile device calls, bit for bit.

gcwt_execute_host and its pooled, band-power and event-locked variants cut a call into channel groups, epochs and time
tiles, and compute every tile with one gcwt_execute into a staging slot.  ``Walk`` restates that geometry
(tile_geometry and the loop of walk_tiles); ``full_rate`` rebuilds the full-rate result from CwtPlan.execute calls on
the same tiles and halos, so every host output has an expected value that does not come from the host path and needs
no tolerance:

* full rate: the host result equals it to the last bit, gaps between epochs are exact zeros, and a strided
  destination keeps its padding;
* pooled bins equal CwtPlan.pool_rows of it, band power CwtPlan.band_reduce of it, and event-locked sums the same
  walk replayed tile by tile through CwtPlan.event_reduce, divided by the event count;
* host_stats() reports the restated tile count and byte count, and whether the destination was pinned.

The expected tiles are staged as the host path stages them, rows ``alloc`` elements apart on an aligned buffer,
because the fused kernels pick some row forms from the row alignment (U = 4 interpolation and the level-4 pairs8
form, tests/test_gpu_fused_kernels.py).  Channel count and store form change no bit (pinned there as well), so all
channels of a tile are computed in one call.

Two cases are large enough to reach the branches that only a result over 1 GiB per call takes: channel groups, and
automatic time tiles across groups.  Bit-identity with a device path cannot see a seam error that the device path
shares, so two forced-tile cases are also compared with the oracle, pointwise, around every tile seam and epoch edge.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

from ghost_b200 import Morse, synth                                      # noqa: E402
from ghost_b200.engine import CwtPlan, scale_tables                      # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402

FS = 1000.0
BUDGET = 1 << 30                       # bytes of coefficients per tile (tile_geometry)
N, NCH = 30001, 3
# 24 scales from 60 Hz down to 2 Hz: L_max = 6974, so the halo is far longer than a 1024-sample tile
FREQS = 60.0 * (2.0 / 60.0) ** (np.arange(24) / 23.0)
# epochs: the first starts after sample 0, gaps, two adjacent epochs, one of 300 samples (shorter than 1024 and than
# L_max), and the last ends at N; with a 2000-sample tile the third ends on a 1-sample tile
EPOCHS = np.array([[700, 5000], [5000, 5300], [9000, 21001], [23000, N]])
# from sample 0, one gap, and a gap after the last epoch up to N
EPOCHS_TAIL = np.array([[0, 12000], [15000, 26000]])
EPOCH_SETS = {"whole": None, "epochs": EPOCHS, "tail": EPOCHS_TAIL}
EPS_D, EPS_I, EPS_64 = 1.2e-6, 1.6e-6, 1e-10
PLANS = {                              # plan dtype, output, input dtype
    "f32-amplitude": (np.float32, "amplitude", np.float32),
    "f32-power": (np.float32, "power", np.float32),
    "f32-complex": (np.float32, "complex", np.float32),
    "f64-amplitude": (np.float64, "amplitude", np.float64),
    "f64-complex": (np.float64, "complex", np.float64),
    "f64in-f32-amplitude": (np.float32, "amplitude", np.float64),
}
SENTINEL = {4: 0x7FC0DEAD, 8: 0x7FF80000DEADBEEF}


def _plan(freqs, dtype, output):
    m = Morse(fs=FS)
    om = np.asarray(freqs, dtype=np.float64) / (FS / 2.0) * np.pi
    L = m.compute_lengths(om)
    plan = CwtPlan(L, *scale_tables(m, om, L), dtype=dtype, output=output)
    assert plan.max_length == int(np.max(L))        # the L_max of tile_geometry: the longest scale of the plan
    return plan


# ------------------------------------------------------------------ the walk, restated
class Walk:
    """tile_geometry and the loop of walk_tiles: groups of ``g`` channels, then epochs, then tiles of ``tile``
    samples, each a tuple (c0, gc, a, len, halo_left, halo_right); staging rows are ``alloc`` elements apart."""

    def __init__(self, plan, nch, n, epochs=None, hint=None, pool_width=0):
        S, lmax = plan.n_scales, plan.max_length
        halo = lmax - 1
        real_el = np.dtype(plan.dtype).itemsize
        self.out_el = 2 * real_el if plan.output == "complex" else real_el
        per_channel = S * n * self.out_el
        self.g = max(1, min(nch, BUDGET // per_channel))
        tile = n
        if per_channel > BUDGET:
            tile = max(BUDGET // (S * self.out_el), min(n, 4 * lmax))
            tile = min(n, -(-tile // 1024) * 1024)
        if hint is not None and hint > 0:
            tile = min(n, max(hint, 1024))
        if pool_width > 0 and tile < n:
            tile = max(pool_width, tile // pool_width * pool_width)
        self.tile, self.alloc, self.halo = tile, (tile + 3) & ~3, halo
        self.epochs = [(0, n)] if epochs is None else [(int(a), int(b)) for a, b in epochs]
        self.tiles = []
        for c0 in range(0, nch, self.g):
            gc = min(self.g, nch - c0)
            for e0, e1 in self.epochs:
                for a in range(e0, e1, tile):
                    ln = min(e1, a + tile) - a
                    self.tiles.append((c0, gc, a, ln, min(halo, a - e0), min(halo, e1 - a - ln)))

    def group_tiles(self):
        """The tiles of one channel group, in walk order: every group walks the same ones."""
        return [t[2:] for t in self.tiles if t[0] == 0]

    def bytes_out(self, rows, el, width=lambda ln: ln):
        """What the streamed outputs send: rows per channel of el-byte elements, width(len) columns per tile."""
        return sum(gc * rows * width(ln) * el for _, gc, _, ln, _, _ in self.tiles)


def full_rate(plan, xd, w, means):
    """The full-rate result rebuilt from one CwtPlan.execute per tile, staged like the host path's slots."""
    nch, n = xd.shape
    want = torch.zeros((nch, plan.n_scales, n), dtype=plan.torch_out_dtype, device=xd.device)
    stage = plan.alloc_out(nch, w.alloc)
    for a, ln, hl, hr in w.group_tiles():
        plan.execute(xd, stage, means=means, start=a, stop=a + ln, halo_left=hl, halo_right=hr, out_start=0)
        want[:, :, a:a + ln] = stage[:, :, :ln]
    del stage
    return want


def _bits(t):
    if t.is_complex():
        t = torch.view_as_real(t)
    return t.contiguous().view(torch.int32)


def _same_bits(got, want):
    """got: a host array (any strides) or a CUDA tensor; compared with want on the device."""
    if isinstance(got, np.ndarray):
        got = torch.from_numpy(got).to(want.device)
    return got.shape == want.shape and torch.equal(_bits(got), _bits(want))


def _recording(nch, n, dtype, offset=10.0):
    return np.stack([synth.chirp_pink(n, FS, c, np.float64) + offset for c in range(nch)]).astype(dtype)


def _check_stats(plan, w, nbytes, pinned=False):
    st = plan.host_stats()
    assert st["tiles"] == len(w.tiles), (st, len(w.tiles))
    assert st["bytes_out"] == nbytes, (st, nbytes)
    assert st["pinned_destination"] == pinned


@pytest.fixture
def env(monkeypatch):
    def set_(tile=None, threads=None):
        for name, v in (("GCWT_HOST_TILE", tile), ("GCWT_HOST_THREADS", threads)):
            if v is None:
                monkeypatch.delenv(name, raising=False)
            else:
                monkeypatch.setenv(name, str(v))
    return set_


# ------------------------------------------------------------------ destinations
def _uint_view(a):
    """a viewed as unsigned integers of its real element size (a complex element is two of them)."""
    el = a.real.dtype.itemsize if a.dtype.kind == "c" else a.dtype.itemsize
    return a.view(np.dtype("u%d" % el)), el


def _fill_sentinel(a):
    v, el = _uint_view(a)
    v[...] = SENTINEL[el]


def _is_sentinel(a):
    v, el = _uint_view(np.ascontiguousarray(a))
    return bool(np.all(v == SENTINEL[el]))


class Dest:
    """The caller's output array for execute_host: None, pageable, strided pageable, torch-pinned, strided pinned, or
    a numpy array registered with cudaHostRegister.  ``big`` is the padded parent of a strided view."""

    def __init__(self, kind, shape, dtype):
        self.kind, self.big, self.registered = kind, None, None
        nch, S, n = shape
        padded = (nch, S + 1, n + 13)
        if kind == "none":
            self.out = None
        elif kind == "pageable":
            self.out = np.empty(shape, dtype)
        elif kind == "pageable-strided":
            self.big = np.empty(padded, dtype)
        elif kind == "pinned":
            self.out = torch.empty(shape, dtype=_torch_dtype(dtype), pin_memory=True).numpy()
        elif kind == "pinned-strided":
            self.big = torch.empty(padded, dtype=_torch_dtype(dtype), pin_memory=True).numpy()
        elif kind == "registered":
            self.out = np.empty(shape, dtype)
            err = torch.cuda.cudart().cudaHostRegister(self.out.ctypes.data, self.out.nbytes, 0)
            assert int(err) == 0, err
            self.registered = self.out
        if self.big is not None:
            _fill_sentinel(self.big)
            self.out = self.big[:, :S, :n]
        elif self.out is not None:
            _fill_sentinel(self.out)

    @property
    def pinned(self):
        return self.kind in ("pinned", "pinned-strided", "registered")

    def padding_intact(self):
        if self.big is None:
            return True
        S, n = self.out.shape[1:]
        return _is_sentinel(self.big[:, S:, :]) and _is_sentinel(self.big[:, :S, n:])

    def close(self):
        if self.registered is not None:
            err = torch.cuda.cudart().cudaHostUnregister(self.registered.ctypes.data)
            self.registered = None
            assert int(err) == 0, err


def _torch_dtype(dtype):
    return {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64,
            np.dtype(np.complex64): torch.complex64, np.dtype(np.complex128): torch.complex128}[np.dtype(dtype)]


def _out_dtype(plan):
    if plan.output == "complex":
        return np.dtype(np.complex64 if plan.dtype == np.float32 else np.complex128)
    return np.dtype(plan.dtype)


def _inputs(X, strided):
    """The host input: X itself, or a row-strided view of it (unit sample stride, row stride != n)."""
    if not strided:
        return X
    big = np.full((X.shape[0], X.shape[1] + 11), np.nan, dtype=X.dtype)
    big[:, 5:5 + X.shape[1]] = X
    v = big[:, 5:5 + X.shape[1]]
    assert v.strides[1] == v.itemsize and v.strides[0] != X.shape[1] * v.itemsize
    return v


# ------------------------------------------------------------------ 1. full-rate calls
# (plan, tile hint, epochs, destination, copier threads, row-strided input, means given)
FULL_CASES = {
    "f32amp-whole-none": ("f32-amplitude", None, "whole", "none", 7, False, False),
    "f32amp-1024-epochs-pageable": ("f32-amplitude", 1024, "epochs", "pageable", 1, True, True),
    "f32amp-2000-epochs-strided": ("f32-amplitude", 2000, "epochs", "pageable-strided", 7, False, False),
    "f32amp-2000-tail-pageable": ("f32-amplitude", 2000, "tail", "pageable", 7, False, False),
    "f32pow-2000-whole-strided": ("f32-power", 2000, "whole", "pageable-strided", 1, False, True),
    "f32pow-2999-epochs-pinned": ("f32-power", 2999, "epochs", "pinned", None, True, True),
    "f32cx-1024-epochs-pinnedstrided": ("f32-complex", 1024, "epochs", "pinned-strided", None, False, False),
    "f32cx-2000-epochs-registered": ("f32-complex", 2000, "epochs", "registered", None, True, False),
    "f64amp-2999-epochs-pageable": ("f64-amplitude", 2999, "epochs", "pageable", 7, False, False),
    "f64amp-whole-epochs-registered": ("f64-amplitude", None, "epochs", "registered", None, False, True),
    "f64cx-2000-epochs-strided": ("f64-complex", 2000, "epochs", "pageable-strided", 1, True, True),
    "f64cx-1024-whole-pinned": ("f64-complex", 1024, "whole", "pinned", None, False, False),
    "f64cx-1024-tail-pinnedstrided": ("f64-complex", 1024, "tail", "pinned-strided", None, True, True),
    "f64in-2000-epochs-pinnedstrided": ("f64in-f32-amplitude", 2000, "epochs", "pinned-strided", None, False, True),
    "f64in-1024-whole-none": ("f64in-f32-amplitude", 1024, "whole", "none", 1, True, False),
}


def test_grid_halo_exceeds_the_smallest_tile():
    plan = _plan(FREQS, np.float32, "amplitude")
    assert plan.max_length - 1 > 1024
    w = Walk(plan, NCH, N, EPOCHS, hint=2000)
    assert any(ln == 1 for _, _, _, ln, _, _ in w.tiles)                  # a 1-sample last tile
    assert any(e1 - e0 < min(1024, plan.max_length) for e0, e1 in w.epochs)
    assert any(b == c for (_, b), (c, _) in zip(w.epochs, w.epochs[1:]))  # adjacent epochs
    assert Walk(plan, NCH, N, hint=2999).tile == 2999                     # no rounding of a hint


@pytest.mark.parametrize("case", list(FULL_CASES))
def test_full_rate_equals_the_tile_walk(case, env):
    name, hint, epoch_set, dest_kind, threads, strided, given = FULL_CASES[case]
    dtype, output, in_dtype = PLANS[name]
    plan = _plan(FREQS, dtype, output)
    S = plan.n_scales
    epochs = EPOCH_SETS[epoch_set]
    X = _recording(NCH, N, in_dtype)
    xd = torch.from_numpy(X).cuda()
    means_d = plan.channel_means(xd)
    means = means_d.cpu().numpy() + 0.25 if given else None           # a caller's means differ from the recording's
    if given:
        means_d = torch.from_numpy(means).cuda()
    w = Walk(plan, NCH, N, epochs, hint=hint)
    want = full_rate(plan, xd, w, means_d)
    env(tile=hint, threads=threads)
    dest = Dest(dest_kind, (NCH, S, N), _out_dtype(plan))
    try:
        got = plan.execute_host(_inputs(X, strided), out=dest.out, means=means, epochs=epochs)
        assert dest.out is None or got is dest.out
        _check_stats(plan, w, NCH * S * sum(b - a for a, b in w.epochs) * w.out_el, dest.pinned)
        assert _same_bits(got, want)
        assert dest.padding_intact()
        if epochs is not None:                                          # exact zeros outside the epochs
            gaps = np.ones(N, bool)
            for a, b in epochs:
                gaps[a:b] = False
            assert np.all(np.asarray(got)[:, :, gaps] == 0)
    finally:
        dest.close()
    plan.close()


# ------------------------------------------------------------------ 2. pooled bins
@pytest.mark.parametrize("pool", ["mean", "max"])
@pytest.mark.parametrize("name,width", [("f32-amplitude", 1), ("f32-power", 3), ("f64-amplitude", 1000),
                                        ("f32-amplitude", 2500), ("f32-power", 40000)])
def test_pooled_bins_equal_pool_rows_of_the_walk(name, width, pool, env):
    """Forced 2000-sample tiles: a tile must end on a bin boundary (width 2500 exceeds the tile, 40000 the
    recording)."""
    dtype, output, in_dtype = PLANS[name]
    plan = _plan(FREQS, dtype, output)
    X = _recording(NCH, N, in_dtype)
    xd = torch.from_numpy(X).cuda()
    w = Walk(plan, NCH, N, hint=2000, pool_width=width)
    want = plan.pool_rows(full_rate(plan, xd, w, plan.channel_means(xd)), width, pool)
    env(tile=2000, threads=3)
    got = plan.execute_host_pooled(X, width, pool)
    _check_stats(plan, w, w.bytes_out(plan.n_scales, 8, lambda ln: -(-ln // width)))
    assert _same_bits(got, want)
    plan.close()


def test_pooled_launch_of_more_than_65535_rows(env):
    """700 channels x 100 scales: one tile's pooling is 70000 rows, split over gridDim.y."""
    nch, n, width = 700, 2048, 16
    plan = _plan(60.0 * (10.0 / 60.0) ** (np.arange(100) / 99.0), np.float32, "amplitude")
    X = (np.random.default_rng(7).standard_normal((nch, n)) + 3.0).astype(np.float32)
    xd = torch.from_numpy(X).cuda()
    w = Walk(plan, nch, n, hint=1024, pool_width=width)
    assert w.g == nch and nch * plan.n_scales > 65535 and len(w.tiles) == 2
    want = plan.pool_rows(full_rate(plan, xd, w, plan.channel_means(xd)), width, "mean")
    env(tile=1024)
    got = plan.execute_host_pooled(X, width, "mean")
    _check_stats(plan, w, w.bytes_out(plan.n_scales, 8, lambda ln: -(-ln // width)))
    assert _same_bits(got, want)
    plan.close()


# ------------------------------------------------------------------ 3. band power
def _bands(S, limits=False):
    """Overlapping bands and a one-scale band; ``limits``: 64 bands holding 1024 (band, scale) entries."""
    if limits:
        count = np.array([1] + [17] * 60 + [1, 1, 1], dtype=np.int32)
        first = np.array([(5 * b) % (S - c + 1) for b, c in enumerate(count)], dtype=np.int32)
        assert count.size == 64 and count.sum() == 1024
    else:
        first = np.array([0, 4, 10, 17, 6], dtype=np.int32)
        count = np.array([8, 8, 1, 7, 12], dtype=np.int32)
    weights = np.random.default_rng(int(count.sum())).uniform(0.1, 1.0, int(count.sum()))
    return first, count, weights


@pytest.mark.parametrize("name,hint,limits", [("f32-amplitude", 1024, True), ("f32-power", 2999, False),
                                              ("f32-complex", 2000, False), ("f64-amplitude", 2000, True),
                                              ("f64-complex", 1024, False)])
def test_band_power_equals_band_reduce_of_the_walk(name, hint, limits, env):
    """The host path reduces 16-byte-aligned tile rows (the vector path), band_reduce of the odd-length full result
    takes the scalar path: band_reduce_kernel promises the same bits."""
    dtype, output, in_dtype = PLANS[name]
    plan = _plan(FREQS, dtype, output)
    X = _recording(NCH, N, in_dtype)
    xd = torch.from_numpy(X).cuda()
    first, count, weights = _bands(plan.n_scales, limits)
    w = Walk(plan, NCH, N, EPOCHS, hint=hint)
    want = plan.band_reduce(full_rate(plan, xd, w, plan.channel_means(xd)), first, count, weights)
    env(tile=hint, threads=2)
    got = plan.execute_host_bands(X, first, count, weights, epochs=EPOCHS)
    _check_stats(plan, w, w.bytes_out(first.size, np.dtype(plan.dtype).itemsize))
    assert _same_bits(got, want)
    plan.close()


# ------------------------------------------------------------------ 4. event-locked sums
def replay_events(plan, want, w, events, lag_first, n_lags):
    """event_reduce over every tile of the walk, in walk order, into one accumulator; then / n_events as the host
    divides."""
    ev = torch.from_numpy(np.asarray(events, dtype=np.int64)).to(want.device)
    power = phase = None
    for a, ln, _, _ in w.group_tiles():
        power, phase = plan.event_reduce(want[:, :, a:a + ln], ev, lag_first, n_lags, sample0=a, power=power,
                                         phase=phase)
    cnt = float(len(events))
    power = power.cpu().numpy() / cnt
    if phase is not None:
        phase = (phase.cpu().numpy().view(np.float64) / cnt).view(np.complex128)
    return power, phase


EVENT_CASES = {     # lag_first, n_lags, events: inside one epoch of EPOCHS each
    # windows of 3500 samples (four 1024-sample tiles) that start or end on epoch bounds, one event twice
    "wide": (-1200, 3500, [1900, 2700, 10200, 10200, 15000, 18701, 27000, 27701]),
    # one lag: the first and last sample of epochs, both sides of the adjacent bound, the 300-sample epoch
    "one-lag": (50, 1, [650, 4949, 4950, 5249, 5249, 20950, 29950]),
    "after": (200, 2500, [500, 9500, 9500, 18301, 27301]),
}


@pytest.mark.parametrize("case", list(EVENT_CASES))
@pytest.mark.parametrize("name,hint", [("f32-amplitude", 1024), ("f32-power", 2999), ("f32-complex", 1024),
                                       ("f64-complex", 2000)])
def test_event_sums_equal_the_replayed_walk(name, hint, case, env):
    dtype, output, in_dtype = PLANS[name]
    lag_first, n_lags, events = EVENT_CASES[case]
    plan = _plan(FREQS, dtype, output)
    X = _recording(NCH, N, in_dtype)
    xd = torch.from_numpy(X).cuda()
    w = Walk(plan, NCH, N, EPOCHS, hint=hint)
    want = full_rate(plan, xd, w, plan.channel_means(xd))
    wp, wph = replay_events(plan, want, w, events, lag_first, n_lags)
    env(tile=hint)
    gp, gph = plan.execute_host_events(X, events, lag_first, n_lags, epochs=EPOCHS)
    _check_stats(plan, w, NCH * plan.n_scales * n_lags * (8 + (16 if output == "complex" else 0)))
    assert np.array_equal(gp.view(np.int64), wp.view(np.int64))
    assert (gph is None) == (output != "complex")
    if gph is not None:
        assert np.array_equal(gph.view(np.int64), wph.view(np.int64))
    plan.close()


# ------------------------------------------------------------------ 5. the 1 GiB branches
def _large_case(plan, nch, n, events, lag_first, n_lags):
    """Full rate, band power and event sums of one fp32 plan, compared on the device (no second host copy)."""
    X = _recording(nch, n, np.float32)
    xd = torch.from_numpy(X).cuda()
    w = Walk(plan, nch, n)
    want = full_rate(plan, xd, w, plan.channel_means(xd))
    got = plan.execute_host(X)
    _check_stats(plan, w, nch * plan.n_scales * n * w.out_el)
    assert _same_bits(got, want)
    del got
    first, count, weights = np.array([0, 3, 20], np.int32), np.array([6, 1, 12], np.int32), np.linspace(0.2, 1, 19)
    bands = plan.execute_host_bands(X, first, count, weights)
    _check_stats(plan, w, w.bytes_out(3, 4))
    assert _same_bits(bands, plan.band_reduce(want, first, count, weights))
    gp, gph = plan.execute_host_events(X, events, lag_first, n_lags)
    _check_stats(plan, w, nch * plan.n_scales * n_lags * (8 + (16 if gph is not None else 0)))
    wp, wph = replay_events(plan, want, w, events, lag_first, n_lags)
    assert np.array_equal(gp.view(np.int64), wp.view(np.int64))
    if gph is not None:
        assert np.array_equal(gph.view(np.int64), wph.view(np.int64))
    return w


def test_channel_groups(env):
    """fp32 amplitude, 64 scales x 2 M samples = 512 MB per channel: 3 channels walk as groups of 2 and 1."""
    env()
    plan = _plan(200.0 * (5.0 / 200.0) ** (np.arange(64) / 63.0), np.float32, "amplitude")
    n = 2_000_000
    w = _large_case(plan, 3, n, [4000, 999_000, 999_000, 1_996_000], -3000, 4001)
    assert (w.g, w.tile) == (2, n) and [t[:2] for t in w.tiles] == [(0, 2), (2, 1)]
    plan.close()


def test_automatic_time_tiles_across_groups(env):
    """fp32 complex, 40 scales x 3.5 M samples = 1.12 GB per channel: groups of one channel, each cut into tiles
    of BUDGET / (S * 8) samples rounded up to 1024."""
    env()
    plan = _plan(150.0 * (4.0 / 150.0) ** (np.arange(40) / 39.0), np.float32, "complex")
    n = 3_500_000
    assert 4 * plan.max_length < BUDGET // (40 * 8)
    w = Walk(plan, 2, n)
    assert w.g == 1 and w.tile < n and w.tile % 1024 == 0 and len(w.tiles) == 2 * -(-n // w.tile)
    seam = w.tile
    _large_case(plan, 2, n, [seam - 5000, seam - 1, seam, seam + 7, 3_400_000], -2000, 6000)
    plan.close()


# ------------------------------------------------------------------ 6. grid splits of the reduction kernels
def test_reduction_grid_splits_beyond_65535_channels():
    """band_reduce and event_reduce on 65539 channels: the c0 += 65535 launch loops.  Power-of-two weights keep
    every product exact, so the fp64 sums equal a sequential numpy sum to the bit."""
    nch, S, n = 65539, 3, 40
    rng = np.random.default_rng(11)
    re = rng.standard_normal((nch, S, n)).astype(np.float32)
    im = rng.standard_normal((nch, S, n)).astype(np.float32)
    W = (re + 1j * im).astype(np.complex64)
    m2 = re.astype(np.float64) ** 2 + im.astype(np.float64) ** 2
    plan = _plan([40.0, 20.0, 10.0], np.float32, "complex")
    amp = _plan([40.0, 20.0, 10.0], np.float32, "amplitude")
    first, count = np.array([0, 1, 0], np.int32), np.array([1, 2, 3], np.int32)
    weights = np.array([1.0, 0.5, 0.5, 0.25, 0.5, 1.0])
    for p, res, mag in ((plan, W, m2), (amp, re, re.astype(np.float64) ** 2)):
        got = p.band_reduce(torch.from_numpy(res).cuda(), first, count, weights).cpu().numpy()
        want = np.zeros((nch, first.size, n))
        o = 0
        for b in range(first.size):
            for k in range(count[b]):
                want[:, b] += weights[o] * mag[:, first[b] + k]
                o += 1
        assert np.array_equal(got, want.astype(np.float32)), p.output
    events, lag_first, n_lags = np.array([3, 3, 10, 25, 38]), -4, 9
    power, phase = plan.event_reduce(torch.from_numpy(W).cuda(), events, lag_first, n_lags)
    wp = np.zeros((nch, S, n_lags))
    wph = np.zeros((nch, S, n_lags), np.complex128)
    u = W.astype(np.complex128) / np.sqrt(m2)
    for lag in range(n_lags):
        for e in events:
            t = e + lag_first + lag
            if 0 <= t < n:
                wp[:, :, lag] += m2[:, :, t]
                wph[:, :, lag] += u[:, :, t]
    assert np.array_equal(power.cpu().numpy(), wp)
    assert np.abs(phase.cpu().numpy() - wph).max() <= 1e-12
    plan.close()
    amp.close()


# ------------------------------------------------------------------ 7. the seams against the oracle
def _bar_families(plan):
    """Per scale: interpolated (checked in the power domain) or direct, as tests/test_gpu_fused_kernels.py sets its
    bars.  The host path's rows are 16-byte aligned, so an interp class runs interpolated."""
    if plan.dtype == np.float64:
        return np.zeros(plan.n_scales, bool)
    classes, of_scale = plan.classes()
    return np.array([ci >= 0 and classes[ci]["kernel"] in ("interp", "wide2") for ci in of_scale])


@pytest.mark.parametrize("name,hint,with_epochs", [("f32-amplitude", 2000, False), ("f64-complex", 2999, True)])
def test_seams_against_the_oracle(name, hint, with_epochs, env):
    """+-300 samples around every tile seam and epoch edge, pointwise against the oracle of the whole recording."""
    dtype, output, in_dtype = PLANS[name]
    plan = _plan(FREQS, dtype, output)
    epochs = EPOCHS if with_epochs else None
    x = _recording(1, N, in_dtype)
    env(tile=hint)
    got = plan.execute_host(x, epochs=epochs)[0]
    w = Walk(plan, 1, N, epochs, hint=hint)
    edges = sorted({a for _, _, a, _, _, _ in w.tiles} | {b for _, b in w.epochs})
    assert len(edges) > 10
    cols = np.unique(np.concatenate([np.arange(max(0, e - 300), min(N, e + 300)) for e in edges]))
    W, _, _ = orc.cwt_complex(x[0].astype(np.float64), FS, frequencies=FREQS,
                              epoch_bounds=EPOCHS if with_epochs else None, parallel=True)
    M = np.abs(W).max(axis=1)[:, None]
    a, b = got[:, cols], W[:, cols]
    if dtype == np.float64:
        ratio = np.abs(a - b) / (EPS_64 * M)
    else:
        interp = _bar_families(plan)[:, None]
        p = a.astype(np.float64)
        ratio = np.where(interp, np.abs(p ** 2 - np.abs(b) ** 2) / (EPS_I * M ** 2), np.abs(p - np.abs(b)) / (EPS_D * M))
    s, t = np.unravel_index(np.argmax(ratio), ratio.shape)
    assert ratio.max() <= 1.0, ("scale", int(s), "column", int(cols[t]), float(ratio.max()))
    plan.close()
