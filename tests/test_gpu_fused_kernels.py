"""Every instance of the fp32 fused kernels (csrc/fast_path.cu, fast_run) against the CPU oracle, pointwise.

fast_run launches one fused kernel per scale class (CwtPlan.classes(), gcwt_plan_classes).  Which kernel and which
form of it runs is decided at launch time from the class, the output pointer and strides and the channel count:

* fused_full_kernel<TIn, KIND, GUARD> for the full-rate class (level -1); with the guard on and >= 64 chunks it runs
  as two launches, the measured chunks (q_mode 1) and the others (q_mode 2);
* fused_banded_kernel<KIND, LP, GUARD> for complex output, for amplitude / power under no_interp, for a level-2
  class that is not wide and for a level-3 U = 4 class whose rows are not 16-byte aligned; LP = 4 at level 2;
* fused_interp_kernel<KIND, GUARD>, whose rows are written by interp_rows_small (U = 4), interp_rows_pairs8 (level 4,
  rows 32-byte aligned, one block per chunk) or the sliding interp_rows<KIND, 3>, interp_rows<KIND, LU = 4 .. 10>,
  and the run-time-LU instance for levels 12 - 14;
* fused_wide2_kernel<KIND, GUARD> (levels 2 - 3, U = D) with scalar, 128-bit or 256-bit stores.

``_launch`` restates those rules, so every case asserts the instance and form it aims at: moving a threshold fails a
test instead of moving it off its target.

Reference: the oracle's complex rows of the exact float64 values the device read (a chirp + pink recording plus an
offset of 10, so that the mean removal matters), for a few scales per class.  Scales above 500 k taps (levels 12 -
14) are checked with a direct float64 sum W[t] = sum_j (x[j] - mean x) psi[t - j + (L - 1) // 2] at chosen columns:
both ends, both sides of every chunk seam of the class, and seeded random columns.

Bars, pointwise per row s with M_s = max|b_s| (b the oracle, a the device):

=========================  ============================  ===========================
kernel                     complex / amplitude           power
=========================  ============================  ===========================
direct (full, banded)      |a - b| <= EPS_D M_s          |a - |b|^2| <= 2 EPS_D M_s^2
interpolated (interp,      |a^2 - |b|^2| <= EPS_I M_s^2  |a - |b|^2| <= EPS_I M_s^2
wide2)
=========================  ============================  ===========================

Amplitude of the interpolated kernels is checked in the power domain: near a zero of |W| the interpolated amplitude
is sqrt|interp(|W|^2)|, whose pointwise error is only bounded by sqrt(EPS_I) M_s.

Every value check runs a plan with the guard on and asserts that the guard re-computed nothing (so the fused result
is what is checked), and the same plan with the guard off, whose bits must be identical: the GUARD instances only
add reductions.

Bars: EPS_D = 1.2e-6 and EPS_I = 1.6e-6, about twice the worst error measured on an NVIDIA B200 (power limit 1000 W):
the worst ratio of error to bar, over output kinds, input dtypes and guard on / off, per instance in
test_every_instance_against_reference, and per family over the whole module (writes, segments, edges, 48 voices):

  full-rate (level -1)                    0.37      interp_rows<KIND, 3> sliding (level 4)   0.33
  banded LP=4 (level 2)                   0.29      interp_rows<KIND, 4 .. 10> (levels 5-11) 0.27 .. 0.47
  banded LP=4, non-wide level-2 class     0.27      run-time LU (levels 12 / 13 / 14)        0.29 / 0.22 / 0.34
  banded LP=0 (levels 3-8 / 9-11 / 12-14) 0.39 / 0.44 / 0.40   wide2 LU 2 / LU 3           0.43 / 0.37
  interp_rows_small (U = 4, level 3)      0.38      whole module, direct kernels             0.51
  interp_rows_pairs8 (level 4)            0.33      whole module, interpolated kernels       0.50

The bars are pointwise: one wrong sample in a row fails them, where a per-row relative L2 bar averages it away.
"""
from multiprocessing import cpu_count
from multiprocessing.pool import ThreadPool

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ghost_b200 import Morse, synth                                      # noqa: E402
from ghost_b200.engine import CwtPlan, scale_tables                      # noqa: E402
from oracle import cwt_oracle as orc                                     # noqa: E402

FS = 1000.0
OFFSET = 10.0
EPS_D, EPS_I = 1.2e-6, 1.6e-6
IN_DTYPES = {"f32in": np.float32, "f64in": np.float64}

# The broad wavelet: gamma = 3, beta = 8 is the first of a (gamma, beta) sweep (gamma 3 / 2 / 1.5, beta 20 / 8 / 4 / 2 /
# 1, 10 voices, 200 k samples) whose level-2 and level-3 bands are too wide for U = D: its level-2 class runs the banded
# kernel and its level-3 class interp_rows_small (U = 4).  test_every_instance_against_reference asserts both.
BROAD = (3, 8)
# levels 9 - 11 (U = 2^8 .. 2^10), two scales each, on the default wavelet at 1 kHz
FREQS_B = (0.28, 0.2, 0.14, 0.1, 0.07, 0.045)
# levels 12, 13 and 14 (run-time U), two scales each; the last has the largest L whose halo fits level 14
FREQS_C = (0.034, 0.022, 0.017, 0.011, 0.0086, 0.0019)
HALO_MAX_14 = int(0.45 * 1024 * 2 ** 14) + 1          # L - 1 <= 0.45 * 1024 * 2^14


def _lengths_c():
    om = np.asarray(FREQS_C) / (FS / 2.0) * np.pi
    L = Morse(gamma=3, beta=20, fs=FS).compute_lengths(om).astype(np.int64)
    L[-1] = HALO_MAX_14
    return L


# recordings: (n, gamma, beta, frequencies or None for the default grid, explicit lengths or None)
GROUPS = {
    "A": (200_000, 3, 20, None, None),                     # full-rate, banded (complex) and levels 2 .. 8
    "broad": (200_000, BROAD[0], BROAD[1], None, None),    # non-wide level-2 and level-3 classes
    "B": (2_000_000, 3, 20, FREQS_B, None),                # levels 9 .. 11, 1 - 4 chunk seams
    "C": (3_600_000, 3, 20, FREQS_C, _lengths_c()),        # levels 12 .. 14 (one seam at level 12), direct sums
}
DIRECT_GROUPS = ("C",)


# ------------------------------------------------------------------ the launcher's rules (fast_run)
def rows_aligned(ptr, s_stride, c_stride):
    """Rows 16-byte aligned (ptr in bytes, strides in float elements): U = 4 interpolation and 128-bit stores."""
    return ptr % 16 == 0 and s_stride % 4 == 0 and c_stride % 4 == 0


def rows_aligned32(ptr, s_stride, c_stride):
    """Rows 32-byte aligned: pairs8 at level 4 and 256-bit stores of fused_wide2_kernel."""
    return ptr % 32 == 0 and s_stride % 8 == 0 and c_stride % 8 == 0


def guard_every(n_chunks, every):
    """Every how many chunks the guard measures one (set_guard_sampling)."""
    return 2 * every if n_chunks >= 512 else (every if n_chunks >= 256 else (every // 2 if n_chunks >= 64 else 1))


def _ilog2_ceil(v):
    return (int(v) - 1).bit_length()


def _launch(cls, n, n_channels, ra, ra32):
    """What fast_run launches for class ``cls`` (a dict of CwtPlan.classes()) on n samples of n_channels channels,
    with the guard on."""
    kernel, level, lu = cls["kernel"], cls["level"], cls["log2u"]
    n_chunks = -(-n // cls["hop"])
    if kernel == "wide2":
        return dict(family="wide2", form="wide2_lu%d" % lu, align=2 if ra32 else (1 if ra else 0), upc=1,
                    n_chunks=n_chunks)
    if kernel == "interp" and (lu >= 3 or ra):
        chunks = n_channels * n_chunks
        upc = max(1, min(-(-1776 // chunks), max(1, (1 << level) // 32)))
        upc = min(upc, 24)
        iters = 2 if ra32 else 1
        if lu == 2:
            form = "small"
        elif lu == 3:
            form = "pairs8" if (iters == 2 and upc == 1) else "sliding3"
        elif lu <= 10:
            form = "lu%d" % lu
        else:
            form = "lu_rt"
        return dict(family="interp", form=form, iters=iters, upc=upc, n_chunks=n_chunks)
    if level >= 0:
        p_cols = (1024 << level) // 256
        assert cls["chunk"] == 1024 << level
        blocks = p_cols // 16
        iters = min(blocks, 16)
        return dict(family="banded", form="banded_lp4" if _ilog2_ceil(p_cols) == 4 else "banded_lp0", iters=iters,
                    upc=-(-blocks // iters), n_chunks=n_chunks, fallback=kernel == "interp")
    ge = guard_every(n_chunks, 16)
    n_meas = -(-n_chunks // ge)
    return dict(family="full", form="full", guard_every=ge, n_chunks=n_chunks, n_meas=n_meas, split=n_chunks > n_meas)


def _interp_bar(launch):
    return launch["family"] in ("interp", "wide2")


# ------------------------------------------------------------------ plans, references, bars
def _tables(freqs, gamma=3, beta=20, lengths=None):
    m = Morse(gamma=gamma, beta=beta, fs=FS)
    om = np.asarray(freqs, dtype=np.float64) / (FS / 2.0) * np.pi
    L = m.compute_lengths(om) if lengths is None else np.asarray(lengths, dtype=np.int64)
    return (L,) + scale_tables(m, om, L)


def _freqs(group):
    n, gamma, beta, freqs, _ = GROUPS[group]
    return orc.frequency_grid(FS, n, gamma, beta) if freqs is None else np.asarray(freqs, dtype=np.float64)


def _recording(n, in_dtype, channel=0):
    return (synth.chirp_pink(n, FS, channel, np.float64) + OFFSET).astype(in_dtype)


def _plan(tables, output, guard=True, no_interp=False):
    return CwtPlan(*tables, dtype=np.float32, output=output, guard=guard, no_interp=no_interp)


def _pick(ids):
    """A few scales of a class: first, middle, last."""
    ids = np.asarray(ids)
    return sorted(set([int(ids[0]), int(ids[len(ids) // 2]), int(ids[-1])]))


def _direct(xm, rev, cols):
    """W[t] = sum_j xm[j] psi[t - j + (L - 1) // 2] at the columns ``cols``, in float64: xm is the recording minus
    its mean, rev = (real, imag) of psi reversed (rev[L - 1 - m] = psi[m])."""
    rr, ri = rev
    L, n = rr.size, xm.size
    h = (L - 1) // 2

    def one(t):
        j0, j1 = max(0, t + h - L + 1), min(n, t + h + 1)
        k0 = L - 1 - t - h + j0
        seg = xm[j0:j1]
        return complex(seg @ rr[k0:k0 + j1 - j0], seg @ ri[k0:k0 + j1 - j0])
    with ThreadPool(cpu_count()) as pool:          # the dot products release the interpreter lock
        return np.array(pool.map(one, [int(t) for t in cols], chunksize=4), dtype=np.complex128)


_KERNELS = {}


def _reversed_kernel(gamma, beta, f, L):
    key = (gamma, beta, float(f), int(L))
    if key not in _KERNELS:
        psi, _ = orc.morse_kernel(gamma, beta, orc.hz_to_rad(f, FS), int(L))
        r = psi[::-1]
        _KERNELS[key] = (np.ascontiguousarray(r.real), np.ascontiguousarray(r.imag))
    return _KERNELS[key]


def _columns(n, hop, seed):
    """Both ends, +-8 columns around every owned-range boundary q hop, and 192 seeded random columns."""
    parts = [np.arange(min(64, n)), np.arange(max(0, n - 64), n)]
    for q in range(1, -(-n // hop)):
        parts.append(np.arange(max(0, q * hop - 8), min(n, q * hop + 8)))
    parts.append(np.random.default_rng(seed).integers(0, n, 192))
    return np.unique(np.concatenate(parts))


WORST = {}


def _record(key, ratio):
    WORST[key] = max(WORST.get(key, 0.0), float(ratio))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(WORST):
        print("worst ratio %-40s %.3f" % (k, WORST[k]))


def _check(got, W, output, interp, row_max, what, key=None):
    """Bars of the module docstring.  got (S, m) device values, W (S, m) complex references at the same columns,
    row_max (S,) = max|b_s| over the whole row."""
    got = np.asarray(got)
    got = got.astype(np.complex128 if np.iscomplexobj(got) else np.float64)
    M = np.asarray(row_max, dtype=np.float64)[:, None]
    p = np.abs(W) ** 2
    if output == "complex":
        assert not interp
        ratio = np.abs(got - W) / (EPS_D * M)
    elif output == "amplitude":
        ratio = np.abs(got ** 2 - p) / (EPS_I * M ** 2) if interp else np.abs(got - np.abs(W)) / (EPS_D * M)
    else:
        ratio = np.abs(got - p) / ((EPS_I if interp else 2 * EPS_D) * M ** 2)
    assert not np.isnan(got).any(), what
    worst = float(ratio.max()) if ratio.size else 0.0
    if key is not None:
        _record(key, worst)
    s, t = np.unravel_index(np.argmax(ratio), ratio.shape)
    assert worst <= 1.0, (what, "row", int(s), "column", int(t), worst)


def _bits(t):
    if t.is_complex():
        t = torch.view_as_real(t)
    return t.contiguous().view(torch.int32)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# ------------------------------------------------------------------ output layouts
SENTINEL = np.uint32(0x7FC0BEEF)          # a quiet NaN with a payload no kernel writes
# name: (out_start, row width): rows are every other row of a (2 C, 2 S + 1, width) buffer, channels every other one
LAYOUTS = {
    "a2": (0, None),        # scale stride = 2 width = 0 mod 8, rows 32-byte aligned
    "a1": (4, 6),           # scale stride = 4 mod 8, 16-byte aligned
    "a0": (1, 1),           # unaligned
}


def _layout_width(layout, n):
    out_start, mod = LAYOUTS[layout]
    w = out_start + n + 8
    if mod is None:
        w += (-w) % 8
    elif mod == 6:
        w += (6 - w) % 8
    else:
        w += (1 - w) % 2
    return w


class Window:
    """A NaN-sentinel buffer and the strided view inside it that a plan writes."""

    def __init__(self, plan, n_channels, n, layout):
        S = plan.n_scales
        self.out_start = LAYOUTS[layout][0]
        self.n = n
        w = _layout_width(layout, n)
        cplx = plan.output == "complex"
        self.buf = torch.empty((2 * n_channels, 2 * S + 1, w * (2 if cplx else 1)), dtype=torch.float32, device="cuda")
        self.buf.view(torch.int32).fill_(int(SENTINEL.view(np.int32)))
        full = torch.view_as_complex(self.buf.view(2 * n_channels, 2 * S + 1, w, 2)) if cplx else self.buf
        self.full = full
        self.view = full[::2, 0:2 * S:2, :]
        esz = self.view.element_size()
        ptr = self.view.data_ptr() + self.out_start * esz
        # fast_run's flags are in float elements for the real kinds (complex output never interpolates)
        self.ra = rows_aligned(ptr, self.view.stride(1), self.view.stride(0))
        self.ra32 = rows_aligned32(ptr, self.view.stride(1), self.view.stride(0))

    def window(self):
        return self.view[:, :, self.out_start:self.out_start + self.n]

    def untouched_outside(self):
        """Nothing outside the window differs from the sentinel bits, nothing inside is NaN."""
        raw = self.buf.view(torch.int32).clone()
        mask = torch.ones(self.full.shape, dtype=torch.bool, device="cuda")
        mask[::2, 0:mask.shape[1] - 1:2, self.out_start:self.out_start + self.n] = False
        if self.full.is_complex():
            mask = mask.unsqueeze(-1).expand(*mask.shape, 2).reshape(raw.shape)
        outside = raw[mask]
        ok = bool((outside == int(SENTINEL.view(np.int32))).all())
        inside_nan = bool(torch.isnan(self.window()).any())
        return ok and not inside_nan


# ------------------------------------------------------------------ recordings, cached per module
class Recording:
    """One recording of a group: samples, plan tables and the references of the scales asked for so far."""

    def __init__(self, group, in_dtype):
        self.group = group
        self.n, self.gamma, self.beta, _, lengths = GROUPS[group]
        self.freqs = _freqs(group)
        self.tables = _tables(self.freqs, self.gamma, self.beta, lengths)
        self.x = _recording(self.n, in_dtype)
        self.x64 = self.x.astype(np.float64)
        self._rows, self._direct = {}, {}

    def rows(self, ids):
        """Oracle rows (len(ids), n) of the whole recording."""
        assert self.group not in DIRECT_GROUPS
        missing = [i for i in ids if i not in self._rows]
        if missing:
            W, _, L = orc.cwt_complex(self.x64, FS, gamma=self.gamma, beta=self.beta,
                                      frequencies=self.freqs[missing], parallel=True)
            np.testing.assert_array_equal(L, self.tables[0][missing])
            self._rows.update(zip(missing, W))
        return np.stack([self._rows[i] for i in ids])

    def direct(self, i, cols):
        """Direct float64 sums of scale i at the columns ``cols`` (cached per column)."""
        have = self._direct.setdefault(i, {})
        missing = [int(t) for t in cols if int(t) not in have]
        if missing:
            rev = _reversed_kernel(self.gamma, self.beta, self.freqs[i], self.tables[0][i])
            have.update(zip(missing, _direct(self.x64 - self.x64.mean(), rev, missing)))
        return np.array([have[int(t)] for t in cols])


@pytest.fixture(scope="module")
def rec():
    cache = {}

    def get(group, in_dtype=np.float32):
        key = (group, np.dtype(in_dtype).name)
        if key not in cache:
            cache[key] = Recording(group, in_dtype)
        return cache[key]
    return get


def _check_class(r, got, cls, ci, of_scale, launch, output, what, key=None):
    """Rows of class ci of the device result ``got`` (S, n) (a torch view) against the references of ``r``."""
    ids = _pick(np.nonzero(of_scale == ci)[0])
    if r.group in DIRECT_GROUPS:
        cols = _columns(r.n, cls["hop"], seed=cls["level"])
        W = np.stack([r.direct(i, cols) for i in ids])
        amp = got[ids].abs().double()
        if output == "power":
            amp = amp.sqrt()
        row_max = np.maximum(np.abs(W).max(axis=1), amp.max(dim=1).values.cpu().numpy())
        rows = got[ids][:, torch.from_numpy(cols).cuda()].cpu().numpy()
    else:
        W = r.rows(ids)
        row_max = np.abs(W).max(axis=1)
        rows = got[ids].cpu().numpy()
    _check(rows, W, output, _interp_bar(launch), row_max, what=what, key=key)


# ------------------------------------------------------------------ 0. the class query
def test_plan_classes_agree_with_levels(rec):
    """gcwt_plan_classes: every fused scale in exactly one class of its level; fp64 plans and plans of generic
    scales report no class."""
    r = rec("A")
    for output, no_interp in (("amplitude", False), ("complex", False), ("power", True)):
        plan = _plan(r.tables, output, no_interp=no_interp)
        classes, of_scale = plan.classes()
        levels = plan.levels()
        assert (of_scale >= 0).all()
        assert sorted({c["level"] for c in classes}) == sorted(set(levels.tolist()))
        for ci, c in enumerate(classes):
            ids = np.nonzero(of_scale == ci)[0]
            assert ids.size == c["n_scales"] <= (64 if c["level"] < 0 else 16) and (levels[ids] == c["level"]).all()
            assert 0 < c["offset"] and 0 < c["hop"] <= c["chunk"] - c["offset"]
            assert c["chunk"] == (4096 if c["level"] < 0 else (1024 << c["level"]) * (2 if c["kernel"] == "wide2" else 1))
            if output == "complex" or no_interp:
                assert c["kernel"] in ("full", "banded") and c["log2u"] == 0
        plan.close()
    for plan in (CwtPlan(*r.tables, dtype=np.float64, output="amplitude"),
                 CwtPlan(*r.tables, dtype=np.float32, output="amplitude", force_generic=True)):
        classes, of_scale = plan.classes()
        assert classes == [] and (of_scale == -1).all()
        plan.close()


# ------------------------------------------------------------------ 1. every instance against the reference
KINDS3, KINDS2 = ("complex", "amplitude", "power"), ("amplitude", "power")
# name: (group, form, level or None, output kinds, layout, no_interp)
INSTANCES = {
    "full": ("A", "full", None, KINDS3, "a2", False),
    "banded_lp4": ("A", "banded_lp4", 2, KINDS3, "a2", True),
    "banded_lp0": ("A", "banded_lp0", None, KINDS3, "a2", True),               # levels 3 .. 8
    "banded_lp0_B": ("B", "banded_lp0", None, ("complex",), "a2", False),      # levels 9 .. 11
    "banded_lp0_C": ("C", "banded_lp0", None, ("complex",), "a2", False),      # levels 12 .. 14
    "banded_lp4_nonwide": ("broad", "banded_lp4", 2, KINDS2, "a2", False),     # a level-2 class too wide for U = D
    "small": ("broad", "small", 3, KINDS2, "a2", False),
    "pairs8": ("A", "pairs8", 4, KINDS2, "a2", False),
    "sliding3": ("A", "sliding3", 4, KINDS2, "a1", False),
    **{"lu%d" % lu: ("A" if lu <= 7 else "B", "lu%d" % lu, lu + 1, KINDS2, "a2", False) for lu in range(4, 11)},
    **{"lu_rt%d" % lv: ("C", "lu_rt", lv, KINDS2, "a2", False) for lv in (12, 13, 14)},
    "wide2_lu2": ("A", "wide2_lu2", 2, KINDS2, "a2", False),
    "wide2_lu3": ("A", "wide2_lu3", 3, KINDS2, "a2", False),
}


def _instance_params():
    out = []
    for name, (_, _, _, kinds, _, _) in INSTANCES.items():
        for output in kinds:
            for in_dtype in IN_DTYPES:
                out.append(pytest.param(name, output, in_dtype, id="%s-%s-%s" % (name, output, in_dtype)))
    return out


@pytest.mark.parametrize("name,output,in_dtype", _instance_params())
def test_every_instance_against_reference(rec, name, output, in_dtype):
    group, form, level, _, layout, no_interp = INSTANCES[name]
    r = rec(group, IN_DTYPES[in_dtype])
    xd = _dev(r.x[None])
    wins = {}
    for guard in (True, False):
        plan = _plan(r.tables, output, guard=guard, no_interp=no_interp)
        if guard:
            classes, of_scale = plan.classes()
        else:
            assert plan.classes()[0] == classes
        win = Window(plan, 1, r.n, layout)
        plan.execute(xd, win.view, out_start=win.out_start)
        if guard:
            assert plan.guard_stats()["last"] == 0, "the guard replaced fused rows"
        plan.close()
        wins[guard] = win
    win = wins[True]
    assert _same_bits(win.window(), wins[False].window()), "guard on and off differ"
    assert win.untouched_outside()
    launches = [_launch(c, r.n, 1, win.ra, win.ra32) for c in classes]
    targets = [i for i, (c, la) in enumerate(zip(classes, launches))
               if la["form"] == form and (level is None or c["level"] == level)]
    assert targets, (name, [(c["level"], c["kernel"], la["form"]) for c, la in zip(classes, launches)])
    got = win.window()[0]
    for ci in targets:
        _check_class(r, got, classes[ci], ci, of_scale, launches[ci], output, what=(name, ci),
                     key="%s/%s" % (name, output))


# ------------------------------------------------------------------ 2. recording edges and chunk seams
EDGE_CASES = {"full": "power", "banded": "complex", "interp": "amplitude", "wide2": "power"}


@pytest.mark.parametrize("family", list(EDGE_CASES))
def test_recording_edges_and_seams(rec, family):
    """One class of each family, its scales alone, on lengths k hop - 1, k hop, k hop + 1, shorter than one chunk
    and odd; every column is checked."""
    output = EDGE_CASES[family]
    r = rec("A")
    plan = _plan(r.tables, output)
    classes, of_scale = plan.classes()
    plan.close()
    ci = [i for i, c in enumerate(classes) if _launch(c, r.n, 1, True, True)["family"] == family][-1]
    cls = classes[ci]
    ids = np.nonzero(of_scale == ci)[0]
    tables = _tables(r.freqs[ids], r.gamma, r.beta)
    plan = _plan(tables, output)
    sub, sub_of = plan.classes()
    assert len(sub) == 1 and (sub_of == 0).all()
    assert {k: sub[0][k] for k in ("level", "kernel", "log2u", "chunk", "offset", "hop")} == \
        {k: cls[k] for k in ("level", "kernel", "log2u", "chunk", "offset", "hop")}
    hop = cls["hop"]
    lengths = [2 * hop - 1, 2 * hop, 2 * hop + 1, 3 * hop + 7, max(64, cls["chunk"] // 3) | 1]
    assert lengths[-1] < cls["chunk"]
    for n in lengths:
        x = _recording(n, np.float32, channel=3)
        win = Window(plan, 1, n, "a2")
        plan.execute(_dev(x[None]), win.view, out_start=0)
        assert plan.guard_stats()["last"] == 0
        assert win.untouched_outside(), n
        la = _launch(sub[0], n, 1, win.ra, win.ra32)
        assert la["family"] == family
        pick = _pick(np.arange(ids.size))
        W, _, _ = orc.cwt_complex(x.astype(np.float64), FS, gamma=r.gamma, beta=r.beta,
                                  frequencies=r.freqs[ids[pick]], parallel=True)
        _check(win.window()[0][pick].cpu().numpy(), W, output, _interp_bar(la), np.abs(W).max(axis=1),
               what=(family, n), key="edges-%s/%s" % (family, output))
    plan.close()


# ------------------------------------------------------------------ 3. where each kernel writes
@pytest.mark.parametrize("output", ["complex", "amplitude"])
@pytest.mark.parametrize("group", ["A", "broad"])
def test_where_each_kernel_writes(rec, group, output):
    """Two channels (x and -2 x, whose coefficients are exactly -2 W) into every other scale row and every other
    channel of a NaN-sentinel buffer, at out_start 0 / 4 / 1 with scale strides 0 / 4 mod 8 and unaligned: 256-bit,
    128-bit and scalar stores, and the banded fallback of a U = 4 class.  Nothing outside the window may change; the
    store form alone must not change a bit, where the form changes the arithmetic each form meets its bar."""
    r = rec(group)
    X = np.stack([r.x, -2 * r.x])
    xd = _dev(X)
    plan = _plan(r.tables, output)
    classes, of_scale = plan.classes()
    flags = {"a2": (True, True), "a1": (True, False), "a0": (False, False)}
    results, forms = {}, {}
    for layout in LAYOUTS:
        win = Window(plan, 2, r.n, layout)
        assert (win.ra, win.ra32) == flags[layout]
        plan.execute(xd, win.view, out_start=win.out_start)
        assert plan.guard_stats()["last"] == 0
        assert win.untouched_outside(), layout
        launches = [_launch(c, r.n, 2, win.ra, win.ra32) for c in classes]
        forms[layout] = launches
        got = win.window()
        for ci, (c, la) in enumerate(zip(classes, launches)):
            for ch, k in ((0, 1.0), (1, -2.0)):
                ids = _pick(np.nonzero(of_scale == ci)[0])
                W = k * r.rows(ids)
                _check(got[ch][ids].cpu().numpy(), W, output, _interp_bar(la), np.abs(W).max(axis=1),
                       what=(layout, ci, ch), key="writes-%s/%s" % (la["form"], output))
        results[layout] = win.window().clone()
        del win
    if output != "complex":
        wide = [la for la in forms["a2"] if la["family"] == "wide2"]
        assert {la["align"] for la in wide} == {2} if wide else True
        assert all(la["align"] == 1 for la in forms["a1"] if la["family"] == "wide2")
        assert all(la["align"] == 0 for la in forms["a0"] if la["family"] == "wide2")
        if group == "broad":
            assert any(la.get("fallback") for la in forms["a0"]), "no U = 4 class fell back to the banded kernel"
            assert any(la["form"] == "small" for la in forms["a2"])
    # the store form alone (256-bit / 128-bit / scalar, units_per_chunk) changes no bit; pairs8 vs the sliding
    # interpolator and interp_rows_small vs the banded fallback compute differently and met their bars above
    for ci in range(len(classes)):
        ids = np.nonzero(of_scale == ci)[0]
        for lay in ("a1", "a0"):
            first = next(f for f in LAYOUTS if forms[f][ci]["form"] == forms[lay][ci]["form"])
            if first != lay:
                assert _same_bits(results[lay][:, ids], results[first][:, ids]), (ci, lay, forms[lay][ci])
    plan.close()


@pytest.mark.parametrize("segment", ["middle", "tail"])
def test_segment_with_clipped_halos(rec, segment):
    """A time segment with halos of L_max - 1 (clipped at the recording's end), checked against the oracle of the
    whole recording."""
    r = rec("A")
    n = r.n
    lmax = int(r.tables[0].max())
    seg = n // 3
    start = (n - seg) // 2 if segment == "middle" else n - seg
    stop = start + seg
    halo_l, halo_r = min(lmax - 1, start), min(lmax - 1, n - stop)
    xb = torch.full((2, n + 41), float("nan"), dtype=torch.float32, device="cuda")
    xv = xb[:, 13:13 + n]
    xv.copy_(_dev(np.stack([r.x, -2 * r.x])))
    for output in ("amplitude", "complex"):
        plan = _plan(r.tables, output)
        classes, of_scale = plan.classes()
        means = plan.channel_means(xv)
        win = Window(plan, 2, seg, "a2")
        plan.execute(xv, win.view, means=means, start=start, stop=stop, halo_left=halo_l, halo_right=halo_r,
                     out_start=0)
        assert plan.guard_stats()["last"] == 0
        assert win.untouched_outside()
        got = win.window()
        for ci, c in enumerate(classes):
            la = _launch(c, seg, 2, win.ra, win.ra32)
            ids = _pick(np.nonzero(of_scale == ci)[0])
            for ch, k in ((0, 1.0), (1, -2.0)):
                W = k * r.rows(ids)
                _check(got[ch][ids].cpu().numpy(), W[:, start:stop], output, _interp_bar(la),
                       np.abs(W).max(axis=1), what=(segment, ci, ch), key="segment-%s/%s" % (la["form"], output))
        plan.close()


# ------------------------------------------------------------------ 4. 64-bit offsets
def test_channel_strides_beyond_2_31():
    """An input and an output whose channel strides exceed 2^31 elements: the second channel's rows must equal
    the first channel's run alone, bit for bit, for every kernel family."""
    n = 60_000
    freqs = orc.frequency_grid(FS, n)
    tables = _tables(freqs)
    x = _recording(n, np.float32)
    big = (1 << 31) + 64
    xb = torch.empty(big + n, dtype=torch.float32, device="cuda")
    xv = xb.as_strided((2, n), (big, 1))
    xv[0].copy_(_dev(x))
    xv[1].copy_(_dev(x))
    families = set()
    for output, no_interp in (("amplitude", False), ("complex", False), ("power", True)):
        plan = _plan(tables, output, no_interp=no_interp)
        classes, _ = plan.classes()
        families |= {_launch(c, n, 2, True, True)["family"] for c in classes}
        S = plan.n_scales
        ob = torch.empty(big + S * n, dtype=plan.torch_out_dtype, device="cuda")
        ov = ob.as_strided((2, S, n), (big, n, 1))
        plan.execute(xv, ov)
        alone = plan.execute(_dev(x[None]))
        assert _same_bits(ov[1], alone[0]), output
        assert _same_bits(ov[0], alone[0]), output
        del ob, ov, alone
        plan.close()
    assert families == {"full", "banded", "interp", "wide2"}, families
    del xb, xv
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 5. bit-for-bit invariants
@pytest.mark.parametrize("k", [63, 64, 255, 256, 511, 512, 513])
def test_full_class_guard_split_bits(rec, k):
    """The full-rate class at k chunks: the guard measures every guard_every-th chunk in a launch of its own (q_mode
    1) and the others in a second one (q_mode 2); without the guard one launch covers all.  Bits must not differ."""
    r = rec("A")
    plan = _plan(r.tables, "amplitude")
    classes, of_scale = plan.classes()
    plan.close()
    ci = [i for i, c in enumerate(classes) if c["kernel"] == "full"][0]
    ids = np.nonzero(of_scale == ci)[0]
    tables = _tables(r.freqs[ids])
    on, off = _plan(tables, "amplitude"), _plan(tables, "amplitude", guard=False)
    assert on.classes()[0] == [classes[ci]]
    on.close()
    off.close()
    n = k * classes[ci]["hop"]
    la = _launch(classes[ci], n, 1, True, True)
    assert la["n_chunks"] == k
    assert la["guard_every"] == {63: 1, 64: 8, 255: 8, 256: 16, 511: 16, 512: 32, 513: 32}[k]
    assert la["split"] == (k >= 64)
    x = _recording(n, np.float32, channel=5)
    xd = _dev(x[None])
    for output in ("complex", "amplitude"):
        on, off = _plan(tables, output), _plan(tables, output, guard=False)
        a, b = on.execute(xd), off.execute(xd)
        assert on.guard_stats()["last"] == 0
        assert _same_bits(a, b), (k, output)
        if k in (64, 513):
            pick = _pick(np.arange(ids.size))
            W, _, _ = orc.cwt_complex(x.astype(np.float64), FS, frequencies=r.freqs[ids[pick]], parallel=True)
            _check(a[0][pick].cpu().numpy(), W, output, False, np.abs(W).max(axis=1), what=(k, output),
                   key="full-split/%s" % output)
        on.close()
        off.close()


def test_channel_alone_equals_batch_of_40(rec):
    """40 channels: the interpolated classes split each chunk over fewer blocks (units_per_chunk) than for one
    channel alone.  Each channel alone must give the same bits."""
    r = rec("B")
    C = 40
    X = np.stack([r.x] + [_recording(r.n, np.float32, channel=c) for c in range(1, C)])
    xd = _dev(X)
    plan = _plan(r.tables, "amplitude")
    classes, _ = plan.classes()
    upc = [(_launch(c, r.n, 1, True, True).get("upc"), _launch(c, r.n, C, True, True).get("upc")) for c in classes
           if c["kernel"] == "interp"]
    assert any(a != b for a, b in upc), upc
    full = plan.execute(xd)
    for c in range(C):
        assert _same_bits(plan.execute(xd[c:c + 1])[0], full[c]), c
    plan.close()


def test_f64_input_of_f32_values(rec):
    """f64 input carrying fp32 values vs the same values as f32: the full-rate class subtracts the mean in double
    before rounding on both, so its rows are identical; the pyramid subtracts in fp32 for f32 input and in fp64 for
    f64 input, so the band classes differ and meet the bars."""
    r = rec("A")
    x32 = r.x
    for output in ("complex", "amplitude"):
        plan = _plan(r.tables, output)
        classes, of_scale = plan.classes()
        a = plan.execute(_dev(x32[None]))[0]
        b = plan.execute(_dev(x32.astype(np.float64)[None]))[0]
        assert plan.guard_stats()["last"] == 0
        band_differs = False
        for ci, c in enumerate(classes):
            ids = np.nonzero(of_scale == ci)[0]
            la = _launch(c, r.n, 1, True, True)
            if c["kernel"] == "full":
                assert _same_bits(a[ids], b[ids]), (output, ci)
            else:
                band_differs |= not _same_bits(a[ids], b[ids])
                pick = _pick(ids)
                W = r.rows(pick)
                _check(b[pick].cpu().numpy(), W, output, _interp_bar(la), np.abs(W).max(axis=1), what=(output, ci))
        assert band_differs, output
        plan.close()


@pytest.mark.parametrize("output", ["complex", "amplitude"])
def test_class_splits_at_48_voices(output):
    """48 voices per octave: more than 16 scales at a level split into several classes, more than 64 full-rate
    scales into several full-rate classes (64 scales each).  Every row against the oracle."""
    n = 60_000
    freqs = orc.frequency_grid(FS, n, voices_per_octave=48)
    tables = _tables(freqs)
    plan = _plan(tables, output)
    classes, of_scale = plan.classes()
    assert (of_scale >= 0).all()
    levels = [c["level"] for c in classes]
    n_full = int((plan.levels() == -1).sum())
    assert n_full > 128 and levels.count(-1) == -(-n_full // 64), (n_full, levels)
    assert any(levels.count(lv) >= 2 for lv in set(levels) if lv >= 0), levels
    x = _recording(n, np.float32, channel=7)
    got = plan.execute(_dev(x[None]))[0]
    assert plan.guard_stats()["last"] == 0
    W, _, L = orc.cwt_complex(x.astype(np.float64), FS, voices_per_octave=48, frequencies=freqs, parallel=True)
    for ci, c in enumerate(classes):
        ids = np.nonzero(of_scale == ci)[0]
        la = _launch(c, n, 1, True, True)
        _check(got[ids].cpu().numpy(), W[ids], output, _interp_bar(la), np.abs(W[ids]).max(axis=1),
               what=(output, ci), key="vpo48-%s/%s" % (la["form"], output))
    plan.close()
