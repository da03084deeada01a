"""Generate tests/golden/* by running the UNMODIFIED reference (/root/reference).

Run in the build container only (the GPU box has no /root/reference):

    python oracle/gen_golden.py

The reference needs two shims to import under numpy 2.x without matplotlib
(SURVEY.md Appendix C): stub ``matplotlib`` modules and explicit ``timestamps``
(which avoids the removed ``np.float``).  Nothing of the reference is copied; only
its outputs are stored.
"""
from __future__ import annotations

import json
import logging
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)


def load_reference(path="/root/reference"):
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, path)
    logging.disable(logging.WARNING)
    import ghost  # noqa: F401
    from ghost import sigtools
    from ghost.wave import ContinuousWaveletTransform, Morse, morseutils
    return ContinuousWaveletTransform, Morse, morseutils, sigtools


def sample_columns(n, k, edge, seed=0):
    """Sorted indices of the columns stored of a length-n output axis (it keeps every golden file under
    1 MB): all of them when n <= k, else the first and last ``edge`` and a seeded draw of the others, k in all."""
    if n <= k:
        return np.arange(n)
    inner = np.random.default_rng(seed).choice(np.arange(edge, n - edge), size=k - 2 * edge, replace=False)
    return np.concatenate([np.arange(edge), np.sort(inner), np.arange(n - edge, n)])


def ref_complex(CWT, Morse, sigtools, x, fs, gamma, beta, freqs_hz):
    """The reference's own wavelet_conv body (transforms.py:187-204) minus abs."""
    cwt = CWT(wavelet=Morse(gamma=gamma, beta=beta))
    cwt.fs = fs
    cwt._wavelet.fs = fs
    xs = x.astype(np.float64) - np.mean(x.astype(np.float64))
    rows = []
    lens = cwt.wavelet.compute_lengths(cwt._hz_to_norm_radians(freqs_hz))
    for f, L in zip(freqs_hz, lens):
        wv = cwt.wavelet.copy()
        wv.norm_radian_freq = cwt._hz_to_norm_radians(f)
        kernel, _ = wv(int(L))
        rows.append(sigtools.fastconv_scipy(xs, kernel))
    return np.array(rows), lens


def main():
    from ghost_b200 import synth
    CWT, Morse, mu, sigtools = load_reference()
    os.makedirs(GOLD, exist_ok=True)

    # ---- scalars over a gamma/beta grid -------------------------------------
    scal = {}
    for g in (1, 2, 3, 6, 9):
        for b in (1, 3, 10, 20, 40, 80):
            scal[f"{g},{b}"] = {"morsefreq": float(mu.morsefreq(g, b)),
                                "morsehigh": float(mu.morsehigh(g, b))}
    json.dump(scal, open(os.path.join(GOLD, "morse_scalars.json"), "w"), indent=0)

    # ---- frequency grids and kernel lengths ---------------------------------
    grids = []
    cases = [
        dict(name="cfg1", fs=1000.0, n=60000, gamma=3, beta=20, freq_limits=None, vpo=10),
        dict(name="cfg2", fs=1250.0, n=2250000, gamma=3, beta=20, freq_limits=[0.40, 300], vpo=10),
        dict(name="cfg3", fs=30000.0, n=18000000, gamma=3, beta=20, freq_limits=[1.7, 15000], vpo=10),
        dict(name="cfg4", fs=30000.0, n=2592000000, gamma=3, beta=20, freq_limits=[1.7, 15000], vpo=10),
        dict(name="short", fs=500.0, n=2000, gamma=3, beta=20, freq_limits=None, vpo=10),
        dict(name="vpo4", fs=1000.0, n=65536, gamma=3, beta=20, freq_limits=None, vpo=4),
        dict(name="vpo48", fs=1000.0, n=65536, gamma=3, beta=20, freq_limits=[5, 400], vpo=48),
    ]
    for g in (1, 2, 3, 6, 9):
        for b in (1, 3, 10, 20, 40, 80):
            cases.append(dict(name=f"gb_{g}_{b}", fs=2000.0, n=131072, gamma=g,
                              beta=b, freq_limits=None, vpo=8))
    for c in cases:
        cwt = CWT(wavelet=Morse(gamma=c["gamma"], beta=c["beta"]))
        cwt.fs = c["fs"]
        ref = cwt._norm_radians_to_hz(cwt.wavelet.compute_freq_bounds(c["n"]))
        if c["freq_limits"] is not None:
            lim = np.sort(c["freq_limits"])
            f_low, f_high = cwt._check_freq_bounds([lim[0], lim[1]], ref)
        else:
            f_low, f_high = ref[0], ref[1]
        J = np.floor(np.log2(f_high / f_low) * c["vpo"])
        f = f_high / 2 ** (np.arange(J + 1) / c["vpo"])
        cwt._wavelet.fs = c["fs"]
        L = cwt.wavelet.compute_lengths(cwt._hz_to_norm_radians(f))
        grids.append(dict(c, ref_bounds=[float(ref[0]), float(ref[1])],
                          frequencies=[float(v) for v in f],
                          lengths=[int(v) for v in L]))
    json.dump(grids, open(os.path.join(GOLD, "plan_grids.json"), "w"))

    # ---- kernels -------------------------------------------------------------
    kern = {}
    meta = []
    for i, (g, b, om, L) in enumerate([
            (3, 20, 2.4629407752267776, 36), (3, 20, 2.2, 40), (3, 20, 1.9, 47),
            (3, 20, 0.5, 176), (3, 20, 0.05, 1753), (3, 20, 0.0123, 7124),
            (2, 5, 0.7, 200), (9, 3, 1.1, 77), (1, 1, 0.4, 64), (6, 40, 0.3, 517),
            (3, 80, 1.0, 141)]):
        m = Morse(gamma=g, beta=b)
        m.norm_radian_freq = om
        psi, psif = m(L)
        kern[f"psi_{i}"] = psi
        kern[f"psif_{i}"] = psif
        meta.append([g, b, om, L])
    kern["meta"] = np.array(meta, dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, "kernels.npz"), **kern)

    # ---- convolution ('same' offset semantics) -------------------------------
    rng = np.random.default_rng(7)
    conv = {}
    for i, (n, m) in enumerate([(1000, 37), (1000, 36), (300, 301), (5000, 1200),
                                (70000, 513), (64, 1)]):
        s = rng.standard_normal(n)
        k = rng.standard_normal(m) + 1j * rng.standard_normal(m)
        cols = sample_columns(n, 6000, 512)
        conv[f"s_{i}"] = s
        conv[f"k_{i}"] = k
        conv[f"y_{i}"] = sigtools.fastconv_scipy(s, k)[cols]
        conv[f"cols_{i}"] = cols
    np.savez_compressed(os.path.join(GOLD, "conv.npz"), **conv)

    # ---- small full transforms -----------------------------------------------
    cw = {}
    # (a) default everything, one epoch
    fs, n = 500.0, 2048
    x = synth.chirp_pink(n, fs, 0, np.float64)
    c = CWT(wavelet=Morse())
    c.transform(x, fs=fs, timestamps=np.arange(n) / fs)
    cw["a_x"], cw["a_amp"], cw["a_f"], cw["a_fs"] = x, c.amplitude, c.frequencies, fs
    # (b) two epochs (gap in timestamps), limits, vpo=6, gamma/beta non-default
    fs, n = 1000.0, 3000
    x = synth.chirp_pink(n, fs, 1, np.float64) + 3.0          # non-zero mean
    ts = np.arange(n) / fs
    ts[1700:] += 0.5
    c = CWT(wavelet=Morse(gamma=6, beta=10))
    c.transform(x, fs=fs, timestamps=ts, freq_limits=[20, 300], voices_per_octave=6)
    cw["b_x"], cw["b_amp"], cw["b_f"], cw["b_ts"], cw["b_fs"] = x, c.amplitude, c.frequencies, ts, fs
    # (c) float32 input, (1, N) shape, parallel=True
    fs, n = 250.0, 1500
    x = synth.chirp_pink(n, fs, 2, np.float32)
    c = CWT(wavelet=Morse(gamma=3, beta=20))
    c.transform(x[None, :], fs=fs, timestamps=np.arange(n) / fs, parallel=True)
    cw["c_x"], cw["c_amp"], cw["c_f"], cw["c_fs"] = x, c.amplitude, c.frequencies, fs
    # (d) complex coefficients through the reference's inner loop
    fs, n = 1000.0, 4096
    x = synth.chirp_pink(n, fs, 3, np.float64)
    fsel = np.array([391.9891989199264, 341.2, 250.0, 97.3, 31.0, 9.7])
    W, lens = ref_complex(CWT, Morse, sigtools, x, fs, 3, 20, fsel)
    cw["d_x"], cw["d_W"], cw["d_f"], cw["d_L"], cw["d_fs"] = x, W, fsel, lens, fs
    # the outputs keep every scale and a sample of their columns, listed in <case>_cols
    for key, k in (("a_amp", 800), ("b_amp", 1200), ("c_amp", 600), ("d_W", 1600)):
        cols = sample_columns(cw[key].shape[1], k, 128)
        cw[key], cw[key[0] + "_cols"] = cw[key][:, cols], cols
    np.savez_compressed(os.path.join(GOLD, "cwt_small.npz"), **cw)

    # ---- sparse samples of a cfg1-sized transform -----------------------------
    fs, n = 1000.0, 60000
    x = synth.chirp_pink(n, fs, 0, np.float32)
    c = CWT(wavelet=Morse())
    c.transform(x, fs=fs, timestamps=np.arange(n) / fs)
    cols = np.unique(np.concatenate([np.arange(0, 64), np.arange(n - 64, n),
                                     np.arange(0, n, 997)]))
    np.savez_compressed(os.path.join(GOLD, "cfg1_samples.npz"),
                        cols=cols, amp=c.amplitude[:, cols], f=c.frequencies,
                        row_l2=np.sqrt((c.amplitude ** 2).sum(axis=1)),
                        row_sum=c.amplitude.sum(axis=1))
    print("golden vectors written to", GOLD)


if __name__ == "__main__":
    main()
