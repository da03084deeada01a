"""Pin the CPU oracle (oracle/cwt_oracle.py) to outputs of the real reference.

The fixtures under tests/golden/ were produced by oracle/gen_golden.py, which
imports /root/reference and runs it; nothing here needs the reference or a GPU.
"""
import json
import os

import numpy as np
import pytest

from oracle import cwt_oracle as orc


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_scalars_bit_exact(golden_dir):
    scal = json.load(open(os.path.join(golden_dir, "morse_scalars.json")))
    assert len(scal) == 30
    for key, val in scal.items():
        g, b = (int(v) for v in key.split(","))
        assert float(orc.morse_peak_freq(g, b)) == val["morsefreq"]
        assert float(orc.morse_high_freq(g, b)) == val["morsehigh"]
    # SURVEY.md section 8(c) known answers
    assert float(orc.morse_peak_freq(3, 20)) == 1.8820720577620569
    assert float(orc.morse_high_freq(3, 20)) == 2.4629407752267776


def test_frequency_grid_and_lengths_bit_exact(golden_dir):
    grids = json.load(open(os.path.join(golden_dir, "plan_grids.json")))
    assert len(grids) >= 37
    for g in grids:
        f = orc.frequency_grid(g["fs"], g["n"], g["gamma"], g["beta"],
                               g["freq_limits"], g["vpo"])
        assert f.tolist() == g["frequencies"], g["name"]
        L = orc.kernel_lengths(g["gamma"], g["beta"], orc.hz_to_rad(f, g["fs"]))
        assert L.tolist() == g["lengths"], g["name"]
    by_name = {g["name"]: g for g in grids}
    assert len(by_name["cfg1"]["frequencies"]) == 84
    assert len(by_name["cfg2"]["frequencies"]) == 96
    assert len(by_name["cfg3"]["frequencies"]) == 128
    assert by_name["cfg3"]["lengths"][0] == 36
    assert by_name["cfg3"]["lengths"][-1] == 236760
    assert sum(by_name["cfg1"]["lengths"]) == 167001


def test_kernels(golden_dir):
    z = _load(golden_dir, "kernels.npz")
    meta = z["meta"]
    for i, (g, b, om, L) in enumerate(meta):
        psi, spec = orc.morse_kernel(g, b, om, int(L))
        ref = z[f"psi_{i}"]
        assert psi.shape == ref.shape
        assert np.max(np.abs(psi - ref)) <= 1e-14 * np.max(np.abs(ref)), (g, b, om, L)
        assert np.max(np.abs(spec - z[f"psif_{i}"])) <= 1e-14 * np.max(spec)


def test_overlap_add_same_offset(golden_dir):
    z = _load(golden_dir, "conv.npz")
    i = 0
    while f"s_{i}" in z:
        s, k, y = z[f"s_{i}"], z[f"k_{i}"], z[f"y_{i}"]
        cols = z[f"cols_{i}"]                  # the columns stored of the reference's output
        got = orc.overlap_add_same(s, k)
        assert got.shape == s.shape
        assert np.max(np.abs(got[cols] - y)) <= 1e-13 * np.max(np.abs(y))
        if len(s) <= 5000:          # definition by direct summation
            d = orc.direct_same(s, k) if len(k) <= len(s) else None
            if d is not None:
                assert np.max(np.abs(d[cols] - y)) <= 1e-12 * np.max(np.abs(y))
        i += 1
    assert i == 6


def test_transform_default(golden_dir):
    z = _load(golden_dir, "cwt_small.npz")
    amp, f, _ = orc.cwt_amplitude(z["a_x"], float(z["a_fs"]))
    assert f.tolist() == z["a_f"].tolist()
    assert amp.shape == (len(z["a_f"]), len(z["a_x"]))
    assert np.max(np.abs(amp[:, z["a_cols"]] - z["a_amp"])) <= 1e-13 * np.max(z["a_amp"])


def test_transform_two_epochs_nonzero_mean(golden_dir):
    z = _load(golden_dir, "cwt_small.npz")
    amp, f, _ = orc.cwt_amplitude(z["b_x"], float(z["b_fs"]), gamma=6, beta=10,
                                  freq_limits=[20, 300], voices_per_octave=6,
                                  timestamps=z["b_ts"])
    assert f.tolist() == z["b_f"].tolist()
    assert amp.shape == (len(z["b_f"]), len(z["b_x"]))
    assert np.max(np.abs(amp[:, z["b_cols"]] - z["b_amp"])) <= 1e-13 * np.max(z["b_amp"])
    ep = orc.contiguous_segments(z["b_ts"], 1 / float(z["b_fs"]))
    assert ep.tolist() == [[0, 1700], [1700, 3000]]


def test_transform_float32_input_parallel(golden_dir):
    z = _load(golden_dir, "cwt_small.npz")
    amp, f, _ = orc.cwt_amplitude(z["c_x"], float(z["c_fs"]), parallel=True)
    assert z["c_x"].dtype == np.float32 and amp.dtype == np.float64
    assert f.tolist() == z["c_f"].tolist()
    assert amp.shape == (len(z["c_f"]), len(z["c_x"]))
    assert np.max(np.abs(amp[:, z["c_cols"]] - z["c_amp"])) <= 1e-13 * np.max(z["c_amp"])


def test_complex_coefficients(golden_dir):
    z = _load(golden_dir, "cwt_small.npz")
    W, f, L = orc.cwt_complex(z["d_x"], float(z["d_fs"]), frequencies=z["d_f"])
    assert L.tolist() == z["d_L"].tolist()
    assert W.shape == (len(z["d_f"]), len(z["d_x"]))
    for s in range(len(f)):
        err = np.max(np.abs(W[s, z["d_cols"]] - z["d_W"][s])) / np.max(np.abs(z["d_W"][s]))
        assert err <= 1e-13, (s, err)


def test_cfg1_samples(golden_dir):
    from ghost_b200 import synth
    z = _load(golden_dir, "cfg1_samples.npz")
    x = synth.chirp_pink(60000, 1000.0, 0, np.float32)
    amp, f, _ = orc.cwt_amplitude(x, 1000.0, parallel=True)
    assert f.tolist() == z["f"].tolist()
    assert amp.shape == (84, 60000)
    ref = z["amp"]
    got = amp[:, z["cols"]]
    assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(ref)
    assert np.allclose(np.sqrt((amp ** 2).sum(axis=1)), z["row_l2"], rtol=1e-12)
    assert np.allclose(amp.sum(axis=1), z["row_sum"], rtol=1e-12)
