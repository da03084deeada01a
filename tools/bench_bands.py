"""GPU box: scale-averaged band power against the full result on config 2 (32 channels x 1.25 kHz x 30 min x
96 scales, fp32 amplitude, 4 bands).  Prints one JSON line.

  a       transform(X, multichannel=True, out=pinned): every coefficient crosses the link
  b       transform(X, multichannel=True, bands=BANDS): only (channels x bands x samples) crosses it
  kernel  band_reduce_kernel alone (plan.band_reduce) on a device-resident 8-channel result, CUDA events over
          repeated launches; bytes = what the kernel must move (the rows inside the bands read once, the
          band rows written) over its time, against the measured 6534.5 GB/s HBM peak (DESIGN.md section 7)
  stages  where b's time goes: CUDA events around each stage of one tile of b's pipeline run on its own
          (compute = gcwt_execute with the accuracy guard, reduction, D2H of the band rows to pinned memory)

a and b are best of 3 after a warm-up, reported as coefficient-equivalents/s (channels x scales x samples over
the call's wall time).  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                            # noqa: E402
from ghost_b200 import ContinuousWaveletTransform, synth               # noqa: E402
from ghost_b200.engine import band_tables                               # noqa: E402

PEAK_GBS = 6534.5
BANDS = [(1.0, 4.0), (6.0, 12.0), (30.0, 80.0), (150.0, 250.0)]        # delta, theta, gamma, ripple


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, limit = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return name, limit


def best_of(fn, reps):
    fn()                                                                # warm-up
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return min(ts), ts


def event_ms(fn, reps):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--channels", type=int, default=32)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-channels", type=int, default=8)
    ap.add_argument("--kernel-launches", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_bands needs a CUDA device")
    name, power_limit = gpu_info()
    wl = bench.WORKLOADS["cfg2"]
    fs, n, C = wl["fs"], wl["n"], args.channels
    X = synth.recording(C, n, fs, np.float32)
    kw = dict(fs=fs, freq_limits=wl["freq_limits"], voices_per_octave=wl["vpo"], multichannel=True)
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=wl["output"])
    cwt.transform(X[:1], **kw)
    S = cwt.frequencies.size
    first, count, weights = band_tables(cwt.frequencies, BANDS)
    B = len(BANDS)
    coeffs = float(C) * S * n

    # (a) the full result into a pinned array; channels per call as bench.py's e2e (a quarter of free host memory)
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    group = int(max(1, min(C, avail // 4 // (S * n * 4))))
    pinned = torch.empty((group, S, n), dtype=torch.float32).pin_memory()
    out = pinned.numpy()
    cols = np.unique(np.concatenate([np.arange(64), n - 64 + np.arange(64),
                                     np.random.default_rng(0).integers(0, n, 4096)]))
    want = np.empty((C, B, cols.size))

    def run_a(check=False):
        for c0 in range(0, C, group):
            g = min(group, C - c0)
            cwt.transform(X[c0:c0 + g], out=out[:g], **kw)
            off = 0
            for b, (f0, k) in enumerate(zip(first, count)):             # numpy band power at sampled columns
                if check:
                    rows = out[:g, f0:f0 + k][:, :, cols].astype(np.float64)
                    want[c0:c0 + g, b] = np.tensordot(weights[off:off + k], rows ** 2, axes=(0, 1))
                off += k

    run_a(check=True)
    ta, tsa = best_of(run_a, args.reps)
    st_a = cwt.last_plan.host_stats()
    del out, pinned

    # (b) band power only
    tb, tsb = best_of(lambda: cwt.transform(X, bands=BANDS, **kw), args.reps)
    st_b = cwt.last_plan.host_stats()
    bp = cwt.band_power
    max_rel = float(np.max(np.abs(bp[:, :, cols] - want) / np.abs(want).max(axis=2, keepdims=True)))

    # stages of one tile of (b): the host path's tile is a group of channels x all scales x all samples
    plan = cwt.last_plan
    g = int(max(1, min(C, (1 << 30) // (S * n * 4))))
    x_dev = torch.from_numpy(X[:g]).cuda()
    means = plan.channel_means(x_dev)
    res = plan.alloc_out(g, n)
    t_compute = event_ms(lambda: plan.execute(x_dev, res, means=means), 5)
    red = plan.band_reduce(res, first, count, weights)
    t_reduce = event_ms(lambda: plan.band_reduce(res, first, count, weights), 10)
    host_bands = torch.empty(red.shape, dtype=red.dtype).pin_memory()
    t_copy = event_ms(lambda: host_bands.copy_(red, non_blocking=True), 10)
    n_tiles = st_b["tiles"]
    del res, red, x_dev

    # (c) the kernel alone on a device-resident result of kernel-channels channels
    K = min(args.kernel_channels, C)
    xk = torch.from_numpy(X[:K]).cuda()
    resk = plan.execute(xk)
    torch.cuda.synchronize()
    t_kernel = event_ms(lambda: plan.band_reduce(resk, first, count, weights), args.kernel_launches)
    rows_read = int(count.sum())
    bytes_kernel = float(K) * n * 4 * (rows_read + B)

    print(json.dumps({
        "tool": "bench_bands", "gpu": name, "power_limit": power_limit,
        "workload": "config 2: %d ch x %.0f Hz x %d samples x %d scales, fp32 %s" % (C, fs, n, S, wl["output"]),
        "bands_hz": BANDS, "scales_per_band": count.tolist(),
        "a_full_pinned": {"best_s": ta, "runs_s": tsa, "coeff_per_s": coeffs / ta, "d2h_bytes": C * S * n * 4,
                          "channels_per_call": group, "tiles_last_call": st_a["tiles"]},
        "b_bands": {"best_s": tb, "runs_s": tsb, "coeff_equiv_per_s": coeffs / tb, "d2h_bytes": st_b["bytes_out"],
                    "tiles": n_tiles, "pinned_destination": st_b["pinned_destination"],
                    "max_rel_diff_vs_numpy_of_a": max_rel},
        "speedup_b_over_a": ta / tb,
        "stages_per_tile_ms": {"channels_per_tile": g, "compute": t_compute, "reduce": t_reduce, "d2h_bands": t_copy,
                               "tiles": n_tiles, "serial_sum_s": (t_compute + t_reduce + t_copy) * n_tiles / 1e3},
        "kernel": {"channels": K, "ms": t_kernel, "bytes": bytes_kernel, "gbs": bytes_kernel / t_kernel / 1e6,
                   "frac_of_measured_peak": bytes_kernel / t_kernel / 1e6 / PEAK_GBS,
                   "bytes_if_all_scales_read": float(K) * n * 4 * (S + B)},
    }), flush=True)


if __name__ == "__main__":
    main()
