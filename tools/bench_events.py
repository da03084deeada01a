"""GPU box: event-locked power and phase against the full result on config 2 (32 channels x 1.25 kHz x 30 min x
96 scales, fp32), 1800 events 1249 samples (0.9992 s) apart, window (-0.5, +1.0) s = 1876 lags.  Prints one JSON line.

  a       transform(X, multichannel=True, out=pinned): every coefficient crosses the link; then the numpy event
          average of that array (float64 sums of |W|^2 over the 1800 windows), timed on its own
  b       transform(X, multichannel=True, events=..., event_window=...): only (channels x scales x lags) means
          cross the link; for an amplitude plan (power) and a complex plan (power and phase)
  kernel  event_reduce_kernel alone (plan.event_reduce) on a device-resident 8-channel amplitude result, CUDA events
          over repeated launches; bytes = what the kernel must move (the samples the windows cover, read once, and the
          fp64 accumulator read and written) over its time, against the measured 6534.5 GB/s HBM peak (DESIGN.md
          section 7); the bytes its loads issue (every window in full) beside it

The events start at 0.5 s and are a whole number of samples apart, so every window lies inside the recording and
consecutive windows overlap by about half a second.  a and b are best of `reps` after a warm-up; the numpy average
runs once.  The GPU's name and power limit are read in the same run.
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
from ghost_b200.engine import event_windows                             # noqa: E402

PEAK_GBS = 6534.5
WINDOW = (-0.5, 1.0)


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


def covered_samples(samples, lag_first, n_lags):
    """Samples of a row that at least one window covers."""
    total, end = 0, -1
    for s in np.sort(samples):
        w0, w1 = s + lag_first, s + lag_first + n_lags
        total += w1 - max(w0, end) if w1 > end else 0
        end = max(end, w1)
    return int(total)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--channels", type=int, default=32)
    ap.add_argument("--events", type=int, default=1800)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-channels", type=int, default=8)
    ap.add_argument("--kernel-launches", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_events needs a CUDA device")
    name, power_limit = gpu_info()
    wl = bench.WORKLOADS["cfg2"]
    fs, n, C = wl["fs"], wl["n"], args.channels
    X = synth.recording(C, n, fs, np.float32)
    ev_s = 0.5 + 1249 / fs * np.arange(args.events)
    kw = dict(fs=fs, freq_limits=wl["freq_limits"], voices_per_octave=wl["vpo"], multichannel=True)
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=wl["output"])
    cwt.transform(X[:1], **kw)
    S = cwt.frequencies.size
    samples, kept, lag_first, n_lags = event_windows(cwt.time, ev_s, WINDOW, [[0, n]], fs)
    assert kept.all(), "every window lies inside the recording"
    E = samples.size
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

    def run_a():
        for c0 in range(0, C, group):
            cwt.transform(X[c0:c0 + group], out=out[:min(group, C - c0)], **kw)

    ta, tsa = best_of(run_a, args.reps)
    st_a = cwt.last_plan.host_stats()
    # the numpy event average of (a): float64 sums of |W|^2 over the windows, group by group, timed once
    want = np.zeros((C, S, n_lags))
    tmp = np.empty((group, S, n_lags))
    t_numpy = 0.0
    for c0 in range(0, C, group):
        g = min(group, C - c0)
        cwt.transform(X[c0:c0 + g], out=out[:g], **kw)
        t1 = time.perf_counter()
        for s in samples:
            np.square(out[:g, :, s + lag_first:s + lag_first + n_lags], out=tmp[:g], dtype=np.float64)
            want[c0:c0 + g] += tmp[:g]
        t_numpy += time.perf_counter() - t1
    want /= E
    del out, pinned

    # (b) the event means only, amplitude and complex plans
    tb, tsb = best_of(lambda: cwt.transform(X, events=ev_s, event_window=WINDOW, **kw), args.reps)
    st_b = cwt.last_plan.host_stats()
    max_rel = float(np.max(np.abs(cwt.event_power - want)) / np.max(want))
    cx = ContinuousWaveletTransform(dtype=np.float32, output="complex")
    tbc, tsbc = best_of(lambda: cx.transform(X, events=ev_s, event_window=WINDOW, **kw), args.reps)
    st_bc = cx.last_plan.host_stats()
    max_rel_cx = float(np.max(np.abs(cx.event_power - want)) / np.max(want))

    # (c) the kernel alone on a device-resident result of kernel-channels channels
    plan = cwt.last_plan
    K = min(args.kernel_channels, C)
    resk = plan.execute(torch.from_numpy(X[:K]).cuda())
    ev_dev = torch.from_numpy(samples).cuda()
    acc, _ = plan.event_reduce(resk, ev_dev, lag_first, n_lags)
    torch.cuda.synchronize()
    t_kernel = event_ms(lambda: plan.event_reduce(resk, ev_dev, lag_first, n_lags, power=acc), args.kernel_launches)
    covered = covered_samples(samples, lag_first, n_lags)
    bytes_kernel = float(K) * S * (covered * 4 + n_lags * 16)
    bytes_issued = float(K) * S * (E * n_lags * 4 + n_lags * 16)

    print(json.dumps({
        "tool": "bench_events", "gpu": name, "power_limit": power_limit,
        "workload": "config 2: %d ch x %.0f Hz x %d samples x %d scales, fp32 %s" % (C, fs, n, S, wl["output"]),
        "events": E, "window_s": list(WINDOW), "lag_first": lag_first, "n_lags": n_lags,
        "a_full_pinned": {"best_s": ta, "runs_s": tsa, "coeff_per_s": coeffs / ta, "d2h_bytes": C * S * n * 4,
                          "channels_per_call": group, "tiles_last_call": st_a["tiles"]},
        "a_numpy_event_average_s": t_numpy,
        "a_total_s": ta + t_numpy,
        "b_events_amplitude": {"best_s": tb, "runs_s": tsb, "coeff_equiv_per_s": coeffs / tb,
                               "d2h_bytes": st_b["bytes_out"], "tiles": st_b["tiles"],
                               "max_rel_diff_vs_numpy_of_a": max_rel},
        "b_events_complex": {"best_s": tbc, "runs_s": tsbc, "coeff_equiv_per_s": coeffs / tbc,
                             "d2h_bytes": st_bc["bytes_out"], "tiles": st_bc["tiles"],
                             "power_max_rel_diff_vs_numpy_of_a": max_rel_cx},
        "speedup_b_amplitude_over_a_total": (ta + t_numpy) / tb,
        "speedup_b_amplitude_over_a_transfer_only": ta / tb,
        "kernel": {"channels": K, "ms": t_kernel, "bytes": bytes_kernel, "gbs": bytes_kernel / t_kernel / 1e6,
                   "frac_of_measured_peak": bytes_kernel / t_kernel / 1e6 / PEAK_GBS,
                   "bytes_issued": bytes_issued, "issued_gbs": bytes_issued / t_kernel / 1e6},
    }), flush=True)


if __name__ == "__main__":
    main()
