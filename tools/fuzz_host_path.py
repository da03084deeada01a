"""GPU box: randomized check of the streamed host path (gcwt_execute_host and its pooled, band-power and event-locked
variants): random channel counts, lengths, epochs, forced tile lengths, pinned / pageable / strided destinations,
random bands and random events, against the device path executed epoch by epoch (pooled in numpy, band-reduced with
plan.band_reduce) and, for the events, plan.event_reduce of the full-rate host result (the same tiles).
       python tools/fuzz_host_path.py [n_cases] [seed]"""
import os
import sys
import numpy as np
import torch
sys.path.insert(0, ".")
from ghost_b200 import Morse
from ghost_b200.engine import CwtPlan, scale_tables
from oracle import cwt_oracle as orc

n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
fails = []
for case in range(n_cases):
    fs = float(rng.choice([200.0, 1000.0, 1250.0]))
    n = int(rng.integers(3000, 120000))
    nch = int(rng.integers(1, 6))
    dtype = np.float32 if rng.random() < 0.7 else np.float64
    output = str(rng.choice(["amplitude", "power", "complex"]))
    n_ep = int(rng.integers(1, 4))
    cuts = np.sort(rng.choice(np.arange(1500, n - 1500), size=2 * (n_ep - 1), replace=False)) if n_ep > 1 else np.array([], int)
    bounds = [0] + cuts.tolist() + [n]
    epochs = np.array([[bounds[2 * i], bounds[2 * i + 1]] for i in range(n_ep)])
    if rng.random() < 0.3:
        epochs[0, 0] = int(rng.integers(0, 500))
    n_min = int(np.min(epochs[:, 1] - epochs[:, 0]))
    f = orc.frequency_grid(fs, n_min, voices_per_octave=8)
    if len(f) == 0:
        continue
    m = Morse(fs=fs)
    om = f / (fs / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    plan = CwtPlan(L, k0, nt, terms, dtype=dtype, output=output)
    X = (rng.standard_normal((nch, n)).cumsum(axis=1) * 0.02 + rng.standard_normal((nch, n)) + 1.0).astype(np.float32)
    tile = int(rng.choice([0, 0, 5000, 12345, 40000]))
    if tile:
        os.environ["GCWT_HOST_TILE"] = str(tile)
    else:
        os.environ.pop("GCWT_HOST_TILE", None)
    S = len(f)
    odt = (np.complex64 if dtype == np.float32 else np.complex128) if output == "complex" else dtype
    dest = str(rng.choice(["none", "pageable", "pinned", "strided"]))
    out = None
    if dest == "pageable":
        out = np.full((nch, S, n), -7, dtype=odt)
    elif dest == "pinned":
        out = torch.empty((nch, S, n), dtype=torch.from_numpy(np.zeros(1, odt)).dtype).pin_memory().numpy()
    elif dest == "strided":
        out = np.full((nch, S + 1, n + 13), -7, dtype=odt)[:, :S, :n]
    got = plan.execute_host(X if dtype == np.float32 else X.astype(np.float64), out=out, epochs=epochs)
    tiles = plan.host_stats()["tiles"]
    # device path, epoch by epoch, global mean
    xd = torch.from_numpy(X if dtype == np.float32 else X.astype(np.float64)).cuda()
    means = plan.channel_means(xd)
    want_d = plan.alloc_out(nch, n)
    want_d.zero_()
    for a, b in epochs:
        plan.execute(xd, want_d, means=means, start=int(a), stop=int(b))
    want = want_d.cpu().numpy()
    num = np.linalg.norm((got - want).reshape(nch, S, -1), axis=2)
    den = np.linalg.norm(want.reshape(nch, S, -1), axis=2)
    err = float((num / den).max())
    bar = (6e-6 if output != "power" else 1.2e-5) if dtype == np.float32 else 1e-11
    gaps_ok = True
    pos = 0
    for a, b in epochs:
        gaps_ok = gaps_ok and bool(np.all(got[:, :, pos:a] == 0))
        pos = b
    ok = err <= bar and gaps_ok
    # pooled variant (one epoch only)
    perr = 0.0
    if output != "complex" and n_ep == 1 and epochs[0, 0] == 0:
        w = int(rng.choice([3, 64, 1000]))
        mode = str(rng.choice(["mean", "max"]))
        pooled = plan.execute_host_pooled(X if dtype == np.float32 else X.astype(np.float64), w, mode)
        nb = -(-n // w)
        pad = nb * w - n
        ap = np.concatenate([want.astype(np.float64), np.full((nch, S, pad), np.nan if mode == "mean" else -np.inf)], axis=2).reshape(nch, S, nb, w)
        ref = np.nanmean(ap, axis=3) if mode == "mean" else ap.max(axis=3)
        # per row, relative to the row's largest bin (tiles round differently at the 1e-7 level of the row's scale)
        perr = float(np.max(np.max(np.abs(pooled - ref), axis=2) / (np.max(np.abs(ref), axis=2) + 1e-300)))
        ok = ok and perr <= (1e-5 if dtype == np.float32 else 1e-11)
    # band power: random (possibly overlapping) bands, same epochs and tiles; the gap columns of want_d are zero
    n_b = int(rng.integers(1, 7))
    first = rng.integers(0, S, n_b).astype(np.int32)
    count = np.array([rng.integers(1, S - f + 1) for f in first], dtype=np.int32)
    weights = rng.uniform(0.1, 2.0, int(count.sum()))
    got_b = plan.execute_host_bands(X if dtype == np.float32 else X.astype(np.float64), first, count, weights, epochs=epochs)
    want_b = plan.band_reduce(want_d, first, count, weights).cpu().numpy()
    berr = float(np.max(np.linalg.norm(got_b - want_b, axis=2) / np.linalg.norm(want_b, axis=2)))
    pos = 0
    for a, b in epochs:
        gaps_ok = gaps_ok and bool(np.all(got_b[:, :, pos:a] == 0))
        pos = b
    gaps_ok = gaps_ok and bool(np.all(got_b[:, :, pos:] == 0))
    ok = ok and gaps_ok and berr <= (1.2e-5 if dtype == np.float32 else 1e-11)
    # event-locked means: ascending events with duplicates, windows of n_lags lags from lag_first (often negative)
    # inside every epoch, some across the forced tile boundaries.  The reference sums the same windows of `got`
    # (the same tiles, so the same coefficients): only the grouping of the fp64 sums differs.
    n_lags = int(rng.integers(1, min(400, n_min) + 1))
    lag_first = int(rng.integers(-n_lags - 50, 50))
    ev = []
    for a, b in epochs:                                              # window starts w0 in [a, b - n_lags]
        ev += (rng.integers(a, b - n_lags + 1, int(rng.integers(1, 6))) - lag_first).tolist()
        bounds_t = np.arange(a + max(tile, 1024), b, max(tile, 1024)) if tile else []
        for t in bounds_t[:3]:                                       # windows that straddle a tile boundary
            lo, hi = max(a, t - n_lags + 1), min(b - n_lags, t - 1)
            if n_lags > 1 and lo <= hi:
                ev.append(int(rng.integers(lo, hi + 1)) - lag_first)
    ev = np.sort(np.array(ev + list(rng.choice(ev, int(rng.integers(1, 4)))), dtype=np.int64))
    Xin = X if dtype == np.float32 else X.astype(np.float64)
    got_p, got_ph = plan.execute_host_events(Xin, ev, lag_first, n_lags, epochs=epochs)
    ref_p, ref_ph = plan.event_reduce(torch.from_numpy(np.ascontiguousarray(got)).cuda(), ev, lag_first, n_lags)
    ref_p = ref_p.cpu().numpy() / ev.size
    eerr = float(np.max(np.abs(got_p - ref_p) / np.maximum(np.abs(ref_p), 1e-300)))
    pherr = 0.0
    if output == "complex":
        pherr = float(np.max(np.abs(got_ph - ref_ph.cpu().numpy() / ev.size)))
    else:
        ok = ok and got_ph is None and ref_ph is None
    ok = ok and eerr <= 1e-12 and pherr <= 1e-12
    print("case %2d %s %s %s ch=%d n=%d epochs=%d S=%d tile=%d tiles=%d dest=%s err=%.2e pooled=%.1e bands=%d %.1e "
          "events=%d lags=%d%+d %.1e %.1e" % (
              case, "ok " if ok else "BAD", np.dtype(dtype).name, output, nch, n, n_ep, S, tile, tiles, dest, err, perr,
              n_b, berr, ev.size, n_lags, lag_first, eerr, pherr), flush=True)
    if not ok:
        fails.append(case)
    plan.close()
print("failures", fails)
sys.exit(1 if fails else 0)
