#!/usr/bin/env python
"""Benchmark of the Morse-wavelet CWT hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo, N ranks via torchrun
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU transform, host cores

A step is one pass of the transform over one batch of synthetic chirp + pink-noise channels.
Workload at N = 1 is config 2 of BASELINE.json (64 channels x 1.25 kHz x 30 min, 96 scales, fp32
amplitude); at N > 1 the headline keeps 64 channels per GPU (weak scaling, channel shards, no data-path
collective) and an `extra` object adds the shapes BASELINE.json names for several GPUs: the same 64
channels split over the ranks (strong scaling), the full config 3 (256 channels, N = 8) and config 4
(one 24 h recording time-sharded over the ranks with NCCL halos, with a seam check).

One JSON line is printed by rank 0 (see the driver contract in the task statement):
  value     device-resident coefficients / s (inputs in HBM, CUDA events, max over ranks)
  e2e       the same through the public API ContinuousWaveletTransform.transform(..., out=pinned) with
            host arrays in and out: H2D of the samples and D2H of every coefficient inside the timed region
  roofline  algorithmic bytes of the dominant kernel family / its event-timed duration vs the measured HBM peak
  cpu_baseline / --impl reference   the UNMODIFIED reference (baseline/_ref, tools/install_reference.sh)
            timed on this host's cores on a bounded sample; the oracle port only if it cannot be imported

--dump-outputs DIR writes what the last timed step left in its result buffer, so that two builds can be
compared output for output on the same (seeded) inputs: DIR/<output>.npy (channels, scales, K) at K sample
columns -- the first and last 64 (K // 2 each when fewer than 128 columns fit) and a seeded random draw of
the others, as many as keep the dump under 64 MB -- (complex results as (..., 2) real / imaginary pairs),
DIR/columns.npy (the K sample indices of this rank's samples) and DIR/frequencies.npy (Hz).  Tiled workloads dump the last tile a step produced.
With several ranks every rank writes its own files, suffixed _rank<r>.
"""
from __future__ import annotations

import argparse
import json
import logging
import os
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cwt_output_coeffs_per_sec"
UNIT = "coeff/s"

WORKLOADS = {
    # name: fs, samples, channels per GPU, freq_limits, voices/octave, output
    "cfg2": dict(fs=1250.0, n=2250000, channels=64, freq_limits=[0.40, 300.0], vpo=10, output="amplitude",
                 desc="64ch x 1.25kHz x 30min, 96 scales, fp32 amplitude"),
    "cfg1": dict(fs=1000.0, n=60000, channels=1, freq_limits=None, vpo=10, output="amplitude",
                 desc="1ch x 1kHz x 60s, 84 scales, fp32 amplitude"),
    # config 3 of BASELINE.json is 256 channels over 8 GPUs = 32 channels per GPU; its result (295 GB
    # per GPU) exceeds HBM, so it is produced in time tiles into a reused buffer (tile = samples per tile)
    # (tile sweep on one shard: 2.25 M samples 91.3 ms, 4.5 M 88.8 ms, 6 M 89.0 ms; 4.5 M = a 74 GB tile buffer)
    "cfg3": dict(fs=30000.0, n=18000000, channels=32, freq_limits=[1.7, 15000.0], vpo=10, output="power",
                 tile=4500000, desc="32ch/GPU x 30kHz x 10min, 128 scales, fp32 power, streamed in 4 time tiles"),
    # config 4 of BASELINE.json: one 24 h recording at 30 kHz (2.592e9 samples) time-sharded over 8 GPUs
    # = 3.24e8 samples per GPU; every step does the mean all-reduce, the NCCL halo exchange with both
    # neighbours and the tiled transform of the shard
    "cfg4": dict(fs=30000.0, n=324000000, channels=1, freq_limits=[1.7, 15000.0], vpo=10, output="power",
                 tile=108000000, time_shard=True, plan_n=2592000000,      # (36 M: 52.2 ms per shard, 81 M: 50.4, 108 M: 49.8)
                 desc="1ch x 30kHz, 3.24e8 samples per GPU (24 h over 8 GPUs), 128 scales, fp32 power, "
                      "time-sharded with NCCL halos, streamed in time tiles"),
    # config 5 of BASELINE.json is the fp64 complex parity sweep; this is its largest single shape as a
    # throughput line for the (default) float64 path of the drop-in class
    "cfg5": dict(fs=1000.0, n=262144, channels=8, freq_limits=None, vpo=10, output="complex", dtype="f64",
                 desc="8ch x 1kHz x 262144 samples, default grid, fp64 complex coefficients"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default=None, choices=["f32", "f64"], help="f64: the float64 path (workload cfg5)")
    ap.add_argument("--samples", type=int, default=None, help="override samples per channel")
    ap.add_argument("--channels", type=int, default=None, help="channels per GPU (default: workload's)")
    ap.add_argument("--tile", type=int, default=None, help="samples per time tile (tiled workloads)")
    ap.add_argument("--no-guard", action="store_true", help="plan without the execute-time accuracy guard")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="N > 1: skip the strong-scaling / config 3 / config 4 entries")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.dtype == "f64" and args.workload == "cfg2":
        args.workload = "cfg5"
    return args


def plan_frequencies(wl):
    from ghost_b200 import ContinuousWaveletTransform
    cwt = ContinuousWaveletTransform(dtype=np.float32)
    cwt.fs = wl["fs"]
    cwt.wavelet.fs = wl["fs"]
    logging.disable(logging.WARNING)                      # the clipping of freq_limits is expected
    try:
        return np.asarray(cwt.plan_frequencies(wl.get("plan_n", wl["n"]), freq_limits=wl["freq_limits"],
                                               voices_per_octave=wl["vpo"]))
    finally:
        logging.disable(logging.NOTSET)


def build_plan(wl, device, guard=True, dtype=np.float32, output=None):
    from ghost_b200 import Morse
    from ghost_b200.engine import CwtPlan, scale_tables
    freqs = plan_frequencies(wl)
    m = Morse(fs=wl["fs"])
    om = freqs / (wl["fs"] / 2.0) * np.pi
    L = m.compute_lengths(om)
    k0, nt, terms = scale_tables(m, om, L)
    return CwtPlan(L, k0, nt, terms, dtype=dtype, output=output or wl["output"], device=device, guard=guard), freqs


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region, through in-process NVML
    (an nvidia-smi subprocess per sample stalls the driver for hundreds of ms)."""

    def __init__(self, index=0, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz, self.power = None, []
        self.nv = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        nv = self.nv
        if nv is None:
            return
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
                if get_reasons is not None:
                    r = int(get_reasons(self.handle))
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        out = {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
               "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
               "source": "nvml" if self.nv is not None else "unavailable"}
        if self.power:
            out["power_w_max"] = float(max(self.power))
        return out


# --------------------------------------------------------------------------- CPU arm
_REF = None


def load_reference():
    """(ContinuousWaveletTransform, Morse) of the UNMODIFIED reference installed under baseline/_ref
    (tools/install_reference.sh; `pip install --target`), imported through the two-line shim of SURVEY.md
    Appendix C: stub matplotlib modules (the reference imports matplotlib at module level but the
    transform never touches it).  Returns (None, reason) when it is not there."""
    global _REF
    if _REF is not None:
        return _REF
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "ghost")):
        _REF = (None, "baseline/_ref is missing (tools/install_reference.sh was not run in the build container)")
        return _REF
    try:
        for name in ("matplotlib", "matplotlib.pyplot"):
            sys.modules.setdefault(name, types.ModuleType(name))
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        sys.path.insert(0, path)
        logging.disable(logging.WARNING)
        from ghost.wave import ContinuousWaveletTransform, Morse
        logging.disable(logging.NOTSET)
        _REF = ((ContinuousWaveletTransform, Morse), "reference")
    except Exception as e:                                       # noqa: BLE001
        logging.disable(logging.NOTSET)
        _REF = (None, "import of baseline/_ref failed: %r" % (e,))
    return _REF


def cpu_transform(wl, x, freqs):
    """One CPU transform of one channel with all host threads: the reference's own
    ContinuousWaveletTransform.transform(parallel=True) (ThreadPool(cpu_count()) over scales,
    transforms.py:206-218), or the oracle port with the same threading when the reference cannot be
    imported.  Returns (seconds, kind, note)."""
    ref, why = load_reference()
    fs = wl["fs"]
    if ref is not None:
        CWT, Morse = ref
        cwt = CWT(wavelet=Morse(gamma=3, beta=20))
        ts = np.arange(x.size) / fs              # explicit timestamps: the reference's default needs np.float (numpy < 1.24)
        logging.disable(logging.WARNING)
        t0 = time.perf_counter()
        cwt.transform(x, fs=fs, timestamps=ts, freq_limits=wl["freq_limits"], voices_per_octave=wl["vpo"], parallel=True)
        dt = time.perf_counter() - t0
        logging.disable(logging.NOTSET)
        amp = cwt.amplitude
        if amp.shape[0] != len(freqs):
            # a shorter sample narrows the reference's own frequency range: count what it computed
            return dt, "reference", "reference grid %d scales" % amp.shape[0], amp.shape[0]
        return dt, "reference", "", amp.shape[0]
    from oracle import cwt_oracle as orc
    t0 = time.perf_counter()
    orc.cwt_amplitude(x, fs, frequencies=freqs, parallel=True)
    return time.perf_counter() - t0, "port", why, len(freqs)


def cpu_sample_size(wl, freqs, seconds_hint, cores):
    """Samples of one channel that keep one CPU transform near `seconds_hint` (the reference needs roughly
    0.3 us per coefficient per core) but long enough for the lowest scale (5 x its kernel)."""
    n = wl["n"]
    est_full = 3.0e-7 * n * len(freqs) / max(1, min(cores, len(freqs)))
    from ghost_b200 import Morse
    lmax = int(Morse(fs=wl["fs"]).compute_lengths(np.array([freqs.min()]) / (wl["fs"] / 2.0) * np.pi)[0])
    n_s = n if est_full <= seconds_hint else max(int(n * seconds_hint / est_full), 5 * lmax + 1000)
    return min(n, n_s)


def cpu_baseline(wl, freqs, seconds_hint):
    from ghost_b200 import synth
    cores = os.cpu_count() or 1
    n_s = cpu_sample_size(wl, freqs, seconds_hint, cores)
    x = synth.chirp_pink(n_s, wl["fs"], 0, np.float32)
    dt, kind, note, n_scales = cpu_transform(wl, x, freqs)
    what = "the unmodified reference from baseline/_ref, ContinuousWaveletTransform.transform(parallel=True), scipy backend" \
        if kind == "reference" else "oracle port of the reference (%s), ThreadPool over scales" % note
    return {"value": n_s * n_scales / dt, "unit": UNIT, "cores": cores, "kind": kind, "seconds": dt,
            "sample": "1 channel x %d samples x %d scales (%s); os.cpu_count() = %d" % (n_s, n_scales, what, cores)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ghost_b200 import synth
    wl = dict(WORKLOADS[args.workload])
    if args.samples:
        wl["n"] = int(args.samples)
    freqs = plan_frequencies(wl)
    cores = os.cpu_count() or 1
    n_s = cpu_sample_size(wl, freqs, 8.0, cores)
    x = synth.chirp_pink(n_s, wl["fs"], 0, np.float32)
    kind = note = ""
    n_scales = len(freqs)
    for _ in range(max(1, args.warmup) if args.warmup else 0):
        cpu_transform(wl, x, freqs)
    t_all = 0.0
    for _ in range(args.steps):
        dt, kind, note, n_scales = cpu_transform(wl, x, freqs)
        t_all += dt
    dt = t_all / max(1, args.steps)
    value = n_s * n_scales / dt
    what = "the unmodified reference from baseline/_ref, transform(parallel=True), scipy backend" if kind == "reference" \
        else "oracle port of the reference: " + note
    sample = "1 channel x %d samples x %d scales per step (%s); os.cpu_count() = %d" % (n_s, n_scales, what, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload + ": " + wl["desc"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------- GPU arm
def synth_channels(wl, nch, n, first_channel, pin=True):
    """(nch, n) fp32 host tensor: distinct seeds for the first 8 channels, then rolled copies (generation cost only)."""
    import torch
    from ghost_b200 import synth
    fs = wl["fs"]
    if n > 50000000:       # very long shards: tile a 2^24-sample block (generation cost only)
        blk = [synth.chirp_pink(1 << 24, fs, first_channel + c, np.float32) for c in range(min(nch, 8))]
        base = [np.tile(b, n // b.size + 1)[:n] for b in blk]
    else:
        base = [synth.chirp_pink(n, fs, first_channel + c, np.float32) for c in range(min(nch, 8))]
    x_host = torch.empty((nch, n), dtype=torch.float32)
    if pin:
        x_host = x_host.pin_memory()
    for c in range(nch):
        x_host[c] = torch.from_numpy(base[c % len(base)])
        if c >= len(base):
            x_host[c] = torch.roll(x_host[c], 1009 * c)
    return x_host


class Timer:
    """K steps between barriers, CUDA events on the current stream, max over ranks."""

    def __init__(self, dev, world):
        import torch
        self.torch, self.dev, self.world = torch, dev, world

    def barrier(self):
        import torch.distributed as dist
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier()
            self.torch.cuda.synchronize(self.dev)

    def run(self, fn, steps, warmup):
        import torch.distributed as dist
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        self.barrier()
        ms = ev0.elapsed_time(ev1)
        if self.world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps


DUMP_BYTES = 48 << 20          # all files of one --dump-outputs call together stay under 64 MB
DUMP_EDGE = 64                 # columns kept at either end: they see the zero padding of the convolution


def dump_outputs(dirname, res, first, output, freqs, rank, world):
    """--dump-outputs: K sample columns of ``res`` (channels, scales, columns), a CUDA tensor that holds
    this rank's samples first, first + 1, ...; the columns are the same from run to run."""
    import torch
    nch, S, ncols = res.shape
    parts = 2 if res.is_complex() else 1
    item = res.element_size() // parts
    k = max(1, min(ncols, (DUMP_BYTES // world - 8 * S) // (nch * S * parts * item + 8)))
    e = min(DUMP_EDGE, k // 2)                            # the edge columns are reserved first, within the k
    edge = np.r_[0:min(e, ncols), max(0, ncols - e):ncols]
    draw = np.random.default_rng(0).integers(0, ncols, size=k - edge.size)
    cols = np.unique(np.concatenate([edge, draw]))
    vals = res.index_select(2, torch.from_numpy(cols).to(res.device))
    if vals.is_complex():
        vals = torch.view_as_real(vals)
    suffix = "_rank%d" % rank if world > 1 else ""
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, ("coefficients" if output == "complex" else output) + suffix + ".npy"), vals.cpu().numpy())
    np.save(os.path.join(dirname, "columns" + suffix + ".npy"), (cols + first).astype(np.float64))
    np.save(os.path.join(dirname, "frequencies" + suffix + ".npy"), np.asarray(freqs, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from ghost_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ.pop("NCCL_DEBUG")                  # keep NCCL's banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    wl = dict(WORKLOADS[args.workload])
    if args.channels:
        wl["channels"] = args.channels
    if args.samples:
        wl["n"] = args.samples
    f64 = wl.get("dtype") == "f64" or args.dtype == "f64"
    fs, n, nch = wl["fs"], wl["n"], wl["channels"]
    plan, freqs = build_plan(wl, local, guard=not args.no_guard, dtype=np.float64 if f64 else np.float32)
    S = len(freqs)

    # synthetic channels of this rank (channel shard: rank r owns channels r*nch .. r*nch+nch-1)
    x_host = synth_channels(wl, nch, n, rank * nch)
    x_dev = x_host.to(dev, non_blocking=True)
    tile = int(args.tile if args.tile else wl.get("tile", 0))
    out = plan.alloc_out(nch, tile if tile else n)
    torch.cuda.synchronize(dev)
    last_tile = [0, n]                 # samples [a, b) that out[:, :, :b - a] holds after a step

    def keep_range(o, a, b):
        last_tile[:] = (a, b)

    def one_pass():
        if wl.get("time_shard"):
            from ghost_b200 import sharding
            sharding.run_time_shard_tiled(plan, x_dev, rank, world, tile, out=out, consumer=keep_range)
        elif tile:
            plan.execute_tiled(x_dev, tile, out=out, consumer=keep_range)   # the mean kernel runs inside the step
        else:
            plan.execute(x_dev, out)

    timer = Timer(dev, world)
    # ---- device-resident timing --------------------------------------------------
    for _ in range(args.warmup):
        one_pass()
    timer.barrier()
    _lib.launch_count(reset=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step = timer.run(one_pass, args.steps, 0)              # the headline: K steps, nothing else inside
    sampler.stop_flag = True
    launches = _lib.launch_count()
    gstats = plan.guard_stats()
    if args.dump_outputs:
        a, b = last_tile
        dump_outputs(args.dump_outputs, out[:, :, :b - a], a, wl["output"], freqs, rank, world)
    # the same K steps again with the library's per-family event spans (they serialise the class launches):
    # what the roofline of each kernel family is computed from
    plan.profile(True)
    plan.profile_read(reset=True)
    ms_step_prof = timer.run(one_pass, args.steps, 0)
    prof = plan.profile_read(reset=True)
    plan.profile(False)
    coeffs_rank = float(nch) * n * S
    value = coeffs_rank * world / (ms_step * 1e-3)

    # ---- roofline of the dominant kernel family -------------------------------------------
    levels = plan.levels()
    out_el = (16 if f64 else 8) if wl["output"] == "complex" else (8 if f64 else 4)
    in_el = 4
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    if f64:
        fam_scales = {"generic": S}
    else:
        interp_on = wl["output"] != "complex"
        # level 2 joins the interpolated classes when its bands allow the wide coarse grid (no direct launches then)
        min_interp_level = 2 if prof["fused_banded"][1] == 0 else 3
        n_interp = int((levels >= min_interp_level).sum()) if interp_on else 0
        n_banded = int((levels >= 0).sum()) - n_interp
        fam_scales = {"fused_interp": n_interp, "fused_banded": n_banded, "fused_full": int((levels == -1).sum())}
    fams = {}
    for fam, ns in fam_scales.items():
        ms_f, ln_f = prof[fam]
        if ns == 0 or ms_f <= 0:
            continue
        # algorithmic bytes of this family's launches in one step: its output rows plus one read of
        # the (decimated) input per class; the input term is bounded by 4 B/sample per launch
        by = float(nch) * n * (ns * out_el + in_el)
        fams[fam] = {"scales": ns, "launches_per_step": ln_f / args.steps, "ms_per_step": ms_f / args.steps,
                     "bytes_per_step": by, "achieved_gbs": by * args.steps / (ms_f * 1e-3) / 1e9,
                     "coeff_per_s": float(nch) * n * ns * args.steps / (ms_f * 1e-3)}
        fams[fam]["frac"] = fams[fam]["achieved_gbs"] / peak
    dom = max(fams, key=lambda k: fams[k]["ms_per_step"]) if fams else None
    whole_gbs = float(nch) * n * (S * out_el + in_el) / (ms_step * 1e-3) / 1e9
    kname = {"generic": "stockham_pass_kernel (generic fp64 path: load, FFT passes, multiply, epilogue)"}.get(dom, (dom or "") + "_kernel")
    roof = {"bound": "hbm", "kernel": kname if dom else None,
            "achieved": fams[dom]["achieved_gbs"] if dom else None, "peak": peak, "unit": "GB/s",
            "frac": fams[dom]["frac"] if dom else None, "traffic": None, "peak_source": peak_src,
            "nominal_peak": 8000.0, "frac_of_nominal": (fams[dom]["achieved_gbs"] / 8000.0) if dom else None,
            "share_of_step": (fams[dom]["ms_per_step"] / ms_step_prof) if dom else None,
            "ms_per_step_with_family_spans": ms_step_prof,
            "families": fams, "mean_pyramid_ms_per_step": prof["mean+pyramid"][0] / args.steps,
            "whole_step": {"achieved": whole_gbs, "frac": whole_gbs / peak, "frac_of_nominal": whole_gbs / 8000.0}}
    # measured DRAM traffic: dram__bytes_read + dram__bytes_write of one ncu --set full capture of this kernel
    # family (profiles/traffic.json names the capture), as a ratio to its algorithmic bytes, scaled to this run
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and dom:
        try:
            tj = json.load(open(traffic_file))
            ratio = tj.get(dom + "_traffic_over_algorithmic")
            if ratio is not None:
                roof["traffic"] = ratio * fams[dom]["bytes_per_step"]
                roof["traffic_note"] = "per step over all %s launches = %.3f x algorithmic bytes; ratio from the ncu capture %s, " \
                                       "not re-measured in this run" % (dom, ratio, tj.get("source", ""))
        except Exception:
            pass

    # ---- end to end through the public API ---------------------------------------------------
    e2e = None
    if not args.no_e2e and not tile and not f64:
        del out
        torch.cuda.empty_cache()
        e2e = run_e2e(args, wl, x_host, dev, local, world, nch, n, S, out_el)

    # ---- CPU baseline (rank 0, N = 1) ------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(wl, freqs, args.cpu_seconds)

    # ---- the shapes BASELINE.json names for several GPUs ------------------------------------
    extra = None
    if world > 1 and not args.no_extra and args.workload == "cfg2" and not args.samples and not args.channels:
        del x_dev, x_host
        plan.close()
        torch.cuda.empty_cache()
        extra = run_extra(args, dev, local, rank, world, peak)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64" if f64 else "f32", "data": "synthetic",
            "config": {"workload": args.workload + ": " + wl["desc"], "channels_per_gpu": nch, "samples": n,
                       "scales": S, "fs": fs, "output": wl["output"],
                       "parallelism": ("time-shard x%d (NCCL halo exchange + mean all-reduce per step)" if wl.get("time_shard")
                                       else "channel-shard x%d") % world,
                       "l2_policy": "inputs (%.2f GB) and outputs (%.1f GB) per step exceed the 126 MB L2" % (
                           nch * n * 4 / 1e9, coeffs_rank * out_el / 1e9),
                       "scale_classes": {"band_limited": int((levels >= 0).sum()), "full_spectrum": int((levels == -1).sum()),
                                         "generic": int((levels == -2).sum())}},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "guard": {"enabled": (not args.no_guard) and not f64, "pairs_checked": gstats["checked"],
                      "pairs_recomputed_fp64": gstats["total"]},
            "clocks": sampler.summary(),
        }
        if extra is not None:
            line["extra"] = extra
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_e2e(args, wl, x_host, dev, local, world, nch, n, S, out_el):
    """Host arrays in, host arrays out through the drop-in class: per step every group of channels goes
    through ContinuousWaveletTransform.transform(X, fs=..., multichannel=True, out=pinned), which is one
    gcwt_execute_host call (H2D of the samples, tiles computed, D2H of every coefficient while the next tile
    is computed); the caller's pinned result buffer is reused from group to group."""
    import torch
    import torch.distributed as dist
    from ghost_b200 import ContinuousWaveletTransform
    # channels per call: as many as a quarter of this rank's share of the free host memory holds pinned (<= 32)
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    group = int(max(1, min(nch, 32, (avail // 4 // max(1, world)) // (S * n * out_el))))
    res = torch.empty((group, S, n), dtype=torch.float32 if out_el == 4 else torch.complex64).pin_memory()
    res_np = res.numpy()
    x_np = x_host.numpy()
    cwt = ContinuousWaveletTransform(dtype=np.float32, output=wl["output"], device=local, guard=not args.no_guard)
    kw = dict(fs=wl["fs"], freq_limits=wl["freq_limits"], voices_per_octave=wl["vpo"], multichannel=True)
    checks = []

    def one_step():
        for c0 in range(0, nch, group):
            g = min(group, nch - c0)
            cwt.transform(x_np[c0:c0 + g], out=res_np[:g], **kw)
            checks.append(float(res_np[0, 0, :64].sum()))        # the caller reads the result before the next group

    logging.disable(logging.WARNING)
    steps = max(1, min(args.steps, 3))
    one_step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    torch.cuda.synchronize(dev)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    sec = float(dt.item()) / steps
    host = cwt.last_plan.host_stats()
    logging.disable(logging.NOTSET)

    # the ceiling of this path: plain pinned D2H copies of the same size class, all ranks at once
    scratch = torch.empty(1 << 28, dtype=torch.float32, device=dev)              # 1 GiB
    tgt = res.view(-1)[:scratch.numel()] if res.numel() >= scratch.numel() and not res.is_complex() else \
        torch.empty(scratch.numel(), dtype=torch.float32).pin_memory()
    tgt.copy_(scratch, non_blocking=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(8):
        tgt.copy_(scratch, non_blocking=True)
    torch.cuda.synchronize(dev)
    d2h = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(d2h, op=dist.ReduceOp.MAX)
    d2h_gbs = 8 * scratch.numel() * 4 * world / float(d2h.item()) / 1e9
    bytes_step = float(nch) * n * (S * out_el + 4) * world
    return {"value": float(nch) * n * S * world / sec, "unit": UNIT, "h2d_bytes_per_step": int(nch * n * 4),
            "d2h_bytes_per_step": int(nch * n * S * out_el), "ms_per_step": sec * 1e3, "steps": steps,
            "api": "ContinuousWaveletTransform.transform(X[%d channels], fs=..., multichannel=True, out=pinned ndarray) "
                   "-> gcwt_execute_host, %d calls per step" % (group, (nch + group - 1) // group),
            "channel_group": group, "tiles_per_call": host["tiles"], "pinned_destination": host["pinned_destination"],
            "link_gbs": bytes_step / sec / 1e9,
            "d2h_ceiling_gbs": d2h_gbs, "frac_of_d2h_ceiling": bytes_step / sec / 1e9 / d2h_gbs,
            "d2h_ceiling_note": "%d ranks x 8 concurrent 1 GiB device -> pinned host copies, aggregate" % world,
            "checksum": float(np.sum(checks[-(nch // group):]))}


def run_extra(args, dev, local, rank, world, peak):
    """N > 1: the multi-GPU shapes BASELINE.json names, each timed like the headline (barriers, CUDA events,
    max over ranks): strong scaling of the 64-channel config 2, the full config 3 at N = 8, and config 4
    (one 24 h recording) time-sharded over the ranks with a seam check against an unsharded transform."""
    import torch
    import torch.distributed as dist
    from ghost_b200 import sharding
    timer = Timer(dev, world)
    extra = {}
    guard = not args.no_guard

    # ---- strong scaling: the named 64 channels split over the ranks ---------------------------
    wl = dict(WORKLOADS["cfg2"])
    lo, hi = sharding.channel_block(64, rank, world)
    plan, freqs = build_plan(wl, local, guard=guard)
    x = synth_channels(wl, hi - lo, wl["n"], lo, pin=False).to(dev)
    out = plan.alloc_out(hi - lo, wl["n"])
    ms = timer.run(lambda: plan.execute(x, out), max(2, min(args.steps, 5)), 2)
    coeffs = 64.0 * wl["n"] * len(freqs)
    extra["cfg2_strong"] = {"workload": "cfg2: the named 64 channels over %d GPUs (%d per GPU), fp32 amplitude" % (world, hi - lo),
                            "scaling": "strong", "ms_per_step": ms, "value": coeffs / (ms * 1e-3), "unit": UNIT,
                            "hbm_frac_of_measured_aggregate": 64.0 * wl["n"] * (len(freqs) * 4 + 4) / (ms * 1e-3) / 1e9 / (peak * world)}
    del x, out
    plan.close()
    torch.cuda.empty_cache()

    # ---- config 3 in full (256 channels need 8 GPUs at 32 per GPU) ----------------------------
    if world == 8:
        wl = dict(WORKLOADS["cfg3"])
        plan, freqs = build_plan(wl, local, guard=guard)
        x = synth_channels(wl, 32, wl["n"], rank * 32, pin=False).to(dev)
        out = plan.alloc_out(32, wl["tile"])
        ms = timer.run(lambda: plan.execute_tiled(x, wl["tile"], out=out), 2, 1)
        coeffs = 256.0 * wl["n"] * len(freqs)
        gbs = 256.0 * wl["n"] * (len(freqs) * 4 + 4) / (ms * 1e-3) / 1e9
        extra["cfg3_full"] = {"workload": "cfg3: 256ch x 30kHz x 10min x 128 scales, fp32 power, 32 channels per GPU, results "
                                          "streamed in %d time tiles per GPU" % (-(-wl["n"] // wl["tile"])), "scaling": "channel-shard x8", "ms_per_step": ms,
                              "value": coeffs / (ms * 1e-3), "unit": UNIT, "achieved_gbs": gbs,
                              "hbm_frac_of_measured_aggregate": gbs / (peak * 8), "hbm_frac_of_nominal_8TBs": gbs / 64000.0,
                              "guard_pairs_recomputed_fp64": plan.guard_stats()["total"]}
        del x, out
        plan.close()
        torch.cuda.empty_cache()

    # ---- config 4: one 24 h recording, time-sharded over the ranks ------------------------------
    wl = dict(WORKLOADS["cfg4"])
    n_total = wl["plan_n"]
    plan, freqs = build_plan(wl, local, guard=guard)
    S = len(freqs)
    halo = sharding.required_halo(plan)
    lo, hi = sharding.time_block(n_total, rank, world, align=16384)
    n_local = hi - lo
    blk = synth_channels(wl, 1, 1 << 24, 0, pin=False)[0].numpy()
    # every rank cuts ITS samples out of the same periodic recording (a 2^24-sample chirp + pink block repeated)
    idx0 = lo % blk.size
    # the shard is stored with room for its halos (sharding.TimeShard): the neighbours' samples are received in place
    shard = sharding.TimeShard(1, n_local, halo, dtype=torch.float32, device=dev)
    shard.core.copy_(torch.from_numpy(np.concatenate([blk[idx0:], np.tile(blk, (n_local + blk.size - 1) // blk.size + 1)])[:n_local].copy())[None, :])
    x = shard.core
    tile = int(wl["tile"])
    out = plan.alloc_out(1, tile)
    M = 20000                                                   # seam check: M samples either side of the rank 0 | rank 1 seam
    keep = {"tail": torch.zeros((S, M), dtype=torch.float32, device=dev), "head": torch.zeros((S, M), dtype=torch.float32, device=dev)}

    def consumer(o, a, b):
        # rank 0 keeps the coefficients of its last M samples, rank 1 those of its first M (whatever tiles hold them)
        if rank == 0:
            lo_, hi_ = max(a, n_local - M), min(b, n_local)
            if hi_ > lo_:
                keep["tail"][:, lo_ - (n_local - M):hi_ - (n_local - M)] = o[0, :, lo_ - a:hi_ - a]
        if rank == 1:
            lo_, hi_ = max(a, 0), min(b, M)
            if hi_ > lo_:
                keep["head"][:, lo_:hi_] = o[0, :, lo_ - a:hi_ - a]

    done = sharding.run_time_shard_tiled(plan, shard, rank, world, tile, out=out, consumer=consumer)
    lens = sharding.gather_shard_lengths(n_local, rank, world, dev)          # the partition is fixed: gathered once
    ms = timer.run(lambda: sharding.run_time_shard_tiled(plan, shard, rank, world, tile, out=out, lens=lens), 3, 1)
    # the same shard with no neighbours (no collectives, zero padding at the seams): what the exchange costs
    ms_alone = timer.run(lambda: plan.execute_tiled(x, tile, out=out), 3, 1)      # (its own mean kernel included)
    # seam check on rank 0: the window [seam - halo - M, seam + halo + M) transformed unsharded
    seam = None
    means = sharding.global_means(plan.channel_means(x) * float(n_local), n_local)
    if rank == 1:
        dist.send(x[0, :halo + M].contiguous(), dst=0)
        dist.send(keep["head"].contiguous(), dst=0)
    if rank == 0:
        right = torch.empty(halo + M, dtype=torch.float32, device=dev)
        head = torch.empty((S, M), dtype=torch.float32, device=dev)
        dist.recv(right, src=1)
        dist.recv(head, src=1)
        win = torch.cat([x[0, n_local - halo - M:], right])[None, :]
        ref = plan.execute(win, means=means)[0][:, halo:halo + 2 * M]
        got = torch.cat([keep["tail"], head], dim=1)
        num = torch.linalg.vector_norm((got - ref).double(), dim=1)
        den = torch.linalg.vector_norm(ref.double(), dim=1)
        seam = {"window": "%d samples either side of the rank 0 | rank 1 seam, all %d scales" % (M, S),
                "rel_l2_max_over_scales": float((num / den).max()), "bar": 1e-5}
    coeffs = float(n_total) * S
    gbs = float(n_total) * (S * 4 + 4) / (ms * 1e-3) / 1e9
    extra["cfg4_time_shard"] = {"workload": "cfg4: 1ch x 30kHz x 24h (%.3e samples) x %d scales, fp32 power, %d time shards of %.3e samples, "
                                            "mean all-reduce + NCCL halo exchange (%d samples per seam) every step, results streamed in "
                                            "tiles of %d" % (n_total, S, world, n_local, halo, tile),
                                "scaling": "time-shard x%d" % world, "ms_per_step": ms, "value": coeffs / (ms * 1e-3), "unit": UNIT,
                                "achieved_gbs": gbs, "hbm_frac_of_measured_aggregate": gbs / (peak * world),
                                "ms_same_shard_no_neighbours": ms_alone, "exchange_overhead": ms / ms_alone - 1.0,
                                "nccl_ranks": world, "seam_check": seam, "coeffs_this_rank": done}
    del x, out
    plan.close()
    return extra


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
