"""bench.py's reference arm runs on the host cores alone: check its JSON line against the driver
contract on the small config (the GPU arm is exercised on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                     # exactly one JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "cwt_output_coeffs_per_sec" and d["unit"] == "coeff/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    have_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "ghost"))
    assert cb["kind"] == ("reference" if have_ref else "port")     # the real reference whenever it is installed
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bad_arguments_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-2000:])
    assert not (tmp_path / "d").exists()


# bench arguments, workload, channels, samples, time tile, name of the coefficient file, runs
DUMP_CASES = {
    "untiled": ([], "cfg2", 2, 300000, None, "amplitude", 2),
    "tiled": (["--tile", "70000"], "cfg2", 2, 300000, 70000, "amplitude", 1),
    "time_shard": (["--workload", "cfg4", "--tile", "150000"], "cfg4", 1, 400000, 150000, "power", 1),
    "f64_complex": (["--dtype", "f64"], "cfg5", 2, 40000, None, "coefficients", 1),
}


def _last_step(bench, wl, nch, n, tile, f64):
    """What the step bench.py times leaves in its result buffer: (coefficients, first sample, frequencies)."""
    from ghost_b200 import sharding
    plan, freqs = bench.build_plan(wl, 0, dtype=np.float64 if f64 else np.float32)
    x = bench.synth_channels(wl, nch, n, 0, pin=False).cuda()
    if not tile:
        return plan.execute(x), 0, freqs
    last = {}

    def keep(o, a, b):
        last["res"], last["a"] = o[:, :, :b - a].clone(), a

    if wl.get("time_shard"):
        sharding.run_time_shard_tiled(plan, x, 0, 1, tile, consumer=keep)
    else:
        plan.execute_tiled(x, tile, consumer=keep)
    return last["res"], last["a"], freqs


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(DUMP_CASES))
def test_dump_outputs_are_the_timed_results(tmp_path, case):
    """--dump-outputs writes a fixed sample of the last timed step: the same files from run to run, and the
    coefficients of the same input transformed directly (for tiled workloads: the last tile of the step)."""
    torch = pytest.importorskip("torch")
    import bench
    extra, workload, nch, n, tile, name, n_runs = DUMP_CASES[case]
    args = extra + ["--channels", str(nch), "--samples", str(n), "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu"]
    runs = []
    for r in range(n_runs):
        d = tmp_path / str(r)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert len([l for l in out.stdout.splitlines() if l.startswith("{")]) == 1
        assert sorted(os.listdir(d)) == sorted([name + ".npy", "columns.npy", "frequencies.npy"])
        assert sum(f.stat().st_size for f in d.iterdir()) <= 64e6
        runs.append({f.stem: np.load(f) for f in d.iterdir()})
    a = runs[0]
    for b in runs[1:]:
        for key in a:
            assert np.array_equal(a[key], b[key]), key
    for key in a:
        assert a[key].dtype in (np.float32, np.float64), key
    wl = dict(bench.WORKLOADS[workload], n=n)
    res, first, freqs = _last_step(bench, wl, nch, n, tile, name == "coefficients")
    assert np.array_equal(a["frequencies"], freqs)
    cols = a["columns"].astype(np.int64)
    last = first + res.shape[2]                                  # the last step ends with samples [first, last)
    assert first == (0 if not tile else (n - 1) // tile * tile)
    assert np.array_equal(cols, np.unique(cols)) and cols[0] == first and cols[-1] == last - 1
    assert set(range(first, first + 64)) | set(range(last - 64, last)) <= set(cols.tolist())
    want = res[:, :, torch.from_numpy(cols - first).cuda()]
    if want.is_complex():
        want = torch.view_as_real(want)
    want = want.cpu().numpy()
    assert a[name].dtype == want.dtype and a[name].shape == want.shape
    assert want.shape[:3] == (nch, freqs.size, cols.size)
    assert want.shape[3:] == ((2,) if name == "coefficients" else ())    # complex: (real, imaginary) pairs
    assert np.max(np.abs(a[name] - want)) <= 1e-6 * np.max(np.abs(want))


def test_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--workload", "cfg1", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
