"""bench.py's reference arm (the CPU leg the driver runs as `--impl reference`):
one JSON line with the contract's keys on rank 0, nothing and exit 0 on the
other ranks; the GPU arm refuses to run without a CUDA device (no CPU fallback)."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, **env):
    e = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        e.pop(k, None)
    e.update({k: str(v) for k, v in env.items()})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=e,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "3"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["metric"].startswith("input Msamples/s") and line["unit"] == "Msamples/s"
    assert line["steps"] == 1 and line["warmup"] >= 3 and line["n_gpus"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["config"]["workload"].startswith("cfg2") and "model" not in line["config"]
    assert line["config"]["sample_dtype"] == "u8" and line["config"]["fft_size"] == 4096
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"],
                           "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_reference_arm_other_ranks_do_nothing():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "3"],
             RANK=1, LOCAL_RANK=1, WORLD_SIZE=2)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "3", "--no-cpu-baseline"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    r = _run(["--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path / "out")])
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_gpu_arm_times_k_steps_and_dumps_their_rows(tmp_path):
    """--steps K times K steps (the kernel launches of the timed region double with K), and
    --dump-outputs writes the rows of the last timed step: float32, one row per frame, the same
    rows from run to run with the same arguments, and the rows the engine returns for the
    (3 + K)-th batch of the same frames -- cfg2 carries its EMA from row to row, and over so few
    rows the rows of the step before still differ."""
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pypanadapter_b200 import synth
    from pypanadapter_b200.engine import ZoomPSD
    w = synth.CFG2
    d_in = torch.from_numpy(synth.make_frames(w, 4)).cuda()
    want = {}
    with ZoomPSD(0) as eng:
        eng.configure(w.fs, w.fft_size, w.fft_ratio, w.frame_len, w.window, dtype=w.dtype, flip=w.flip,
                      f_demod=w.f_demod, crop=w.crop, ema_alpha=w.ema_alpha, mode="fast")
        d_rows = torch.empty((4, eng.row_width), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        for batch in range(1, 3 + 4 + 1):
            eng.process_device(d_in.data_ptr(), 4, d_rows.data_ptr())
            eng.synchronize()
            want[batch] = d_rows.cpu().numpy()
    assert not np.array_equal(want[4], want[5])
    lines, rows = [], []
    for i, steps in enumerate((2, 2, 4)):
        out = tmp_path / str(i)
        r = _run(["--frames", "4", "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline",
                  "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-3000:]
        lines.append(json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]))
        rows.append(np.load(out / "rows.npy"))
    assert [ln["steps"] for ln in lines] == [2, 2, 4]
    assert lines[2]["gpu_launches"] == 2 * lines[0]["gpu_launches"] > 0
    assert rows[0].dtype == np.float32 and rows[0].shape == (4, lines[0]["config"]["row_width"])
    assert np.isfinite(rows[0]).all()
    assert np.array_equal(rows[0], rows[1])
    assert np.array_equal(rows[0], want[3 + 2]) and np.array_equal(rows[2], want[3 + 4])


def test_committed_gpu_arm_line_carries_the_contract():
    """The line the GPU arm printed on the B200 for the build the round ends on (profiles/r02am_*):
    every key the bench contract names, with consistent arithmetic."""
    with open(os.path.join(ROOT, "profiles", "r02am_bench_cfg2.json")) as f:
        line = json.loads([ln for ln in f if ln.startswith("{")][-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline",
              "roofline_fp32", "cpu_baseline", "clocks"):
        assert k in line, k
    assert line["higher_is_better"] is True and line["scaling"] == "weak" and line["vs_baseline"] is None
    assert line["data"] == "synthetic" and line["config"]["workload"].startswith("cfg2") and "model" not in line["config"]
    assert line["warmup"] >= 3 and line["n_gpus"] == 1 and line["gpu_launches"] > 0
    e = line["e2e"]
    assert e["value"] > 0 and e["unit"] == line["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert e["value"] < line["value"]                       # host buffers cross PCIe: never the device-resident figure
    r = line["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s" and r["peak"] > 0
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] >= r["algorithmic_bytes_per_launch"]
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    c = line["clocks"]
    assert c["sm_mhz"] and c["sm_max_mhz"] and not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    samples = line["config"]["frames_per_step_per_gpu"] * line["config"]["frame_len"]
    assert abs(line["value"] - samples / (line["ms_per_step"] * 1e-3) / 1e6) / line["value"] < 1e-6
