"""bench.py contract on CPU: the reference arm (oracle port on the host cores) prints ONE JSON
line with the agreed keys; a tiny operand keeps it to a few seconds."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import ROOT, rel_err


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, BL_BENCH_N="20000", BL_BENCH_DEPTH="12", BL_REF_DEPTH="6")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, env=env, timeout=300)  # fmt: skip
    assert out.returncode == 0, out.stderr
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, BL_BENCH_N="20000", BL_BENCH_DEPTH="12", RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, timeout=120)  # fmt: skip
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_the_same_way_every_time(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    small = np.arange(12, dtype=np.float64).reshape(3, 4)
    large = np.random.default_rng(5).standard_normal((3, 2000)).astype(np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "large": large})
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    a, b = np.load(tmp_path / "a" / "large.npy"), np.load(tmp_path / "b" / "large.npy")
    assert a.dtype == np.float32 and a.shape == (1000,) and np.array_equal(a, b)
    assert np.isin(a, large).all() and len(np.unique(a)) == 1000
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "c"), {"ints": np.arange(3)})


def _bench_small(steps, dump_dir):
    env = dict(os.environ, BL_BENCH_N="20000", BL_BENCH_DEPTH="12")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                          "--quick", "--dump-outputs", str(dump_dir)], capture_output=True, text=True, env=env,
                         timeout=600)  # fmt: skip
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {k: np.load(dump_dir / f"{k}.npy") for k in ("H", "dv", "dparams")}


@pytest.mark.gpu
def test_dumped_outputs_are_those_of_the_last_of_steps_timed_steps(tmp_path):
    """Two lanes of four probes: `H` and `dv` are the same after one timed step and after three, the parameter
    cotangent accumulates over the timed steps (three times that of one), and more steps launch more kernels."""
    one, out1 = _bench_small(1, tmp_path / "one")
    three, out3 = _bench_small(3, tmp_path / "three")
    assert out1["H"].shape == (2, 4, 12, 12) and out1["dv"].shape == (2, 4, 20000)
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in (*out1.values(), *out3.values()))
    assert rel_err(out3["H"], out1["H"]) < 1e-5 and rel_err(out3["dv"], out1["dv"]) < 1e-4
    assert rel_err(out3["dparams"], 3 * out1["dparams"]) < 1e-4 and np.abs(out1["dparams"]).max() > 0
    assert rel_err(out1["dv"][0, 0], out1["dv"][1, 0]) > 1e-3  # the lanes run different probes
    assert three["gpu_launches"] > one["gpu_launches"]
