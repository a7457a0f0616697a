"""The bench.py contract. Reference arm (`--impl reference`, CPU): one JSON line on stdout with the keys a reader of
the result needs; non-zero ranks print nothing. CUDA arm (gpu): `--dump-outputs` writes the last timed step's grid."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from conftest import assert_parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["value"] > 0
    # the faster of the two CPU implementations is reported: the oracle port of backend='vectorized' or, when
    # oracle/_ref is built, the reference's compiled backend='C' twin
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert "other_cpu_implementation" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # a non-zero rank of the reference arm exits 0 without output
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"],
                         capture_output=True, text=True, env=env, timeout=60)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_ours_arm_dumps_the_last_timed_step(tmp_path):
    """`--dump-outputs DIR`: the headline grid of the last timed step as (ny, nx) float64 arrays, in execute('grid')
    orientation (checked against the CPU oracle on a few cells); `--steps` is the number of timed steps reported."""
    from oracle import krige_oracle as ko
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--configs", "none", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, env=env, timeout=1200)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    z, ss = np.load(tmp_path / "zvalues.npy"), np.load(tmp_path / "sigmasq.npy")
    assert z.shape == ss.shape == (1000, 1000) and z.dtype == ss.dtype == np.float64
    assert sorted(p.name for p in tmp_path.iterdir()) == ["sigmasq.npy", "zvalues.npy"]
    xyz, val = cases.synth_data(1002, 5000, 2)
    gx = gy = np.linspace(0.0, 1000.0, 1000)
    rng = np.random.default_rng(5)
    iy, ix = rng.integers(0, 1000, 32), rng.integers(0, 1000, 32)
    zo, so = ko.krige(xyz, val, "exponential", ko.stored_parameters("exponential", [1.0, 300.0, 0.05]),
                      np.column_stack([gx[ix], gy[iy]]))
    assert_parity(z[iy, ix], zo, 1e-5, "z")
    assert_parity(ss[iy, ix], so, 1e-5, "ss")
