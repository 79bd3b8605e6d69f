"""bench.py's JSON contract, checked on CPU through the reference arm at a reduced geometry; --dump-outputs on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    env = dict(os.environ)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--hw", "80x144"], capture_output=True, text=True, env=env, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpixels/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert "80x144" in d["metric"] and "NOT the BASELINE geometry" in d["metric"]  # a shrunk run says so itself


def test_non_zero_ranks_of_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--hw", "80x144"], capture_output=True, text=True, env=env, timeout=120, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_same_for_the_same_arguments(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same float32 / float64 arrays, 64 MB at most, and the
    JSON line reports the requested number of timed steps.  6 pairs per step: every output is small enough to be
    written whole, in its own shape."""
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--hw",
                              "80x144", "--global-batch", "6", "--micro-batch", "4", "--no-cpu-baseline",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
        dumps.append({f: np.load(d / f) for f in os.listdir(d)})
    a, b = dumps
    assert {"y_dec.npy", "y_syn.npy", "x_dec.npy", "x_with_si.npy", "symbols.npy", "bits_sum.npy", "row.npy"} <= set(a)
    assert sorted(a) == sorted(b) and sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["x_with_si.npy"].shape == (6, 3, 80, 144) and a["row.npy"].shape[0] == 6
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
