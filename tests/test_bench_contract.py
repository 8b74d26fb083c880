"""bench.py contract.  Without a GPU: the reference arm (`--impl reference`) times the oracle's faithful mode on the
host cores and prints ONE JSON line with the same metric / unit / config as the GPU arm; bad arguments are rejected.
On the GPU: --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS=str(os.cpu_count() or 1))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "audio-sec/sec" and d["unit"] == "audio-s/s"
    assert d["vs_baseline"] is None and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bad_arguments_are_rejected():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", args


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's outputs; seeded inputs make two runs agree bit for bit."""
    dumps = []
    for steps in (1, 2):
        d = tmp_path / ("s%d" % steps)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "cfg1", "--steps", str(steps), "--warmup", "1",
                              "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout)["steps"] == steps
        dumps.append({n: np.load(str(d / (n + ".npy"))) for n in ("out_i16", "out_f32", "out_offsets")})
        assert sorted(os.listdir(str(d))) == ["out_f32.npy", "out_i16.npy", "out_offsets.npy"]     # 1 x 4 s: no sampling
    a, b = dumps
    n = len(a["out_f32"])
    assert a["out_f32"].dtype == a["out_i16"].dtype == np.float32 and a["out_offsets"].dtype == np.float64
    assert list(a["out_offsets"]) == [0, n] and len(a["out_i16"]) == n
    assert np.array_equal(a["out_i16"], np.round(a["out_i16"])) and np.abs(a["out_i16"]).max() > 0
    assert np.isfinite(a["out_f32"]).all() and np.abs(a["out_f32"]).max() > 0
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
