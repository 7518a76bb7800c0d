"""The bench.py output contract, checked on the CPU through the reference arm (tiny workload): exactly one JSON line
on stdout with the keys its readers expect; non-zero ranks of a multi-process launch print nothing and exit 0.  On the
GPU: the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--arch", "XS", "--size", "128",
        "--ref-frames", "1", "--people", "2", "--steps", "1", "--warmup", "0"]


def test_reference_arm_prints_one_json_line():
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run(ARGS, capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("frames/sec LitePose") and d["value"] > 0 and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run(ARGS, capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_repeat(tmp_path):
    """--dump-outputs: float32 payloads of the last timed step, the same for the same arguments whatever --steps is"""
    import numpy as np
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    dumps = []
    for steps in (1, 3):
        out = tmp_path / ("steps%d" % steps)
        args = [sys.executable, os.path.join(ROOT, "bench.py"), "--arch", "XS", "--size", "128", "--batch", "2",
                "--people", "2", "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)]
        r = subprocess.run(args, capture_output=True, text=True, cwd=ROOT, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({n: np.load(str(out / (n + ".npy"))) for n in ("packed", "e2e_packed")})
    for d in dumps:
        assert all(a.dtype == np.float32 for a in d.values())
        assert d["packed"].shape[0] == 2 and d["e2e_packed"].shape[:2] == (1, 2)
        assert np.array_equal(d["e2e_packed"][0], d["packed"])
        assert (d["packed"][:, -1] >= 1).all()                  # the planted persons are found
    assert all(np.array_equal(dumps[0][n], dumps[1][n]) for n in dumps[0])
