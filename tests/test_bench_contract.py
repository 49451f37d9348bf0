"""bench.py contract: the reference arm (`--impl reference`) prints one JSON line with the agreed keys on rank 0 and nothing
on the other ranks; `--dump-outputs` writes the outputs of the last timed step (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                          cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_json_line():
    r = _run({"RANK": "0", "WORLD_SIZE": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "ray-samples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_are_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_needs_the_c2_workload_and_a_step():
    for extra in (["--impl", "reference", "--dump-outputs", "x"], ["--workload", "c5", "--dump-outputs", "x"], ["--steps", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, cwd=ROOT, capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-500:])


def _dump(out, steps):
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--quick",
                        "--dump-outputs", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return {p.stem: np.load(p) for p in out.glob("*.npy")}


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """The dump is what the timed step computed: complete, reproducible bit for bit from run to run (seeded inputs, fixed-order
    reductions), and taken after the requested number of steps (a different --steps trains the parameters further)."""
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    arrays = _dump(tmp_path / "a", 2)
    for k in ("loss", "out.color", "out.weights", "grad.udf.lin0.weight_v", "param.udf.lin0.weight_v", "param.beta.beta"):
        assert k in arrays, k
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["out.color"].shape == (512, 3) and np.isfinite(arrays["loss"]).all()
    assert np.abs(arrays["grad.udf.lin0.weight_v"]).max() > 0
    again = _dump(tmp_path / "b", 2)
    assert sorted(again) == sorted(arrays)
    assert [k for k in arrays if not np.array_equal(arrays[k], again[k])] == []
    longer = _dump(tmp_path / "c", 3)
    assert not np.array_equal(longer["param.udf.lin0.weight_v"], arrays["param.udf.lin0.weight_v"])
