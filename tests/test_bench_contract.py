"""bench.py's driver contract on the CPU side: the reference arm prints ONE well-formed JSON line (also under
torchrun-style environments, where only rank 0 works), and the GPU arm refuses to run without a CUDA device instead of
falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                          cwd=ROOT, timeout=300)


@pytest.mark.timeout(400)
def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "windows/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("ChebyNet K=5 training windows/sec") and d["config"]["workload"].startswith("config2")
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 1 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "window" in cb["sample"] and cb["cpu"]
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_same_outputs_run_after_run(tmp_path):
    """--dump-outputs writes the last timed step's results; two runs with the same arguments see the same inputs, so
    they agree up to the order of floating-point sums.  --steps sets the step count of every timed region."""
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    runs = []
    for k in range(2):
        out = tmp_path / ("run%d" % k)
        r = _run(["--steps", "3", "--warmup", "2", "--no-cpu-baseline", "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert d["steps"] == 3 and d["e2e"]["steps"] == 3
        runs.append({f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)})
    assert sorted(runs[0]) == ["grads", "logits", "loss", "params"]
    assert runs[0]["logits"].shape == (512, 22) and runs[0]["loss"].shape == (1,)
    assert sum(a.nbytes for a in runs[0].values()) <= 64 << 20
    for name, a in runs[0].items():
        b = runs[1][name]
        assert a.dtype in (np.float32, np.float64) and np.all(np.isfinite(a)), name
        assert a.shape == b.shape and np.abs(a - b).max() <= 1e-4 * max(np.abs(b).max(), 1e-30), name


@pytest.mark.gpu
@pytest.mark.parametrize("config,shapes", [("1", {"logits": (128, 22), "pred": (128,)}),
                                           ("5", {"y": (64, 2048, 32), "dx": (64, 2048, 15), "dW": (375, 32),
                                                  "db": (32,)})])
def test_gpu_arm_dumps_predict_and_vertex_outputs(tmp_path, config, shapes):
    """The predict path dumps the outputs of its CUDA graph (the predictions are the arg-max of the dumped logits, so
    both come from the same step); the vertex-level layer dumps dW, db and a 2048-vertex sample of y and dx."""
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    r = _run(["--config", config, "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    got = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert {k: a.shape for k, a in got.items()} == shapes
    assert all(a.dtype in (np.float32, np.float64) and np.all(np.isfinite(a)) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    if config == "1":
        assert np.array_equal(got["pred"], got["logits"].argmax(1).astype(np.float64))
    else:
        assert np.abs(got["y"]).max() > 0 and np.abs(got["dW"]).max() > 0
