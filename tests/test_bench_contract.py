"""bench.py's reference arm runs without a GPU: check its JSON line against the contract (one line, the device arm's
metric / unit / config keys, `impl`, `cpu_baseline`, `e2e`) on a tiny grid, its --dump-outputs files, that a run
writes nothing into the tree, and that the device arm refuses to run without a CUDA device instead of falling back to
the CPU."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*argv, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, cwd=ROOT,
                          env=e, timeout=600)


def test_reference_arm_line():
    r = _run("--impl", "reference", "--size", "32", "--cpu-sub", "2", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "parsdmm_iterations_per_second" and d["unit"] == "iterations/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    assert d["config"]["grid"] == [32, 32, 32] and d["config"]["ran_on_grid"] == [32, 32, 16]
    assert d["config"]["extrapolated"] is True and d["config"]["extrapolation_factor"] == 2.0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sub-volume" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def _tree_state():
    """(path, size, mtime) of every file where a run could leave bytecode or a build of the CPU baseline."""
    out = set()
    for top in ("__pycache__", "oracle", "setintersectionprojection.jl_b200", "tests"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                st = os.stat(os.path.join(dirpath, f))
                out.add((os.path.join(dirpath, f), st.st_size, st.st_mtime_ns))
    return out


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs: x, l_<i>, y_<i> and the log's arrays of the last step as finite float32 / float64 .npy files, the
    same on a second run with the same arguments; neither run writes into the tree."""
    before = _tree_state()
    outs = []
    for run in ("a", "b"):
        r = _run("--impl", "reference", "--size", "32", "--cpu-sub", "2", "--steps", "1", "--warmup", "0",
                 "--dump-outputs", str(tmp_path / run), env={"PYTHONDONTWRITEBYTECODE": ""})
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append({p.stem: np.load(p) for p in (tmp_path / run).glob("*.npy")})
    assert _tree_state() == before
    a, b = outs
    assert {"x", "l_0", "y_0", "log_obj", "log_rho", "log_cg_it"} <= set(a) and set(a) == set(b)
    assert a["x"].shape == (32 * 32 * 16,) and a["log_evol_x"].shape == (a["log_obj"].size - 1,)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.all(np.isfinite(a[k])), k
        assert np.allclose(a[k], b[k], rtol=1e-5, atol=0), k


def test_reference_arm_other_ranks_exit_silently():
    r = _run("--impl", "reference", "--gpus", "2", "--size", "32", "--steps", "1", "--warmup", "0",
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29999"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_device_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run("--size", "32", "--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert "CUDA device" in (r.stderr + r.stdout)
