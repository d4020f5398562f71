"""bench.py's output contract: exactly ONE JSON line on stdout with the result keys (everything else goes to stderr) and,
with --dump-outputs, what the last timed solve returned. The reference arm (the CPU oracle on the benchmarked scene) is
checked on the CPU tier, the CUDA arm on a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("camera", "views", "points", "iteration_cost")


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    return json.loads(lines[0])


def _load_dump(d):
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in DUMPED)
    out = {n: np.load(os.path.join(d, n + ".npy")) for n in DUMPED}
    assert all(a.dtype == np.float64 for a in out.values())
    return out


def test_reference_arm_prints_one_json_line(tmp_path):
    d = _bench("--impl", "reference", "--workload", "cfg1", "--steps", "4", "--warmup", "1",
               "--dump-outputs", str(tmp_path))
    assert d["steps"] == 4 and d["warmup"] == 1
    assert d["impl"] == "reference" and d["metric"] == "lm_residual_jacobian_evals_per_s" and d["unit"] == "M evals/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["dtype"] == "f64" and d["gpu_launches"] == 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["same_scene"] is True and "sample" in cb
    assert d["config"]["workload"].startswith("cfg1")
    out = _load_dump(tmp_path)
    assert out["camera"].shape == (17,) and out["views"].shape[1] == 6 and out["points"].shape[1] == 3
    assert out["iteration_cost"][-1] == d["final_cost"]


@pytest.mark.parametrize("flags", [("--steps", "0"), ("--warmup", "-1")])
def test_step_counts_out_of_range_are_refused(flags):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *flags],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and flags[0] in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_gpu_arm_dumps_what_its_last_timed_solve_returned(built, tmp_path):
    """The CUDA arm's dump holds the solution of the benchmarked scene: the CPU oracle's dump of the same scene agrees
    with it to the bars of the parity tests (rows and final parameters within 1e-9 relative) and of smoke() (camera)."""
    d = _bench("--workload", "cfg1", "--steps", "2", "--warmup", "0", "--no-cpu-baseline", "--no-e2e",
               "--dump-outputs", str(tmp_path / "gpu"))
    assert d["steps"] == 2 and d["lm_iterations_per_solve"] == len(np.load(tmp_path / "gpu" / "iteration_cost.npy"))
    _bench("--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "0",
           "--dump-outputs", str(tmp_path / "cpu"))
    gpu, cpu = _load_dump(tmp_path / "gpu"), _load_dump(tmp_path / "cpu")
    assert gpu["iteration_cost"][-1] == d["final_cost"]
    for n in DUMPED:
        assert gpu[n].shape == cpu[n].shape, n
    assert np.allclose(gpu["iteration_cost"], cpu["iteration_cost"], rtol=1e-9, atol=0)
    assert np.allclose(gpu["camera"], cpu["camera"], rtol=1e-7, atol=1e-12)
    for n in ("views", "points"):
        assert np.max(np.abs(gpu[n] - cpu[n])) <= 1e-9 * max(1.0, np.max(np.abs(cpu[n]))), n


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                        "--gpus", "2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT,
                       env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
