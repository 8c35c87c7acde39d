"""The bench.py contract as far as it can be exercised without a GPU: the reference arm (the CPU port on the host cores) prints
ONE JSON line with the keys the driver reads, and behaves under a multi-rank launch (rank 0 prints, the others exit 0)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "cpu_baseline", "e2e")


def _run(extra_env=None, extra_args=()):
    env = dict(os.environ); env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--workload", "cfg2",
                        *extra_args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "BA residual+Jacobian evals/sec" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["steps"] == 2 and d["warmup"] == 1 and d["dtype"] == "f64"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_reference_arm_dumps_the_timed_result(tmp_path, oracle):
    """--dump-outputs: the cameras, points and focal length after the 2 timed LM iterations, which start from the seeded problem."""
    assert len(_run(extra_args=("--dump-outputs", str(tmp_path / "out")))) == 1
    out = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("cameras", "points", "focal")}
    from sfm_toy_library_b200 import synth
    p = synth.make_ba_problem(seed=0, **synth.BA_CONFIGS["cfg2"])
    o = oracle.ba_default_options(max_num_iterations=2, max_solver_time_in_seconds=0.0, function_tolerance=-1.0, parameter_tolerance=-1.0,
                                  gradient_tolerance=-1.0, jacobian_mode=0, num_threads=1)
    cams, pts, f, s = oracle.ba_solve(p["cams"], p["pts"], p["focal"], p["obs_xy"], p["obs_cam"], p["pt_off"], o)
    assert s["num_iterations"] == 2
    assert all(x.dtype == np.float64 for x in out.values())
    assert out["cameras"].shape == (20, 6) and out["points"].shape == (10_000, 3) and out["focal"].shape == (1,)
    assert np.abs(out["cameras"] - p["cams"]).max() > 1e-6                     # the solver moved the cameras
    np.testing.assert_allclose(out["cameras"], cams, rtol=0, atol=1e-9)
    np.testing.assert_allclose(out["points"], pts, rtol=0, atol=1e-9 * np.abs(pts).max())
    assert abs(out["focal"][0] - f) < 1e-9 * f


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""
