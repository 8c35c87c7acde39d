"""bench.py on the GPU: `--steps K` times exactly K LM iterations of the seeded problem, and `--dump-outputs` holds what they returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from sfm_toy_library_b200 import capi, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(900)
def test_dump_outputs_hold_the_timed_iterations(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--workload", "cfg2",
                        "--no-stages", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    out = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("cameras", "points", "focal")}
    assert all(x.dtype == np.float64 for x in out.values())
    p = synth.make_ba_problem(seed=0, **synth.BA_CONFIGS["cfg2"])
    ctx = capi.Context(0)
    prob = ctx.ba_problem(p["cams"], p["pts"], p["focal"], p["obs_xy"], p["obs_cam"], p["pt_off"])
    s = prob.run(capi.ba_default_options(max_num_iterations=3, max_solver_time_in_seconds=0.0, function_tolerance=-1.0,
                                         parameter_tolerance=-1.0, gradient_tolerance=-1.0))
    cams, pts, f = prob.download()
    prob.close(); ctx.close()
    assert s["num_iterations"] == 3
    assert out["cameras"].shape == cams.shape and out["points"].shape == pts.shape and out["focal"].shape == (1,)
    np.testing.assert_allclose(out["cameras"], cams, rtol=0, atol=1e-9)
    np.testing.assert_allclose(out["points"], pts, rtol=0, atol=1e-9 * np.abs(pts).max())
    assert abs(out["focal"][0] - f) < 1e-9 * f
