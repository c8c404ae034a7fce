"""bench.py --dump-outputs: the last timed step's outputs land as float32 .npy files of the documented
shapes, and two runs with the same arguments compute from the same seeded inputs, weights and draws."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu

NAMES = ("losses", "params", "param_grads", "step_preds", "step_log_probas", "step_values", "step_pos")


def _bench_dump(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", "3",
           "--no-secondary", "--no-cpu-baseline", "--no-roofline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    assert sorted(os.listdir(out_dir)) == sorted(f"{n}.npy" for n in NAMES)
    return {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in NAMES}


def test_dump_outputs_repeat_for_the_same_arguments(tmp_path):
    import bench

    w = bench.WORKLOADS["c1"]
    a = _bench_dump(tmp_path / "a", 4)
    b = _bench_dump(tmp_path / "b", 4)
    T, na, nb = w["T"], w["na"], w["B"]
    assert a["losses"].shape == (5,) and a["params"].shape == a["param_grads"].shape
    assert a["step_preds"].shape == (T, na, nb, w["nc"]) and a["step_pos"].shape == (T, na, nb, 2)
    assert a["step_values"].shape == a["step_log_probas"].shape == (T, na, nb)
    for n in NAMES:
        assert a[n].dtype == np.float32 and np.isfinite(a[n]).all(), n
    assert np.array_equal(a["step_pos"], b["step_pos"])
    for n in NAMES:
        den = max(float(np.linalg.norm(b[n].astype(np.float64))), 1e-30)
        assert float(np.linalg.norm(a[n].astype(np.float64) - b[n])) / den < 1e-5, n
