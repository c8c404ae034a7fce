"""bench.py's reference arm runs on the host cores only (the driver launches it on the GPU box, but it needs no
GPU): its JSON line must carry the contract's keys, the SAME `config` as the GPU arm would print for the workload,
and exactly the requested number of steps."""
import json
import os
import subprocess
import sys

from tests.conftest import ROOT


def _run(*args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_json_contract():
    d = _run("--impl", "reference", "--workload", "c1", "--steps", "3", "--warmup", "1")
    assert d["impl"] == "reference" and d["metric"] == "image_episodes_per_sec" and d["unit"] == "image-episodes/s"
    assert d["steps"] == d["steps_requested"] == 3 and d["value"] > 0 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "image-episodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cfg = d["config"]
    assert cfg["workload"].startswith("c1:") and cfg["agents"] == 3 and cfg["steps_per_episode"] == 5
    assert cfg["global_batch"] == 32 and cfg["parallelism"] == "dp1" and "l2" in cfg


def test_unusable_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and out.stdout == "", (args, out.stderr[-500:])


def test_default_workload_is_config_4_strong_scaling():
    sys.path.insert(0, ROOT)
    import bench

    w = bench.WORKLOADS["c4"]
    assert w["B"] == 256 and w.get("strong") and w["na"] == 16 and w["T"] == 16 and (w["H"], w["W"], w["f"]) == (256, 256, 12)
    # bounded CPU sample: never more images per iteration than fit the time budget, never zero
    assert 1 <= bench.cpu_sample_batch(w, 25, 170.0) <= 256
    assert bench.cpu_sample_batch(bench.WORKLOADS["c1"], 20, 170.0) == 32
