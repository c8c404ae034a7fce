"""CPU-side checks: the C-ABI library loads and exports every declared symbol,
the flat parameter layout matches the reference's state_dict (names + shapes),
host-side logic (config, meters, returns helper) behaves like the reference."""
import ctypes as C
import os
import re

import pytest
import torch

from marlclassification_b200 import _lib
from marlclassification_b200.config import ModelConfig
from tests.conftest import GOLDEN_NAMES, ROOT, load_golden


def test_library_loads_and_exports_header_symbols():
    lib = _lib.lib()
    assert lib.marlc_version() >= 1
    header = open(os.path.join(ROOT, "include", "marlc.h")).read()
    declared = set(re.findall(r"\b(marlc_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed from include/marlc.h"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in marlc.h but not exported"
    assert declared == set(_lib.exported_symbols())


def test_engine_create_rejects_bad_geometry():
    cfg = _lib.MarlcConfig()
    handle = C.c_void_p()
    assert _lib.lib().marlc_engine_create(C.byref(cfg), C.byref(handle)) != 0
    assert b"geometry" in _lib.lib().marlc_last_error()


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_state_dict_matches_reference(name):
    fx = load_golden(name)
    model = ModelConfig(**fx["model_config"]).build_networks()
    sd = model.state_dict()
    assert list(sd) == list(fx["state_dict"])  # same keys, same order
    for k, v in fx["state_dict"].items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    model.load_state_dict(fx["state_dict"])  # strict
    layout, total = model._layout()
    assert [n for n, _, _ in layout] == list(sd)
    for n, off, shape in layout:
        assert shape == tuple(sd[n].shape) and off % 64 == 0 and off + sd[n].numel() <= total


def test_no_cpu_fallback():
    from marlclassification_b200.core import Environment

    env = Environment([[1, 0], [-1, 0]], 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        env.reset(torch.zeros(2, 1, 8, 8), 2)
    model = ModelConfig(**load_golden("single_agent")["model_config"]).build_networks()
    with pytest.raises(RuntimeError, match="CUDA"):
        model.ensure_flat()


def test_marl_json_roundtrip(tmp_path):
    fx = load_golden("mnist_ckpt")
    cfg = ModelConfig(**fx["model_config"])
    p = tmp_path / "marl.json"
    cfg.save_marl_config(str(p))
    assert ModelConfig.load_marl_config(str(p)) == cfg


def test_functions_match_oracle():
    from marlclassification_b200.training import functions as Fn
    from oracle import marl_oracle as O

    g = torch.Generator().manual_seed(3)
    preds = torch.randn(5, 3, 4, 7, generator=g)
    y = torch.randint(7, (4,), generator=g)
    assert torch.allclose(Fn.classification_rewards(preds, y), O.classification_rewards(preds, y), atol=1e-6)
    r = torch.randn(5, 3, 4, generator=g)
    assert torch.allclose(Fn.discounted_returns(r, 0.9), O.discounted_returns(r, 0.9), atol=1e-5)
    assert torch.allclose(Fn.standardize(r), O.standardize(r))


def test_confusion_meter():
    from marlclassification_b200.metrics import ConfusionMeter, LossMeter

    cm = ConfusionMeter(3, None)
    proba = torch.eye(3)
    cm.add(proba, torch.tensor([0, 1, 1]))
    assert cm.conf_mat().tolist() == [[1, 0, 0], [0, 1, 1], [0, 0, 0]]
    assert torch.allclose(cm.precision(), torch.tensor([1.0, 1.0, 0.0]))
    assert torch.allclose(cm.recall(), torch.tensor([1.0, 0.5, 0.0]))
    lm = LossMeter(2)
    for v in (1.0, 2.0, 3.0):
        lm.add(v)
    assert lm.loss() == 2.5


def test_input_pipeline_has_no_cpu_path():
    """Device-side ToTensor and the prefetcher refuse host tensors / a CPU device loudly."""
    import pytest
    import torch

    from marlclassification_b200.input_pipeline import DevicePrefetcher, images_u8_to_f32

    with pytest.raises(RuntimeError):
        images_u8_to_f32(torch.zeros(1, 4, 4, 3, dtype=torch.uint8))
    with pytest.raises(RuntimeError):
        DevicePrefetcher([], "cpu")


def test_to_tensor_restatement_matches_torchvision():
    """oracle.to_tensor_batch == torchvision ToTensor (what registry.py:56-57 composes) on PIL images,
    checked live when torchvision / PIL are importable (the recorded fixture covers the other case)."""
    import pytest
    import torch

    tv = pytest.importorskip("torchvision.transforms")
    Image = pytest.importorskip("PIL.Image")
    from oracle import marl_oracle as O

    g = torch.Generator().manual_seed(11)
    u8 = torch.randint(0, 256, (3, 13, 10, 3), dtype=torch.uint8, generator=g)
    ref = torch.stack([tv.ToTensor()(Image.fromarray(u8[i].numpy())) for i in range(3)])
    assert torch.equal(O.to_tensor_batch(u8), ref)


def test_bench_reference_arm_runs_without_a_gpu():
    """`bench.py --impl reference` times the CPU port and prints the contract's JSON line; every
    other rank of a multi-process launch exits 0 without output."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "image_episodes_per_sec" and line["value"] > 0
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_fastdiv_reciprocal_division_is_exact_within_its_bound():
    """The element-wise kernels (gather, CNN backward, im2col) index with multiply-high by a
    host-computed reciprocal; the library's host twin of that code must agree with `/` for every
    divisor up to 4096 over the whole range the launchers admit (n * d < 2^32)."""
    assert _lib.lib().marlc_selftest_fastdiv(4096, 9973) == 0
    assert _lib.lib().marlc_selftest_fastdiv(64, 1 << 12) == 0


@pytest.mark.parametrize("name", ["conftest_odd", "resisc_small", "aid_small", "single_agent"])
def test_same_seed_gives_the_reference_initialisation(name):
    """Drop-in property of construction (init.py:6-29, models.py:30-76): under the same
    ``torch.manual_seed`` our ModelsWrapper consumes the RNG exactly like the reference's, so a run
    started from a seed begins from bit-identical weights.  The fixture's ``state_dict`` is the
    reference's ``build_marl`` under the case's seed plus a perturbation drawn from a separate seeded
    generator (oracle/make_golden.py ``run_case``); the same recipe on our side must give it bit for bit."""
    from oracle.make_golden import CASES

    fx = load_golden(name)
    seed = CASES[name]["seed"]
    torch.manual_seed(seed)
    model, _, _ = ModelConfig(**fx["model_config"]).build_marl(fx["na"])
    g = torch.Generator().manual_seed(seed + 1000)
    with torch.no_grad():
        for prm in model.parameters():
            prm.add_(0.1 * torch.randn(prm.shape, generator=g))
    ours = model.state_dict()
    assert list(ours) == list(fx["state_dict"])
    for k, ref in fx["state_dict"].items():
        assert torch.equal(ours[k], ref), k


def test_every_environment_switch_is_documented():
    """Every MARLC_* variable the library or the Python package reads is listed in INTEGRATION.md section 3, and
    every MARLC_* name in the first column of that table is still read by the code or tested by an #ifdef in csrc/."""
    import glob
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names, macros = set(), set()
    for path in glob.glob(os.path.join(root, "marlclassification_b200", "csrc", "*.cu*")):
        src = open(path).read()
        names |= set(re.findall(r'getenv\("(MARLC_[A-Z0-9_]+)"\)', src))
        macros |= set(re.findall(r"#\s*ifn?def\s+(MARLC_[A-Z0-9_]+)", src))
        macros |= set(re.findall(r"defined\s*\(?\s*(MARLC_[A-Z0-9_]+)", src))
    for path in glob.glob(os.path.join(root, "marlclassification_b200", "**", "*.py"), recursive=True) + [os.path.join(root, "bench.py")]:
        names |= set(re.findall(r'environ(?:\.get)?[\(\[]"(MARLC_[A-Z0-9_]+)"', open(path).read()))
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    missing = sorted(n for n in names if n not in doc)
    assert names and not missing, f"undocumented switches: {missing}"
    section = re.search(r"^## 3\..*?$(.*?)(?=^## |\Z)", doc, re.M | re.S)
    assert section, "INTEGRATION.md has no section 3"
    listed = set()
    for line in section.group(1).splitlines():
        if line.startswith("|"):
            listed |= set(re.findall(r"MARLC_[A-Z0-9_]+", line.split("|")[1]))
    assert listed, "no switches parsed from INTEGRATION.md section 3"
    stale = sorted(listed - names - macros)
    assert not stale, f"documented switches the code no longer reads: {stale}"
