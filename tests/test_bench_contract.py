"""bench.py's contract: the reference arm prints exactly one JSON line with the agreed keys (under torchrun only rank 0 prints), our arm refuses to run
without a CUDA device instead of falling back to the CPU, and --dump-outputs writes the last timed step's results from identical inputs on every run
(on a GPU: our arm's dump agrees with the reference arm's)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)


def test_reference_arm_prints_one_json_line_with_the_contract_keys(libs):
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--bodies", "3000", "--substeps", "2", "--iterations", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["steps"] == 2 and line["warmup"] == 1 and line["higher_is_better"] is True
    assert line["metric"].startswith("constraint-iterations/sec") and line["unit"] == "constraint-iterations/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "3000 bodies" in line["config"]["workload"] and line["config"]["substeps"] == 2


def test_reference_arm_is_silent_on_ranks_other_than_zero(libs):
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--bodies", "500", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


DUMP_NAMES = ("accumulated_impulses", "body_poses", "body_velocities", "body_world_inverse_inertias")
SMALL = ["--bodies", "2000", "--substeps", "2", "--iterations", "2", "--steps", "2", "--warmup", "3"]


def _dump(args, directory):
    r = _run(args + ["--dump-outputs", str(directory)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(directory)) == sorted(n + ".npy" for n in DUMP_NAMES)
    out = {n: np.load(os.path.join(directory, n + ".npy")) for n in DUMP_NAMES}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def test_reference_arm_dumps_the_same_outputs_on_every_run(libs, tmp_path):
    a = _dump(["--impl", "reference"] + SMALL, tmp_path / "a")
    b = _dump(["--impl", "reference"] + SMALL, tmp_path / "b")
    assert a["body_poses"].shape == (2000, 7) and a["body_velocities"].shape == (2000, 6) and a["body_world_inverse_inertias"].shape == (2000, 14)
    assert a["accumulated_impulses"].size > 2000 and np.abs(a["accumulated_impulses"]).max() > 0
    for n in DUMP_NAMES:
        assert np.array_equal(a[n], b[n]), n


@pytest.mark.gpu
def test_our_arm_dumps_what_the_reference_arm_computes(libs, tmp_path):
    """Same arguments, same number of solves (warm-up 3 + 2 timed steps) on both arms: the strict build's last step agrees with the oracle's within fp32 tolerance."""
    ours = _dump(SMALL + ["--strict", "--no-configs", "--no-cpu-baseline"], tmp_path / "ours")
    ref = _dump(["--impl", "reference"] + SMALL, tmp_path / "reference")
    for n in DUMP_NAMES:
        assert ours[n].shape == ref[n].shape, n
        d = np.abs(ours[n].astype(np.float64) - ref[n].astype(np.float64))
        assert np.sqrt((d ** 2).sum() / max((ref[n].astype(np.float64) ** 2).sum(), 1e-30)) <= 1e-3 and d.max() <= 5e-2, n


def test_our_arm_has_no_cpu_fallback(libs):
    import torch

    if torch.cuda.is_available():
        return  # on a GPU box the -m gpu suite and the bench itself cover this arm
    r = _run(["--steps", "1", "--warmup", "1", "--bodies", "500"])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
