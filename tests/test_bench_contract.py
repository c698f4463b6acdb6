"""bench.py's reference arm runs on the CPU, so its JSON contract can be checked without a GPU; the GPU arm's
--dump-outputs is checked on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "3", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "80 pyramids x 20 levels" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dumped_outputs_are_the_states_after_the_last_timed_step(built, tmp_path):
    """--dump-outputs writes the body states each timed scene holds after warm-up + --steps timed steps, bit for bit
    what a PhysicsWorld stepped as many times returns."""
    from rapier_b200 import scenes
    from rapier_b200.world import PhysicsWorld
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4", "--warmup", "3",
                        "--cpu-seconds", "0.1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 4
    for name, scene in (("b3d_many_pyramids_80x20", scenes.pyramids(8, 10, 20)), ("b3d_many_pyramids", scenes.pyramids(14, 14, 10))):
        w = PhysicsWorld(scene)
        for _ in range(3 + 4):
            w.step()
        for part, want in zip(("pose", "vel"), w.body_states()):
            got = np.load(tmp_path / f"{name}_{part}.npy")
            assert got.dtype == np.float32 and got.shape == want.shape, (name, part, got.dtype, got.shape)
            assert (got.view(np.uint32) == want.view(np.uint32)).all(), (name, part)
