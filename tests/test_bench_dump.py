"""bench.py --dump-outputs: what every workload's timed path returned in its last step, float32 / float64 only, identical from
run to run with the same arguments (seeded inputs), so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import philox  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS, WARMUP, FUSE, ENVS = 2, 3, 8, 65536
SMALL = ["--steps", str(STEPS), "--warmup", str(WARMUP), "--fuse", str(FUSE), "--envs-per-gpu", str(ENVS), "--ppo-envs", "4096",
         "--no-cpu", "--no-e2e", "--sustain-s", "0"]


def _bench(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *SMALL, "--dump-outputs", str(out)],
                       stdout=subprocess.PIPE, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_of_the_last_timed_step_are_reproducible(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    lines = [_bench(tmp_path / f"run{i}") for i in range(2)]
    assert lines[0]["steps"] == STEPS and all(w["steps"] == STEPS for w in lines[0]["workloads"].values())
    files = sorted(os.listdir(tmp_path / "run0"))
    assert files == sorted(os.listdir(tmp_path / "run1"))
    assert {f"{wl}_{k}.npy" for wl in ("c4", "c2", "c3", "c5") for k in ("env_index", "reward", "done")} <= set(files)
    assert "c5_params.npy" in files
    total = 0
    for f in files:
        a, b = np.load(tmp_path / "run0" / f), np.load(tmp_path / "run1" / f)
        assert a.dtype in (np.float32, np.float64), f
        assert np.array_equal(a, b, equal_nan=True), f
        total += a.nbytes
    assert total <= 64 << 20
    # c4: a fixed sample of env columns; its random-policy actions are the Philox draws of the LAST timed launch
    d = tmp_path / "run0"
    idx = np.load(d / "c4_env_index.npy")
    assert 0 < idx.size < ENVS and np.load(d / "c4_next_obs.npy").shape == (FUSE, idx.size, 15)
    acts, t0 = np.load(d / "c4_actions.npy"), (WARMUP + STEPS - 1) * FUSE
    for k in range(FUSE):
        want = philox.action_uniforms(0, idx.astype(np.uint64), t0 + k).astype(np.float32) * np.float32(7.3575)
        assert np.array_equal(acts[k], want), k
