"""GPU: bench.py times exactly --steps steps, and --dump-outputs writes what the last timed step returned -- the same
files on every run with the same arguments, equal to the outputs of the same step sequence replayed here, within the
64 MB budget (a fixed sample of instances when the batch is larger)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

NAMES = ("current_state", "next_state", "policy_state", "reward", "is_terminal", "terminal_flag", "time", "instance_index")
N, WARMUP, STEPS, BLOCKS = 65536, 3, 7, [2, 2, 1, 1, 1]


def _bench(out):
    # ugvo at 65,536 instances: 1 kB of outputs per instance, so the dump has to sample
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(STEPS), "--warmup", str(WARMUP),
           "--workload", "ugvo", "--envs", str(N), "--no-extras", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _replayed():
    """The step sequence of bench.py on its own inputs: the warm-up steps, then the timed blocks, every block after the
    first preceded by one untimed step.  Returns the env after the last timed step."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    dev = torch.device("cuda", 0)
    env = bench.make_env("ugvo", N, dev, 0)
    env.reset(True)
    pool = bench.action_pool(env, N, 4, dev, torch.float64, seed=1)
    for r, k in enumerate(BLOCKS):
        w = WARMUP if r == 0 else 1
        for j in range(w + k):
            env.step_soa(pool[j % pool.shape[0]])
    torch.cuda.synchronize()
    return env


def test_bench_times_the_given_steps_and_dumps_the_same_outputs_every_run(tmp_path):
    lines = [_bench(tmp_path / f"run{k}") for k in range(2)]
    for line in lines:
        assert line["steps"] == STEPS and line["gpu_launches"] == STEPS
        assert line["repeats"]["steps_per_block"] == BLOCKS
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        assert sorted(os.listdir(d)) == sorted(f"{n}.npy" for n in NAMES)
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64_000_000
        dumps.append({n: np.load(d / f"{n}.npy") for n in NAMES})
    a, b = dumps
    idx = a["instance_index"]
    assert 0 < idx.size < N and np.all(np.diff(idx) > 0) and idx[-1] < N
    for n in NAMES:
        assert a[n].dtype in (np.float32, np.float64), n
        assert a[n].shape[0] == idx.size, n
        assert np.array_equal(a[n], b[n]), n
    assert a["next_state"].shape[1] == 41
    assert np.all(np.isfinite(a["next_state"])) and np.any(a["time"] > 0)
    env = _replayed()
    sel = idx.astype(np.int64)
    for n in NAMES[:-1]:
        want = getattr(env, n).cpu().numpy()[sel]
        assert np.array_equal(a[n], want.astype(a[n].dtype)), n
