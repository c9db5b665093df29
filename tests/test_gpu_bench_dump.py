"""`bench.py --dump-outputs`: the files hold what the last of the `--steps` timed steps returned, the same on every run
with the same arguments, and equal to the oracle replaying the bench's own inputs for warm-up + timed steps."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import OracleMapfGym

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = {"status": np.float32, "reward": np.float32, "cost": np.float32, "train_valid": np.float32,
          "goals_reached": np.float32, "violated": np.float32, "shadow_goals": np.float64, "fixed_actions": np.float32,
          "obs": np.float32, "vec": np.float32}


def test_gpu_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    W, K, WU = 1024, 4, 3
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(WU),
                            "--worlds", str(W), "--no-extras", "--cpu-budget", "0", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in DTYPES)
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
        dumps.append({n: np.load(d / (n + ".npy")) for n in DTYPES})
    for n, dt in DTYPES.items():
        assert dumps[0][n].dtype == dt, n
        np.testing.assert_array_equal(dumps[0][n], dumps[1][n], err_msg=f"{n} differs between two runs")

    sys.path.insert(0, ROOT)
    import bench
    sc, ring = bench.bench_inputs(W, torch.device("cuda", 0), rank=0)
    orc = OracleMapfGym(sc, seed=1234, threads=8, use_tape=False)
    for i in list(range(WU)) + list(range(K)):
        ref = orc.step_observe(ring[i % 8].cpu().numpy())
    idx = np.sort(np.random.default_rng(0).choice(W, size=bench.DUMP_WORLDS, replace=False))
    for n, key in (("status", "status"), ("reward", "reward"), ("cost", "cost"), ("train_valid", "train_valid"),
                   ("goals_reached", "goals_reached"), ("violated", "violated"), ("shadow_goals", "shadow"),
                   ("fixed_actions", "fixed"), ("obs", "obs"), ("vec", "vec")):
        np.testing.assert_array_equal(dumps[0][n], ref[key][idx].astype(DTYPES[n]), err_msg=n)
