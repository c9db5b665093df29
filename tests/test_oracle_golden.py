"""Pins the C oracle (oracle/mapf_oracle.c) bit-for-bit against traces of the UNMODIFIED reference
(tests/golden/*.npz, produced by tests/golden/make_golden.py running /root/reference/mapf_gym.py).
Integer / byte outputs and f32 outputs are all compared with exact equality."""
import numpy as np
import pytest

from golden_util import ENV_CASES, Golden
from oracle import OracleMapfGym, gae_oracle


def _check_oracle_against(g, case):
    env = OracleMapfGym(g.scenario, threads=2)
    s0 = env.state()
    np.testing.assert_array_equal(s0["pos"], g["pos"][0])
    np.testing.assert_array_equal(s0["goal"], g["goal"][0])
    obs, vec = env.getAllObservations()
    np.testing.assert_array_equal(obs, g.obs[0].astype(np.float32))
    np.testing.assert_array_equal(vec.view(np.uint32), g["vec"][0].view(np.uint32))
    np.testing.assert_array_equal(env.bfs_maps()[:len(g["bfs0"])], g["bfs0"])
    for t in range(g.T):
        out = env.step(g["actions"][t])
        for key, ref in (("status", "status"), ("goals_reached", "goals_reached"), ("violated", "violated"),
                         ("shadow", "shadow"), ("fixed", "fixed")):
            np.testing.assert_array_equal(out[key], g[ref][t], err_msg=f"{case} t={t} {key}")
        for key in ("reward", "cost", "train_valid"):
            np.testing.assert_array_equal(out[key].view(np.uint32), g[key][t].view(np.uint32),
                                          err_msg=f"{case} t={t} {key}")
        s = env.state()
        assert not s["err"].any(), (case, t, s["err"])
        np.testing.assert_array_equal(s["pos"], g["pos"][t + 1], err_msg=f"{case} t={t} pos")
        np.testing.assert_array_equal(s["goal"], g["goal"][t + 1], err_msg=f"{case} t={t} goal")
        obs, vec = env.getAllObservations()
        np.testing.assert_array_equal(obs, g.obs[t + 1].astype(np.float32), err_msg=f"{case} t={t} obs")
        np.testing.assert_array_equal(vec.view(np.uint32), g["vec"][t + 1].view(np.uint32), err_msg=f"{case} t={t} vec")
    np.testing.assert_array_equal(env.bfs_maps()[:len(g["bfsT"])], g["bfsT"])


@pytest.mark.parametrize("case", ENV_CASES)
def test_oracle_matches_reference_trace(case):
    _check_oracle_against(Golden(case), case)


def test_oracle_gae_matches_reference_runner():
    import os
    from golden_util import GOLDEN_DIR
    d = np.load(os.path.join(GOLDEN_DIR, "gae_runner.npz"))
    ret, _ = gae_oracle(d["rewards"], d["values"], d["last_values"], float(d["gamma"]), float(d["lam"]))
    np.testing.assert_array_equal(ret.view(np.uint32), d["returns"].view(np.uint32))
    cret, _ = gae_oracle(d["cost_rewards"], d["cost_values"], d["last_cost_values"], float(d["gamma"]), float(d["lam"]))
    np.testing.assert_array_equal(cret.view(np.uint32), d["cost_returns"].view(np.uint32))


def test_oracle_fused_step_observe_equals_separate_calls():
    g = Golden("g_8x8_n8_dense")
    e1, e2 = OracleMapfGym(g.scenario, threads=2), OracleMapfGym(g.scenario, threads=3)
    for t in range(g.T):
        a = e1.step(g["actions"][t])
        o1, v1 = e1.getAllObservations()
        b = e2.step_observe(g["actions"][t])
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow", "fixed"):
            np.testing.assert_array_equal(a[key], b[key], err_msg=f"t={t} {key}")
        np.testing.assert_array_equal(o1, b["obs"])
        np.testing.assert_array_equal(v1.view(np.uint32), b["vec"].view(np.uint32))
