"""On-device goal sampling (SURVEY §8 f1): the oracle's restatement of `MapfGym.getNextGoal` at arrival
(mapf_gym.py:189-190, 623-627 -> util.getFreeCell, util.py:67-76 on worldWithAgentsAndGoals(), :200-209).

The CUDA path is held bit-exact to this restatement (same Philox stream; tests/test_gpu_round2.py).  Here, on the CPU:
properties of the restatement — the reference draws from NumPy's global MT19937, so only the distribution can agree."""
import numpy as np

from oracle import OracleMapfGym
from oracle.oracle import checksum_rows
from primal_ppo_b200.scenario import Scenario


def _one_world_many_times(W, seed=0):
    """W copies of one 10x10 world with 3 agents; agent 0 stands next to its goal."""
    rng = np.random.default_rng(seed)
    H = Wd = 10
    ob = (rng.random((H, Wd)) < 0.2).astype(np.uint8)
    for c in ((1, 1), (1, 2), (5, 5), (8, 8), (2, 7), (7, 2), (0, 0), (0, 1)):
        ob[c] = 0
    starts = np.array([[1, 1], [5, 5], [8, 8]], dtype=np.int16)
    goals = np.array([[[1, 2]], [[2, 7]], [[7, 2]]], dtype=np.int16)            # Q = 1: only the first goal comes from the queue
    htrace = np.array([[0, 0, 0, 1], [0, 1, 0, 1]], dtype=np.int16)
    rep = lambda a: np.ascontiguousarray(np.broadcast_to(a[None], (W,) + a.shape))
    sc = Scenario(obst=rep(ob), starts=rep(starts), goal_queue=rep(goals), htrace=rep(htrace),
                  hlen=np.full((W,), 2, dtype=np.int32))
    return sc, ob, starts, goals


def _expected_free(ob, pos, goal):
    free = ob == 0
    for p in pos:
        free[tuple(p)] = False
    for g in goal:
        free[tuple(g)] = False
    return free


def test_oracle_goal_sampling_draws_free_cells_only_and_all_of_them():
    W = 20000
    sc, ob, starts, goals = _one_world_many_times(W)
    orc = OracleMapfGym(sc, seed=5, threads=4, use_tape=False, goal_sampling=True)
    a = np.zeros((W, 3), dtype=np.int8)
    a[:, 0] = 1                                             # agent 0 steps east onto its goal
    out = orc.step(a)
    assert out["goals_reached"][:, 0].all() and not out["goals_reached"][:, 1:].any()
    s = orc.state()
    assert not s["err"].any()
    np.testing.assert_array_equal(s["goal"][:, 1:], np.broadcast_to(goals[None, 1:, 0], (W, 2, 2)))   # others keep theirs
    # world at the moment agent 0 samples: agent 0 has moved to (1,2); agents 1, 2 have not moved yet (they stay anyway)
    pos = np.array([[1, 2], [5, 5], [8, 8]])
    free = _expected_free(ob.copy(), pos, goals[:, 0])
    g = s["goal"][:, 0].astype(np.int64)
    assert free[g[:, 0], g[:, 1]].all(), "a sampled goal is never an obstacle, an agent's cell or a goal"
    hist = np.zeros((10, 10), dtype=np.int64)
    np.add.at(hist, (g[:, 0], g[:, 1]), 1)
    assert (hist[free] > 0).all(), "every free cell is reachable by the sampler"
    n = int(free.sum())
    chi2 = float((((hist[free] - W / n) ** 2) / (W / n)).sum())
    assert chi2 < n + 6 * np.sqrt(2 * n), (chi2, n)          # uniform over the free cells (chi-square, ~6 sigma)
    # the same worlds with different world_offset / seed give different draws; same key gives the same bits
    o2 = OracleMapfGym(sc, seed=5, threads=2, use_tape=False, goal_sampling=True)
    o2.step(a)
    np.testing.assert_array_equal(o2.state()["goal"], s["goal"])
    o3 = OracleMapfGym(sc, seed=6, threads=2, use_tape=False, goal_sampling=True)
    o3.step(a)
    assert (o3.state()["goal"][:, 0] != s["goal"][:, 0]).any()


def test_oracle_goal_sampling_sequential_occupancy():
    """Two agents arrive in the same step: the second one's draw sees the first one's NEW goal as taken and the first
    one's new cell as occupied (jointStep's loop is sequential, mapf_gym.py:620-627)."""
    W = 4000
    H = Wd = 3
    ob = np.zeros((H, Wd), dtype=np.uint8)
    ob[2, :] = 1                                            # 6 free cells
    starts = np.array([[0, 0], [1, 2]], dtype=np.int16)
    goals = np.array([[[0, 1]], [[1, 1]]], dtype=np.int16)
    htrace = np.array([[2, 2, 2, 2]], dtype=np.int16)       # the human is parked on a shelf cell
    rep = lambda a: np.ascontiguousarray(np.broadcast_to(a[None], (W,) + a.shape))
    sc = Scenario(obst=rep(ob), starts=rep(starts), goal_queue=rep(goals), htrace=rep(htrace), hlen=np.ones((W,), np.int32))
    orc = OracleMapfGym(sc, seed=11, threads=2, use_tape=False, goal_sampling=True)
    a = np.tile(np.array([[1, 3]], dtype=np.int8), (W, 1))  # 0: east onto (0,1); 1: west onto (1,1)
    out = orc.step(a)
    assert out["goals_reached"].all()
    g = orc.state()["goal"]
    # agent 0 samples with agent 1 still at (1,2): free = {(0,0) left behind? no: agent 0 is at (0,1) now} ...
    free0 = {(0, 0), (0, 2), (1, 0)}                        # not (0,1) [own cell/goal], (1,2) [agent 1], (1,1) [goal 1]
    assert set(map(tuple, g[:, 0].tolist())) == free0
    for w in range(0, W, 97):
        g0 = tuple(g[w, 0])
        free1 = {(0, 0), (0, 2), (1, 0), (1, 2)} - {g0}     # agent 1 is at (1,1) now; (0,1) agent 0; g0 is agent 0's new goal
        assert tuple(g[w, 1]) in free1


def test_oracle_checksum_is_position_sensitive():
    a = np.arange(64, dtype=np.uint32).reshape(2, 32)
    b = a.copy()
    b[0, [3, 4]] = b[0, [4, 3]]
    s1, s2 = checksum_rows(a), checksum_rows(b)
    assert s1[0] != s2[0] and s1[1] == s2[1]
    z = np.zeros((3, 8), dtype=np.float32)
    assert len(set(checksum_rows(z).tolist())) == 1 and checksum_rows(z)[0] != 0


def test_packed_results_decoder_matches_oracle_outputs():
    """mapf_decode_results_host (a HOST function of the C-ABI library; no GPU involved) on words packed from the oracle's
    outputs per the MAPF_PACKED_* definition: every decoded array equals the oracle's, bit for bit — in particular
    reward = base(status) (+1.5 on arrival) and cost = f(d2) are reproduced from the 16-bit record."""
    import torch
    from primal_ppo_b200 import decode_results, random_actions, random_scenario
    sc = random_scenario(64, 12, 12, 8, density=(0.1, 0.3), queue_len=3, seed=4)
    orc = OracleMapfGym(sc, threads=2, use_tape=False)
    acts = random_actions(24, 64, 8, seed=1)
    DR, DC = np.array([0, 0, 1, 0, -1]), np.array([0, 1, 0, -1, 0])
    code = {-1: 0, -2: 1, -3: 2, -4: 3, 1: 4}
    for t in range(24):
        pos = orc.state()["pos"].astype(np.int64)
        tick = t % sc.hlen
        nxt = sc.htrace[np.arange(64), tick, 2:].astype(np.int64)
        out = orc.step(acts[t])
        a = acts[t].astype(np.int64)
        tr, tc = pos[..., 0] + DR[a], pos[..., 1] + DC[a]
        d2 = np.minimum((nxt[:, None, 0] - tr) ** 2 + (nxt[:, None, 1] - tc) ** 2, 25)
        sc_ = np.vectorize(code.get)(out["status"].astype(np.int64))
        packed = (sc_ | (out["goals_reached"].astype(np.int64) << 3) | (out["violated"].astype(np.int64) << 4) |
                  (out["fixed"].astype(np.int64) << 5) | (d2 << 8)).astype(np.uint16)
        dec = decode_results(torch.from_numpy(packed.view(np.int16)))
        np.testing.assert_array_equal(dec["status"].numpy(), out["status"])
        np.testing.assert_array_equal(dec["reward"].numpy().view(np.uint32), out["reward"].view(np.uint32))
        np.testing.assert_array_equal(dec["cost"].numpy().view(np.uint32), out["cost"].view(np.uint32))
        np.testing.assert_array_equal(dec["goals_reached"].numpy(), out["goals_reached"])
        np.testing.assert_array_equal(dec["violated"].numpy(), out["violated"])
        np.testing.assert_array_equal(dec["fixed_actions"].numpy(), out["fixed"])
