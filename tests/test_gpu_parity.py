"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI, against
  (1) the reference-generated golden traces (tests/golden/*.npz) and
  (2) the C oracle on seeded synthetic scenarios at sizes the oracle finishes in seconds,
plus size-independent properties at BASELINE.json's full size.
Bar: bit-exact for every integer / byte output AND for every f32 output (rewards, cost, trainValid, obs, vec, GAE)."""
import numpy as np
import pytest
import torch

from golden_util import ENV_CASES, GOLDEN_DIR, Golden
from oracle import OracleMapfGym, gae_oracle
from ppo_loss_ref import gae_masked_ref
from primal_ppo_b200 import random_actions, random_scenario

pytestmark = pytest.mark.gpu


def _env(sc, **kw):
    from primal_ppo_b200 import BatchedMapfGym
    return BatchedMapfGym(sc, **kw)


def _np(t):
    return t.detach().cpu().numpy()


def _eq(a, b, msg):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.float32:
        a, b = a.view(np.uint32), np.asarray(b, dtype=np.float32).view(np.uint32)
    np.testing.assert_array_equal(a, b, err_msg=msg)


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("case", ENV_CASES)
def test_gpu_matches_reference_trace(case, fused):
    g = Golden(case)
    env = _env(g.scenario)
    s = env.state()
    _eq(_np(s["pos"]), g["pos"][0], "pos0")
    _eq(_np(s["goal"]), g["goal"][0], "goal0")
    obs, vec = env.getAllObservations()
    _eq(_np(obs), g.obs[0].astype(np.float32), "obs0")
    _eq(_np(vec), g["vec"][0], "vec0")
    _eq(_np(env.bfs_maps())[:len(g["bfs0"])], g["bfs0"], "bfs0")
    for t in range(g.T):
        if fused:
            out, obs, vec = env.step_observe(torch.from_numpy(g["actions"][t]))
        else:
            out = env.step(torch.from_numpy(g["actions"][t]))
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated"):
            _eq(_np(getattr(out, key)), g[key][t], f"{case} t={t} {key}")
        _eq(_np(out.shadow_goals), g["shadow"][t], f"{case} t={t} shadow")
        _eq(_np(out.fixed_actions), g["fixed"][t], f"{case} t={t} fixed")
        s = env.state()
        assert not _np(s["err"]).any(), (case, t)
        _eq(_np(s["pos"]), g["pos"][t + 1], f"{case} t={t} pos")
        _eq(_np(s["goal"]), g["goal"][t + 1], f"{case} t={t} goal")
        if not fused:
            obs, vec = env.getAllObservations()
        _eq(_np(obs), g.obs[t + 1].astype(np.float32), f"{case} t={t} obs")
        _eq(_np(vec), g["vec"][t + 1], f"{case} t={t} vec")
    _eq(_np(env.bfs_maps())[:len(g["bfsT"])], g["bfsT"], "bfsT")


@pytest.mark.parametrize("case", ["g_10x10_n8", "g_8x8_n8_dense"])
def test_gpu_five_call_api_matches_reference_trace(case):
    """The reference's own call order (runner.py:64-91) through the split entry points."""
    g = Golden(case)
    env = _env(g.scenario)
    for t in range(g.T):
        a = torch.from_numpy(g["actions"][t]).cuda()
        st = env.getActionStatus(a)
        rw, sg = env.calculateActionReward(a, st)
        cost = env.calculateCostReward(a)
        tv = env.getTrainValid(a)
        _eq(_np(st), g["status"][t], f"t={t} status")
        _eq(_np(cost), g["cost"][t], f"t={t} cost")
        _eq(_np(tv), g["train_valid"][t], f"t={t} tv")
        _eq(_np(sg), g["shadow"][t], f"t={t} shadow")
        rw = rw.clone()
        gr, cv = env.jointStep(a, st)
        rw[gr == 1] += 1.5
        _eq(_np(rw), g["reward"][t], f"t={t} reward")
        _eq(_np(gr), g["goals_reached"][t], f"t={t} goals")
        _eq(_np(cv), g["violated"][t], f"t={t} violated")
        _eq(_np(env.state()["pos"]), g["pos"][t + 1], f"t={t} pos")


def _run_vs_oracle(sc, T, seed=1234, check_obs_every=1, threads=8, fused=False):
    orc = OracleMapfGym(sc, seed=seed, threads=threads, use_tape=False)
    env = _env(sc, seed=seed, use_tape=False)
    acts = random_actions(T, sc.num_worlds, sc.num_agents, seed=seed)
    o_obs, o_vec = orc.getAllObservations()
    obs, vec = env.getAllObservations()
    assert torch.equal(obs, torch.from_numpy(o_obs).cuda()) and torch.equal(vec, torch.from_numpy(o_vec).cuda())
    for t in range(T):
        ref = orc.step(acts[t])
        if fused:       # mapf_step_observe: one launch for the step and the observations of the new state
            out, obs, vec = env.step_observe(torch.from_numpy(acts[t]))
        else:
            out = env.step(torch.from_numpy(acts[t]))
        # worlds where the reference would have hung or raised carry an error flag; since round 2 every agent of such a world
        # stays for that step, the world remains valid, and it is compared like any other
        ok_w = np.ones_like(orc.state()["err"], dtype=bool)
        e_gpu = _np(env.state()["err"]).astype(np.uint32)
        np.testing.assert_array_equal(e_gpu, orc.state()["err"], err_msg=f"t={t} err flags")
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated"):
            _eq(_np(getattr(out, key))[ok_w], ref[key][ok_w], f"t={t} {key}")
        _eq(_np(out.shadow_goals)[ok_w], ref["shadow"][ok_w], f"t={t} shadow")
        _eq(_np(out.fixed_actions)[ok_w], ref["fixed"][ok_w], f"t={t} fixed")
        s, so = env.state(), orc.state()
        _eq(_np(s["pos"])[ok_w], so["pos"][ok_w], f"t={t} pos")
        _eq(_np(s["goal"])[ok_w], so["goal"][ok_w], f"t={t} goal")
        _eq(_np(s["rep"])[ok_w], so["rep"][ok_w], f"t={t} rep")
        if t % check_obs_every == 0 or t == T - 1:
            o_obs, o_vec = orc.getAllObservations(out=(o_obs, o_vec))
            if not fused:
                obs, vec = env.getAllObservations()
            okd = torch.from_numpy(ok_w).cuda()
            assert torch.equal(obs[okd], torch.from_numpy(o_obs).cuda()[okd]), f"t={t} obs"
            assert torch.equal(vec[okd], torch.from_numpy(o_vec).cuda()[okd]), f"t={t} vec"
    _eq(_np(env.bfs_maps())[ok_w], orc.bfs_maps()[ok_w], "bfs")
    return env, orc


def test_gpu_matches_oracle_config2_4096x20x20x8():
    """BASELINE.json configs[1]: 4096 worlds 20x20, 8 agents, replayed actions, bit-exact step+obs."""
    sc = random_scenario(4096, 20, 20, 8, density=(0.2, 0.2), queue_len=8, seed=11, unique_maps=256)
    env, orc = _run_vs_oracle(sc, T=64, check_obs_every=4)
    # counters accumulated on device equal the sums over the trace (util.py:56-65)
    assert int(env.counters()[:, 0].sum()) > 0


def test_gpu_matches_oracle_config3_shape_40x40x32():
    sc = random_scenario(768, 40, 40, 32, density=(0.0, 0.3), queue_len=8, seed=12, unique_maps=96)
    _run_vs_oracle(sc, T=32, check_obs_every=4)


@pytest.mark.parametrize("shape", [(1024, 40, 40, 32, 6), (512, 20, 20, 8, 6), (300, 8, 8, 8, 5), (64, 33, 65, 5, 6),
                                   (40, 64, 64, 31, 6), (7, 7, 11, 1, 6), (5, 96, 80, 12, 6), (3, 128, 128, 32, 5)])
def test_gpu_fused_step_observe_matches_oracle(shape):
    """mapf_step_observe (the fused launch) against the oracle, every step, incl. crowded worlds and odd shapes."""
    W, H, Wd, N, C = shape
    dens = (0.2, 0.3) if H == 8 else (0.0, 0.3)
    sc = random_scenario(W, H, Wd, N, density=dens, queue_len=4, seed=W + N, num_channel=C, unique_maps=min(W, 64))
    _run_vs_oracle(sc, T=24, fused=True)


def test_gpu_fused_step_observe_equals_two_calls_and_falls_back():
    """Same bits from the fused launch and from step + getAllObservations; shapes the fused kernel does not cover
    (N > 32, FOV 31 with 32 agents) go through the two kernels behind the same entry point."""
    for (W, H, N, fov) in ((2048, 40, 32, 9), (16, 40, 32, 31), (12, 48, 48, 9), (64, 20, 8, 15)):
        sc = random_scenario(W, H, H, N, density=(0.0, 0.3), queue_len=4, seed=fov + N, fov=fov, unique_maps=min(W, 32))
        a = torch.from_numpy(random_actions(12, W, N, seed=4)).cuda()
        e1, e2 = _env(sc, use_tape=False), _env(sc, use_tape=False)
        for t in range(12):
            o1 = e1.step(a[t]); obs1, vec1 = e1.getAllObservations()
            o2, obs2, vec2 = e2.step_observe(a[t])
            for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow_goals",
                        "fixed_actions"):
                assert torch.equal(getattr(o1, key), getattr(o2, key)), (W, H, N, fov, t, key)
            assert torch.equal(obs1, obs2) and torch.equal(vec1, vec2), (W, H, N, fov, t)
        s1, s2 = e1.state(), e2.state()
        assert all(torch.equal(s1[k], s2[k]) for k in s1)
        assert torch.equal(e1.counters(), e2.counters())


def test_gpu_matches_oracle_crowded_fixactions_philox():
    """8x8, 8 agents, density up to 0.3: fixActions branch 3 (Philox stand-in) and error flags agree."""
    sc = random_scenario(2048, 8, 8, 8, density=(0.2, 0.3), queue_len=6, seed=13, unique_maps=256)
    _run_vs_oracle(sc, T=48)


@pytest.mark.parametrize("shape", [(1, 7, 11, 1), (3, 12, 9, 6), (13, 10, 10, 2), (9, 33, 65, 5), (5, 64, 64, 31),
                                   (4, 80, 80, 8), (3, 128, 128, 16), (6, 65, 64, 32)])
def test_gpu_matches_oracle_ragged_shapes(shape):
    W, H, Wd, N = shape
    sc = random_scenario(W, H, Wd, N, density=(0.05, 0.2), queue_len=3, seed=W * 7 + N, num_channel=5 if N == 6 else 6)
    _run_vs_oracle(sc, T=24)


def test_gpu_eval_channels_and_large_fov_observe_only():
    """use_da / use_hp channels and a FOV sweep; N = 128 agents (observe and BFS only: config 5 shape)."""
    for fov in (9, 15, 21, 31):
        sc = random_scenario(6, 80, 80, 128, density=(0.0, 0.3), queue_len=2, seed=fov, fov=fov, use_da=True, use_hp=True)
        orc = OracleMapfGym(sc, threads=8, use_tape=False)
        env = _env(sc, use_tape=False)
        o_obs, o_vec = orc.getAllObservations()
        obs, vec = env.getAllObservations()
        assert torch.equal(obs, torch.from_numpy(o_obs).cuda()), fov
        assert torch.equal(vec, torch.from_numpy(o_vec).cuda()), fov
        if fov == 9:
            _eq(_np(env.bfs_maps()), orc.bfs_maps(), "bfs 80x80")


def test_gpu_matches_oracle_config5_shape_80x80x128():
    """BASELINE.json configs[4] shape: 80x80 worlds, 128 agents (the lane-loops-over-agents step kernel)."""
    sc = random_scenario(48, 80, 80, 128, density=(0.0, 0.3), queue_len=4, seed=51, unique_maps=12)
    _run_vs_oracle(sc, T=24, check_obs_every=4)
    sc = random_scenario(64, 16, 16, 48, density=(0.1, 0.25), queue_len=4, seed=52, unique_maps=16)   # crowded, N = 48
    _run_vs_oracle(sc, T=32, check_obs_every=4)


def test_gpu_maximum_sizes_and_empty_inputs():
    """The limits include/mapf_b200.h states: 128x128 cells, 128 agents for the joint step, 254 for observe / BFS;
    empty work lists are accepted; sizes beyond the limits are refused with an error code, not a crash."""
    from primal_ppo_b200 import BatchedMapfGym, gae
    from primal_ppo_b200._cabi import MapfError
    sc = random_scenario(3, 128, 128, 128, density=(0.0, 0.25), queue_len=3, seed=71, fov=31)
    _run_vs_oracle(sc, T=6)
    sc = random_scenario(2, 128, 128, 254, density=(0.0, 0.2), queue_len=2, seed=72, fov=9, use_da=True, use_hp=True)
    orc = OracleMapfGym(sc, threads=8, use_tape=False)
    env = _env(sc, use_tape=False)
    o_obs, o_vec = orc.getAllObservations()
    obs, vec = env.getAllObservations()
    assert torch.equal(obs, torch.from_numpy(o_obs).cuda()) and torch.equal(vec, torch.from_numpy(o_vec).cuda())
    _eq(_np(env.bfs_maps()), orc.bfs_maps(), "bfs 128x128x254")
    with pytest.raises(MapfError):                       # joint step beyond 128 agents is refused, not mis-computed
        env.step(torch.zeros((2, 254), dtype=torch.int8))
    # empty inputs
    empty = env.bfs_maps(agent_ids=torch.zeros((0,), dtype=torch.int32, device="cuda"))
    assert empty.shape == (0, 128, 128)
    r = gae(torch.zeros((0, 8), device="cuda"), torch.zeros((0, 8), device="cuda"), torch.zeros((8,), device="cuda"))
    assert r.shape == (0, 8)
    with pytest.raises(MapfError):
        BatchedMapfGym(random_scenario(1, 8, 8, 2, seed=1, fov=33))       # fov must be <= 31
    with pytest.raises(ValueError):
        env.step(torch.zeros((3, 254), dtype=torch.int8))                  # wrong shape (mapf_gym.py:437 assert)


@pytest.mark.parametrize("shape", [(512, 40, 40, 32, 9), (33, 20, 20, 8, 9), (7, 12, 9, 5, 9), (6, 64, 64, 31, 15),
                                   (4, 80, 80, 128, 21), (3, 9, 9, 3, 3)])
def test_gpu_bf16_observations_equal_f32(shape):
    """Optional bf16 output format: the same 0/1 values (exact in bf16), from both the stand-alone and the fused launch."""
    W, H, Wd, N, F = shape
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.3), queue_len=3, seed=W + F, fov=F, unique_maps=min(W, 32))
    e1, e2 = _env(sc, use_tape=False), _env(sc, use_tape=False)
    a = torch.from_numpy(random_actions(4, W, N, seed=1)).cuda()
    ob16 = torch.empty((W, N, 6, F, F), dtype=torch.bfloat16, device="cuda")
    v16 = torch.empty((W, N, 4), device="cuda")
    obs, vec = e1.getAllObservations()
    e2.getAllObservations(out=(ob16, v16))
    assert torch.equal(ob16.float(), obs) and torch.equal(v16, vec)
    for t in range(4):
        o1, obs, vec = e1.step_observe(a[t])
        o2, _, _ = e2.step_observe(a[t], obs_out=(ob16, v16))
        assert torch.equal(ob16.float(), obs) and torch.equal(v16, vec), (shape, t)
        assert torch.equal(o1.reward, o2.reward) and torch.equal(o1.status, o2.status)


def test_gpu_checkpoint_resume_reproduces_the_rollout():
    """save_state / load_state: resuming from a checkpoint replays the same steps bit for bit (incl. Philox draws, goal
    queues, human ticks, counters); a blob can be carried to another env built from the same scenario."""
    sc = random_scenario(300, 8, 8, 8, density=(0.2, 0.3), queue_len=6, seed=91, unique_maps=64)
    a = torch.from_numpy(random_actions(16, 300, 8, seed=3)).cuda()
    env = _env(sc, use_tape=False, seed=7)
    for t in range(6):
        env.step_observe(a[t])
    blob = env.save_state().clone()

    def run(e):
        rec = []
        for t in range(6, 16):
            o, obs, vec = e.step_observe(a[t])
            rec.append([x.clone() for x in (o.status, o.reward, o.cost, o.train_valid, o.goals_reached, o.violated,
                                            o.shadow_goals, o.fixed_actions, obs, vec)])
        rec.append([e.counters(), e.state()["err"], e.state()["pos"], e.state()["goal"]])
        return rec
    first = run(env)
    env.load_state(blob)
    second = run(env)
    other = _env(sc, use_tape=False, seed=7)
    other.load_state(blob.cpu().cuda())
    third = run(other)
    for r1, r2, r3 in zip(first, second, third):
        for x, y, z in zip(r1, r2, r3):
            assert torch.equal(x, y) and torch.equal(x, z)


def test_gpu_unaligned_output_buffers():
    """Outputs that are not 16-byte aligned take the scalar-store paths (obs f32 / bf16, BFS tiles) and give the same
    bits; a misaligned vec is refused."""
    from primal_ppo_b200._cabi import MapfError
    sc = random_scenario(37, 20, 20, 8, density=(0.1, 0.25), queue_len=3, seed=5, unique_maps=16)
    env = _env(sc, use_tape=False)
    a = torch.from_numpy(random_actions(3, 37, 8, seed=2)).cuda()
    n = 37 * 8 * 6 * 81
    big = torch.zeros(n + 8, device="cuda")
    big16 = torch.zeros(n + 8, dtype=torch.bfloat16, device="cuda")
    vec = torch.empty((37, 8, 4), device="cuda")
    for t in range(3):
        _, obs, v = env.step_observe(a[t])
        o1 = big[1:1 + n].view(37, 8, 6, 9, 9)                     # 4-byte aligned only
        env.getAllObservations(out=(o1, vec))
        assert torch.equal(o1, obs) and torch.equal(vec, v) and float(big[0]) == 0 and float(big[1 + n]) == 0
        o2 = big16[1:1 + n].view(37, 8, 6, 9, 9)                   # 2-byte aligned only
        env.getAllObservations(out=(o2, vec))
        assert torch.equal(o2.float(), obs) and float(big16[0]) == 0 and float(big16[1 + n]) == 0
    ref = env.bfs_maps()
    raw = torch.zeros(ref.numel() + 4, dtype=torch.int16, device="cuda")
    out = raw[1:1 + ref.numel()].view(ref.shape)
    env.bfs_maps(out=out)
    assert torch.equal(out, ref) and int(raw[0]) == 0 and int(raw[-1]) == 0
    vraw = torch.zeros(37 * 8 * 4 + 4, device="cuda")
    with pytest.raises(MapfError):
        env.getAllObservations(out=(big[0:n].view(37, 8, 6, 9, 9), vraw[1:1 + 37 * 8 * 4].view(37, 8, 4)))


def test_gpu_sharded_worlds_equal_unsharded():
    """World w gives the same bits whichever rank owns it: run worlds [0,W) in one env and as two shards
    (world_offset keys the Philox draws), compare every output."""
    sc = random_scenario(512, 8, 8, 8, density=(0.2, 0.3), queue_len=6, seed=61, unique_maps=64)
    acts = random_actions(32, 512, 8, seed=62)
    full = _env(sc, use_tape=False, seed=77)
    lo = _env(sc.slice(0, 200), use_tape=False, seed=77, world_offset=0)
    hi = _env(sc.slice(200, 512), use_tape=False, seed=77, world_offset=200)
    for t in range(32):
        a = torch.from_numpy(acts[t]).cuda()
        o = full.step(a); o1 = lo.step(a[:200]); o2 = hi.step(a[200:])
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "fixed_actions"):
            assert torch.equal(getattr(o, key), torch.cat([getattr(o1, key), getattr(o2, key)])), (t, key)
        obs, vec = full.getAllObservations()
        ob1, _ = lo.getAllObservations(); ob2, _ = hi.getAllObservations()
        assert torch.equal(obs, torch.cat([ob1, ob2]))
    assert torch.equal(full.state()["err"], torch.cat([lo.state()["err"], hi.state()["err"]]))


def test_gpu_bfs_deep_mazes():
    """Serpentine corridors next to ordinary maps in one batch: distances of several hundred (far beyond a byte), and
    warps whose maps finish after very different numbers of levels."""
    from primal_ppo_b200.scenario import Scenario, looping_trace
    W, H, N = 12, 40, 6
    base = random_scenario(W, H, H, N, density=(0.0, 0.2), queue_len=3, seed=4)
    obst = base.obst.copy()
    for w in range(0, W, 2):                                  # every other world becomes a serpentine maze
        m = np.zeros((H, H), dtype=np.uint8)
        for r in range(1, H, 2):
            m[r, :] = 1
            m[r, H - 1 if (r // 2) % 2 == 0 else 0] = 0
        obst[w] = m
    starts = base.starts.copy(); queue = base.goal_queue.copy(); htrace = base.htrace.copy(); hlen = base.hlen.copy()
    for w in range(0, W, 2):                                  # agents, goals and the human on open rows of the maze
        for i in range(N):
            starts[w, i] = (2 * i, 3 + i)
            queue[w, i, :] = (38 - 2 * i, 5 + i)
        tr = looping_trace([(0, 0), (0, 1), (0, 0)])
        htrace[w, :3] = tr; htrace[w, 3:] = tr[-1]; hlen[w] = 3
    sc = Scenario(obst=obst, starts=starts, goal_queue=queue, htrace=htrace, hlen=hlen)
    sc.validate()
    orc = OracleMapfGym(sc, threads=4, use_tape=False)
    env = _env(sc, use_tape=False)
    ref = orc.bfs_maps()
    assert ref[0].max() > 600 and ref[1].max() < 200
    _eq(_np(env.bfs_maps()), ref, "deep + shallow maps")
    ids = torch.tensor([0, 7, 13, 2 * N + 1, 5], dtype=torch.int32).cuda()
    _eq(_np(env.bfs_maps(agent_ids=ids)), ref.reshape(W * N, H, H)[ids.cpu().numpy()], "listed maps")


@pytest.mark.parametrize("fused", [False, True])
def test_gpu_fix_actions_livelock_world(fused):
    """The reference's `while problemAgents` loop (mapf_gym.py:563) never ends for two boxed-in agents whose only
    viable actions collide: A at (1,1) can only move right (its stay is the human's next cell, its move down a swap
    with the human), B at (1,2) can only stay (its move left is the human's next cell).  Both implementations stop
    after the same number of iterations, flag the world with MAPF_ERR_FIX_ITER_CAP and leave identical state and
    outputs — compared here for EVERY world, the flagged one included."""
    from primal_ppo_b200.scenario import Scenario, looping_trace
    W, H, N = 4, 8, 2
    base = random_scenario(W, H, H, N, density=(0.0, 0.2), queue_len=3, seed=9)
    obst = base.obst.copy(); starts = base.starts.copy(); queue = base.goal_queue.copy()
    htrace = base.htrace.copy(); hlen = base.hlen.copy()
    m = np.ones((H, H), dtype=np.uint8)
    m[1, 1] = 0; m[1, 2] = 0; m[2, 1] = 0
    obst[0] = m
    starts[0, 0] = (1, 1); starts[0, 1] = (1, 2)
    queue[0, 0, :] = (2, 1); queue[0, 1, :] = (1, 1)
    tr = looping_trace([(2, 1), (1, 1), (2, 1)])
    htrace[0, :len(tr)] = tr; htrace[0, len(tr):] = tr[-1]; hlen[0] = len(tr)
    sc = Scenario(obst=obst, starts=starts, goal_queue=queue, htrace=htrace, hlen=hlen)
    sc.validate()
    orc = OracleMapfGym(sc, seed=1234, threads=2, use_tape=False)
    env = _env(sc, seed=1234, use_tape=False)
    rng = np.random.default_rng(3)
    for t in range(4):
        acts = rng.integers(0, 5, size=(W, N)).astype(np.int8)
        if t % 2 == 0:
            acts[0] = (1, 0)                                   # A right, B stay: vertex conflict -> fixActions
        ref = orc.step(acts)
        if fused:
            out, obs, vec = env.step_observe(torch.from_numpy(acts))
        else:
            out = env.step(torch.from_numpy(acts))
            obs, vec = env.getAllObservations()
        e_ref = orc.state()["err"]
        np.testing.assert_array_equal(_np(env.state()["err"]).astype(np.uint32), e_ref, err_msg=f"t={t} err flags")
        if t == 0:
            assert e_ref[0] & 2 and not e_ref[1:].any()        # MAPF_ERR_FIX_ITER_CAP on the livelock world only
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated"):
            _eq(_np(getattr(out, key)), ref[key], f"t={t} {key}")
        _eq(_np(out.fixed_actions), ref["fixed"], f"t={t} fixed")
        s, so = env.state(), orc.state()
        for key in ("pos", "goal", "rep"):
            _eq(_np(s[key]), so[key], f"t={t} {key}")
        o_obs, o_vec = orc.getAllObservations()
        assert torch.equal(obs, torch.from_numpy(o_obs).cuda()) and torch.equal(vec, torch.from_numpy(o_vec).cuda()), f"t={t} obs"


@pytest.mark.parametrize("shape", [(8, 5), (8, 8), (6, 12), (16, 31), (8, 32), (24, 33), (40, 40), (17, 40), (12, 64),
                                   (9, 96), (30, 100), (8, 127), (25, 128), (64, 64), (100, 72), (7, 9), (11, 13)])
def test_gpu_bfs_map_shapes(shape):
    """Row lengths on both sides of every 32-bit word boundary (the row-neighbour shift of the cell-string kernel is
    32*(Wd/32) + Wd%32 bits), cell counts that do and do not fill the last word, and shapes whose maps cannot leave as
    16-byte vectors (H*Wd % 8 != 0: the row-word kernel takes them)."""
    H, Wd = shape
    W, N = 6, 5
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.35), queue_len=2, seed=1000 + H * 131 + Wd, fov=3)
    orc = OracleMapfGym(sc, threads=4, use_tape=False)
    env = _env(sc, use_tape=False)
    ref = orc.bfs_maps()
    _eq(_np(env.bfs_maps()), ref, f"bfs {H}x{Wd}")
    ids = torch.tensor([W * N - 1, 0, 7, 7, 3], dtype=torch.int32).cuda()      # listed (and repeated) maps
    _eq(_np(env.bfs_maps(agent_ids=ids)), ref.reshape(W * N, H, Wd)[ids.cpu().numpy()], f"listed maps {H}x{Wd}")


def test_gpu_bfs_refresh_in_place():
    sc = random_scenario(256, 40, 40, 32, density=(0.0, 0.3), queue_len=8, seed=21, unique_maps=32)
    orc = OracleMapfGym(sc, threads=8, use_tape=False)
    env = _env(sc, use_tape=False)
    maps = env.bfs_maps()
    rng = np.random.default_rng(0)
    total = 0
    for t in range(24):
        # walk down the BFS field so that goals are reached
        m = _np(maps)
        s = orc.state()
        acts = rng.integers(0, 5, size=(sc.num_worlds, sc.num_agents)).astype(np.int8)
        pos = s["pos"].astype(np.int64)
        for k, (dr, dc) in enumerate([(0, 1), (1, 0), (0, -1), (-1, 0)], start=1):
            rr = np.clip(pos[..., 0] + dr, 0, 39)
            cc = np.clip(pos[..., 1] + dc, 0, 39)
            w_i = np.arange(sc.num_worlds)[:, None]
            a_i = np.arange(sc.num_agents)[None, :]
            here = m[w_i, a_i, pos[..., 0], pos[..., 1]]
            nxt = m[w_i, a_i, rr, cc]
            acts = np.where((nxt >= 0) & (nxt < here), k, acts).astype(np.int8)
        orc.step(acts)
        out = env.step(torch.from_numpy(acts))
        total += int(out.goals_reached.sum())
        env.refresh_bfs(maps)
        _eq(_np(maps), orc.bfs_maps(), f"t={t} refreshed maps")
    assert total > 100


def test_gpu_gae_bit_exact():
    d = np.load(GOLDEN_DIR + "/gae_runner.npz")
    from primal_ppo_b200 import gae
    ret = gae(torch.from_numpy(d["rewards"]).cuda(), torch.from_numpy(d["values"]).cuda(),
              torch.from_numpy(d["last_values"]).cuda(), float(d["gamma"]), float(d["lam"]))
    _eq(_np(ret), d["returns"], "golden returns")
    cret = gae(torch.from_numpy(d["cost_rewards"]).cuda(), torch.from_numpy(d["cost_values"]).cuda(),
               torch.from_numpy(d["last_cost_values"]).cuda(), float(d["gamma"]), float(d["lam"]))
    _eq(_np(cret), d["cost_returns"], "golden cost returns")
    rng = np.random.default_rng(5)
    for T, cols in ((256, 4096 * 8), (256, 1000 * 3), (1, 64), (7, 5)):
        r = rng.normal(size=(T, cols)).astype(np.float32)
        v = rng.normal(size=(T, cols)).astype(np.float32)
        lv = rng.normal(size=(cols,)).astype(np.float32)
        ref, radv = gae_oracle(r, v, lv)
        ret, adv = gae(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(lv).cuda(),
                       return_advantages=True)
        _eq(_np(ret), ref, f"gae returns {T}x{cols}")
        _eq(_np(adv), radv, f"gae adv {T}x{cols}")


def test_gpu_gae_with_terminal_mask():
    """nonterminal[t] = 0 cuts the bootstrap and the advantage carry at step t (the reference always uses 1.0,
    runner.py:123; the mask is the generalisation to episodic envs).  NumPy f32 restatement, op by op."""
    from primal_ppo_b200 import gae
    rng = np.random.default_rng(9)
    T, cols = 37, 203
    r = rng.normal(size=(T, cols)).astype(np.float32); v = rng.normal(size=(T, cols)).astype(np.float32)
    lv = rng.normal(size=(cols,)).astype(np.float32)
    nt = (rng.random((T, cols)) > 0.1).astype(np.uint8)
    ret, adv = gae_masked_ref(r, v, lv, nt)
    out, a = gae(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(lv).cuda(),
                 nonterminal=torch.from_numpy(nt).cuda(), return_advantages=True)
    _eq(_np(out), ret, "masked returns"); _eq(_np(a), adv, "masked advantages")


def test_gpu_host_buffer_call_equals_device_call():
    sc = random_scenario(512, 20, 20, 8, density=(0.1, 0.2), queue_len=4, seed=31, unique_maps=64)
    a = random_actions(6, 512, 8, seed=3)
    e1, e2 = _env(sc, use_tape=False), _env(sc, use_tape=False)
    hb = e2.make_host_buffers(with_obs=True, with_train_valid=True)
    obs2 = torch.empty((512, 8, 6, 9, 9), device="cuda")
    vec2 = torch.empty((512, 8, 4), device="cuda")
    for t in range(6):
        o1 = e1.step(torch.from_numpy(a[t]))
        obs1, vec1 = e1.getAllObservations()
        hb["actions"].copy_(torch.from_numpy(a[t]))
        e2.step_observe_host(hb, obs2, vec2)
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow_goals"):
            _eq(_np(getattr(o1, key)), hb[key].numpy(), key)
        assert torch.equal(obs1, obs2) and torch.equal(vec1, vec2)
        assert torch.equal(obs1.cpu(), hb["obs"]) and torch.equal(vec1.cpu(), hb["vec"])


def test_gpu_host_buffer_call_large_batch_equals_fused_device_call():
    """The host-buffer call (two kernels, results copied back on a second stream while the observations are written)
    against the fused device call on a larger batch: every output and the state must be equal."""
    W, N = 16500, 4            # not a multiple of the range size
    sc = random_scenario(W, 10, 10, N, density=(0.1, 0.25), queue_len=3, seed=77, unique_maps=128)
    a = random_actions(5, W, N, seed=8)
    e1, e2 = _env(sc, use_tape=False, seed=5), _env(sc, use_tape=False, seed=5)
    hb = e2.make_host_buffers(with_obs=False, with_train_valid=True)
    obs2 = torch.empty((W, N, 6, 9, 9), device="cuda")
    vec2 = torch.empty((W, N, 4), device="cuda")
    for t in range(5):
        o1, obs1, vec1 = e1.step_observe(torch.from_numpy(a[t]))
        hb["actions"].copy_(torch.from_numpy(a[t]))
        e2.step_observe_host(hb, obs2, vec2)
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow_goals"):
            _eq(_np(getattr(o1, key)), hb[key].numpy(), f"t={t} {key}")
        assert torch.equal(obs1, obs2) and torch.equal(vec1, vec2), t
    s1, s2 = e1.state(), e2.state()
    assert all(torch.equal(s1[k], s2[k]) for k in s1) and torch.equal(e1.counters(), e2.counters())


def test_gpu_full_size_properties_65536x40x40x32():
    """BASELINE.json configs[2] at full size: properties that do not need the oracle."""
    W, N, H = 65536, 32, 40
    sc = random_scenario(W, H, H, N, density=(0.0, 0.3), queue_len=8, seed=41, unique_maps=128)
    env = _env(sc, use_tape=False)
    obst = torch.from_numpy(sc.obst).cuda()
    acts = torch.from_numpy(random_actions(4, W, N, seed=9)).cuda()
    widx = torch.arange(W, device="cuda")[:, None].expand(W, N)
    for t in range(4):
        out = env.step(acts[t])
        s = env.state()
        ok = s["err"] == 0
        pos = s["pos"].long()
        cell = pos[..., 0] * H + pos[..., 1]
        # in bounds, never on an obstacle, no two agents of a world on one cell
        assert bool(((pos >= 0) & (pos < H)).all())
        assert bool((obst[widx, pos[..., 0], pos[..., 1]] == 0)[ok].all())
        srt = cell.sort(dim=1).values
        assert bool((srt[:, 1:] != srt[:, :-1])[ok].all())
        # fixActions post-condition (mapf_gym.py:600-610): executed actions have status 1 or -4 -> moved agents
        # either stayed or moved exactly one cell
        assert set(torch.unique(out.status).tolist()) <= {-4, -3, -2, -1, 1}
        assert set(torch.unique(out.reward).tolist()) <= {float(np.float32(x)) for x in (-2, -0.35, -0.3, -0.5, np.float32(-0.35) + np.float32(1.5), np.float32(-0.3) + np.float32(1.5))}
        obs, vec = env.getAllObservations()
        assert bool(((obs == 0) | (obs == 1)).all())
        assert bool((obs[:, :, 0, 4, 4] == 1).all())          # own cell marked in channel 0
        assert bool((obs[:, :, 2].sum(dim=(2, 3)) <= 1).all())  # own goal at most once
        assert bool((obs[:, :, 5] == 0).all())                # channel 5 is all-zero in training
        # channel 1 never overlaps channel 0
        assert bool(((obs[:, :, 0] * obs[:, :, 1]) == 0).all())
    assert float((env.state()["err"] != 0).float().mean()) < 0.01
