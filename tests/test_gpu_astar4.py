"""astar_4 on the device (csrc/astar4.cuh): `mapf_astar4_paths` and `human_path="astar4"` generation bit-exact with
`episode_io.astar_path`, the default walk unchanged, fixture conversion on the device byte-identical to the host one."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

from astar_util import GOLDEN, golden_cases, human_legs, random_cases
from primal_ppo_b200 import _cabi
from primal_ppo_b200.episode_io import astar_path, load_fixed_episode_infos, scenario_from_fixed_episode_infos

gpu = pytest.mark.gpu


# ---- ABI (no GPU needed) ------------------------------------------------------------------------------------------------
def test_gen_config_layout_keeps_its_offsets():
    G = _cabi.MapfGenConfig
    assert ctypes.sizeof(G) == 72
    assert G.human_loops.offset == 48 and G.human_path.offset == 52
    assert G.seed.offset == 56 and G.world_offset.offset == 64 and G.device.offset == 68


def test_misuse_codes_without_gpu():
    from primal_ppo_b200.build import build
    build()
    lib = _cabi.load_library()
    p = ctypes.c_void_p(64)                      # never dereferenced: every call below fails its argument checks first
    assert lib.mapf_astar4_paths(None, 1, 8, 8, p, 4, p, p, None) == -2                # MAPF_E_NULL
    assert lib.mapf_astar4_paths(p, 1, 8, 8, p, 4, p, None, None) == -2
    for n, H, Wd, L in ((-1, 8, 8, 4), (1, 0, 8, 4), (1, 8, 129, 4), (1, 129, 8, 4), (1, 8, 8, 0)):
        assert lib.mapf_astar4_paths(p, n, H, Wd, p, L, p, p, None) == -1, (n, H, Wd, L)   # MAPF_E_BAD_CONFIG
        assert b"mapf_astar4_paths" in lib.mapf_last_error()
    cfg = _cabi.MapfGenConfig(num_worlds=4, height=8, width=8, num_agents=2, kind=0, density_lo=0.1, density_hi=0.2,
                              queue_len=2, trace_len=8, human_loops=1, human_path=2)
    assert lib.mapf_generate_scenario(ctypes.byref(cfg), p, p, p, p, p, p, p, p, None) == -1
    assert b"human_path" in lib.mapf_last_error()


# ---- mapf_astar4_paths ---------------------------------------------------------------------------------------------------
def _solve(cases, H, Wd, max_len=None):
    """cases: (world [h,w] with -1 = wall, start, goal), each padded with walls to H x Wd."""
    import torch
    from primal_ppo_b200.device_scenario import astar_paths_device
    obst = np.ones((len(cases), H, Wd), dtype=np.uint8)
    for i, (m, _, _) in enumerate(cases):
        obst[i, :m.shape[0], :m.shape[1]] = m == -1
    sg = np.array([[s, g] for _, s, g in cases], dtype=np.int16)
    paths, lens = astar_paths_device(torch.from_numpy(obst).cuda(), torch.from_numpy(sg).cuda(), max_len)
    return paths.cpu().numpy(), lens.cpu().numpy()


def _expect(cases, paths, lens, max_len):
    codes = set()
    for i, (m, s, g) in enumerate(cases):
        inside = all(0 <= r < m.shape[0] and 0 <= c < m.shape[1] for r, c in (s, g))
        ref = astar_path(m, s, g) if inside else None
        want = -3 if not inside else -1 if ref is None else 0 if ref == [] else -2 if len(ref) > max_len else len(ref)
        assert lens[i] == want, (i, m.shape, s, g, lens[i], want)
        k = max(want, 0)
        if k:
            assert [tuple(x) for x in paths[i, :k].tolist()] == ref, (i, m.shape, s, g)
        assert (paths[i, k:] == -1).all(), i
        codes.add(int(np.sign(want)) if want > 0 else int(want))
    return codes


def _training_legs():
    G = np.load(os.path.join(GOLDEN, "training_env.npz"))
    out = []
    for ci in range(int(G["n_cases"])):
        for w in range(G[f"c{ci}_obst"].shape[0]):
            rows, cols = (int(x) for x in G[f"c{ci}_dims"][w])
            world = -(G[f"c{ci}_obst"][w, :rows, :cols] != 0).astype(np.int64)
            out += [(world, ent, turn) for ent, turn, _ in human_legs(G[f"c{ci}_htrace"][w])]
    return out


@gpu
def test_gpu_astar4_paths_match_astar_path():
    small = golden_cases() + [c for c in random_cases() if c[0].shape[0] <= 64] + _training_legs()
    H, Wd = max(c[0].shape[0] for c in small), max(c[0].shape[1] for c in small)
    # cells outside the (padded) map (-3) and start == goal (0)
    m = np.zeros((H, Wd), dtype=np.int64)
    small += [(m, (H, 0), (0, 0)), (m, (0, 0), (0, Wd)), (m, (-1, 2), (3, 3)), (m, (2, 2), (2, -1)), (m, (4, 4), (4, 4))]
    paths, lens = _solve(small, H, Wd)
    assert _expect(small, paths, lens, H * Wd) == {-3, -1, 0, 1}
    # a short max_len: the longer paths report -2, the rest are unchanged
    paths, lens = _solve(small, H, Wd, max_len=12)
    assert -2 in _expect(small, paths, lens, 12)


@gpu
def test_gpu_astar4_paths_128x128():
    rng = np.random.default_rng(3)
    big = [c for c in random_cases() if c[0].shape[0] == 128]
    open_ = np.zeros((128, 128), dtype=np.int64)
    big += [(open_, (0, 0), (127, 127)), (open_, (127, 0), (0, 127)), (open_, (64, 64), (0, 0))]
    for _ in range(6):                           # long detours: walls with one gap each
        m = np.zeros((128, 128), dtype=np.int64)
        for r in range(4, 128, 8):
            m[r, :] = -1
            m[r, int(rng.integers(128))] = 0
        big.append((m, (0, int(rng.integers(128))), (127, int(rng.integers(128)))))
    paths, lens = _solve(big, 128, 128)
    assert 1 in _expect(big, paths, lens, 128 * 128)
    assert lens.max() > 800


# ---- generation ------------------------------------------------------------------------------------------------------
GEN = {
    "warehouse_l1": dict(num_worlds=600, height=40, width=60, num_agents=8, kind="warehouse", size_range=(10, 40), queue_len=4, seed=3),
    "warehouse_l3": dict(num_worlds=300, height=40, width=60, num_agents=8, kind="warehouse", queue_len=2, human_loops=3, seed=4),
    "density_l1": dict(num_worlds=512, height=40, width=40, num_agents=16, kind="density", density=(0.0, 0.45), queue_len=2, seed=6),
    "density_l3_sizes": dict(num_worlds=400, height=40, width=40, num_agents=6, kind="density", density=(0.0, 0.25),
                             size_range=(10, 40), queue_len=3, human_loops=3, seed=5),
    "density_128_offset": dict(num_worlds=64, height=128, width=128, num_agents=16, kind="density", density=(0.0, 0.4),
                               queue_len=2, seed=7, world_offset=1000),
}

# SHA-256 of every output array of the default walk, computed on a B200 with the build before human_path existed
PARENT_SHA = {
    "warehouse_l1": {
        "obst": "19d31ce81d18d7092cf185b4ede7f9688fd784e0bd4930401c531b6a698e2d9d",
        "dims": "82b7702f9492459680abb0cd2580a6d21fa8be8d3bab9e86ea0a2ea176c9d973",
        "starts": "03a759c4116fd2cef256e80dd8a67b973dd5a9e8d97c84dfaef52dcc125de9d9",
        "goal_queue": "e642f5f6e76a0f39a56e56c34847fc45db9f8e6c69f53588866be5b8440bdca5",
        "htrace": "19fcb6ef8f5b564bfc05a9a9b6c662c0394d8b0ba0991cf08e425f7e6346c779",
        "hlen": "81602b9dfa9a0f808b43c07022d38467e587c9a6ad1a631690396af5ea372c8f",
        "hp5": "ecbe1ac5a4aaae0ff35f044d45ba1ab2349b22ab68927750c9091658de6793be",
        "gen_err": "a0ee989ed2a0a2e3626520afa4032e06144865c8c8f6357293c9f4cd2069eaf2",
    },
    "warehouse_l3": {
        "obst": "fb73332bdd37e6f12f871ac99c11665bf4a79bad44c193db5754589ff078df53",
        "dims": "b4693f3fb06585b806a4cc7a4af62d66717b671918c36cf0cc25829b7a6e9234",
        "starts": "47ac316c117d1aaca8b6bdacdfb18b2a3e83e97067aa0680390d23ffd7adb654",
        "goal_queue": "129305182a89e350f7869a89b81845fdbf0d4297d039960f4759f64ac225e4ca",
        "htrace": "9f71132570488eaf335bb7b5600d965be533f9c54831c76b3e4a4f11194c54ad",
        "hlen": "1de8f5ecd85297df66feddfdfd426d88f79d9073db13e3ee449e8eb57be39b11",
        "hp5": "abaef4cfcfa7255fd3f4f2e5b6d91188ce6735767b38e2da1bf54139a4e6221e",
        "gen_err": "655a3ef0465a9f30fddf25f4dde0c19a05c6f9069b83961800c1944165955273",
    },
    "density_l1": {
        "obst": "ce4455c3848dd07d1bcad60bbad60c3e25f49e44f70c8e27517c80b5d521dfce",
        "dims": "48aac49fa2b255d1c82df1e7b7cb4d56995712f3f4024a72303676b0d9671cd4",
        "starts": "2a1d7e10c9036f1aea32b3d6f21e9395feb365b6935da4bbe2df786109189c6c",
        "goal_queue": "e047b2f1d69a6980dc37a9fff36e8cef1566655a3940ab6f88748cf4ad2047c0",
        "htrace": "5279d26a08f675ec0fd6bf553c38fb98ea6473f228a7c8613865eb7757bc2d9c",
        "hlen": "962615714f46391c541b763b95b275c3da6fc294b4f75f76729ffdd89bcb62fc",
        "hp5": "49d0c68745cf35f9d724f7aef073fa675e953493e4b46690e7774ca570b79f10",
        "gen_err": "75f0bb7b5ea63a7451ad241413db8bbe8fadadc3d3dca2d9ab83819f5dbd63cc",
    },
    "density_l3_sizes": {
        "obst": "5c302549e2b66a38df061b5b2ffc1b6134853cb5a438e1a782d1216c0cbf1a92",
        "dims": "7b88c6e6071d0205851f1cb15a6823cc110e1a2d587a89e28244ec51aa17162f",
        "starts": "efdb1c66f32f4b5daf06cb3657f4f539db905fabf66a3b389a2ece6927ffa663",
        "goal_queue": "9cd086fb598cd4c934d6170c3cd70f2b53903715b1cdb926a6fa4c2fec191ade",
        "htrace": "d01094bd69e478e4ae372f9a103a0ba8b7115536e281b1839e3d33d448d881c5",
        "hlen": "3cc4f7e3a3989900ba39f405027e7cbf74ea71e884d155955071ebd1c3339d8c",
        "hp5": "a288385539f7474e02ccc8b0810e30e46734a2b63fc3066b19ca696ad12bfd1d",
        "gen_err": "8879bb0b71de1786871eea9c6ed1de96fedd0f5778c053f51f79fba87b47515f",
    },
    "density_128_offset": {
        "obst": "44a361f0450ee403de22dcb7cfedf7a97a0da715bc1e5317b15ca3ada0742a29",
        "dims": "9b19bbe6bb1726ee2f4fe74a7acc3f2fcfb38e83433f6ea8ef24c46fb39191ce",
        "starts": "a3d22a88266085ecadf6f8f571624a278d28188b7b4a560f055c6d2f18dd2722",
        "goal_queue": "f07fb819a8efc2797b99c9fb26cb609553cc89e294d313659ec73689727b3a97",
        "htrace": "d9eb65fd40a579b3f48d2360225fc1c207e5b1876f7d5c3db744c385a2819ba4",
        "hlen": "c91b690bf6d4ddafa6f89f7ee01d9c4e12ffdfa173e5c6db29ed6932e5c12cd2",
        "hp5": "3e3f578da2d4924de7b4f49a1e9bdfc0f7f48c1bbbd24342566b68081b1d111b",
        "gen_err": "1e5ef7a0e82e092b7175c01cae5e393348670216cc360270748fee0c5dfc58ee",
    },
}


def _gen(name, **kw):
    import torch
    from primal_ppo_b200 import generate_scenario_device
    d = generate_scenario_device(**{**GEN[name], **kw})
    torch.cuda.synchronize()
    return {k: getattr(d, k).cpu().numpy() for k in ("obst", "dims", "starts", "goal_queue", "htrace", "hlen", "hp5", "gen_err")}, d


@gpu
@pytest.mark.parametrize("name", sorted(GEN))
def test_gpu_astar4_generation_walks_astar_path(name):
    a, d = _gen(name, human_path="astar4")
    assert d.meta["human_path"] == "astar4"
    b, _ = _gen(name)
    for k in ("obst", "dims", "starts", "goal_queue", "hlen", "gen_err"):
        assert np.array_equal(a[k], b[k]), k
    legs = 0
    for w in range(a["obst"].shape[0]):
        L = int(a["hlen"][w])
        ta, tb = a["htrace"][w, :L, :2], b["htrace"][w, :L, :2]
        if a["gen_err"][w] & 4:
            assert np.array_equal(ta, tb)
            continue
        rows, cols = (int(x) for x in a["dims"][w])
        world = -(a["obst"][w, :rows, :cols] != 0).astype(np.int64)
        la, lb = human_legs(a["htrace"][w, :L]), human_legs(b["htrace"][w, :L])
        assert [(e, t, len(o)) for e, t, o in la] == [(e, t, len(o)) for e, t, o in lb], w
        for ent, turn, out in la:
            assert astar_path(world, ent, turn) == out, (name, w, ent, turn)
        legs += len(la)
        # the two walks agree at every entrance and turning tick
        key = [t for t in range(L) if tuple(tb[t]) == tuple(tb[0]) or 0 < t < L - 1 and tuple(tb[t + 1]) == tuple(tb[t - 1])]
        assert np.array_equal(ta[key], tb[key]), w
        if GEN[name].get("human_loops", 1) == 1:
            k = min(5, L - 1)
            assert (a["hp5"][w, :k] == ta[1:1 + k]).all() and (a["hp5"][w, k:] == -1).all()
            assert (a["htrace"][w, :L - 1, 2:] == a["htrace"][w, 1:L, :2]).all()
    assert legs >= a["obst"].shape[0] // 2


@gpu
@pytest.mark.parametrize("name", sorted(GEN))
def test_gpu_default_walk_is_unchanged(name):
    got, _ = _gen(name)
    assert {k: hashlib.sha256(v.tobytes()).hexdigest() for k, v in got.items()} == PARENT_SHA[name]


@gpu
def test_gpu_env_on_astar4_worlds_matches_oracle():
    import torch
    from oracle import OracleMapfGym
    from primal_ppo_b200 import BatchedMapfGym, generate_scenario_device, random_actions
    d = generate_scenario_device(128, 40, 60, 8, kind="warehouse", queue_len=4, seed=21, human_path="astar4")
    env = BatchedMapfGym(d, use_tape=False, seed=9)
    sc = d.to_host()
    sc.validate()
    orc = OracleMapfGym(sc, seed=9, threads=4, use_tape=False)
    acts = random_actions(16, 128, 8, seed=2)
    for t in range(16):
        out, obs, vec = env.step_observe(torch.from_numpy(acts[t]))
        ref = orc.step(acts[t])
        for key in ("status", "reward", "cost", "train_valid", "goals_reached", "violated"):
            assert np.array_equal(getattr(out, key).cpu().numpy(), ref[key]), (t, key)
        o_obs, o_vec = orc.getAllObservations()
        assert np.array_equal(obs.cpu().numpy(), o_obs) and np.array_equal(vec.cpu().numpy(), o_vec), t


# ---- fixture conversion ------------------------------------------------------------------------------------------------
def _synthetic_infos(n, seed):
    """n fixture episodes on density maps: 3 agents, a human start / goal and a pose sequence in the start's component."""
    from collections import deque
    rng = np.random.default_rng(seed)
    infos = {k: [] for k in ("obstacleMap", "agentsSequence", "humanSequence", "humanStart", "humanGoal")}
    while len(infos["obstacleMap"]) < n:
        h, w = (int(x) for x in rng.integers(6, 33, 2))
        m = -(rng.random((h, w)) < rng.uniform(0.0, 0.35)).astype(np.int64)
        free = np.argwhere(m == 0)
        if len(free) < 12:
            continue
        s = tuple(int(x) for x in free[rng.integers(len(free))])
        seen, q = {s}, deque([s])
        while q:
            r, c = q.popleft()
            for nb in ((r + 1, c), (r - 1, c), (r, c + 1), (r, c - 1)):
                if 0 <= nb[0] < h and 0 <= nb[1] < w and m[nb] == 0 and nb not in seen:
                    seen.add(nb)
                    q.append(nb)
        comp = sorted(seen)
        if len(comp) < 6:
            continue
        seq = [s]
        while len(seq) < int(rng.integers(2, 9)):
            p = comp[rng.integers(len(comp))]
            if p != seq[-1]:
                seq.append(p)
        infos["obstacleMap"].append(m)
        infos["humanStart"].append(s)
        infos["humanGoal"].append(seq[1])
        infos["humanSequence"].append(seq)
        infos["agentsSequence"].append([[tuple(int(x) for x in free[rng.integers(len(free))]) for _ in range(int(rng.integers(2, 5)))]
                                        for _ in range(3)])
    infos["numEpisodes"] = n
    return infos


def _same_scenario(a, b):
    for k in ("obst", "starts", "goal_queue", "htrace", "hlen", "hp5", "dims"):
        x, y = getattr(a, k), getattr(b, k)
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), k
    assert a.meta == b.meta


@gpu
@pytest.mark.parametrize("mtype", [0, 1])
def test_gpu_fixture_conversion_on_device_is_byte_identical(mtype):
    for infos, max_steps in ((load_fixed_episode_infos(os.path.join(GOLDEN, "fixed_episode_infos")), 48),
                             (load_fixed_episode_infos(os.path.join(GOLDEN, "fixed_episode_infos")), 256),
                             (_synthetic_infos(2000, 1 + mtype), 256)):
        kw = dict(human_movement_type=mtype, max_steps=max_steps, use_da=True, use_hp=True)
        _same_scenario(scenario_from_fixed_episode_infos(infos, **kw),
                       scenario_from_fixed_episode_infos(infos, device="cuda:0", **kw))


@gpu
def test_gpu_fixture_conversion_on_device_raises_what_the_host_raises():
    base = _synthetic_infos(4, 7)

    agents = [[(1, 1), (2, 2)], [(3, 1), (5, 2)], [(6, 6), (1, 6)]]

    def variant(ep, **items):
        infos = {k: (list(v) if isinstance(v, list) else v) for k, v in base.items()}
        for k, v in items.items():
            infos[k][ep] = v
        return infos
    m = np.zeros((8, 8), dtype=np.int64)
    m[:, 4] = -1                                  # two halves, no way across
    cases = [
        (0, variant(1, obstacleMap=m, agentsSequence=agents, humanStart=(0, 0), humanGoal=(0, 7))),                    # unreachable goal
        (0, variant(2, humanStart=base["humanStart"][2], humanGoal=base["humanStart"][2])),      # start == goal
        (0, variant(1, obstacleMap=m, agentsSequence=agents, humanStart=(0, 0), humanGoal=(0, 4))),                    # goal on a wall
        (0, variant(3, humanGoal=(40, 1))),                                                      # goal off the map
        (1, variant(1, obstacleMap=m, agentsSequence=agents, humanSequence=[(0, 0), (3, 3), (0, 7)])),                 # unreachable pose
        (1, variant(0, humanSequence=[base["humanSequence"][0][0]] * 2)),                       # empty leg
    ]
    for mtype, infos in cases:
        kw = dict(human_movement_type=mtype, max_steps=64)
        with pytest.raises(Exception) as host:
            scenario_from_fixed_episode_infos(infos, **kw)
        with pytest.raises(type(host.value)):
            scenario_from_fixed_episode_infos(infos, device="cuda:0", **kw)
    # a start one row above the map: astar_path walks in from there, and so does the device conversion
    infos = variant(2, humanStart=(-1, 0), humanGoal=(3, 0), obstacleMap=np.zeros((5, 5), dtype=np.int64), agentsSequence=agents[:1] * 3)
    _same_scenario(scenario_from_fixed_episode_infos(infos), scenario_from_fixed_episode_infos(infos, device="cuda:0"))
    # an unreachable pose after the last tick: neither conversion plans that leg
    infos = variant(1, obstacleMap=m, agentsSequence=agents, humanSequence=[(0, 0), (7, 3), (0, 3), (7, 3), (0, 7)])
    kw = dict(human_movement_type=1, max_steps=4)
    _same_scenario(scenario_from_fixed_episode_infos(infos, **kw), scenario_from_fixed_episode_infos(infos, device="cuda:0", **kw))
