"""The split-phase host call (mapf_step_observe_host_begin / _wait) with bf16 and bit-packed observations, and with the
step's observations delivered in the host result slot (MAPF_HOST_OBS): bit-exact against a twin env driven by the
device-resident step_observe in the same format, for every observation kernel family."""
import ctypes

import pytest
import torch

from primal_ppo_b200 import random_actions, random_scenario

pytestmark = pytest.mark.gpu

GUARD = 0x5A
RESULTS = ("status", "reward", "cost", "goals_reached", "violated", "shadow_goals", "fixed_actions")

# (W, H, Wd, N, F, MAPF_DBG_FLAGS): lane groups of 4 agents, warp per world (the bench shape), CTA per world at 128 agents,
# FOV 31, and the two-launch step + observe fallback (flags 1)
SHAPES = [(64, 12, 12, 4, 9, 0), (256, 40, 40, 32, 9, 0), (8, 80, 80, 128, 9, 0), (6, 64, 64, 32, 31, 0),
          (33, 20, 20, 8, 9, 1)]


def _ids(s):
    return "W{}_{}x{}_N{}_F{}_f{}".format(*s)


def _env(sc, **kw):
    from primal_ppo_b200 import BatchedMapfGym
    return BatchedMapfGym(sc, use_tape=False, seed=5, **kw)


def _obs_buf(env, fmt):
    if fmt == "bits":
        return torch.empty(env.obs_bits_shape, dtype=torch.int32, device="cuda")
    dt = torch.bfloat16 if fmt == "bf16" else torch.float32
    return torch.empty((env.W, env.N, env.C, env.F, env.F), dtype=dt, device="cuda")


def _ring_obs(fmt):
    return {"f32": torch.float32, "bf16": torch.bfloat16, "bits": "bits"}[fmt]


def _setup(shape, monkeypatch):
    W, H, Wd, N, F, flags = shape
    if flags:
        monkeypatch.setenv("MAPF_DBG_FLAGS", str(flags))       # read when the env is created
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.3), queue_len=4, seed=W + N + F, fov=F, unique_maps=min(W, 32))
    return sc, _env(sc), _env(sc)


def _twin_steps(twin, acts, fmt):
    """What the device-resident call gives for each joint action of `acts`, computed before the split-phase loop runs so
    that nothing synchronises the device between its begins."""
    obs, vec = _obs_buf(twin, fmt), torch.empty((twin.W, twin.N, 4), device="cuda")
    want = []
    for a in acts:
        o, _, _ = twin.step_observe(a.cuda(), obs_out=(obs, vec))
        w = {k: getattr(o, k).cpu() for k in RESULTS + ("train_valid",)}
        w.update(obs=obs.clone(), vec=vec.clone())
        want.append(w)
    return want


def _check_slot(slot, want, what, with_tv=False):
    from primal_ppo_b200 import decode_results
    if "packed" in slot:
        dec = decode_results(slot["packed"])
        for k in ("status", "reward", "cost", "goals_reached", "violated", "fixed_actions"):
            assert torch.equal(dec[k], want[k]), (what, k)
    else:
        for k in ("status", "reward", "cost", "goals_reached", "violated", "fixed_actions"):
            assert torch.equal(slot[k], want[k]), (what, k)
    assert torch.equal(slot["shadow_goals"], want["shadow_goals"]), (what, "shadow_goals")
    if with_tv:
        assert torch.equal(slot["train_valid"], want["train_valid"]), (what, "train_valid")


@pytest.mark.parametrize("fmt", ["bf16", "bits"])
@pytest.mark.parametrize("shape", SHAPES, ids=_ids)
def test_gpu_split_phase_obs_format_equals_device_call(shape, fmt, monkeypatch):
    """obs_dev in bf16 / bits: every step's obs_dev and vec_dev equal the twin's, and the result slots decode to its
    results (full and compact wire formats, two begins in flight)."""
    sc, twin, env = _setup(shape, monkeypatch)
    W, N, T = env.W, env.N, 5
    acts = torch.from_numpy(random_actions(2 * T, W, N, seed=3))
    obs_t = [_obs_buf(env, fmt) for _ in range(2)]
    vec_t = [torch.empty((W, N, 4), device="cuda") for _ in range(2)]
    for part, compact in enumerate((False, True)):
        ring = env.make_host_ring(slots=2, action_slots=2, compact=compact)
        want = _twin_steps(twin, acts[part * T:(part + 1) * T], fmt)
        for t in range(T):
            ring["action_ring"][t & 1].copy_(acts[part * T + t])
            env.step_observe_host_begin(ring["action_ring"][t & 1], ring["slots"][t & 1], obs_t[t & 1], vec_t[t & 1])
            assert torch.equal(obs_t[t & 1], want[t]["obs"]) and torch.equal(vec_t[t & 1], want[t]["vec"]), (compact, t)
            if t >= 1:
                env.host_wait(1)
                _check_slot(ring["slots"][(t - 1) & 1], want[t - 1], (compact, t - 1))
        env.host_wait(0)
        _check_slot(ring["slots"][(T - 1) & 1], want[T - 1], (compact, T - 1))


@pytest.mark.parametrize("fmt", ["f32", "bf16", "bits"])
@pytest.mark.parametrize("shape", SHAPES, ids=_ids)
def test_gpu_host_obs_in_result_slot(shape, fmt, monkeypatch):
    """MAPF_HOST_OBS: the host obs / vec of every slot equal the twin's observations of that step.  Every step writes
    the SAME obs_dev / vec_dev, and the begins are issued back to back with nothing on the host between them (every
    step has its own host slot and action buffer; the slots are read after the last step), so at every begin the
    previous step's copy out of obs_dev may still run: a missing wait on that copy would show up as a later step's
    observations in an earlier slot.  Also with the compact wire format and with trainValid; the bytes of the pinned slab
    around the slots in use stay untouched."""
    from primal_ppo_b200 import unpack_observations
    sc, twin, env = _setup(shape, monkeypatch)
    W, N, C, F, T = env.W, env.N, env.C, env.F, 5
    acts = torch.from_numpy(random_actions(4 * T, W, N, seed=4))
    obs_dev, vec_dev = _obs_buf(env, fmt), torch.empty((W, N, 4), device="cuda")
    tv = torch.empty((W, N, 5), device="cuda")
    for part, (compact, with_tv) in enumerate(((False, False), (True, False), (False, True), (True, True))):
        ring = env.make_host_ring(slots=T + 2, action_slots=T, compact=compact, with_train_valid=with_tv,
                                  obs=_ring_obs(fmt))
        ring["_slab"].fill_(GUARD)
        sb = ring["slot_bytes"]
        off_obs = int(env.host_layout(with_tv, compact).slot_bytes)
        n_obs = obs_dev.numel() * obs_dev.element_size()
        off_vec = off_obs + (n_obs + 255) // 256 * 256
        assert sb == off_vec + (W * N * 16 + 255) // 256 * 256
        assert sb == int(env.host_layout(with_tv, compact, obs=_ring_obs(fmt)).slot_bytes)
        slots = ring["slots"][1:T + 1]                    # the first and the last slot are guards
        want = _twin_steps(twin, acts[part * T:(part + 1) * T], fmt)
        ring["action_ring"].copy_(acts[part * T:(part + 1) * T])
        for t in range(T):
            h2d, d2h = env.step_observe_host_begin(ring["action_ring"][t], slots[t], obs_dev, vec_dev,
                                                   train_valid_dev=tv if with_tv else None, with_train_valid=with_tv)
            assert h2d == W * N and d2h == sb
        env.host_wait(0)                                  # the copy stream is in order: every slot has landed
        for t, s in enumerate(slots):
            what = (compact, with_tv, t)
            _check_slot(s, want[t], what, with_tv)
            assert torch.equal(s["obs"], want[t]["obs"].cpu()), what
            assert torch.equal(s["vec"], want[t]["vec"].cpu()), what
        if fmt == "bits":                                 # the host expansion equals the device's
            assert torch.equal(unpack_observations(slots[-1]["obs"], C, F),
                               unpack_observations(want[-1]["obs"], C, F).cpu())
        for g in (ring["slots"][0]["_raw"], ring["slots"][T + 1]["_raw"]):
            assert bool((g == GUARD).all()), (compact, with_tv)
        for s in slots:                                   # padding after the observation block and after vec
            raw = s["_raw"]
            assert bool((raw[off_obs + n_obs:off_vec] == GUARD).all()) and bool((raw[off_vec + W * N * 16:] == GUARD).all())


def test_gpu_host_obs_bits_full_size_equals_device_call():
    """65 536 worlds of 40x40 with 32 agents, bit-packed observations, compact wire format with MAPF_HOST_OBS, 8
    split-phase steps into alternating obs_dev buffers (a rollout buffer's pattern: no step waits for a copy): the
    per-world checksums of obs_dev, vec_dev, the decoded results and the host observations equal the device call."""
    from primal_ppo_b200 import checksum_rows
    W, N, T = 65536, 32, 8
    sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256)
    twin, env = _env(sc), _env(sc)
    obs_t = [_obs_buf(env, "bits") for _ in range(2)]
    vec_t = [torch.empty((W, N, 4), device="cuda") for _ in range(2)]
    ring = env.make_host_ring(slots=2, action_slots=2, compact=True, obs="bits")
    g = torch.Generator().manual_seed(1)
    acts = [torch.randint(0, 5, (W, N), generator=g, dtype=torch.int8) for _ in range(T)]
    want = _twin_steps(twin, acts, "bits")
    for t in range(T):
        ring["action_ring"][t & 1].copy_(acts[t])
        env.step_observe_host_begin(ring["action_ring"][t & 1], ring["slots"][t & 1], obs_t[t & 1], vec_t[t & 1])
        assert torch.equal(checksum_rows(obs_t[t & 1]), checksum_rows(want[t]["obs"])), t
        assert torch.equal(vec_t[t & 1], want[t]["vec"]), t
        if t >= 1:
            env.host_wait(1)
            s = ring["slots"][(t - 1) & 1]
            _check_slot(s, want[t - 1], t - 1)
            assert torch.equal(s["obs"], want[t - 1]["obs"].cpu()) and torch.equal(s["vec"], want[t - 1]["vec"].cpu()), t - 1
            want[t - 1] = None
    env.host_wait(0)
    s = ring["slots"][(T - 1) & 1]
    _check_slot(s, want[T - 1], T - 1)
    assert torch.equal(s["obs"], want[T - 1]["obs"].cpu()) and torch.equal(s["vec"], want[T - 1]["vec"].cpu())


def test_gpu_host_obs_misuse_raises():
    from primal_ppo_b200 import _cabi
    from primal_ppo_b200._cabi import MapfError
    W, N = 16, 8
    sc = random_scenario(W, 20, 20, N, density=(0.0, 0.3), queue_len=4, seed=2)
    env, twin = _env(sc), _env(sc)
    ring = env.make_host_ring(slots=2, action_slots=2, obs="bits")
    bits, vec = _obs_buf(env, "bits"), torch.empty((W, N, 4), device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    act = ring["action_ring"][0]
    slot = ring["slots"][0]

    def begin(flags, obs_ptr):
        return env._lib.mapf_step_observe_host_begin(env._h, ctypes.c_void_p(act.data_ptr()),
                                                     ctypes.c_void_p(slot["_raw"].data_ptr()), flags, obs_ptr,
                                                     ctypes.c_void_p(vec.data_ptr()), None, stream)
    both = _cabi.HOST_OBS_BF16 | _cabi.HOST_OBS_BITS
    with pytest.raises(MapfError, match="exclusive"):
        _cabi.check(begin(both, ctypes.c_void_p(bits.data_ptr())), "begin")
    with pytest.raises(MapfError, match="exclusive"):
        _cabi.check(env._lib.mapf_host_layout(env._h, both | _cabi.HOST_OBS, ctypes.byref(_cabi.MapfHostLayout())), "layout")
    raw = torch.empty((bits.numel() * 4 + 16,), dtype=torch.uint8, device="cuda")
    with pytest.raises(MapfError, match="4-byte aligned"):
        _cabi.check(begin(_cabi.HOST_OBS_BITS | _cabi.HOST_OBS, ctypes.c_void_p(raw.data_ptr() + 2)), "begin")
    with pytest.raises(MapfError, match="ring holds"):
        env.step_observe_host_begin(act, slot, torch.empty((W, N, 6, 9, 9), device="cuda"), vec)
    with pytest.raises(MapfError, match="train_valid"):     # the slot has no room for trainValid
        env.step_observe_host_begin(act, slot, bits, vec, with_train_valid=True)
    tv_ring = env.make_host_ring(slots=2, action_slots=2, with_train_valid=True, obs="bits")
    with pytest.raises(MapfError, match="train_valid"):     # its observation block starts after trainValid
        env.step_observe_host_begin(act, tv_ring["slots"][0], bits, vec)
    with pytest.raises(MapfError):
        env.host_wait(0)                                  # none of the refused calls started a step
    # the env is unaffected: the next begin gives the twin's first step
    a = torch.from_numpy(random_actions(1, W, N, seed=9))
    want = _twin_steps(twin, a, "bits")[0]
    act.copy_(a[0])
    env.step_observe_host_begin(act, slot, bits, vec)
    env.host_wait(0)
    _check_slot(slot, want, "after misuse")
    assert torch.equal(slot["obs"], want["obs"].cpu()) and torch.equal(slot["vec"], want["vec"].cpu())
