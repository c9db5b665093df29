"""Bit-packed observations on the GPU: every observation kernel family writes the same bits as the f32 path (which the
parity tests pin to the oracle), unpack_observations gathers and expands them exactly, and a VecPPOTrainer whose rollout
buffer stores bits reproduces the f32 trainer's rollout."""
import numpy as np
import pytest
import torch

from obs_bits_util import pack_obs
from oracle import OracleMapfGym
from primal_ppo_b200 import random_actions, random_scenario

pytestmark = pytest.mark.gpu

GUARD = 0x5A5A5A5A


def _env(sc, **kw):
    from primal_ppo_b200 import BatchedMapfGym
    return BatchedMapfGym(sc, use_tape=False, **kw)


def _same_step(o1, o2):
    for k in ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow_goals", "fixed_actions"):
        assert torch.equal(getattr(o1, k), getattr(o2, k)), k


def _unpacked_equal(bits, obs, C, F, chunk=4096):
    from primal_ppo_b200 import unpack_observations
    for lo in range(0, bits.shape[0], chunk):
        if not torch.equal(unpack_observations(bits[lo:lo + chunk], C, F), obs[lo:lo + chunk]):
            return False
    return True


# (W, H, Wd, N, F, C, eval channels, MAPF_DBG_FLAGS): the shapes of the bf16 test, lane groups of 8 / 16 agents, the
# CTA-per-world kernels at 128 agents and FOV 9..31 with the danger / human-path channels, five channels (AW = 13: the
# scalar store path), a single world, the stand-alone warp kernel with several chunks per world (flags 2: no CTA-per-world
# observe; flags 1: the two-launch step + observe fallback), and the two-launch fallback on lane-group worlds
CASES = [(512, 40, 40, 32, 9, 6, False, 0), (33, 20, 20, 8, 9, 6, False, 0), (7, 12, 9, 5, 9, 6, False, 0),
         (6, 64, 64, 31, 15, 6, False, 0), (4, 80, 80, 128, 21, 6, False, 0), (3, 9, 9, 3, 3, 6, False, 0),
         (64, 20, 20, 8, 9, 6, False, 0), (48, 24, 24, 16, 9, 6, False, 0),
         (6, 80, 80, 128, 9, 6, True, 0), (6, 80, 80, 128, 15, 6, True, 0), (6, 80, 80, 128, 21, 6, True, 0),
         (6, 80, 80, 128, 31, 6, True, 0), (40, 20, 20, 8, 9, 5, False, 0), (1, 40, 40, 32, 9, 6, False, 0),
         (6, 64, 64, 32, 31, 6, False, 3), (33, 20, 20, 8, 9, 6, False, 1)]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "W{}_{}x{}_N{}_F{}_C{}{}_f{}".format(*c[:6], "_eval" if c[6] else "", c[7]))
def test_gpu_bits_equal_f32_every_kernel_family(case, monkeypatch):
    W, H, Wd, N, F, C, ev, flags = case
    if flags:
        monkeypatch.setenv("MAPF_DBG_FLAGS", str(flags))       # read when the env is created
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.3), queue_len=3, seed=W + F + C, fov=F, num_channel=C,
                         use_da=ev, use_hp=ev, unique_maps=min(W, 32))
    e1, e2 = _env(sc), _env(sc)
    bits = torch.empty(e2.obs_bits_shape, dtype=torch.int32, device="cuda")
    vb = torch.empty((W, N, 4), device="cuda")
    obs, vec = e1.getAllObservations()
    e2.getAllObservations(out=(bits, vb))
    assert torch.equal(vb, vec) and _unpacked_equal(bits, obs, C, F)
    a = torch.from_numpy(random_actions(3, W, N, seed=1)).cuda()
    for t in range(3):
        o1, obs, vec = e1.step_observe(a[t])
        o2, _, _ = e2.step_observe(a[t], obs_out=(bits, vb))
        _same_step(o1, o2)
        assert torch.equal(vb, vec) and _unpacked_equal(bits, obs, C, F), (case, t)
    e1.getAllObservations(out=(obs, vec))
    e2.getAllObservations(out=(bits, vb))
    assert torch.equal(vb, vec) and _unpacked_equal(bits, obs, C, F)


@pytest.mark.parametrize("shape", [(64, 20, 20, 8, 9), (6, 64, 64, 31, 15)])
def test_gpu_bits_equal_packed_oracle_words(shape):
    """The raw words, padding bits included, equal the oracle's observations packed by the NumPy reference packer."""
    W, H, Wd, N, F = shape
    sc = random_scenario(W, H, Wd, N, density=(0.05, 0.3), queue_len=3, seed=7 + F, fov=F, unique_maps=min(W, 16))
    env, orc = _env(sc), OracleMapfGym(sc, threads=2, use_tape=False)
    bits = torch.empty(env.obs_bits_shape, dtype=torch.int32, device="cuda")
    vec = torch.empty((W, N, 4), device="cuda")
    env.getAllObservations(out=(bits, vec))
    assert np.array_equal(bits.cpu().numpy().view(np.uint32), pack_obs(orc.getAllObservations()[0]))
    acts = random_actions(3, W, N, seed=2)
    for t in range(3):
        env.step_observe(torch.from_numpy(acts[t]), obs_out=(bits, vec))
        orc.step(acts[t])
        o_obs, o_vec = orc.getAllObservations()
        assert np.array_equal(bits.cpu().numpy().view(np.uint32), pack_obs(o_obs)), t
        assert np.array_equal(vec.cpu().numpy(), o_vec)


@pytest.mark.parametrize("shape", [(64, 40, 40, 32, 9), (6, 80, 80, 128, 15), (40, 20, 20, 8, 9)])
def test_gpu_bits_guard_words_and_scalar_path(shape):
    """Words before and after the buffer stay untouched; a 4-byte-aligned (not 16-byte) buffer takes the scalar store path
    and gives the same words as the aligned one, from the stand-alone and the fused launch."""
    W, H, Wd, N, F = shape
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.3), queue_len=3, seed=5, fov=F, unique_maps=min(W, 16))
    envs = [_env(sc) for _ in range(2)]
    shp = envs[0].obs_bits_shape
    n = shp[0] * shp[1] * shp[2]
    raws = [torch.full((n + 8,), GUARD, dtype=torch.int32, device="cuda") for _ in range(2)]
    views = [raws[0][4:4 + n].view(shp), raws[1][1:1 + n].view(shp)]     # 16-byte aligned / 4-byte aligned
    assert views[0].data_ptr() % 16 == 0 and views[1].data_ptr() % 16 == 4
    vec = torch.empty((W, N, 4), device="cuda")
    a = torch.from_numpy(random_actions(3, W, N, seed=3)).cuda()
    for t in range(4):
        for e, b in zip(envs, views):
            if t == 0:
                e.getAllObservations(out=(b, vec))
            else:
                e.step_observe(a[t - 1], obs_out=(b, vec))
        assert torch.equal(views[0], views[1]), t
        assert bool((raws[0][:4] == GUARD).all() and (raws[0][4 + n:] == GUARD).all())
        assert bool((raws[1][:1] == GUARD).all() and (raws[1][1 + n:] == GUARD).all())


@pytest.mark.parametrize("shape", [(300, 40, 40, 32, 9), (5, 80, 80, 128, 31), (40, 20, 20, 7, 9)])
def test_gpu_unpack_gather_equals_index_select(shape):
    from primal_ppo_b200 import unpack_observations
    W, H, Wd, N, F = shape
    sc = random_scenario(W, H, Wd, N, density=(0.0, 0.3), queue_len=3, seed=11, fov=F, unique_maps=min(W, 16))
    e1, e2 = _env(sc), _env(sc)
    bits = torch.empty(e2.obs_bits_shape, dtype=torch.int32, device="cuda")
    vec = torch.empty((W, N, 4), device="cuda")
    a = torch.from_numpy(random_actions(1, W, N, seed=4)).cuda()
    _, obs, _ = e1.step_observe(a[0])
    e2.step_observe(a[0], obs_out=(bits, vec))
    g = torch.Generator(device="cuda").manual_seed(0)
    rows = torch.randint(0, W, (3 * W + 1,), generator=g, device="cuda")
    ref = obs.index_select(0, rows)
    assert torch.equal(unpack_observations(bits, 6, F, rows=rows), ref)
    assert torch.equal(unpack_observations(bits, 6, F, rows=rows, dtype=torch.bfloat16), ref.to(torch.bfloat16))
    assert torch.equal(unpack_observations(bits, 6, F, dtype=torch.bfloat16), obs.to(torch.bfloat16))
    # out-of-range indices give zero rows; the in-range ones are unaffected
    bad = torch.tensor([-1, 0, W, W + 1000, W - 1, -(1 << 40)], device="cuda")
    got = unpack_observations(bits, 6, F, rows=bad)
    assert torch.equal(got[1], obs[0]) and torch.equal(got[4], obs[W - 1])
    assert not bool(got[[0, 2, 3, 5]].any())
    # into a caller's (unaligned, scalar-path) buffer
    raw = torch.empty(rows.numel() * obs[0].numel() + 1, device="cuda")
    out = raw[1:].view(rows.numel(), *obs.shape[1:])
    unpack_observations(bits, 6, F, rows=rows, out=out)
    assert torch.equal(out, ref)


def test_gpu_bits_full_size_fused_steps():
    """65 536 worlds of 40x40 with 32 agents (the headline shape, W > 1024: the batched L2 prefetch path), 8 fused steps."""
    W, N = 65536, 32
    sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256)
    e1, e2 = _env(sc), _env(sc)
    obs = torch.empty((W, N, 6, 9, 9), device="cuda")
    vec = torch.empty((W, N, 4), device="cuda")
    bits = torch.empty(e2.obs_bits_shape, dtype=torch.int32, device="cuda")
    vb = torch.empty((W, N, 4), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    for t in range(8):
        a = torch.randint(0, 5, (W, N), generator=g, device="cuda", dtype=torch.int8)
        o1, _, _ = e1.step_observe(a, obs_out=(obs, vec))
        o2, _, _ = e2.step_observe(a, obs_out=(bits, vb))
        _same_step(o1, o2)
        assert torch.equal(vb, vec) and _unpacked_equal(bits, obs, 6, 9, chunk=8192), t


def test_gpu_trainer_bits_rollout_equals_f32():
    """fp32, deterministic cuDNN: a bit-packed rollout buffer gives the f32 trainer's rollout.  The env-side tensors are
    compared exactly.  The policy sees bit-identical inputs in both trainers (the bits trainer runs it on an expanded
    scratch tensor, the f32 trainer on a slice of its buffer); its outputs are compared with a tolerance of a few ulps,
    since cuDNN may pick its kernel by the address of the input as well as by its shape."""
    from primal_ppo_b200 import BatchedMapfGym
    from primal_ppo_b200.ppo import PPOConfig, ScrimpPolicy, VecPPOTrainer
    torch.backends.cudnn.deterministic = True
    W, N, T = 48, 8, 6
    sc = random_scenario(W, 20, 20, N, density=(0.05, 0.2), queue_len=4, seed=8, unique_maps=16)
    torch.manual_seed(0)
    p1 = ScrimpPolicy().cuda().eval()
    p2 = ScrimpPolicy().cuda().eval()
    p2.load_state_dict(p1.state_dict())
    cfg = PPOConfig(n_steps=T, n_epochs=1, minibatch_size=16)
    kw = dict(rows_per_minibatch=16, seed=11, forward_chunk_rows=128)       # several forward chunks per step
    t1 = VecPPOTrainer(BatchedMapfGym(sc, use_tape=False, seed=1), p1, cfg, **kw)
    t2 = VecPPOTrainer(BatchedMapfGym(sc, use_tape=False, seed=1), p2, cfg, obs_dtype="bits", **kw)
    assert t2.buf.obs.dtype == torch.int32 and tuple(t2.buf.obs.shape) == (T + 1, W, N, 16)
    perf1, perf2 = t1.collect(), t2.collect()
    b1, b2 = t1.buf, t2.buf
    for k in ("actions", "rewards", "cost_rewards", "status", "train_valid", "goals_reached", "violated", "shadow_goals",
              "fixed_actions", "vec"):
        assert torch.equal(getattr(b1, k), getattr(b2, k)), k
    for t in range(T + 1):
        assert _unpacked_equal(b2.obs[t], b1.obs[t], 6, 9), t
    for k in ("ps", "values", "cost_values", "returns", "cost_returns"):
        torch.testing.assert_close(getattr(b2, k), getattr(b1, k), rtol=1e-6, atol=1e-6, msg=k)
    assert perf1 == perf2
    rows = torch.randperm(T * W, device="cuda")[:20]
    m1, m2 = b1.minibatch(rows), b2.minibatch(rows)
    assert m2["obs"].dtype == torch.float32 and torch.equal(m1["obs"], m2["obs"])
    for k in m1:
        assert torch.equal(m1[k], m2[k]) or k in ("ps", "values", "cost_values", "returns", "cost_returns"), k
    stats = t2.update(perf2, max_minibatches=2)
    assert len(stats) == 2 and all(np.isfinite(s["all_loss"]) for s in stats)


def test_gpu_trainer_bits_bf16_autocast_expands_to_bf16():
    from primal_ppo_b200 import BatchedMapfGym
    from primal_ppo_b200.ppo import PPOConfig, ScrimpPolicy, VecPPOTrainer
    W, N, T = 16, 8, 3
    sc = random_scenario(W, 20, 20, N, density=(0.05, 0.2), queue_len=4, seed=9, unique_maps=8)
    tr = VecPPOTrainer(BatchedMapfGym(sc, use_tape=False, seed=1), ScrimpPolicy().cuda().eval(),
                       PPOConfig(n_steps=T, n_epochs=1, minibatch_size=8), amp_dtype=torch.bfloat16, obs_dtype="bits",
                       rows_per_minibatch=8)
    perf = tr.collect()
    mb = tr.buf.minibatch(torch.arange(8, device="cuda"))
    assert mb["obs"].dtype == torch.bfloat16 and mb["obs"].shape == (8, N, 6, 9, 9)
    stats = tr.update(perf, max_minibatches=1)
    assert len(stats) == 1 and np.isfinite(stats[0]["all_loss"])
