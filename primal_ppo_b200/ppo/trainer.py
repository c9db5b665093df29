"""Rollout + update loop over the GPU vector env (BASELINE.json configs[3]; reference: `runner.py:28-150` rollouts in 16
Ray actors, `driver.py:77-134` update loop, `model.py:78-199` minibatch step).

Design (one process per GPU, `torchrun`):
  * `RolloutBuffer` is the reference's `BatchValues` (`util.py:41-54`) as device tensors with a leading [T, W] shape.  The
    env kernels write straight into its slices (`mapf_step_observe` gets pointers to `reward[t]`, `obs[t+1]`, ...): there
    is no per-step stacking or host round trip.  `hiddenState` is not stored (the network ignores it, `net.py:102`).
  * actions are sampled on device by `mapf_sample_actions` (reference: per-agent `np.random.choice` on the host,
    `model.py:38-40`); returns come from the `mapf_gae` reverse-scan kernel (`runner.py:120-149`).
  * `PPOLearner.train_minibatch` is `Model.train`: loss -> backward -> gradient all-reduce -> Lagrange update -> clip ->
    Adam.  Gradients live in ONE flat fp32 buffer (parameters' `.grad` are views of it), so the multi-GPU exchange is a
    single NCCL all-reduce of 33 MB over NVLink; the loss is formed as a share of the global-minibatch mean
    (`loss.py`), so the summed gradient equals the single-process gradient on the concatenated minibatch.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.distributed as dist

from .lagrange import make_lagrangian
from .loss import PPOConfig, ppo_lagrange_loss, reduce_stats
from .policy import ScrimpPolicy


class PPOLearner:
    """`Model(global_model=True)` (`model.py:16-24`): network + Adam + Lagrange multiplier, data-parallel over `group`."""

    def __init__(self, policy: ScrimpPolicy, cfg: PPOConfig = PPOConfig(), group=None, amp_dtype=None, fused_loss=None):
        """fused_loss: compute the elementwise part of the loss and its gradients with the fused CUDA kernel
        (`fused_loss.py`, `csrc/ppo_loss.cu`) instead of the eager PyTorch statement in `loss.py`; default: on CUDA."""
        self.policy, self.cfg, self.group, self.amp_dtype = policy, cfg, group, amp_dtype
        self.params = [p for p in policy.parameters() if p.requires_grad]
        dev = self.params[0].device
        self.fused_loss = (dev.type == "cuda") if fused_loss is None else bool(fused_loss)
        n = sum(p.numel() for p in self.params)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:                       # .grad of every parameter is a view into the flat buffer
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.opt = torch.optim.Adam(self.params, lr=cfg.lr, fused=True if dev.type == "cuda" else None)
        self.lagrange = make_lagrangian(cfg.lagrangian_type, cfg.cost_limit_per_agent)

    def compute_gradients(self, batch: Dict[str, torch.Tensor]) -> Dict[str, float]:
        """Forward + loss + backward + all-reduce; leaves the global-minibatch gradient in `flat_grad`."""
        self.flat_grad.zero_()
        dev_type = self.flat_grad.device.type
        with torch.autocast(dev_type, dtype=self.amp_dtype, enabled=self.amp_dtype is not None):
            out = self.policy(batch["obs"], batch["vec"])
        out = type(out)(*[o.float() for o in out])
        if self.fused_loss:
            from .fused_loss import fused_ppo_lagrange_loss as loss_fn
        else:
            loss_fn = ppo_lagrange_loss
        loss, stats = loss_fn(out, returns=batch["returns"], cost_returns=batch["cost_returns"],
                                        old_v=batch["values"], old_cv=batch["cost_values"], actions=batch["actions"],
                                        old_ps=batch["ps"], train_valid=batch["train_valid"],
                                        lagrangian=self.lagrange.value(), cfg=self.cfg, group=self.group)
        loss.backward()
        if self.group is not None:
            dist.all_reduce(self.flat_grad, group=self.group)       # the one collective of the training loop
        return reduce_stats(stats, self.group)

    def train_minibatch(self, batch: Dict[str, torch.Tensor], episode_cost: float, n_agents: int) -> Dict[str, float]:
        stats = self.compute_gradients(batch)
        self.lagrange.update(episode_cost / n_agents)                # model.py:180
        gn = self.flat_grad.norm()                                   # clip_grad_norm_ over all parameters (:182)
        stats["grad_norm"] = float(gn)
        stats["lagrangian"] = self.lagrange.value()
        if not torch.isfinite(gn):
            # the reference's GradScaler skips a step whose gradients are inf / NaN (model.py:178-186); without this
            # guard one bad minibatch would poison Adam's moments and the weights for good.  The all-reduced gradient is
            # the same on every rank, so every rank skips together.
            self.skipped_steps = getattr(self, "skipped_steps", 0) + 1
            stats["skipped"] = 1.0
            return stats
        self.flat_grad.mul_(torch.clamp(self.cfg.max_grad_norm / (gn + 1e-6), max=1.0))
        self.opt.step()
        return stats

    # ---- checkpoints in the reference's layout (driver.py:164-208) ---------------------------------------------------
    def save_checkpoint(self, path: str, step: int = 0, episode: int = 0, reward: float = 0.0) -> None:
        """`net_checkpoint.pkl`: {"model", "optimizer", "step", "episode", "reward"} with "model" keyed like the
        reference's SCRIMPNet, so the reference's `evaluate.py` / `RETRAIN` path can load it; "lagrange" is an extra key."""
        torch.save({"model": self.policy.reference_state_dict(), "optimizer": self.opt.state_dict(), "step": int(step),
                    "episode": int(episode), "reward": float(reward), "lagrange": self.lagrange.state_dict()}, path)

    def load_checkpoint(self, path: str, load_optimizer: bool = True) -> dict:
        """Loads a checkpoint written by `save_checkpoint` OR by the reference (`driver.py:189-194`).  The reference's Adam
        state is indexed by ITS parameter order and is therefore only restored from checkpoints written here."""
        ck = torch.load(path, map_location=self.flat_grad.device, weights_only=True)   # tensors / dicts / scalars only
        self.policy.load_reference_state_dict(ck["model"])
        if load_optimizer and "lagrange" in ck:
            self.opt.load_state_dict(ck["optimizer"])
            self.lagrange.load_state_dict(ck["lagrange"])
        return {k: ck[k] for k in ("step", "episode", "reward") if k in ck}

    def state_dict(self):
        return {"model": self.policy.state_dict(), "optimizer": self.opt.state_dict(),
                "lagrange": self.lagrange.state_dict()}

    def load_state_dict(self, sd):
        self.policy.load_state_dict(sd["model"])
        self.opt.load_state_dict(sd["optimizer"])
        self.lagrange.load_state_dict(sd["lagrange"])


@dataclass
class RolloutBuffer:
    obs: torch.Tensor            # f32 [T+1, W, N, C, F, F] (or bf16; or bit-packed int32 [T+1, W, N, AW])
    vec: torch.Tensor            # f32 [T+1, W, N, 4]
    actions: torch.Tensor        # i8  [T, W, N]
    ps: torch.Tensor             # f32 [T, W, N, 5]
    values: torch.Tensor         # f32 [T, W, N]
    cost_values: torch.Tensor
    rewards: torch.Tensor
    cost_rewards: torch.Tensor
    train_valid: torch.Tensor    # f32 [T, W, N, 5]
    status: torch.Tensor         # i8  [T, W, N]
    goals_reached: torch.Tensor  # u8  [T, W, N]
    violated: torch.Tensor       # u8  [T, W, N]
    shadow_goals: torch.Tensor   # i32 [T, W]
    fixed_actions: torch.Tensor  # i8  [T, W, N]
    returns: Optional[torch.Tensor] = None
    cost_returns: Optional[torch.Tensor] = None
    obs_cf: tuple = (0, 0)                        # (C, F) of the observations (what bit-packed rows expand to)
    unpack_dtype: torch.dtype = torch.float32     # dtype bit-packed observations expand to (f32, or bf16 under bf16 autocast)

    @staticmethod
    def allocate(T, W, N, C, F, device, obs_dtype=torch.float32, unpack_dtype=torch.float32):
        """obs_dtype: torch.float32 (the reference's layout), torch.bfloat16, or "bits" (one bit per cell: int32
        [T+1, W, N, AW], 64 B per agent at 6 x 9 x 9 instead of 1944 B; expanded to `unpack_dtype` when read)."""
        from .._cabi import obs_bits_words
        z = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device=device)
        obs = (z(T + 1, W, N, obs_bits_words(C, F), dt=torch.int32) if obs_dtype == "bits"
               else z(T + 1, W, N, C, F, F, dt=obs_dtype))
        return RolloutBuffer(obs=obs, vec=z(T + 1, W, N, 4), actions=z(T, W, N, dt=torch.int8),
                             ps=z(T, W, N, 5), values=z(T, W, N), cost_values=z(T, W, N), rewards=z(T, W, N),
                             cost_rewards=z(T, W, N), train_valid=z(T, W, N, 5), status=z(T, W, N, dt=torch.int8),
                             goals_reached=z(T, W, N, dt=torch.uint8), violated=z(T, W, N, dt=torch.uint8),
                             shadow_goals=z(T, W, dt=torch.int32), fixed_actions=z(T, W, N, dt=torch.int8),
                             obs_cf=(C, F), unpack_dtype=unpack_dtype)

    def minibatch(self, rows: torch.Tensor) -> Dict[str, torch.Tensor]:
        """rows: flat indices into the [T*W] (time, world) rows; a row carries all N agents of one world."""
        T, W = self.actions.shape[:2]

        def g(x):
            return x[:T].reshape(T * W, *x.shape[2:]).index_select(0, rows)
        if self.obs.dtype == torch.int32:        # bit-packed: gather and expand in one kernel pass
            from ..vec_env import unpack_observations
            obs = unpack_observations(self.obs[:T].reshape(T * W, *self.obs.shape[2:]), *self.obs_cf, rows=rows,
                                      dtype=self.unpack_dtype)
        else:
            obs = g(self.obs)
        return dict(obs=obs, vec=g(self.vec), actions=g(self.actions), ps=g(self.ps), values=g(self.values),
                    cost_values=g(self.cost_values), returns=g(self.returns), cost_returns=g(self.cost_returns),
                    train_valid=g(self.train_valid))


class VecPPOTrainer:
    """Rollouts of T steps over the W lockstep worlds of a `BatchedMapfGym`, then `n_epochs` passes of minibatch updates.

    `rows_per_minibatch` (time, world) rows of N agents form one minibatch PER RANK; the reference uses
    MINIBATCH_SIZE = 256 rows of one env (`driver.py:121-131`; its index set only ever covers the first env's rows)."""

    def __init__(self, env, policy: ScrimpPolicy, cfg: PPOConfig = PPOConfig(), group=None, amp_dtype=None,
                 rows_per_minibatch: Optional[int] = None, forward_chunk_rows: int = 1 << 15, seed: int = 1234,
                 obs_dtype=torch.float32, fresh_worlds=None):
        """fresh_worlds: callable(rollout_index) -> scenario with the env's shapes; when given, every rollout starts on
        new worlds, as the reference does (`env = MapfGym()` in `Runner.run`, runner.py:30).
        obs_dtype=torch.bfloat16 stores the rollout's observations in the env's optional bf16 format (same values, half
        the memory and half the env's store traffic); it needs amp_dtype=torch.bfloat16.
        obs_dtype="bits" stores them bit-packed (one bit per cell, 1/30 of the f32 memory); each forward chunk and each
        minibatch is expanded by one kernel pass into bf16 when amp_dtype is torch.bfloat16, f32 otherwise."""
        if obs_dtype == torch.bfloat16 and amp_dtype != torch.bfloat16:
            raise ValueError("bf16 observations need amp_dtype=torch.bfloat16 (the fp32 convolution would reject them)")
        self.env, self.policy, self.cfg, self.group = env, policy, cfg, group
        self.learner = PPOLearner(policy, cfg, group, amp_dtype)
        self.amp_dtype = amp_dtype
        self.T = cfg.n_steps
        self.rows_per_minibatch = rows_per_minibatch or cfg.minibatch_size
        self.chunk = forward_chunk_rows
        self.seed, self.sample_calls = seed, 0
        self.fresh_worlds, self.rollouts = fresh_worlds, 0
        self.unpack_dtype = torch.bfloat16 if amp_dtype == torch.bfloat16 else torch.float32
        self.buf = RolloutBuffer.allocate(self.T, env.W, env.N, env.C, env.F, env.device, obs_dtype, self.unpack_dtype)
        self._obs_scratch = None         # expanded observations of one forward chunk (bit-packed rollouts only)
        self.gen = torch.Generator(device=env.device); self.gen.manual_seed(seed)
        env.getAllObservations(out=(self.buf.obs[0], self.buf.vec[0]))

    @torch.no_grad()
    def _forward(self, obs, vec, ps, values, cost_values):
        W, N = obs.shape[:2]
        step = max(1, self.chunk // N)
        if obs.dtype == torch.int32 and self._obs_scratch is None:
            C, F = self.buf.obs_cf
            self._obs_scratch = torch.empty((min(W, step), N, C, F, F), dtype=self.unpack_dtype, device=obs.device)
        for lo in range(0, W, step):
            hi = min(W, lo + step)
            x = obs[lo:hi]
            if obs.dtype == torch.int32:
                from ..vec_env import unpack_observations
                x = unpack_observations(x, *self.buf.obs_cf, dtype=self.unpack_dtype, out=self._obs_scratch[:hi - lo])
            with torch.autocast(obs.device.type, dtype=self.amp_dtype, enabled=self.amp_dtype is not None):
                o = self.policy(x, vec[lo:hi])
            if ps is not None:
                ps[lo:hi] = o.policy.float()
            values[lo:hi] = o.value.float().squeeze(-1)
            cost_values[lo:hi] = o.cost_value.float().squeeze(-1)

    @torch.no_grad()
    def collect(self) -> Dict[str, float]:
        """`Runner.run` (`runner.py:28-150`) for all worlds at once."""
        from ..vec_env import StepOut, gae2, sample_actions
        b, env = self.buf, self.env
        if self.fresh_worlds is not None and self.rollouts > 0:
            env.reset(self.fresh_worlds(self.rollouts))
            env.getAllObservations(out=(b.obs[0], b.vec[0]))
        elif self.sample_calls:      # continue from the last observation of the previous rollout
            b.obs[0].copy_(b.obs[self.T]); b.vec[0].copy_(b.vec[self.T])
        self.rollouts += 1
        for t in range(self.T):
            self._forward(b.obs[t], b.vec[t], b.ps[t], b.values[t], b.cost_values[t])
            sample_actions(b.ps[t], seed=self.seed, draw=self.sample_calls, out=b.actions[t])
            self.sample_calls += 1
            out = StepOut(status=b.status[t], reward=b.rewards[t], cost=b.cost_rewards[t], train_valid=b.train_valid[t],
                          goals_reached=b.goals_reached[t], violated=b.violated[t], shadow_goals=b.shadow_goals[t],
                          fixed_actions=b.fixed_actions[t])
            env.step_observe(b.actions[t], out=out, obs_out=(b.obs[t + 1], b.vec[t + 1]))
        last_v = torch.empty_like(b.values[0]); last_cv = torch.empty_like(b.values[0])
        self._forward(b.obs[self.T], b.vec[self.T], None, last_v, last_cv)
        b.returns, b.cost_returns = gae2(b.rewards, b.values, last_v, b.cost_rewards, b.cost_values, last_cv,
                                         self.cfg.gamma, self.cfg.lam)          # both streams, one launch
        # OneEpPerformance means over worlds (driver.py:101-112)
        perf = dict(episodeReward=float(b.rewards.sum(dim=(0, 2)).mean()),
                    episodeCostReward=float(b.cost_rewards.sum(dim=(0, 2)).mean()),
                    totalGoals=float(b.goals_reached.sum(dim=(0, 2), dtype=torch.float32).mean()),
                    constraintViolations=float(b.violated.sum(dim=(0, 2), dtype=torch.float32).mean()),
                    staticCollide=float((b.status == -1).sum(dim=(0, 2), dtype=torch.float32).mean()),
                    humanCollide=float((b.status == -2).sum(dim=(0, 2), dtype=torch.float32).mean()),
                    agentCollide=float((b.status == -3).sum(dim=(0, 2), dtype=torch.float32).mean()),
                    shadowGoals=float(b.shadow_goals.sum(dim=0, dtype=torch.float32).mean()))
        if self.group is not None:
            # mean over ALL worlds of the job: ranks may own different numbers of worlds (shard_range), so the per-rank
            # means are weighted by the rank's world count
            keys = sorted(perf)
            t = torch.tensor([perf[k] * env.W for k in keys] + [float(env.W)], dtype=torch.float64, device=env.device)
            dist.all_reduce(t, group=self.group)
            perf = {k: float(v) / float(t[-1]) for k, v in zip(keys, t[:-1])}
        return perf

    def update(self, perf: Dict[str, float], max_minibatches: Optional[int] = None):
        """`driver.py:121-131`: n_epochs shuffled passes over the rollout rows."""
        rows_total = self.T * self.env.W
        per_epoch = rows_total // self.rows_per_minibatch
        if self.group is not None:
            # every minibatch issues collectives (advantage statistics, gradient all-reduce): all ranks must run the SAME
            # number of them even when shard_range gave some ranks one world more than others
            t = torch.tensor([per_epoch], dtype=torch.int64, device=self.env.device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
            per_epoch = int(t.item())
        stats, done = [], 0
        for _ in range(self.cfg.n_epochs):
            perm = torch.randperm(rows_total, generator=self.gen, device=self.env.device)
            for mb in range(per_epoch):
                lo = mb * self.rows_per_minibatch
                batch = self.buf.minibatch(perm[lo:lo + self.rows_per_minibatch])
                stats.append(self.learner.train_minibatch(batch, perf["episodeCostReward"], self.env.N))
                done += 1
                if max_minibatches is not None and done >= max_minibatches:
                    return stats
        return stats
