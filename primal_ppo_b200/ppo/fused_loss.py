"""PPO-Lagrangian minibatch loss through the fused elementwise kernel (`csrc/ppo_loss.cu`, `mapf_adv_moments` +
`mapf_ppo_loss`): the same function as `loss.ppo_lagrange_loss` (reference: `model.py:104-164`), which remains the
checked PyTorch statement of it (`tests/test_gpu_ppo.py` compares values and gradients).

One autograd node: forward computes the loss statistics AND the gradients with respect to the four network outputs in a
single pass over the minibatch; backward hands those gradients (scaled by the incoming gradient) to autograd, which
continues into the network.  CUDA only — there is no CPU fallback; CPU runs (the gloo tests) use `loss.py`."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Tuple

import torch
import torch.distributed as dist

from .. import _cabi
from .loss import PPOConfig


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _mean_std(s: float, s2: float, n: float) -> Tuple[float, float]:
    """Mean and unbiased std of n values from their sum and sum of squares.  The std of a single value is NaN, as
    `x.std()` gives it in model.py:106 and loss.py, so a one-element minibatch yields a NaN loss instead of an error."""
    mean = s / n
    if n <= 1.0:
        return mean, float("nan")
    return mean, max((s2 - n * mean * mean) / (n - 1.0), 0.0) ** 0.5


class _FusedPPOLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, policy, value, cost_value, policy_sig, returns, cost_returns, old_v, old_cv, actions, old_ps, train_valid,
                lagrangian: float, cfg: PPOConfig, group):
        lib = _cabi.load_library()
        dev = policy.device
        f = lambda t: t.detach().contiguous().float()
        policy, value, cost_value, policy_sig = f(policy), f(value).reshape(-1), f(cost_value).reshape(-1), f(policy_sig)
        returns, cost_returns, old_v, old_cv = (f(t).reshape(-1) for t in (returns, cost_returns, old_v, old_cv))
        old_ps, train_valid = f(old_ps), f(train_valid)
        actions = actions.detach().contiguous().to(torch.int8).reshape(-1)
        n = int(returns.numel())
        assert policy.numel() == n * 5 and policy_sig.numel() == n * 5 and value.numel() == n and actions.numel() == n
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with torch.cuda.device(dev):
            pm = torch.empty((_cabi.PPO_LOSS_MAX_BLOCKS, 4), dtype=torch.float64, device=dev)
            _cabi.check(lib.mapf_adv_moments(_ptr(returns), _ptr(cost_returns), _ptr(old_v), _ptr(old_cv), n, _ptr(pm), stream),
                        "mapf_adv_moments")
            m = torch.cat([pm.sum(0), torch.tensor([float(n)], dtype=torch.float64, device=dev)])
            if group is not None:
                dist.all_reduce(m, group=group)            # (sum a, sum a^2, sum c, sum c^2, count) of the GLOBAL minibatch
            m = m.tolist()
            ng = m[4]
            am, astd = _mean_std(m[0], m[1], ng)
            cm, cstd = _mean_std(m[2], m[3], ng)
            kc = _cabi.MapfPpoLossConfig(clip_range=cfg.clip_range, entropy_coef=cfg.entropy_coef, value_coef=cfg.value_coef,
                                         valid_coef=cfg.valid_coef, cost_value_coef=cfg.cost_value_coef, cost_coef=cfg.cost_coef,
                                         lagrangian=float(lagrangian), minus_adv_with_cadv=int(cfg.minus_adv_with_cadv),
                                         n_global=ng, adv_mean=am, adv_std=astd, cadv_mean=cm, cadv_std=cstd)
            g_policy, g_sig = torch.empty_like(policy), torch.empty_like(policy_sig)
            g_value, g_cv = torch.empty_like(value), torch.empty_like(cost_value)
            part = torch.empty((_cabi.PPO_LOSS_MAX_BLOCKS, _cabi.PPO_LOSS_STATS), dtype=torch.float64, device=dev)
            _cabi.check(lib.mapf_ppo_loss(C.byref(kc), n, _ptr(policy), _ptr(value), _ptr(cost_value), _ptr(policy_sig), _ptr(returns),
                                          _ptr(cost_returns), _ptr(old_v), _ptr(old_cv), _ptr(actions), _ptr(old_ps),
                                          _ptr(train_valid), _ptr(g_policy), _ptr(g_value), _ptr(g_cv), _ptr(g_sig), _ptr(part),
                                          stream), "mapf_ppo_loss")
            st = part.sum(0) / ng                           # this rank's share of every global-minibatch mean
        policy_loss, entropy, critic, cost_critic = st[0], st[1], st[2], st[3]
        valid_loss = -st[4] / 5.0
        cost_loss = st[5]
        loss = (-policy_loss - entropy * cfg.entropy_coef + cfg.value_coef * critic + cfg.valid_coef * valid_loss
                + cfg.cost_value_coef * cost_critic + cfg.cost_coef * float(lagrangian) * cost_loss)
        ctx.save_for_backward(g_policy, g_value, g_cv, g_sig)
        stats = torch.stack([loss, policy_loss, entropy, critic, valid_loss, cost_critic, cost_loss, st[6], st[7], st[8]]).float()
        ctx.mark_non_differentiable(stats)
        return loss.float(), stats

    @staticmethod
    def backward(ctx, g_loss, _g_stats):
        g_policy, g_value, g_cv, g_sig = ctx.saved_tensors
        return (g_policy * g_loss, g_value * g_loss, g_cv * g_loss, g_sig * g_loss) + (None,) * 10


_STAT_NAMES = ("all_loss", "policy_loss", "policy_entropy", "critic_loss", "valid_loss", "cost_critic_loss", "cost_loss",
               "clipfrac", "advantage", "cost_advantage")


def fused_ppo_lagrange_loss(out, *, returns, cost_returns, old_v, old_cv, actions, old_ps, train_valid, lagrangian: float,
                            cfg: PPOConfig, group=None) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """Drop-in for `loss.ppo_lagrange_loss` on CUDA tensors: (loss, stats) with the same meaning — `loss` is this rank's
    share of the global-minibatch loss, `stats` the shares of its terms."""
    if not out.policy.is_cuda:
        raise _cabi.MapfError("fused_ppo_lagrange_loss needs CUDA tensors; there is no CPU fallback (use loss.ppo_lagrange_loss)")
    shp = out.policy.shape[:-1]
    loss, stats = _FusedPPOLoss.apply(out.policy.reshape(-1, 5), out.value.reshape(shp).reshape(-1), out.cost_value.reshape(shp).reshape(-1),
                                      out.policy_sig.reshape(-1, 5), returns, cost_returns, old_v, old_cv, actions, old_ps, train_valid,
                                      lagrangian, cfg, group)
    return loss, {k: stats[i] for i, k in enumerate(_STAT_NAMES)}
