"""The float64 reference of the fused PPO loss (tests/ppo_loss_ref.py) against float64 autograd through ppo/loss.py, the
PyTorch statement of model.py:104-164 that tests/test_ppo_parity.py pins.  CPU only.

The reference uses the kernel's f32 constants; here loss.py is given the same numbers (coefficients that are exact in
f32, a clip range on the 2^-23 grid so that 1 -/+ clip is exact in f32 too) and inputs on which the two can only differ by
double rounding: differences returns - old_v exact in f32, sig on the 2^-24 grid (so f32(1 - sig) is exact), p and sig
away from the clamp bounds, and no element near a decision boundary."""
import dataclasses

import numpy as np
import pytest
import torch

import ppo_loss_ref as ref
from primal_ppo_b200.ppo.loss import PPOConfig, ppo_lagrange_loss
from primal_ppo_b200.ppo.policy import PolicyOutput

VARIANTS = {"default": PPOConfig(), "cost_terms": PPOConfig(cost_value_coef=0.05, cost_coef=0.2),
            "no_mix": PPOConfig(minus_adv_with_cadv=False, cost_coef=0.3, cost_value_coef=0.1)}


def f32_exact(cfg: PPOConfig) -> PPOConfig:
    f = lambda x: float(np.float32(x))
    return dataclasses.replace(cfg, clip_range=round(cfg.clip_range * 2 ** 23) / 2 ** 23, entropy_coef=f(cfg.entropy_coef),
                               value_coef=f(cfg.value_coef), valid_coef=f(cfg.valid_coef),
                               cost_value_coef=f(cfg.cost_value_coef), cost_coef=f(cfg.cost_coef))


def random_inputs(rng, n):
    f32 = np.float32
    grid = lambda x, q: (np.round(x * q) / q).astype(f32)
    logits = rng.standard_normal((n, 5)) * 2
    p = np.exp(logits) / np.exp(logits).sum(1, keepdims=True)
    d = dict(policy=((p + 1e-3) / (1 + 5e-3)).astype(f32),
             old_ps=((np.exp(logits + 0.3 * rng.standard_normal((n, 5))) + 1e-3)).astype(f32),
             sig=grid(np.clip(1 / (1 + np.exp(-3 * rng.standard_normal((n, 5)))), 1e-4, 1 - 1e-4), 2 ** 24),
             value=grid(rng.standard_normal(n), 2 ** 12), cost_value=grid(rng.standard_normal(n), 2 ** 12),
             returns=grid(rng.standard_normal(n), 2 ** 12), cost_returns=grid(rng.standard_normal(n), 2 ** 12),
             actions=rng.integers(0, 5, n).astype(np.int8),
             train_valid=(rng.random((n, 5)) < 0.6).astype(f32))
    d["old_ps"] = (d["old_ps"] / d["old_ps"].sum(1, keepdims=True)).astype(f32)
    # old values near and far from the new ones: the value clip active and inactive
    d["old_v"] = grid(d["value"] + rng.choice([0.05, 0.5], n) * rng.standard_normal(n), 2 ** 12)
    d["old_cv"] = grid(d["cost_value"] + rng.choice([0.05, 0.5], n) * rng.standard_normal(n), 2 ** 12)
    return d


def autograd_f64(cfg, lag, d):
    t = {k: torch.from_numpy(np.asarray(v)) for k, v in d.items()}
    leaves = [t[k].double().requires_grad_(True) for k in ("policy", "value", "cost_value", "sig")]
    kw = {f: None for f in PolicyOutput._fields}
    kw.update(policy=leaves[0], value=leaves[1].unsqueeze(-1), cost_value=leaves[2].unsqueeze(-1), policy_sig=leaves[3])
    loss, stats = ppo_lagrange_loss(PolicyOutput(**kw), returns=t["returns"].double(), cost_returns=t["cost_returns"].double(),
                                    old_v=t["old_v"].double(), old_cv=t["old_cv"].double(), actions=t["actions"].long(),
                                    old_ps=t["old_ps"].double(), train_valid=t["train_valid"].double(), lagrangian=lag,
                                    cfg=cfg, group=None)
    loss.backward()
    return float(loss.detach()), {k: float(v) for k, v in stats.items()}, [x.grad.numpy() for x in leaves]


@pytest.mark.parametrize("lag", [0.0, 0.7, 3.0])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_reference_equals_float64_autograd_through_loss_py(variant, lag):
    cfg = f32_exact(VARIANTS[variant])
    lag = float(np.float32(lag))
    rng = np.random.default_rng(17)
    d = random_inputs(rng, 6000)
    rc = ref.loss_config(cfg, lag, d["returns"], d["cost_returns"], d["old_v"], d["old_cv"])
    args = {k: d[k] for k in ("policy", "value", "cost_value", "sig", "returns", "cost_returns", "old_v", "old_cv",
                              "actions", "old_ps")}
    keep = ~ref.near_boundary(rc, **args)
    assert keep.mean() > 0.99
    d = {k: v[keep] for k, v in d.items()}
    rc = ref.loss_config(cfg, lag, d["returns"], d["cost_returns"], d["old_v"], d["old_cv"])
    r = ref.ppo_loss_ref(rc, **{k: d[k] for k in args}, train_valid=d["train_valid"])
    # the data exercise both sides of every decision
    assert 0.05 < r["clipped"].mean() < 0.95
    delta = np.abs(d["value"].astype(np.float64) - d["old_v"])
    assert 0.05 < (delta > cfg.clip_range).mean() < 0.95

    loss, stats, grads = autograd_f64(cfg, lag, d)
    sums, mags = r["stats"].sum(0), r["stats_mag"].sum(0)
    mine, mine_mag = ref.stat_means(rc, sums), ref.stat_mags(rc, mags)
    assert abs(mine["all_loss"] - loss) <= 1e-12 * mine_mag["all_loss"], (mine["all_loss"], loss)
    n = len(d["actions"])
    assert round(stats["clipfrac"] * n) == r["clipped"].sum() == sums[6]     # loss.py takes this mean in f32
    for k in ref.STAT_NAMES:
        if k == "clipfrac":
            continue
        assert abs(mine[k] - stats[k]) <= 1e-12 * mine_mag[k] + 1e-300, (k, mine[k], stats[k])
    assert r["stats"][:, 9].sum() == 0
    for name, g in zip(("g_policy", "g_value", "g_cost_value", "g_sig"), grads):
        err = np.abs(r[name] - g.reshape(r[name].shape))
        bound = 1e-12 * r[name + "_mag"] + 1e-300
        assert (err <= bound).all(), (name, float((err / np.maximum(bound, 1e-300)).max()))
