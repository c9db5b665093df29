"""The fused PPO-loss kernels (csrc/ppo_loss.cu: mapf_adv_moments, mapf_ppo_loss) against the float64 reference of
tests/ppo_loss_ref.py at the sizes where the grid-stride loop and the block tails change, at the clamp and tie edges,
through shards, and with their buffer contracts; plus the masked GAE scan on the float4 path and action sampling past
one pass of its grid.

Random elements are kept 1e-5 (relative) away from every decision boundary that is taken on a computed value, so the
tolerances follow from f32 arithmetic alone: per gradient element 2^-17 of its magnitude (the sum of the absolute values
of the terms that make it up), per statistic 2^-18 of the mean magnitude, and the clip count exactly."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import ppo_loss_ref as ref
from oracle import gae_oracle, sample_actions_oracle
from primal_ppo_b200 import _cabi
from primal_ppo_b200.ppo.loss import PPOConfig

pytestmark = pytest.mark.gpu

F32 = np.float32
MAXB, NS = _cabi.PPO_LOSS_MAX_BLOCKS, _cabi.PPO_LOSS_STATS
GRAD_TOL, STAT_TOL = 2.0 ** -17, 2.0 ** -18
VARIANTS = [("default", PPOConfig(), 0.7), ("cost_terms", PPOConfig(cost_value_coef=0.05, cost_coef=0.2), 3.0),
            ("no_mix", PPOConfig(minus_adv_with_cadv=False, cost_coef=0.3, cost_value_coef=0.1), 0.0)]
GRADS = ("g_policy", "g_value", "g_cost_value", "g_sig")
INPUTS = ("policy", "value", "cost_value", "sig", "returns", "cost_returns", "old_v", "old_cv", "actions", "old_ps",
          "train_valid")
GUARDED = INPUTS[:-1]


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- data --------------------------------------------------------------------------------------------------------------

def _draw(rng, n):
    logits = rng.standard_normal((n, 5)) * 3
    p = np.exp(logits) / np.exp(logits).sum(1, keepdims=True)
    lo = logits + 0.3 * rng.standard_normal((n, 5))
    op = np.exp(lo) / np.exp(lo).sum(1, keepdims=True)
    value, cost_value = rng.standard_normal(n), rng.standard_normal(n)
    d = dict(policy=p, old_ps=op, sig=1 / (1 + np.exp(-4 * rng.standard_normal((n, 5)))), value=value, cost_value=cost_value,
             returns=rng.standard_normal(n), cost_returns=0.5 * rng.standard_normal(n) + 0.3,
             old_v=value + rng.choice([0.05, 0.5], n) * rng.standard_normal(n),
             old_cv=cost_value + rng.choice([0.05, 0.5], n) * rng.standard_normal(n),
             actions=rng.integers(0, 5, n), train_valid=rng.random((n, 5)) < 0.6)
    d = {k: np.asarray(v, np.int8 if k == "actions" else F32) for k, v in d.items()}
    same = rng.random(n) < 0.05                      # ratio exactly 1: old_ps == policy
    d["old_ps"][same] = d["policy"][same]
    return d


def random_batch(rng, n, clip):
    """n random elements, none within 1e-5 of a decision boundary (offending elements are redrawn)."""
    d = _draw(rng, n)
    for _ in range(20):
        bad = np.flatnonzero(ref.near_boundary(dict(clip_range=clip), **{k: d[k] for k in GUARDED}))
        if bad.size == 0:
            return d
        fresh = _draw(rng, bad.size)
        for k in d:
            d[k][bad] = fresh[k]
    raise AssertionError("could not draw a batch away from the boundaries")


def edge_rows(rng, clip, adv_mean, cadv_mean):
    """Elements placed exactly on the kernel's edges; each starts from a clean random element and changes only the
    fields its edge needs.  adv_mean / cadv_mean (f32 values) are the statistics the caller will pass, so that
    returns - old_v == adv_mean gives an advantage of exactly 0."""
    L = F32(ref.P_LO)
    S_HI = F32(ref.SIG_HI)
    c = F32(clip)
    rows = []

    def base():
        return {k: v[0].copy() for k, v in random_batch(rng, 1, clip).items()}
    # probabilities on and around the clamp bound and at 0 and 1, for each action, with ratio exactly 1 or far from 1 -/+ clip
    for x in (F32(0), L, np.nextafter(L, F32(0)), np.nextafter(L, F32(1)), F32(1)):
        for a in range(5):
            for old in ("same", "half"):
                r = base()
                r["policy"][:] = (F32(1) - x) / F32(4)
                r["policy"][a] = x
                r["actions"] = np.int8(a)
                r["old_ps"][:] = r["policy"] if old == "same" else F32(0.125)
                if old == "half":
                    r["old_ps"][a] = F32(0.5)
                rows.append(r)
    for a in range(5):                               # one-hot rows; old probability of the action 1, or 0
        for old_p in (F32(1), F32(0)):
            r = base()
            r["policy"][:] = 0
            r["policy"][a] = 1
            r["actions"] = np.int8(a)
            r["old_ps"][:] = (F32(1) - old_p) / F32(4)
            r["old_ps"][a] = old_p
            rows.append(r)
    # sigmoid outputs on the clamp bounds, their f32 neighbours, 0 and 1
    sv = [F32(0), F32(1), L, S_HI, np.nextafter(L, F32(0)), np.nextafter(L, F32(1)), np.nextafter(S_HI, F32(0)),
          np.nextafter(S_HI, F32(1)), np.nextafter(F32(0), F32(1)), np.nextafter(F32(1), F32(0))]
    for i in range(0, len(sv), 5):
        for tv in (0.0, 1.0):
            r = base()
            r["sig"][:] = sv[i:i + 5]
            r["train_valid"][:] = tv
            rows.append(r)
    # value deltas exactly -/+ clip (old = 0, so the delta is exact): the closed-interval mask decides
    h = F32(2.0 ** -6)
    for sgn in (F32(1), F32(-1)):
        for which in (("value", "old_v", "returns"), ("cost_value", "old_cv", "cost_returns")):
            r = base()
            v, o, t = which
            r[o], r[v], r[t] = F32(0), sgn * c, sgn * (c + F32(0.3))
            rows.append(r)
            # a value-loss tie e1 == e2 with the clip active: the target half way between the value and the clipped value
            r = base()
            r[o], r[v], r[t] = F32(0), sgn * (c + 2 * h), sgn * (c + h)
            assert (r[v] - r[t]) == -(sgn * c - r[t]) and r[t] - sgn * c == sgn * h
            rows.append(r)
    # advantage exactly 0 (and cost advantage exactly 0, so that the mixed advantage is 0 too)
    for _ in range(5):
        r = base()
        r["old_v"], r["returns"], r["old_cv"], r["cost_returns"] = F32(0), F32(adv_mean), F32(0), F32(cadv_mean)
        r["value"], r["cost_value"] = F32(adv_mean) + F32(0.05), F32(cadv_mean) - F32(0.05)
        rows.append(r)
    e = {k: np.stack([r[k] for r in rows]) for k in rows[0]}
    assert not ref.near_boundary(dict(clip_range=clip), **{k: e[k] for k in GUARDED}, inputs=False).any()
    return e


def batch(rng, n, clip, edges=True):
    """n elements: random ones with (if n allows) the edge rows scattered among them.  Returns (data, rounded means),
    where the means are the data's, rounded to f32, and the zero-advantage rows were built against them."""
    d = random_batch(rng, n, clip)
    am = float(F32((d["returns"].astype(np.float64) - d["old_v"]).mean()))
    cm = float(F32((d["cost_returns"].astype(np.float64) - d["old_cv"]).mean()))
    if edges:
        e = edge_rows(rng, clip, am, cm)
        assert n >= 2 * len(e["actions"])
        at = np.sort(rng.choice(n, size=len(e["actions"]), replace=False))
        for k in d:
            d[k][at] = e[k]
    return d, am, cm


def abi_config(variant, n, d, am=None, cm=None):
    """The reference's config: the PPOConfig, n_global = n, the data's two-pass statistics (means replaced by am, cm)."""
    _, cfg, lag = variant
    rc = ref.loss_config(cfg, lag, d["returns"], d["cost_returns"], d["old_v"], d["old_cv"])
    rc["n_global"] = float(n)
    if am is not None:
        rc["adv_mean"], rc["cadv_mean"] = am, cm
    return rc


def kernel_config(rc):
    f = {k: rc[k] for k in ("clip_range", "entropy_coef", "value_coef", "valid_coef", "cost_value_coef", "cost_coef",
                            "lagrangian", "n_global", "adv_mean", "adv_std", "cadv_mean", "cadv_std")}
    return _cabi.MapfPpoLossConfig(minus_adv_with_cadv=int(rc["minus_adv_with_cadv"]), **f)


def to_dev(d):
    return {k: torch.from_numpy(np.ascontiguousarray(v.astype(np.float32) if k == "train_valid" else v)).cuda()
            for k, v in d.items()}


def nan_outputs(n):
    g = dict(g_policy=torch.full((n, 5), float("nan"), device="cuda"), g_value=torch.full((n,), float("nan"), device="cuda"),
             g_cost_value=torch.full((n,), float("nan"), device="cuda"), g_sig=torch.full((n, 5), float("nan"), device="cuda"))
    return g, torch.full((MAXB, NS), float("nan"), dtype=torch.float64, device="cuda")


def call_moments(t, n=None, lo=0):
    lib = _cabi.load_library()
    n = int(t["returns"].numel()) - lo if n is None else n
    pm = torch.full((MAXB, 4), float("nan"), dtype=torch.float64, device="cuda")
    s = lambda k: t[k][lo:]
    _cabi.check(lib.mapf_adv_moments(_ptr(s("returns")), _ptr(s("cost_returns")), _ptr(s("old_v")), _ptr(s("old_cv")), n,
                                     _ptr(pm), _stream()), "mapf_adv_moments")
    return pm


def call_loss(rc, t, g, part, n=None, lo=0):
    """mapf_ppo_loss on elements [lo, lo + n) of the device inputs t, into the gradient buffers g (entries may be None)."""
    lib = _cabi.load_library()
    n = int(t["returns"].numel()) - lo if n is None else n
    s = lambda k: t[k][lo:]
    gs = lambda k: None if g.get(k) is None else g[k][lo:]
    kc = kernel_config(rc)
    _cabi.check(lib.mapf_ppo_loss(C.byref(kc), n, *[_ptr(s(k)) for k in INPUTS], *[_ptr(gs(k)) for k in GRADS], _ptr(part),
                                  _stream()), "mapf_ppo_loss")


def blocks(n):
    return min((n + 255) // 256, MAXB)


def assert_grads_close(r, got, what=""):
    for k in GRADS:
        x = got[k].double().cpu().numpy().reshape(r[k].shape)
        err = np.abs(x - r[k])
        bound = GRAD_TOL * r[k + "_mag"] + 1e-30
        bad = ~(err <= bound)
        assert not bad.any(), (what, k, np.argwhere(bad)[:5].tolist(), x[bad][:5], r[k][bad][:5], r[k + "_mag"][bad][:5])


def assert_stats_close(rc, r, sums, what=""):
    """Kernel partial sums (10) against the reference: means within 2^-18 of the mean magnitude, the clip count exact."""
    n = rc["n_global"]
    want, mag = r["stats"].sum(0), r["stats_mag"].sum(0)
    sums = np.asarray(sums, np.float64)
    assert sums[6] == r["clipped"].sum(), (what, sums[6], r["clipped"].sum())
    assert sums[9] == 0.0
    for j in (0, 1, 2, 3, 4, 5, 7, 8):
        assert abs(sums[j] - want[j]) / n <= STAT_TOL * mag[j] / n + 1e-12, (what, j, sums[j] / n, want[j] / n, mag[j] / n)


# ---- through the C ABI: grid sizes, edges, moments, contracts ------------------------------------------------------------

SIZES = [1, 255, 256, 257, 262143, 262144, 262145, 3 * 10 ** 6 + 77]


@pytest.mark.parametrize("n", SIZES)
def test_abi_loss_and_moments_match_float64_reference(n):
    """mapf_adv_moments and mapf_ppo_loss at sizes around the block size and the 1024-block grid-stride wrap, edges mixed in:
    moment sums to 1e-12, gradients per element, statistics, the clip count, and the unused partial rows zeroed."""
    variant = VARIANTS[SIZES.index(n) % 3]
    rng = np.random.default_rng(1000 + n)
    d, am, cm = batch(rng, n, variant[1].clip_range, edges=n >= 255)
    rc = abi_config(variant, n, d, am, cm)
    if n == 1:                                            # the ABI takes the statistics as given; one value has no std
        rc["adv_std"], rc["cadv_std"] = 1.0, 1.0
    t = to_dev(d)
    pm = call_moments(t).cpu().numpy()
    want = ref.adv_moments(d["returns"], d["cost_returns"], d["old_v"], d["old_cv"])
    a = (d["returns"] - d["old_v"]).astype(np.float64)
    c = (d["cost_returns"] - d["old_cv"]).astype(np.float64)
    scale = np.array([np.abs(a).sum(), (a * a).sum(), np.abs(c).sum(), (c * c).sum()])
    assert (np.abs(pm.sum(0) - want) <= 1e-12 * scale).all(), (pm.sum(0), want)
    assert (pm[blocks(n):] == 0).all()

    g, part = nan_outputs(n)
    call_loss(rc, t, g, part)
    r = ref.ppo_loss_ref(rc, **d)
    assert_grads_close(r, g, f"n={n}")
    p = part.cpu().numpy()
    assert np.isfinite(p).all() and (p[blocks(n):] == 0).all()
    assert_stats_close(rc, r, p.sum(0), f"n={n}")


def test_abi_contracts_null_gradients_determinism_and_empty_call():
    """Any subset of the four gradient pointers may be NULL: statistics and the remaining gradients are bit-identical and
    the NULL buffers untouched; two calls are bit-identical; n = 0 zeroes every partial row and writes no gradient."""
    variant = VARIANTS[1]
    for n in (257, 262145):
        rng = np.random.default_rng(n)
        d, am, cm = batch(rng, n, variant[1].clip_range)
        rc = abi_config(variant, n, d, am, cm)
        t = to_dev(d)
        g0, p0 = nan_outputs(n)
        call_loss(rc, t, g0, p0)
        g1, p1 = nan_outputs(n)
        call_loss(rc, t, g1, p1)
        assert torch.equal(p0, p1) and all(torch.equal(g0[k], g1[k]) for k in GRADS)
        for mask in range(16):
            g, p = nan_outputs(n)
            passed = {k: (g[k] if mask >> i & 1 else None) for i, k in enumerate(GRADS)}
            call_loss(rc, t, passed, p)
            assert torch.equal(p, p0), mask
            for i, k in enumerate(GRADS):
                if mask >> i & 1:
                    assert torch.equal(g[k], g0[k]), (mask, k)
                else:
                    assert torch.isnan(g[k]).all(), (mask, k)
    g, p = nan_outputs(4)
    t = to_dev(random_batch(np.random.default_rng(0), 4, 0.2))
    call_loss(abi_config(variant, 4, {k: v.cpu().numpy() for k, v in t.items()}), t, g, p, n=0)
    assert (p == 0).all() and all(torch.isnan(g[k]).all() for k in GRADS)
    assert (call_moments(t, n=0) == 0).all()


def test_abi_shards_equal_the_unsharded_call():
    """One global minibatch cut into uneven shards (an empty one and a one-element one among them): the shards' moment
    sums equal the unsharded ones, per-shard mapf_ppo_loss calls with the one global config give bit-identical
    gradients, and the summed statistics equal the unsharded ones."""
    variant = VARIANTS[0]
    n = 300007
    rng = np.random.default_rng(7)
    d, am, cm = batch(rng, n, variant[1].clip_range)
    rc = abi_config(variant, n, d, am, cm)
    r = ref.ppo_loss_ref(rc, **d)
    t = to_dev(d)
    g0, p0 = nan_outputs(n)
    call_loss(rc, t, g0, p0)
    m0 = call_moments(t).sum(0).cpu().numpy()
    cuts = [0, 0, 1, 40000, 40017, 262161, n]              # shards: empty, 1, 39999, 17, 222144, 37846
    g, _ = nan_outputs(n)
    msum, psum = np.zeros(4), np.zeros(NS)
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        pm = call_moments(t, n=hi - lo, lo=lo)
        msum += pm.sum(0).cpu().numpy()
        _, p = nan_outputs(1)
        call_loss(rc, t, g, p, n=hi - lo, lo=lo)
        psum += p.sum(0).cpu().numpy()
    a = (d["returns"] - d["old_v"]).astype(np.float64)
    c = (d["cost_returns"] - d["old_cv"]).astype(np.float64)
    scale = np.array([np.abs(a).sum(), (a * a).sum(), np.abs(c).sum(), (c * c).sum()])
    assert (np.abs(msum - m0) <= 1e-12 * scale).all()
    assert all(torch.equal(g[k], g0[k]) for k in GRADS)
    p0s = p0.sum(0).cpu().numpy()
    assert (np.abs(psum - p0s) <= 1e-12 * np.abs(r["stats"]).sum(0)).all(), (psum, p0s)


def test_single_pass_variance_on_episode_like_returns():
    """Returns around -300 with a standard deviation of 0.5: the wrapper's single-pass variance from the kernel's sums
    agrees with a two-pass float64 variance to 1e-9."""
    from primal_ppo_b200.ppo.fused_loss import _mean_std
    n = 10 ** 6 + 3
    rng = np.random.default_rng(21)
    ret = (-300 + 0.5 * rng.standard_normal(n)).astype(F32)
    old_v = (0.01 * rng.standard_normal(n)).astype(F32)
    cret = (-40 + 2 * rng.standard_normal(n)).astype(F32)
    t = {k: torch.from_numpy(v).cuda() for k, v in (("returns", ret), ("old_v", old_v), ("cost_returns", cret),
                                                     ("old_cv", np.zeros(n, F32)))}
    s = call_moments(t).sum(0).cpu().numpy()
    for (s1, s2), x in (((s[0], s[1]), ret - old_v), ((s[2], s[3]), cret)):
        mean, std = _mean_std(float(s1), float(s2), float(n))
        x = x.astype(np.float64)
        assert abs(mean - x.mean()) <= 1e-12 * np.abs(x).mean()
        assert abs(std ** 2 - ref.two_pass_std(x) ** 2) <= 1e-9 * ref.two_pass_std(x) ** 2, (std, ref.two_pass_std(x))


# ---- through the wrapper -------------------------------------------------------------------------------------------------

def run_loss(fn, d, variant, group=None, lo=0, hi=None):
    """fn(out, ...) on elements [lo, hi) of d as CUDA tensors; returns (loss, stats, gradients of the four outputs)."""
    from primal_ppo_b200.ppo.policy import PolicyOutput
    _, cfg, lag = variant
    hi = len(d["actions"]) if hi is None else hi
    t = {k: torch.from_numpy(np.ascontiguousarray(v[lo:hi])).cuda() for k, v in d.items()}
    leaves = [t["policy"].clone().requires_grad_(True), t["value"].unsqueeze(-1).clone().requires_grad_(True),
              t["cost_value"].unsqueeze(-1).clone().requires_grad_(True), t["sig"].clone().requires_grad_(True)]
    kw = {f: None for f in PolicyOutput._fields}
    kw.update(policy=leaves[0], value=leaves[1], cost_value=leaves[2], policy_sig=leaves[3])
    loss, stats = fn(PolicyOutput(**kw), returns=t["returns"], cost_returns=t["cost_returns"], old_v=t["old_v"],
                     old_cv=t["old_cv"], actions=t["actions"], old_ps=t["old_ps"], train_valid=t["train_valid"].float(),
                     lagrangian=lag, cfg=cfg, group=group)
    loss.backward()
    grads = {k: x.grad.detach().reshape(-1, 5) if k in ("g_policy", "g_sig") else x.grad.detach().reshape(-1)
             for k, x in zip(GRADS, leaves)}
    return float(loss.detach()), {k: float(v) for k, v in stats.items()}, grads


def assert_named_stats_close(rc, r, loss, stats, what=""):
    want = ref.stat_means(rc, r["stats"].sum(0))
    mag = ref.stat_mags(rc, r["stats_mag"].sum(0))
    assert abs(loss - want["all_loss"]) <= STAT_TOL * mag["all_loss"] + 1e-12, (what, loss, want["all_loss"])
    assert round(stats["clipfrac"] * rc["n_global"]) == r["clipped"].sum(), what
    for k in ref.STAT_NAMES:
        if k != "clipfrac":
            # the f32 result of the wrapper adds one rounding of the value itself
            tol = STAT_TOL * mag[k] + 2.0 ** -24 * abs(want[k]) + 1e-12
            assert abs(stats[k] - want[k]) <= tol, (what, k, stats[k], want[k], mag[k])


@pytest.mark.parametrize("n", [255, 262145])
@pytest.mark.parametrize("vi", [0, 1, 2])
def test_wrapper_matches_float64_reference(vi, n):
    """fused_ppo_lagrange_loss end to end (moments, wrapper statistics, kernel, autograd hand-off) against the reference."""
    from primal_ppo_b200.ppo.fused_loss import fused_ppo_lagrange_loss
    variant = VARIANTS[vi]
    rng = np.random.default_rng(50 + vi + n)
    d, _, _ = batch(rng, n, variant[1].clip_range)
    rc = abi_config(variant, n, d)
    r = ref.ppo_loss_ref(rc, **d)
    loss, stats, grads = run_loss(fused_ppo_lagrange_loss, d, variant)
    assert_grads_close(r, grads, variant[0])
    assert_named_stats_close(rc, r, loss, stats, variant[0])


class _EmulatedAllReduce:
    """torch.distributed.all_reduce for K ranks in one process.  Pass 1 records every shard's inputs, call by call; pass 2
    replaces each input with the sum over the shards of the inputs recorded at the same call index."""

    def __init__(self):
        self.recorded, self.shard, self.call, self.replay = [], 0, 0, False

    def start(self, shard):
        self.shard, self.call = shard, 0
        if not self.replay:
            self.recorded.append([])

    def __call__(self, tensor, op=None, group=None, async_op=False):
        if not self.replay:
            self.recorded[self.shard].append(tensor.detach().clone())
        else:
            mine = self.recorded[self.shard][self.call]
            assert torch.equal(tensor, mine), "a shard's all-reduce input changed between the passes"
            tensor.copy_(sum(rec[self.call] for rec in self.recorded))
        self.call += 1


@pytest.mark.parametrize("K", [2, 3])
@pytest.mark.parametrize("which", ["fused", "eager"])
def test_group_path_with_emulated_all_reduce(monkeypatch, which, K):
    """The collective-dependent code of fused_loss.py / loss.py: K unequal shards of one minibatch, normalised with the
    emulated all-reduce of their moments.  The loss shares add up to the single-process loss and the concatenated
    gradients equal the single-process gradients."""
    import torch.distributed as dist
    from primal_ppo_b200.ppo.fused_loss import fused_ppo_lagrange_loss
    from primal_ppo_b200.ppo.loss import ppo_lagrange_loss
    fn = fused_ppo_lagrange_loss if which == "fused" else ppo_lagrange_loss
    variant = VARIANTS[1]
    n = 70001
    rng = np.random.default_rng(K)
    d, _, _ = batch(rng, n, variant[1].clip_range)
    rc = abi_config(variant, n, d)
    r = ref.ppo_loss_ref(rc, **d)
    loss1, stats1, grads1 = run_loss(fn, d, variant)
    cuts = [0, 1, 30000, n] if K == 3 else [0, 50001, n]
    fake = _EmulatedAllReduce()
    monkeypatch.setattr(dist, "all_reduce", fake)
    group = object()
    for replay in (False, True):
        fake.replay = replay
        shards = []
        for i, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
            fake.start(i)
            shards.append(run_loss(fn, d, variant, group=group, lo=lo, hi=hi))
    loss_k = sum(s[0] for s in shards)
    mag = ref.stat_mags(rc, r["stats_mag"].sum(0))
    assert abs(loss_k - loss1) <= 2 * STAT_TOL * mag["all_loss"] + 1e-12, (loss_k, loss1)
    for k in ref.STAT_NAMES:
        total = sum(s[1][k] for s in shards)
        assert abs(total - stats1[k]) <= 2 * STAT_TOL * mag[k] + 2.0 ** -22 * abs(stats1[k]) + 1e-12, (k, total, stats1[k])
    cat = {k: torch.cat([s[2][k] for s in shards]) for k in GRADS}
    for k in GRADS:
        err = (cat[k] - grads1[k]).double().abs().cpu().numpy().reshape(r[k].shape)
        assert (err <= 2 * GRAD_TOL * r[k + "_mag"] + 1e-30).all(), k
    assert_grads_close(r, cat, which)


def test_single_element_minibatch_gives_nan_like_loss_py():
    """A global minibatch of one element: the unbiased std is NaN, so the loss, the advantage statistics and the policy
    gradient of the taken action are NaN through the fused path exactly where they are NaN through loss.py, and the
    rest agree.  The fused path must not raise."""
    from primal_ppo_b200.ppo.fused_loss import fused_ppo_lagrange_loss
    from primal_ppo_b200.ppo.loss import ppo_lagrange_loss
    d = random_batch(np.random.default_rng(3), 1, 0.2)
    for variant in VARIANTS:
        with warnings.catch_warnings():                   # torch.std of one element warns about the degrees of freedom
            warnings.simplefilter("ignore")
            l1, s1, g1 = run_loss(ppo_lagrange_loss, d, variant)
        l2, s2, g2 = run_loss(fused_ppo_lagrange_loss, d, variant)
        assert np.isnan(l1) and np.isnan(l2)
        for k in s1:
            assert np.isnan(s1[k]) == np.isnan(s2[k]), k
            if not np.isnan(s1[k]):
                assert abs(s1[k] - s2[k]) <= 1e-5 + 1e-5 * abs(s1[k]), k
        for k in GRADS:
            a, b = g1[k].cpu().numpy(), g2[k].cpu().numpy()
            assert np.array_equal(np.isnan(a), np.isnan(b)), k
            assert np.allclose(a[~np.isnan(a)], b[~np.isnan(b)], rtol=1e-5, atol=1e-9), k
        assert np.isnan(g2["g_policy"][0, int(d["actions"][0])].item())


# ---- GAE: the terminal mask on the float4 path, misaligned views, adv = NULL -------------------------------------------

def _gae_case(rng, T, cols):
    r, v = (rng.normal(size=(T, cols)).astype(F32) for _ in range(2))
    lv = rng.normal(size=(cols,)).astype(F32)
    nt = (rng.random((T, cols)) > 0.2).astype(np.uint8)
    return r, v, lv, nt


def _offset_view(x):
    """A CUDA copy of x whose data starts 4 bytes past a 16-byte boundary."""
    buf = torch.zeros(x.size + 1, dtype=torch.float32, device="cuda")
    view = buf[1:].view(x.shape)
    view.copy_(torch.from_numpy(x))
    assert view.data_ptr() % 16 == 4
    return view


@pytest.mark.parametrize("T", [1, 7, 8, 9, 17])
def test_gae_terminal_mask_on_float4_path(T):
    """cols % 4 == 0 and aligned (4 columns per thread), around the unroll of 8 time steps; then the same data through a
    4-byte-offset view, which forces one column per thread.  Both bit-exact with the f32 restatement."""
    from primal_ppo_b200 import gae
    rng = np.random.default_rng(T)
    r, v, lv, nt = _gae_case(rng, T, 4 * 301)
    want_ret, want_adv = ref.gae_masked_ref(r, v, lv, nt)
    cu = lambda x: torch.from_numpy(x).cuda()
    ret, adv = gae(cu(r), cu(v), cu(lv), nonterminal=cu(nt), return_advantages=True)
    assert ret.cpu().numpy().tobytes() == want_ret.tobytes() and adv.cpu().numpy().tobytes() == want_adv.tobytes()
    ret, adv = gae(_offset_view(r), _offset_view(v), _offset_view(lv), nonterminal=cu(nt), return_advantages=True)
    assert ret.cpu().numpy().tobytes() == want_ret.tobytes() and adv.cpu().numpy().tobytes() == want_adv.tobytes()
    # adv = NULL gives the same returns
    assert torch.equal(gae(cu(r), cu(v), cu(lv), nonterminal=cu(nt)), ret)


def test_gae2_with_one_misaligned_stream_and_mask():
    """mapf_gae2 with only the cost stream misaligned (so the launch falls back to one column per thread for both) and
    a terminal mask: each stream bit-exact with the f32 restatement; without a mask, with the oracle."""
    from primal_ppo_b200 import gae2
    rng = np.random.default_rng(4)
    T, cols = 13, 4 * 257
    r, v, lv, nt = _gae_case(rng, T, cols)
    cr, cv, lcv, _ = _gae_case(rng, T, cols)
    cu = lambda x: torch.from_numpy(x).cuda()
    for mask in (nt, None):
        ret, cret = gae2(cu(r), cu(v), cu(lv), _offset_view(cr), _offset_view(cv), _offset_view(lcv),
                         nonterminal=None if mask is None else cu(mask))
        m = np.ones_like(nt) if mask is None else mask
        assert ret.cpu().numpy().tobytes() == ref.gae_masked_ref(r, v, lv, m)[0].tobytes()
        assert cret.cpu().numpy().tobytes() == ref.gae_masked_ref(cr, cv, lcv, m)[0].tobytes()
        if mask is None:
            assert ret.cpu().numpy().tobytes() == gae_oracle(r, v, lv)[0].tobytes()
            assert cret.cpu().numpy().tobytes() == gae_oracle(cr, cv, lcv)[0].tobytes()


# ---- action sampling past one pass of its grid ----------------------------------------------------------------------------

@pytest.mark.parametrize("rows", [148 * 8 * 256 + 1, 10 ** 6 + 9])
def test_sample_actions_bit_exact_past_one_grid_pass(rows):
    """The sampling kernel grid-strides over 148*8 blocks of 256 threads: actions and chosen_p bit-exact with the oracle
    past the first pass, with a seed whose high bits are set and a draw index >= 2^31."""
    from primal_ppo_b200 import sample_actions
    rng = np.random.default_rng(rows)
    logits = rng.standard_normal((rows, 5)) * 2
    ps = (np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)).astype(F32)
    ps[::13, 1] = 0
    seed, draw = 0xF00DFACE12345678, 2 ** 31 + 12345
    cp = torch.empty(rows, device="cuda")
    a = sample_actions(torch.from_numpy(ps).cuda(), seed=seed, draw=draw, chosen_p=cp)
    ra, rcp = sample_actions_oracle(ps, seed=seed, draw=draw)
    np.testing.assert_array_equal(a.cpu().numpy(), ra)
    np.testing.assert_array_equal(cp.cpu().numpy().view(np.uint32), rcp.view(np.uint32))
    assert (ps[np.arange(rows), ra] > 0).all()
